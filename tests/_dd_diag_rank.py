"""Worker of tests/test_domains_diagnostics.py: ONE rank of an N-rank engine that asks for the on-demand diagnostics
(`sph_conserved`, `sph_column_density`, `simulate(drift=...)`) under the Morton-domain decomposition.  Not a test module.

  python tests/_dd_diag_rank.py RANK WORLD COMM DEVICE TOKEN OUT.npz SPEC_JSON

COMM = nccl (one GPU per rank) | host (shared-memory collectives: ranks may share a device); WORLD = 1 runs the same
scenario on a single rank (no communicator).  SPEC keys: scenario, mode, n, steps, sinks.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

IMG_FRAME = (-120.0, 120.0, -120.0, 120.0)


def case(spec):
    """The disc of tests/_mp_rank.py: plain, or with the accretion + bounds set-up (and optionally a second sink)."""
    from summersph_b200 import default_params, ics, Sinks
    mode, n = spec["mode"], spec.get("n", 60_000)
    b, s = ics.keplerian_disc(n, seed=12)
    if spec["scenario"] == "removals":
        p = default_params(mode, bounding_size=95.0, decomposition=1)
        s.radius[:] = 12.0
        if spec.get("sinks", 1) == 2:      # a second accreting sink (as in test_widen_conserved's two-sink case)
            s = Sinks([s.x[0], 40.0], [s.y[0], 0.0], [s.z[0], 0.0], [s.vx[0], 0.0], [s.vy[0], 6.0], [s.vz[0], 0.0], [s.m[0], 0.01], [12.0, 6.0])
    elif spec["scenario"] == "image":
        p = default_params(mode, h_fixed=2.5, decomposition=1)
    elif spec["scenario"] == "simulate":
        p = default_params(mode, end_time=1.0, decomposition=1)
    else:
        p = default_params(mode, decomposition=1)
    return p, b, s


def cons_array(d):
    from summersph_b200._abi import CONSERVED
    return np.array([d[k] for k in CONSERVED])


def open_engine(spec, rank, world, comm, device, token):
    from summersph_b200.engine import Engine
    p, b, s = case(spec)
    e = Engine(p, device=device)
    if world > 1:
        if comm == "nccl":
            e.comm_init(rank, world, bytes.fromhex(token))
        else:
            e.comm_init_host(rank, world, token)
    return e, p, b, s


def main():
    rank, world, comm, device, token, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], int(sys.argv[4]), sys.argv[5], sys.argv[6]
    spec = json.loads(sys.argv[7])
    sc = spec["scenario"]
    res = {}
    if sc == "ask":      # the same run without and with sph_conserved before and between the steps (two engines, two segments)
        for ask in (0, 1):
            e, p, b, s = open_engine(spec, rank, world, comm, device, f"{token}_{ask}")
            with e:
                e.upload(b, s)
                dt, t = 0.01, 0.0
                if ask:
                    e.conserved()
                for _ in range(spec["steps"]):
                    dt, t = e.step(dt, t)
                    if ask:
                        e.conserved()
                h, _ = e.state_hash()
                res[f"run{ask}"] = np.array([float(h & 0xffffffff), float(h >> 32), dt, t])
    else:
        e, p, b, s = open_engine(spec, rank, world, comm, device, token)
        with e:
            if sc == "simulate":
                from summersph_b200.simulate import simulate
                rep = {}
                _, _, t, dt, steps = simulate(b, s, p, engine=e, max_steps=spec["steps"], log=lambda line: None, drift=rep)
                res["first"] = cons_array(rep["first"]); res["last"] = cons_array(rep["last"])
                res["report"] = np.array([rep[k] if rep[k] is not None else np.nan for k in ("energy_rel", "momentum_rel", "angular_momentum_rel", "mass_rel")])
                res["meta"] = np.array([steps, rep["steps"], t, dt])
            else:
                e.upload(b, s)
                dt, t = 0.01, 0.0
                for _ in range(spec.get("steps", 0)):
                    dt, t = e.step(dt, t)
                res["cons"] = cons_array(e.conserved())      # straight after the upload: the tree (domains: migration, halo, LET) is built inside
                res["meta"] = np.array([dt, t, float(e.sizes()[0]), float(e.sizes()[1])])
                if sc == "image":      # rows have migrated and the halo is filled by the build above: images of the own rows only
                    res["img_z"] = e.column_density("z", IMG_FRAME, (192, 160))
                    res["img_x"] = e.column_density("x", IMG_FRAME, (128, 144))
                    res["img_big"] = e.column_density("z", IMG_FRAME, (1024, 1024))      # 8 MB: more than one host-communicator slot
                    res["mass"] = np.array([b.m.sum()])
                    if world > 1:
                        res["halo"] = np.array([e.domain_stats()["halo"]])
    np.savez(out, **res)


if __name__ == "__main__":
    main()
