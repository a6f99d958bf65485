"""Worker of tests/test_widen_interpolate.py: ONE rank of an N-rank engine that calls `sph_interpolate` (collective under
the Morton-domain decomposition, local in the replicated form).  Not a test module.

  python tests/_dd_interp_rank.py RANK WORLD COMM DEVICE TOKEN OUT.npz SPEC_JSON

COMM = nccl (one GPU per rank) | host (shared-memory collectives: ranks may share a device); WORLD = 1 runs the same
scenario on a single rank (no communicator).  SPEC keys: scenario (values | mismatch | ask), mode, decomposition, steps.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

COLS = ("rho", "vx", "vy", "vz", "u", "alpha", "count")


def points(seed=5):
    """The same probe points on every rank: a mid-plane slice, random points in the disc, and a few far outside."""
    rng = np.random.default_rng(seed)
    g = np.linspace(-110.0, 110.0, 48)
    X, Y = np.meshgrid(g, g, indexing="ij")
    sl = np.stack([X.ravel(), Y.ravel(), np.zeros(X.size)], 1)
    r = np.sqrt(rng.uniform(8.0 ** 2, 104.0 ** 2, 3000)); phi = rng.uniform(0.0, 2.0 * np.pi, 3000)
    disc = np.stack([r * np.cos(phi), r * np.sin(phi), rng.normal(0.0, 2.5, 3000)], 1)
    far = rng.uniform(150.0, 300.0, (20, 3))
    return np.concatenate([sl, disc, far])


def make_engine(spec, rank, world, comm, device, token):
    from summersph_b200 import default_params, ics
    from summersph_b200.engine import Engine
    p = default_params(spec["mode"], decomposition=spec.get("decomposition", 1))
    b, s = ics.keplerian_disc(spec.get("n", 20_000), seed=12)
    e = Engine(p, device=device)
    if world > 1:
        if comm == "nccl":
            e.comm_init(rank, world, bytes.fromhex(token))
        else:
            e.comm_init_host(rank, world, token)
    return e, b, s


def main():
    rank, world, comm, device, token, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], int(sys.argv[4]), sys.argv[5], sys.argv[6]
    spec = json.loads(sys.argv[7])
    sc = spec["scenario"]
    from summersph_b200.engine import SphError
    pts = points()
    res = {}
    if sc == "ask":      # the same run without and with interpolation before and between the steps (two engines, two segments)
        for ask in (0, 1):
            e, b, s = make_engine(spec, rank, world, comm, device, f"{token}_{ask}")
            with e:
                e.upload(b, s)
                dt, t = 0.01, 0.0
                if ask:
                    e.interpolate(pts)
                for _ in range(spec["steps"]):
                    dt, t = e.step(dt, t)
                    if ask:
                        e.interpolate(pts)
                h, _ = e.state_hash()
                res[f"run{ask}"] = np.array([float(h & 0xffffffff), float(h >> 32), dt, t, float(e.far_reuse_count())])
    elif sc == "mismatch":      # rank 2 passes other points; then rank 1 passes a NaN; then every rank passes the same points
        e, b, s = make_engine(spec, rank, world, comm, device, token)
        codes = []
        with e:
            e.upload(b, s)
            for call in range(3):
                q = pts.copy()
                if call == 0 and rank == 2:
                    q[7, 0] += 1e-9
                if call == 1 and rank == 1:
                    q[3, 2] = np.nan
                try:
                    e.interpolate(q)
                    codes.append(0)
                except SphError as err:
                    assert err.code == -1, err      # SPH_ERR_ARG on every rank
                    codes.append(1)
        res["codes"] = np.array(codes)
    else:
        e, b, s = make_engine(spec, rank, world, comm, device, token)
        with e:
            e.upload(b, s)
            got = e.interpolate(pts)      # domains: the tree (migration, halo, LET) is built inside the call
            for k in COLS:
                res["up_" + k] = got[k]
            dt, t = 0.01, 0.0
            for _ in range(spec.get("steps", 2)):
                dt, t = e.step(dt, t)
            got = e.interpolate(pts)
            for k in COLS:
                res["st_" + k] = got[k]
            res["halo"] = np.array([e.domain_stats()["halo"] if world > 1 else 0])
    np.savez(out, **res)


if __name__ == "__main__":
    main()
