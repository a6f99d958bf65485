"""Worker of tests/test_multi_gpu.py: ONE rank of an N-rank engine run, in its own process (the way bench.py and a
production host run it: one process per rank, CUDA-IPC peers).  Not a test module.

  python tests/_mp_rank.py RANK WORLD COMM DEVICE MODE STEPS OUT.npz [UID_HEX | SHM_NAME] [N] [DOMAINS] [EXTRA] [ICS] [CASE.npz]

CASE.npz: run this input instead of the disc (`params` bytes and the in_* gas and sink columns, as tests/_cases.load_golden
reads them); DOMAINS still sets the decomposition.

COMM = nccl (needs one GPU per rank) | host (shared-memory collectives: ranks may share a device).
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def case(mode, n=60_000, decomposition=0):
    from summersph_b200 import default_params, ics
    if os.environ.get("SPH_TEST_QUIET"):    # nothing is removed: evaluation A keeps evaluation B's far-field gravity (sph_far_reuse_count > 0)
        p = default_params(mode, decomposition=decomposition)
        b, s = ics.keplerian_disc(n, seed=12)
        return p, b, s
    p = default_params(mode, bounding_size=95.0, decomposition=decomposition)
    b, s = ics.keplerian_disc(n, seed=12)
    s.radius[:] = 12.0                      # accretion + bounds removals exercised too
    return p, b, s


def main():
    rank, world, comm, device, mode, steps, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], int(sys.argv[4]), int(sys.argv[5]), int(sys.argv[6]), sys.argv[7]
    token = sys.argv[8] if len(sys.argv) > 8 else ""
    n = int(sys.argv[9]) if len(sys.argv) > 9 else 60_000
    domains = int(sys.argv[10]) if len(sys.argv) > 10 else 0
    from summersph_b200.engine import Engine, SphError
    from summersph_b200.state import GAS_FIELDS
    if len(sys.argv) > 13 and sys.argv[13] != "-":
        from _cases import load_golden
        _, p, b, s = load_golden(os.path.splitext(os.path.abspath(sys.argv[13]))[0])
        p = p.copy(decomposition=domains)
    else:
        p, b, s = case(mode, n, domains)
    with Engine(p, device=device) as e:
        if world > 1:
            if comm == "nccl":
                e.comm_init(rank, world, bytes.fromhex(token))
            else:
                e.comm_init_host(rank, world, token)
        if len(sys.argv) > 12 and sys.argv[12] == "devics":
            e.ics_disc(n, seed=12)           # every rank generates its own rows on the device
        elif len(sys.argv) > 12 and sys.argv[12] == "rank0":
            e.upload_local(n, b if rank == 0 else b.take(slice(0, 0)), s)      # domains: rank 0 owns every row, the others none
        else:
            e.upload(b, s)
        dt, t = 0.01, 0.0
        for k in range(steps):
            if k > 0 and os.environ.get("SPH_TEST_ROUNDTRIP"):      # the host takes the state and hands it back before every step
                if domains:
                    numbers, bl = e.download_local(); sl = e.sinks_only()
                    e.upload_local(n, bl, sl, numbers=numbers)
                else:
                    bl, sl = e.download(); e.upload(bl, sl)
            dt, t = e.step(dt, t)
        bb, ss = e.download()
        d = e.diag()
        c = e.counters()
        extra = {"far_reuse": np.array([e.far_reuse_count()]), "resident_hits": np.array([e.resident_hits()])}
        if len(sys.argv) > 11 and sys.argv[11] == "tree":      # one more evaluation on the end state with exact counters: tree + neighbour sets
            e.set_exact_counters(True); e.evaluate(); e.set_exact_counters(False)
            tr = e.tree(); cnt, hsh, _, _ = e.neighbours(with_list=False)
            extra.update({"t_" + k: v for k, v in tr.items()})
            extra.update({"n_count": cnt, "n_hash": hsh})
            d2 = e.diag(); extra.update({"e_" + k: v for k, v in d2.items()})
            c2 = e.counters(); extra["e_counters"] = np.array([c2[k] for k in sorted(c2)], dtype=np.int64)
            extra["local_n"] = np.array([e.local_size()])
        if len(sys.argv) > 11 and sys.argv[11] == "nblist":      # the neighbour list form after an evaluation: its error code, 0 if it worked
            e.evaluate()
            try:
                e.neighbours(with_list=True)
                extra["nblist_code"] = np.array([0])
            except SphError as err:
                extra["nblist_code"] = np.array([err.code]); extra["nblist_msg"] = np.array([str(err)])
        res = {k: getattr(bb, k) for k in GAS_FIELDS}
        res.update({"s_" + k: getattr(ss, k) for k in ("x", "y", "z", "vx", "vy", "vz", "m")})
        res.update({"d_" + k: v for k, v in d.items()})
        res["meta"] = np.array([dt, t, float(e.sizes()[0]), float(e.sizes()[1])])
        res["counters"] = np.array([c[k] for k in sorted(c)], dtype=np.int64)
        res.update(extra)
        np.savez(out, **res)


if __name__ == "__main__":
    main()
