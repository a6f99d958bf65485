#!/usr/bin/env python
"""Energy / momentum / angular-momentum drift of the flagship disc under the Morton-domain decomposition.

  python -m torch.distributed.run --nproc-per-node N scripts/drift_domains.py [--particles P] [--steps K]

The engine of bench.py (variable h, the Keplerian disc generated on the device by Engine.ics_disc with bench.py's
seed; decomposition = 1 when N > 1): sph_conserved, K loop bodies, sph_conserved again.  sph_conserved is collective
under the decomposition (every rank calls it and gets the same sums).  Rank 0 prints one JSON line: the drift_report
fields, both sums, the wall-clock time of each sph_conserved call (synchronous: it returns with the sums on the host;
the first call also builds the tree, migration, halo and LET), the rank and particle counts, and the card name and
power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(local):
    """(name, power limit) of the GPU this rank runs on, read now."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1] if len(q) > 1 else None
    except Exception:
        import torch
        return torch.cuda.get_device_name(local), None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, default=16_000_000)
    ap.add_argument("--steps", type=int, default=3)
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))

    import torch
    import torch.distributed as dist
    from summersph_b200 import default_params, MODE_VARIABLE_H
    from summersph_b200._abi import drift_report
    from summersph_b200.engine import Engine
    from summersph_b200.parallel import init_comm, torch_broadcast_bytes

    if not torch.cuda.is_available():
        raise SystemExit("drift_domains.py needs a CUDA device")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    p = default_params(MODE_VARIABLE_H)
    p.n_ranks = world
    p.decomposition = 1 if world > 1 else 0
    with Engine(p, device=local) as e:
        if world > 1:
            init_comm(e, rank, world, torch_broadcast_bytes)
        e.ics_disc(args.particles, seed=20251018)

        def timed_conserved():
            t0 = time.perf_counter(); d = e.conserved(); return d, time.perf_counter() - t0

        first, t_first = timed_conserved()
        dt, t = 0.01, 0.0
        for _ in range(args.steps):
            dt, t = e.step(dt, t)
        last, t_last = timed_conserved()
        n_gas = e.sizes()[0]
    if world > 1:
        dist.barrier()
    if rank == 0:
        name, power = card(local)
        line = {"ranks": world, "decomposition": p.decomposition, "particles": args.particles, "particles_end": n_gas,
                "steps": args.steps, "t": t, "dt": dt, "first": first, "last": last, **drift_report(first, last),
                "conserved_call_s": {"first": t_first, "last": t_last}, "gpu": name, "power_limit": power}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
