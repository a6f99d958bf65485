#!/usr/bin/env python
"""Cost of `sph_interpolate` on the flagship disc.

  python scripts/interpolate_bench.py [--particles 16000000] [--repeats 5] [--out FILE]

The engine of bench.py (variable h, the Keplerian disc generated on the device by Engine.ics_disc with bench.py's seed),
two loop bodies (h iterated, the tree of evaluation B is then reused by the calls).  After one warm-up call each, the
median of `--repeats` calls of:
  slice   a 1024 x 1024 mid-plane slice (z = 0, |x|, |y| < 100, pixel centres)
  grid    a 128^3 grid over the same box (|z| < 100 too)
  random  1M random points inside the disc (r in [10, 100], z ~ N(0, 0.05 r))
  one     a single point: the fixed part of a call (private BVH over the walk groups, launches, copies)
and, for scale, sph_column_density at 1024 x 1024 and one sph_step.  Each call is timed with a host clock around the
synchronous call and with the context's device timer (CUDA events on its stream).  Prints one JSON line (also appended
to --out) with the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    """(name, power limit) of GPU 0, read now (read-only query)."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1] if len(q) > 1 else None
    except Exception:
        return None, None


def timed(e, fn, repeats):
    """Median host and device milliseconds of `repeats` calls after one warm-up call."""
    fn()
    host, dev = [], []
    for _ in range(repeats):
        e.timer_start()
        t0 = time.perf_counter()
        fn()
        host.append((time.perf_counter() - t0) * 1e3)
        dev.append(e.timer_stop())
    return float(np.median(host)), float(np.median(dev))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, default=16_000_000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from summersph_b200 import default_params, MODE_VARIABLE_H
    from summersph_b200.engine import Engine

    g = (np.arange(1024) + 0.5) * (200.0 / 1024) - 100.0
    X, Y = np.meshgrid(g, g, indexing="xy")
    slice_pts = np.stack([X.ravel(), Y.ravel(), np.zeros(X.size)], 1)
    g3 = (np.arange(128) + 0.5) * (200.0 / 128) - 100.0
    X, Y, Z = np.meshgrid(g3, g3, g3, indexing="ij")
    grid_pts = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1)
    rng = np.random.default_rng(7)
    r = np.sqrt(rng.uniform(10.0 ** 2, 100.0 ** 2, 1 << 20)); phi = rng.uniform(0.0, 2.0 * np.pi, 1 << 20)
    rand_pts = np.stack([r * np.cos(phi), r * np.sin(phi), rng.standard_normal(1 << 20) * 0.05 * r], 1)
    one_pt = np.array([[50.0, 0.0, 0.0]])

    p = default_params(MODE_VARIABLE_H)
    with Engine(p, device=0) as e:
        e.ics_disc(args.particles, seed=20251018)
        dt, t = 0.01, 0.0
        for _ in range(2):
            dt, t = e.step(dt, t)
        res = {}
        for name, pts in (("slice", slice_pts), ("grid", grid_pts), ("random", rand_pts), ("one", one_pt)):
            h, d = timed(e, lambda: e.interpolate(pts), args.repeats)
            res[name] = {"points": len(pts), "host_ms": h, "device_ms": d, "points_per_s": len(pts) / (h * 1e-3)}
        out = e.interpolate(slice_pts)
        h, d = timed(e, lambda: e.column_density("z", (-100.0, 100.0, -100.0, 100.0), (1024, 1024)), args.repeats)
        res["column_density_1024"] = {"host_ms": h, "device_ms": d}
        e.timer_start(); t0 = time.perf_counter()
        dt, t = e.step(dt, t)
        res["step"] = {"host_ms": (time.perf_counter() - t0) * 1e3, "device_ms": e.timer_stop()}
        name, plim = card()
        line = {"what": "sph_interpolate", "particles": args.particles, "mode": "variable_h", "repeats": args.repeats,
                **res,
                "fixed_share_of_slice": res["one"]["host_ms"] / res["slice"]["host_ms"],
                "slice_members_mean": float(np.mean(out["count"])), "slice_rho_max": float(np.max(out["rho"])),
                "gpu": name, "power_limit": plim}
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
