#!/usr/bin/env python
"""Cost of `sph_gravity_at` on the flagship disc.

  python scripts/gravity_at_bench.py [--particles 16000000] [--repeats 5] [--out FILE]

The engine of bench.py (variable h, the Keplerian disc generated on the device by Engine.ics_disc with bench.py's seed),
two loop bodies (h iterated, the tree of evaluation B is then reused by the calls).  After one warm-up call each, the
median of `--repeats` calls of:
  slice   a 1024 x 1024 mid-plane slice (z = 0, |x|, |y| < 100, pixel centres)
  random  1M random points inside the disc (r in [10, 100], z ~ N(0, 0.05 r))
  rings   the rotation-curve rings of summersph_b200.rotation_curve (46 radii from 10 to 100, 256 points each)
  one     a single point: the fixed part of a call (sort, launches, copies)
Each call is timed with a host clock around the synchronous call and with the context's device timer (CUDA events on its
stream); ns per point is the device time over the points.  Beside them, in the same run: the gravity stage of an
evaluation that walks the whole tree (sph_evaluate(GRAVITY) on the tree of the same state with exact counters,
which switch the far-field reuse off: the walk and its sink sums) per particle.  Prints one JSON line (also appended to --out) with the card name and power limit read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from interpolate_bench import card, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, default=16_000_000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from summersph_b200 import default_params, MODE_VARIABLE_H, EVAL_TREE, EVAL_GRAVITY
    from summersph_b200.engine import Engine
    from summersph_b200.rotation_curve import ring_points

    g = (np.arange(1024) + 0.5) * (200.0 / 1024) - 100.0
    X, Y = np.meshgrid(g, g, indexing="xy")
    slice_pts = np.stack([X.ravel(), Y.ravel(), np.zeros(X.size)], 1)
    rng = np.random.default_rng(7)
    r = np.sqrt(rng.uniform(10.0 ** 2, 100.0 ** 2, 1 << 20)); phi = rng.uniform(0.0, 2.0 * np.pi, 1 << 20)
    rand_pts = np.stack([r * np.cos(phi), r * np.sin(phi), rng.standard_normal(1 << 20) * 0.05 * r], 1)
    ring_pts, _ = ring_points(np.linspace(10.0, 100.0, 46), 256)
    one_pt = np.array([[50.0, 0.0, 0.0]])

    p = default_params(MODE_VARIABLE_H)
    with Engine(p, device=0) as e:
        e.ics_disc(args.particles, seed=20251018)
        dt, t = 0.01, 0.0
        for _ in range(2):
            dt, t = e.step(dt, t)
        res = {}
        for name, pts in (("slice", slice_pts), ("random", rand_pts), ("rings", ring_pts), ("one", one_pt)):
            h, d = timed(e, lambda: e.gravity_at(pts), args.repeats)
            res[name] = {"points": len(pts), "host_ms": h, "device_ms": d, "ns_per_point": d * 1e6 / len(pts)}
        acc = e.gravity_at(slice_pts)["accepted"]
        # exact counters switch the far-field reuse off: every evaluation walks the whole tree (k_gravity<2>)
        e.set_exact_counters(True)
        e.evaluate(EVAL_TREE | EVAL_GRAVITY)
        ev = []
        for _ in range(args.repeats):
            e.timer_start()
            e.evaluate(EVAL_GRAVITY)
            ev.append(e.timer_stop())
        ms = float(np.median(ev))
        res["full_walk"] = {"particles": args.particles, "evaluate_device_ms": ms, "ns_per_particle": ms * 1e6 / args.particles}
        name, plim = card()
        line = {"what": "sph_gravity_at", "particles": args.particles, "mode": "variable_h", "repeats": args.repeats,
                "kernel": "k_gravity_at (thread per point)", **res,
                "slice_accepted_mean": float(np.mean(acc)), "gpu": name, "power_limit": plim}
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
