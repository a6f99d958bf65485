"""Developer script: how often the FP32 screens of the walks decide against the FP64 tests behind them.

Needs the audit build (scripts/build_variant.sh audit -DSCREEN_AUDIT): after every evaluation and step the engine prints
`SCREEN_AUDIT <call> density D pair P gravity G` on stderr, the contradictions since the last line (0 for a correct screen).
Runs the clustered cases of tests/test_widen_screen_edges.py (one evaluation, one density + SPH evaluation, one step in
fixed h), then `steps` steps of an N-particle device-generated disc (bench.py's state).  usage: screen_audit.py [N] [steps]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from summersph_b200 import default_params, MODE_VARIABLE_H, MODE_FIXED_H, EVAL_TREE, EVAL_DENSITY, EVAL_SPH  # noqa: E402
from summersph_b200.engine import Engine  # noqa: E402
from test_widen_screen_edges import MODES, SCALES, build_case  # noqa: E402

LIB = os.path.join(ROOT, "summersph_b200", "variants", "libsph_audit.so")
n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 16_000_000
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 3


def say(msg):
    sys.stdout.flush(); sys.stderr.write(msg + "\n"); sys.stderr.flush()


for mode in MODES:
    for scale in SCALES:
        c = build_case(mode, scale)
        p, b, s = c["params"], c["bodies"], c["sinks"]
        say(f"case {mode} {scale}: {len(b)} gas, {len(c['pairs'])} binaries, {len(c['probes'])} probes")
        with Engine(p, lib_path=LIB) as e:
            e.upload(b, s); e.evaluate()
            e.evaluate(EVAL_TREE | EVAL_DENSITY | EVAL_SPH)
            if p.mode == MODE_FIXED_H or scale == "h1e-3":
                e.upload(b, s); e.step(0.01, 0.0)
say(f"disc {n}, {steps} steps")
with Engine(default_params(MODE_VARIABLE_H), lib_path=LIB) as e:
    e.ics_disc(n, seed=20251018)
    dt, t = 0.01, 0.0
    for _ in range(steps):
        dt, t = e.step(dt, t)
