"""Host-side `simulate` shell (SUMMER_SPH.f90:863-930 | "SUMMER_SPH - Variable.f90":1076-1164).

The loop shell, save cadence and per-step print stay on the host exactly as in the reference; the loop
body (F:886-928 | V:1120-1162) is one call into the CUDA engine through the C-ABI (`sph_step`).
"""
from ._abi import SphParams, drift_report
from .state import Bodies, Sinks
from .io import make_save


def simulate(bodies: Bodies, sinks: Sinks, params: SphParams, engine=None, save_dir=None, max_steps=None,
             log=print, device=0, drift=None):
    """Run until t >= params.end_time (no final-step clipping, no final save: F:879).

    `engine` defaults to a new CUDA `Engine` (there is no CPU fallback). Saves `save<k>.txt` into
    `save_dir` when `t > k*end_time/1000` (F:874,881; the reference reads t_list(0) out of bounds on
    the first pass, here t_list(0) := 0 so save0 is written at the first step with t > 0).
    `drift`: pass a dict to get the run's conservation report (north_star: "energy/momentum drift reported
    over the full run"): the engine's conserved sums (`sph_conserved`) are taken before the first and after the
    last step, the dict receives `first`, `last` and the relative drifts, and two extra lines are logged.  The
    reference itself prints nothing of the kind, so the default leaves its output untouched.  `drift=` works on a
    multi-rank engine of either form when every rank calls `simulate` (under the Morton domains `sph_conserved` is
    collective); every rank then gets the same report.
    Returns (bodies, sinks, t, dt, steps)."""
    own = engine is None
    if own:
        from .engine import Engine
        engine = Engine(params, device=device)
    try:
        engine.upload(bodies, sinks)
        t, dt = 0.0, 1.0e-2                                                  # F:872,875
        first = engine.conserved() if drift is not None else None
        end_time = params.end_time
        t_test, steps = 0, 0
        while t < end_time:                                                  # F:879
            if save_dir is not None and t > t_test * end_time / 1000.0:      # F:881
                b, s = engine.download()
                make_save(b, s, t_test, params, save_dir)
                t_test += 1
            n, _ = engine.sizes()
            log(f" SPH Particles: {n} dt : {dt!r} time :  {t!r}")            # F:891
            dt, t = engine.step(dt, t)
            steps += 1
            if max_steps is not None and steps >= max_steps:
                break
        if drift is not None:
            last = engine.conserved()
            drift.update(first=first, last=last, steps=steps, t=t, **drift_report(first, last))
            log(f" Conserved sums: E = {first['e_total']!r} -> {last['e_total']!r}  (kin {last['e_kin']!r} int {last['e_int']!r} pot {last['e_pot']!r})")
            fmt = lambda v: "n/a" if v is None else f"{v:.3e}"   # noqa: E731
            log(f" Drift over {steps} steps: dE/|E0| = {fmt(drift['energy_rel'])}  |dP|/sqrt(2 E_kin M) = {fmt(drift['momentum_rel'])}"
                f"  |dL|/|L| = {fmt(drift['angular_momentum_rel'])}  dM/M0 = {fmt(drift['mass_rel'])}")
        b, s = engine.download()
        return b, s, t, dt, steps
    finally:
        if own:
            engine.close()
