"""The benchmark's own evaluation path at the size the metric is quoted on, held to the oracle and to the exact path.

bench.py generates the 16M Keplerian disc on the device (`sph_ics_disc`, seed 20251018) and steps it resident; from the
third step on, evaluation A keeps the far-field gravity sums of the step before and adds only the near terms - from the
pairs the full walk recorded (`k_gravity_near`), or by the near-only walk (`k_gravity<1>`) for the runs whose records
overflowed - and the density and pair loops decide membership through their FP32 screens.  tests/test_gpu_scale_parity.py
holds a host-generated disc to the oracle with exact counters on (count-all screens, the plain gravity walk `k_gravity<2>`),
so none of that runs there.  Here, on the bench's own state after 4 resident steps:
  1. the near-only production evaluation against the exact-counter evaluation of the same state over all N rows (1e-12),
     and against the oracle's `sample_eval` per stratum (uniform, smallest h, largest h, widest leaf cells for h, next to
     the sink's accretion radius) at 1e-10 with neighbour counts and hashes bit for bit;
  2. the same whole-array comparison with forced record overflow, the near field walked, and a candidate-list pool too small;
  3. 6 resident steps with and without the far-field reuse (variable h at N, also with the cutoff at h where k_far_check
     must refuse; fixed h at N / 4): equal dt / t / counts, 1e-12;
  4. 4 host round trips (`sph_step_host`) against 4 resident steps: bit for bit, 3 recognised uploads;
  5. a -DSCREEN_AUDIT build of the engine: no FP32 screen decision contradicts the FP64 test behind it.

SPH_SCALE_PARITY_N overrides the size (default 16e6; 64e6 is config5: ~75 GB of device memory with the records and about
as much host memory for the oracle's tree - a developer run, not part of the default suite).
GPU wall time of this module at 16M: 84 s on one B200 (1000 W power limit, 16 host cores), of which the audit build
takes 20 s and the oracle's `sample_eval` on the 16M tree 9 s."""
import os
import re
import subprocess
import sys
import time

import numpy as np
import pytest

from summersph_b200 import default_params, MODE_VARIABLE_H, MODE_FIXED_H, Bodies, Sinks
from summersph_b200.state import GAS_FIELDS, SINK_FIELDS

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = int(float(os.environ.get("SPH_SCALE_PARITY_N", "16e6")))
SEED = 20251018                     # bench.py's disc
DIAG = ("rho", "omega", "P", "c", "ax", "ay", "az", "udot", "alphadot")
EXACT_TOL = 1e-12                   # two evaluations of one state that add the same terms in another order
ORACLE_TOL = 1e-10
N_UNIFORM, N_STRATUM = 2000, 300
ENV_SWITCHES = ("SPH_B200_FAR_SLOTS", "SPH_B200_NO_FAR_LISTS", "SPH_B200_LIST_POOL_BLOCKS", "SPH_B200_NO_FAR_REUSE", "SPH_B200_FAR_HCUT")


def _rel(a, b, scale_of=None):
    """max |a - b| / max(|b|, RMS): the RMS of `scale_of` (default b) - one stratum's own values."""
    ref = b if scale_of is None else scale_of
    scale = np.maximum(np.abs(b), np.sqrt(np.mean(ref * ref)))
    scale = np.where(scale > 0, scale, 1.0)
    return float(np.max(np.abs(a - b) / scale)) if len(b) else 0.0


def _clear_env(monkeypatch):
    for k in ENV_SWITCHES:
        monkeypatch.delenv(k, raising=False)


def _steps(e, k, dt=0.01, t=0.0):
    """k resident loop bodies; (dt, t, [(n_gas, n_sink) before the first and after every step])"""
    sizes = [e.sizes()]
    for _ in range(k):
        dt, t = e.step(dt, t)
        sizes.append(e.sizes())
    return dt, t, sizes


def _expected_reuse(sizes):
    """Evaluation A of step k >= 3 keeps the far sums stored by evaluation B of step k - 1 (step 1 starts on a new state,
    so step 2's evaluation B is the first to store) unless step k - 1 removed particles: the tree does not stand then."""
    return sum(1 for k in range(3, len(sizes)) if sizes[k - 1][0] == sizes[k - 2][0])


def _reuse_note(sizes, got):
    return (f"far-field reuses {got}, expected {_expected_reuse(sizes)} from the gas counts {[s[0] for s in sizes]}: where no step "
            "removed particles, a missing reuse means k_far_check found some h beyond its cutoff, an extra one a stale tree")


def _production_and_exact(e, sizes):
    """The near-only evaluation of the state the steps left (exact counters off, as bench.py steps), then the exact-counter
    evaluation of the same state; it has to come second: it walks without the split and voids the stored sums."""
    n_ovf = e.far_overflow_runs()
    f0 = e.far_reuse_count()
    e.evaluate()
    near_only = e.far_reuse_count() - f0
    assert near_only == 1, (f"the evaluation after the steps did not keep the far sums (gas counts {[s[0] for s in sizes]}: "
                            "a removal in the last step, or k_far_check found some h beyond its cutoff)")
    d_prod = e.diag()
    e.set_exact_counters(True)
    e.evaluate()
    e.set_exact_counters(False)
    assert e.far_reuse_count() == f0 + 1
    return d_prod, e.diag(), n_ovf


def _whole_array(d_prod, d_exact, tag):
    worst = {k: _rel(d_prod[k], d_exact[k]) for k in DIAG}
    print(f"{tag}: production vs exact counters over all {len(d_exact['rho'])} rows, worst relerr per field", worst)
    assert max(worst.values()) < EXACT_TOL, (tag, worst)
    for k in ("sink_ax", "sink_ay", "sink_az"):
        assert _rel(d_prod[k], d_exact[k]) < EXACT_TOL, (tag, k)
    return worst


@pytest.fixture(scope="module")
def bench_state(built_engine):
    """Part 1's GPU side: bench.py's state after 4 resident steps, its production and its exact-counter evaluation."""
    from summersph_b200.engine import Engine
    mp = pytest.MonkeyPatch()
    _clear_env(mp)
    t0 = time.perf_counter()
    p = default_params(MODE_VARIABLE_H)
    with Engine(p) as e:
        e.ics_disc(N, seed=SEED)
        dt, t, sizes = _steps(e, 4)
        reuse = e.far_reuse_count()
        assert reuse == _expected_reuse(sizes), _reuse_note(sizes, reuse)      # no removal: 2, evaluation A of steps 3 and 4
        b, s = e.download()
        d_prod, d_exact, n_ovf = _production_and_exact(e, sizes)
        ce, he, _, _ = e.neighbours(with_list=False)
        tr = e.tree()
        leaf_size = tr["size"]
        del tr
    mp.undo()
    print(f"bench state: N {N} -> {sizes[-1][0]} gas, {sizes[-1][1]} sinks after 4 steps, dt {dt} t {t}, far-field reuses {reuse}, "
          f"overflowing runs with 128 slots (natural): {n_ovf}  [{time.perf_counter() - t0:.1f} s]")
    return dict(params=p, b=b, s=s, d_prod=d_prod, d_exact=d_exact, count=ce, hash=he, leaf_size=leaf_size, n_ovf=n_ovf)


def test_production_evaluation_matches_exact_counters_on_every_row(bench_state):
    """Near-only gravity (recorded pairs + walked overflow runs) against the plain walk, screened and listed density / pair
    sums against count-all: the same terms in another order, over all N rows."""
    _whole_array(bench_state["d_prod"], bench_state["d_exact"], "default")


def _strata(st):
    b, s, p = st["b"], st["s"], st["params"]
    n = len(b)
    rng = np.random.default_rng(SEED)
    k = min(N_STRATUM, n)
    rs = s.radius[0] if np.isfinite(s.radius[0]) else p.sink_radius
    dist = np.sqrt((b.x - s.x[0]) ** 2 + (b.y - s.y[0]) ** 2 + (b.z - s.z[0]) ** 2)
    return {
        "uniform": np.sort(rng.choice(n, min(N_UNIFORM, n), replace=False)),
        "smallest_h": np.argsort(b.h, kind="stable")[:k],                          # inner disc by the sink: deepest tree, most near pairs
        "largest_h": np.argsort(-b.h, kind="stable")[:k],                          # outer disc: sparse cells, loosest screen bounds
        "wide_leaf": np.argsort(-(st["leaf_size"] / b.h), kind="stable")[:k],      # isolated particles in wide cells
        "sink_edge": np.argsort(np.abs(dist - rs), kind="stable")[:k],             # next to the accretion radius
    }


def test_production_evaluation_matches_oracle_by_stratum(bench_state):
    """The production evaluation against the oracle's on the downloaded state, one `sample_eval` for all strata (it
    builds the whole-set tree on the host); each stratum's error is scaled by its own RMS, so a stratum of small values is
    not hidden behind the large ones.  Neighbour counts and hashes bit for bit."""
    from oracle.oracle import Oracle
    st = bench_state
    strata = _strata(st)
    targets = np.unique(np.concatenate(list(strata.values()))).astype(np.int32)
    t0 = time.perf_counter()
    o = Oracle(st["params"], threads=os.cpu_count() or 1)
    o.upload(st["b"], st["s"])
    so = o.sample_eval(targets)
    o.close()
    print(f"oracle sample_eval of {len(targets)} targets on {len(st['b'])} rows: {time.perf_counter() - t0:.1f} s")
    d = st["d_prod"]
    assert np.array_equal(st["count"][targets], so["count"]), "neighbour counts differ"
    assert np.array_equal(st["hash"][targets], so["hash"]), "neighbour sets differ"
    report = {}
    for name, idx in strata.items():
        pos = np.searchsorted(targets, idx)
        worst = {k: _rel(d[k][idx], so[k][pos], so[k][pos]) for k in DIAG}
        report[name] = worst
        print(f"stratum {name} ({len(idx)} targets, h {st['b'].h[idx].min():.3g}..{st['b'].h[idx].max():.3g}, "
              f"pairs {int(so['pairs'][pos].sum())}): worst relerr {max(worst.values()):.2e}", worst)
    bad = {name: w for name, w in report.items() if max(w.values()) >= ORACLE_TOL}
    assert not bad, bad


VARIANTS = {
    "forced_overflow": {"SPH_B200_FAR_SLOTS": "32"},           # a large share of runs through k_gravity<1>
    "near_by_walk": {"SPH_B200_NO_FAR_LISTS": "1"},            # no records: the near-only walk serves every run
    "list_fallback": {"SPH_B200_LIST_POOL_BLOCKS": "64"},      # the candidate-list pool overflows: k_force<false> walks
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_recorded_pair_variants_match_exact_counters(variant, bench_state, built_engine, monkeypatch):
    """The bench state under each switch (read in sph_create: one context each): the near-only evaluation against the
    exact-counter evaluation of the same context over all rows.  The overflow switch has to send runs to the walk."""
    from summersph_b200.engine import Engine
    _clear_env(monkeypatch)
    for k, v in VARIANTS[variant].items():
        monkeypatch.setenv(k, v)
    with Engine(default_params(MODE_VARIABLE_H)) as e:
        e.ics_disc(N, seed=SEED)
        _, _, sizes = _steps(e, 4)
        reuse = e.far_reuse_count()
        assert reuse == _expected_reuse(sizes), _reuse_note(sizes, reuse)
        d_prod, d_exact, n_ovf = _production_and_exact(e, sizes)
    print(f"{variant}: overflowing runs {n_ovf} (natural, 128 slots: {bench_state['n_ovf']})")
    if variant == "forced_overflow":
        assert n_ovf > 0, "32 recorded slots per particle overflowed no run: the near-only walk was not exercised"
        assert n_ovf > bench_state["n_ovf"]
    _whole_array(d_prod, d_exact, variant)


def _trajectory(p, n, steps, env, monkeypatch):
    from summersph_b200.engine import Engine
    _clear_env(monkeypatch)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    with Engine(p) as e:
        e.ics_disc(n, seed=SEED)
        dt, t, sizes = _steps(e, steps)
        reuse = e.far_reuse_count()
        b, s = e.download()
    return dict(dt=dt, t=t, sizes=sizes, reuse=reuse, b=b, s=s)


def _same_trajectory(a, off, tag, refused=False):
    """`a` (far-field reuse on) against `off` (every evaluation walks the whole tree).  refused: the near / far cutoff is
    h itself, so k_far_check has to turn the reuse down after some step (an h grew) - stale far sums would pass it."""
    assert (a["dt"], a["t"]) == (off["dt"], off["t"]), tag
    assert a["sizes"] == off["sizes"], (tag, a["sizes"], off["sizes"])
    assert off["reuse"] == 0, tag
    worst = {k: _rel(getattr(a["b"], k), getattr(off["b"], k)) for k in GAS_FIELDS}
    worst.update({"sink_" + k: _rel(getattr(a["s"], k), getattr(off["s"], k)) for k in SINK_FIELDS if k != "radius"})
    print(f"{tag}: {a['sizes'][-1]} after {len(a['sizes']) - 1} steps, far-field reuses {a['reuse']} (without refusals "
          f"{_expected_reuse(a['sizes'])}), worst relerr {max(worst.values()):.2e}", worst)
    assert max(worst.values()) < EXACT_TOL, (tag, worst)
    assert np.array_equal(a["s"].radius, off["s"].radius, equal_nan=True), tag
    if refused:
        assert a["reuse"] < _expected_reuse(a["sizes"]), (tag, "k_far_check never refused the reuse although h grew past the cutoff")
    else:
        assert a["reuse"] == _expected_reuse(a["sizes"]), (tag, _reuse_note(a["sizes"], a["reuse"]))


def test_trajectory_with_far_reuse_matches_full_walks(built_engine, monkeypatch):
    """6 resident steps of the bench disc with and without the far-field reuse (one context after the other), and once
    more with the near / far cutoff at h itself (SPH_B200_FAR_HCUT=1), where k_far_check must refuse stale far sums."""
    p = default_params(MODE_VARIABLE_H)
    off = _trajectory(p, N, 6, {"SPH_B200_NO_FAR_REUSE": "1"}, monkeypatch)
    on = _trajectory(p, N, 6, {}, monkeypatch)
    _same_trajectory(on, off, f"variable h, N {N}")
    del on
    low = _trajectory(p, N, 6, {"SPH_B200_FAR_HCUT": "1"}, monkeypatch)
    _same_trajectory(low, off, f"variable h, N {N}, cutoff 1 h", refused=True)


def test_trajectory_with_far_reuse_matches_full_walks_fixed_h(built_engine, monkeypatch):
    """The same in fixed h at N / 4, where h never changes and the reuse always stands.  h_fixed = the median of the
    disc's variable-h smoothing lengths, so the neighbour counts stay near those of the variable-h disc."""
    from summersph_b200.engine import Engine
    n = N // 4
    _clear_env(monkeypatch)
    with Engine(default_params(MODE_VARIABLE_H)) as e:
        e.ics_disc(n, seed=SEED)
        h_fixed = float(np.median(e.download()[0].h))
    p = default_params(MODE_FIXED_H, h_fixed=h_fixed)
    off = _trajectory(p, n, 6, {"SPH_B200_NO_FAR_REUSE": "1"}, monkeypatch)
    on = _trajectory(p, n, 6, {}, monkeypatch)
    _same_trajectory(on, off, f"fixed h {h_fixed:.4g}, N {n}")


def test_host_round_trips_match_resident_steps(built_engine, monkeypatch):
    """The loop bench.py's e2e leg times: 4 `sph_step_host` round trips, each output fed back as the next input, against
    4 resident steps from the same uploaded rows - bit for bit; the 3 uploads after the first are recognised."""
    from summersph_b200.engine import Engine
    _clear_env(monkeypatch)
    p = default_params(MODE_VARIABLE_H)
    with Engine(p) as e:
        e.ics_disc(N, seed=SEED)
        b0, s0 = e.download()
    with Engine(p) as e:
        b, s, dt, t = b0, s0, 0.01, 0.0
        ns_hist = [len(b)]
        for _ in range(4):
            ob, os_ = Bodies.empty(len(b)), Sinks.empty(len(s) + 8)
            dt, t, n2, ns2 = e.step_host(b, s, dt, t, into=(ob, os_))
            b = ob.take(slice(0, n2)) if n2 < len(ob) else ob
            s = Sinks(*[getattr(os_, k)[:ns2].copy() for k in SINK_FIELDS])
            ns_hist.append(n2)
        hits = e.resident_hits()
        host = (dt, t, b, s)
    with Engine(p) as e:
        e.upload(b0, s0)
        dt, t, sizes = _steps(e, 4)
        rb, rs = e.download()
    assert (host[0], host[1]) == (dt, t)
    assert [z[0] for z in sizes] == ns_hist, (ns_hist, sizes)
    for k in GAS_FIELDS:
        assert np.array_equal(getattr(host[2], k), getattr(rb, k)), f"gas column {k} differs"
    for k in SINK_FIELDS:
        assert np.array_equal(getattr(host[3], k), getattr(rs, k), equal_nan=True), f"sink column {k} differs"
    expected = sum(1 for k in range(1, 4) if ns_hist[k] == ns_hist[k - 1])     # a removal makes the next upload a new state
    assert hits == expected, f"recognised uploads {hits}, expected {expected} from the gas counts {ns_hist}"
    if ns_hist[-1] == len(b0):
        assert hits == 3
    print(f"host round trips: {ns_hist}, recognised uploads {hits}, bit-identical to resident steps")


AUDIT_RUN = r"""
import sys
sys.path.insert(0, sys.argv[1])
from summersph_b200 import default_params, MODE_VARIABLE_H
from summersph_b200.engine import Engine
with Engine(default_params(MODE_VARIABLE_H), lib_path=sys.argv[3]) as e:
    e.ics_disc(int(sys.argv[2]), seed=int(sys.argv[4]))
    dt, t = 0.01, 0.0
    for _ in range(4):
        dt, t = e.step(dt, t)
    f0 = e.far_reuse_count()
    e.evaluate()
    print("near_only", e.far_reuse_count() - f0, "gas", e.sizes()[0])
"""
AUDIT_LINE = re.compile(r"^SCREEN_AUDIT (\S+) density (\d+) pair (\d+) gravity (\d+)$")


@pytest.fixture(scope="module")
def audit_lib(tmp_path_factory):
    """The engine built with -DSCREEN_AUDIT (the flags of the in-tree build) into a temporary directory."""
    from summersph_b200.build import nvcc_command
    d = tmp_path_factory.mktemp("screen_audit")
    so = str(d / "libsph_audit.so")
    t0 = time.perf_counter()
    res = subprocess.run(nvcc_command(so, ["-DSCREEN_AUDIT"]), capture_output=True, text=True, cwd=str(d))
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    print(f"audit build: {time.perf_counter() - t0:.1f} s")
    return so


def test_screen_audit_counts_no_contradiction(audit_lib):
    """Every FP32 screen decision of the walks (density, pair loop, gravity classification and far entries) checked against
    the FP64 test behind it, on the bench state's 4 steps and the near-only evaluation after them: none may disagree.  A
    member dropped at q ~ 2 changes rho by far less than the field tolerances; this counts membership itself."""
    res = subprocess.run([sys.executable, "-B", "-c", AUDIT_RUN, ROOT, str(N), audit_lib, str(SEED)],
                         capture_output=True, text=True, cwd=ROOT, env=dict(os.environ))
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    lines = [AUDIT_LINE.match(ln.strip()) for ln in res.stderr.splitlines() if ln.startswith("SCREEN_AUDIT")]
    assert all(lines), res.stderr[-4000:]
    for m in lines:
        print(m.group(0))
    print(res.stdout.strip())
    calls = [m.group(1) for m in lines]
    assert calls.count("step") == 4 and calls.count("evaluate") == 1, calls
    assert "near_only 1" in res.stdout, res.stdout
    bad = [m.group(0) for m in lines if any(int(m.group(g)) != 0 for g in (2, 3, 4))]
    assert not bad, bad
