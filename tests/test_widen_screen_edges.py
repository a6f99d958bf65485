"""The FP32 screens of the walks (density prefilter, pair-loop prefilter, gravity run-box classification and mixed-node
MAC) on clustered inputs, against the CPU oracle.

The screens compare float coordinates taken relative to the centre of a walk group or gravity run, so their rounding
grows with the group's width, not with h or with the distance they decide on.  Smooth inputs keep groups a few h wide;
these cases do not.  A sparse background (30k particles in a 200 AU cube, groups many AU wide) holds a few hundred
planted binaries whose members sit just inside each other's kernel, q = r / h = 2 (1 - eps) with eps log-uniform in
[1e-9, 1e-3], at h ~ 1e-3 (one-word keys) and h ~ 1e-7 (two-word keys, leaf levels > 21).  Gravity probes sit just on
either side of the opening test of a binary's parent node: size / sqrt(d^2 + soft) = theta (1 + eps), eps of both signs.

What must hold, with one evaluation in the default counter mode: the exact integers (order, leaves, neighbour counts
and hashes), the default-mode counters `density_contributing` and `grav_accepted` (read before any exact-counter
evaluation: the exact mode bypasses the walk screens), and per planted particle every field against |oracle value|."""
import numpy as np
import pytest

from conftest import relerr
from summersph_b200 import (default_params, MODE_FIXED_H, MODE_VARIABLE_H, FLAG_SOFT_USES_HI, Bodies, Sinks,
                            EVAL_ALL, EVAL_TREE, EVAL_DENSITY, EVAL_SPH)
from summersph_b200.state import GAS_FIELDS, SINK_FIELDS

MODES = {"fixed": MODE_FIXED_H, "variable": MODE_VARIABLE_H, "soft_hi": MODE_VARIABLE_H | FLAG_SOFT_USES_HI}
SCALES = {"h1e-3": 1e-3, "h1e-7": 1e-7}
N_BG, HALF, N_PAIRS, N_PROBES = 30_000, 100.0, 300, 60
TOL = 1e-10
FIELDS = ("rho", "omega", "ax", "ay", "az", "udot", "alphadot")


# ---------------------------------------------------------------------------------------------------------------------
# builder
# ---------------------------------------------------------------------------------------------------------------------
def _directions(rng, n):
    u = rng.normal(size=(n, 3))
    return u / np.linalg.norm(u, axis=1)[:, None]


def _parent_cell(pos, level, root_center, root_size):
    """Centre and size of the level-(level - 1) cell holding `pos`, descended the way the oracle builds its tree."""
    c = np.array(root_center, dtype=float); s = float(root_size)
    for _ in range(level - 1):
        c = c + np.where(pos > c, 0.25 * s, -0.25 * s)
        s = s * 0.5
    return c, s


def _tree(p, b, s):
    from oracle.oracle import Oracle
    o = Oracle(p); o.upload(b, s); o.evaluate(EVAL_TREE)
    return o.tree()


def _bodies(x, v, h, m):
    n = len(x)
    return Bodies(x[:, 0].copy(), x[:, 1].copy(), x[:, 2].copy(), v[:, 0].copy(), v[:, 1].copy(), v[:, 2].copy(),
                  np.full(n, 0.25), m, np.full(n, 0.1), h)


def build_case(mode_name, scale_name, seed=0, probes=True):
    """The clustered input of one mode and h scale.  Returns a dict: params, bodies, sinks, `pairs` (k, 2) row numbers of
    the binary members, `probes` the rows of the gravity probes that survived the tree check, `n_probe_planned`."""
    mode, hs = MODES[mode_name], SCALES[scale_name]
    variable = bool(mode & MODE_VARIABLE_H)
    # variable h: h_fixed only sets the softening (0.001 h_fixed); small, so soft << d^2 at the probes
    p = default_params(mode, h_fixed=hs if not variable else hs * hs)
    eta = p.eta
    rng = np.random.default_rng(1000 * seed + 10 * list(MODES).index(mode_name) + list(SCALES).index(scale_name))
    from scipy.spatial import cKDTree

    xb = rng.uniform(-HALF, HALF, (N_BG, 3))
    hb = rng.uniform(0.8, 1.2, N_BG) if variable else np.full(N_BG, hs)
    mb = np.full(N_BG, 1e-7)
    # binary centres: inside the cube, farther than 2 h of every background particle and from one another
    cand = rng.uniform(-0.9 * HALF, 0.9 * HALF, (8 * N_PAIRS, 3))
    cand = cand[cKDTree(xb).query(cand)[0] > 3.0]
    centres = []
    for c in cand:
        if all(np.linalg.norm(c - q) > 3.0 for q in centres):
            centres.append(c)
        if len(centres) == N_PAIRS:
            break
    centres = np.array(centres)
    k = len(centres)
    eps = 10.0 ** rng.uniform(-9, -3, k)
    u = _directions(rng, k)
    half = np.arange(k) % 3 == 2 if variable else np.zeros(k, bool)      # h_j = h_i / 2: only max(h_i, h_j) admits the pair
    r = 2.0 * hs * (rng.uniform(0.8, 1.2, k) if variable else 1.0 - eps)
    xa = centres - 0.5 * r[:, None] * u
    xc = centres + 0.5 * r[:, None] * u
    if variable:                 # h from the separation the rounded coordinates really have: q = 2 (1 - eps) to rounding
        ha = np.sqrt(np.sum((xa - xc) ** 2, 1)) / (2.0 * (1.0 - eps))
        hb2 = np.where(half, 0.5 * ha, ha)
    else:                        # one h for all: at h ~ 1e-7 the coordinates' ulp moves q by ~1e-7, past 2 for some pairs
        ha = hb2 = np.full(k, hs)
    hm = lambda h: 0.2 * h ** 3 / eta ** 3          # m (eta / h)^3 = 0.2 <= 0.5: no sink is created (V:549)
    x = np.concatenate([xb, xa, xc])
    h = np.concatenate([hb, ha, hb2])
    m = np.concatenate([mb, hm(ha), hm(hb2)])
    v = rng.normal(0.0, 0.1, (len(x), 3))
    pairs = np.stack([N_BG + np.arange(k), N_BG + k + np.arange(k)], 1)
    s = Sinks.dummy()
    case = {"params": p, "pairs": pairs, "pair_eps": eps, "half": half, "probes": np.zeros(0, np.int64), "n_probe_planned": 0}
    if not probes:
        case.update(bodies=_bodies(x, v, h, m), sinks=s)
        return case

    # gravity probes at the opening test of the binaries' parent nodes (the two members are siblings)
    t = _tree(p, _bodies(x, v, h, m), s)
    lvl = t["level"]
    hp = hs if not (mode & FLAG_SOFT_USES_HI) else min(hs, 1e3 * hs * hs)    # soft = 0.001 h_probe << d^2
    soft = 0.001 * (hp if mode & FLAG_SOFT_USES_HI else p.h_fixed)
    theta = p.theta
    kd = cKDTree(x)
    px, owner, peps = [], [], []
    for q in range(k):
        ia, ic = pairs[q]
        if lvl[ia] != lvl[ic] or lvl[ia] < 2:
            continue
        ca, S = _parent_cell(x[ia], lvl[ia], t["root_center"], t["root_size"])
        cc, _ = _parent_cell(x[ic], lvl[ic], t["root_center"], t["root_size"])
        if not np.array_equal(ca, cc):
            continue
        e = (1 if len(px) % 2 else -1) * 10.0 ** rng.uniform(-9, -3)
        d2 = (S / (theta * (1.0 + e))) ** 2 - soft
        if d2 <= 0.0:
            continue
        com = (m[ia] * x[ia] + m[ic] * x[ic]) / (m[ia] + m[ic])
        pos = com + np.sqrt(d2) * _directions(rng, 1)[0]
        if not np.any(np.abs(pos - ca) > 0.5 * S):
            continue                                               # inside the parent cell: it would change the node
        near = kd.query_ball_point(pos, 3.0)
        if any(j not in (ia, ic) for j in near):
            continue
        if min(np.linalg.norm(pos - x[ia]), np.linalg.norm(pos - x[ic])) <= 2.2 * max(h[ia], h[ic], hp):
            continue                                               # no density or pair term with the members
        px.append(pos); owner.append(q); peps.append(e)
        if len(px) == N_PROBES:
            break
    n_plan = len(px)
    px = np.array(px).reshape(-1, 3)
    owner = np.array(owner, np.int64); peps = np.array(peps)
    vp = rng.normal(0.0, 0.1, (n_plan, 3))
    keep = np.ones(n_plan, bool)
    for _ in range(4):          # rebuild: drop the probes that change a binary's leaves, until none does
        kept = int(keep.sum())
        b = _bodies(np.concatenate([x, px[keep]]), np.concatenate([v, vp[keep]]),
                    np.concatenate([h, np.full(kept, hp)]), np.concatenate([m, np.full(kept, hm(hp))]))
        t2 = _tree(p, b, s)
        rows = np.flatnonzero(keep)
        bad = [i for i, q in enumerate(owner[keep]) if t2["level"][pairs[q, 0]] != lvl[pairs[q, 0]] or t2["level"][pairs[q, 1]] != lvl[pairs[q, 1]]]
        if not bad:
            break
        keep[rows[bad]] = False
    else:
        raise RuntimeError(f"{mode_name} {scale_name}: the probes still change a binary's leaves after 4 rebuilds")
    n0 = len(x)
    case.update(bodies=b, sinks=s, probes=n0 + np.arange(int(keep.sum())), probe_owner=owner[keep], probe_eps=peps[keep],
                n_probe_planned=n_plan)
    return case


_CACHE = {}


def case_of(mode_name, scale_name):
    key = (mode_name, scale_name)
    if key not in _CACHE:
        _CACHE[key] = build_case(mode_name, scale_name)
    return _CACHE[key]


def pair_q(case):
    """q = r / max(h_i, h_j) of every planted pair (the pair's kernel with the larger support)."""
    b, (ia, ic) = case["bodies"], case["pairs"].T
    r = np.sqrt((b.x[ia] - b.x[ic]) ** 2 + (b.y[ia] - b.y[ic]) ** 2 + (b.z[ia] - b.z[ic]) ** 2)
    hh = np.maximum(b.h[ia], b.h[ic]) if case["params"].mode & MODE_VARIABLE_H else np.full(len(ia), case["params"].h_fixed)
    return r / hh


def planted_tolerance(case, gravity):
    """Per member: 1e-10, plus the conditioning of the pair's terms.  One rounding of q changes a kernel value that
    vanishes at q = 2 (W, dW ~ (2 - q)^k near the edge) by about 2^-52 q / |2 - q| of itself.  With gravity, the
    partner's term is taken from its one-particle node's centre of mass, and one rounding of that changes the
    separation r by 2^-52 |x| / r of itself: at h ~ 1e-7 and |x| ~ 100 that is ~1e-7, which no summation order or
    arithmetic can remove.  (Without gravity r comes from x_i - x_j, exact for two members this close.)"""
    b, (ia, ic) = case["bodies"], case["pairs"].T
    q = pair_q(case)
    cond = q / np.maximum(np.abs(2.0 - q), 1e-300)
    if gravity:
        xmax = np.max(np.abs(np.stack([b.x[ia], b.y[ia], b.z[ia]], 1)), 1)
        cond = cond + xmax / (q * np.maximum(b.h[ia], b.h[ic]))
    tol = TOL + 16 * 2.0 ** -52 * cond
    return np.concatenate([tol, tol])


def assert_planted(got, ref, rows, tol, what):
    """Each planted particle: |got - ref| <= tol |ref|, and the same zeros."""
    for k in FIELDS:
        a, b = got[k][rows], ref[k][rows]
        assert np.array_equal(a == 0.0, b == 0.0), (what, k, "zero pattern", rows[np.flatnonzero((a == 0.0) != (b == 0.0))][:5])
        err = np.abs(a - b) / np.where(b != 0.0, np.abs(b), 1.0)
        bad = np.flatnonzero(err > tol)
        assert bad.size == 0, (what, k, rows[bad][:5], err[bad][:5])


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the builder, through the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale", list(SCALES))
def test_builder_plants_what_it_says(scale):
    """Fixed h, h_fixed below the background spacing: every density term other than the self terms belongs to a planted
    pair with q <= 2, so the oracle's contributing count is n + 2 x those pairs.  Every planned probe survives the
    rebuild with the binary's leaves unchanged and sits outside the parent cell."""
    from oracle.oracle import Oracle
    c = case_of("fixed", scale)
    p, b, s = c["params"], c["bodies"], c["sinks"]
    q = pair_q(c)
    assert np.all(np.abs(q - 2.0) < 2.2e-3) and np.mean(q <= 2.0) > 0.8
    o = Oracle(p); o.upload(b, s); o.evaluate(EVAL_TREE | EVAL_DENSITY)
    assert o.counters()["density_contributing"] == len(b) + 2 * int(np.sum(q <= 2.0))
    assert len(c["probes"]) == c["n_probe_planned"]
    if scale == "h1e-3":
        assert c["n_probe_planned"] >= N_PROBES // 2
        assert np.any(c["probe_eps"] > 0) and np.any(c["probe_eps"] < 0)
    lv = o.tree()["level"]
    assert lv[c["pairs"]].max() > 21 if scale == "h1e-7" else lv[c["pairs"]].max() <= 21


@pytest.mark.parametrize("scale", list(SCALES))
@pytest.mark.parametrize("mode", list(MODES))
def test_builder_probes(mode, scale):
    """Every mode and scale: the planned probes all survive the rebuild, on both sides of the opening test."""
    c = case_of(mode, scale)
    assert len(c["probes"]) == c["n_probe_planned"] >= N_PROBES // 2
    assert len(c["bodies"]) == N_BG + 2 * len(c["pairs"]) + len(c["probes"])
    assert np.any(c["probe_eps"] > 0) and np.any(c["probe_eps"] < 0)
    assert np.any(c["half"]) == (mode != "fixed")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _engine(p):
    from summersph_b200.engine import Engine
    return Engine(p)


def _compare_integers(o, e):
    to, te = o.tree(), e.tree()
    assert np.array_equal(to["order"], te["order"])
    assert np.array_equal(to["level"], te["level"])
    for k in ("cx", "cy", "cz", "size"):
        assert np.array_equal(to[k], te[k]), k
    co, ho, _, _ = o.neighbours(with_list=False); ce, he, _, _ = e.neighbours(with_list=False)
    assert np.array_equal(co, ce), np.flatnonzero(co != ce)[:5]
    assert np.array_equal(ho, he)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", list(SCALES))
@pytest.mark.parametrize("mode", list(MODES))
def test_evaluation_matches_oracle(mode, scale, built_engine):
    from oracle.oracle import Oracle
    c = case_of(mode, scale)
    p, b, s = c["params"], c["bodies"], c["sinks"]
    o = Oracle(p); o.record_neighbours(True); o.upload(b, s); o.evaluate()
    with _engine(p) as e:
        e.upload(b, s); e.evaluate()
        co, ce = o.counters(), e.counters()         # default mode: the screens decided
        assert ce["density_contributing"] == co["density_contributing"], (ce["density_contributing"], co["density_contributing"])
        assert ce["grav_accepted"] == co["grav_accepted"], (ce["grav_accepted"], co["grav_accepted"])
        _compare_integers(o, e)
        do, de = o.diag(), e.diag()
    for k in do:
        assert relerr(de[k], do[k]) < TOL, k
    members = c["pairs"].T.reshape(-1)
    assert_planted(de, do, members, planted_tolerance(c, gravity=True), "members")
    if len(c["probes"]):
        assert_planted(de, do, c["probes"], TOL, "probes")


@pytest.mark.gpu
@pytest.mark.parametrize("scale", list(SCALES))
@pytest.mark.parametrize("mode", ["fixed", "variable"])
def test_pair_loop_planted_terms(mode, scale, built_engine):
    """Density and SPH only: a member's a, du/dt and d(alpha)/dt are its partner's term alone, so a dropped pair shows
    as a zero where the oracle has a value."""
    from oracle.oracle import Oracle
    c = case_of(mode, scale)
    p, b, s = c["params"], c["bodies"], c["sinks"]
    mask = EVAL_TREE | EVAL_DENSITY | EVAL_SPH
    o = Oracle(p); o.upload(b, s); o.evaluate(mask)
    with _engine(p) as e:
        e.upload(b, s); e.evaluate(mask)
        assert e.counters()["density_contributing"] == o.counters()["density_contributing"]
        do, de = o.diag(), e.diag()
    members = c["pairs"].T.reshape(-1)
    inside = np.tile(pair_q(c) < 2.0, 2)
    assert np.all(do["ax"][members[inside]] != 0.0)
    assert_planted(de, do, members, planted_tolerance(c, gravity=False), "members")
    for k in do:
        assert relerr(de[k], do[k]) < TOL, k


def _one_step(c, built_engine):
    from oracle.oracle import Oracle
    p, b, s = c["params"], c["bodies"], c["sinks"]
    o = Oracle(p); o.upload(b, s)
    with _engine(p) as e:
        e.upload(b, s)
        dto, to = o.step(0.01, 0.0); dte, te = e.step(0.01, 0.0)
        assert (dto, to) == (dte, te)
        assert o.sizes() == e.sizes()
        if p.mode & MODE_VARIABLE_H:
            assert o.counters()["h_iterations"] == e.counters()["h_iterations"]
        bo, so = o.download(); be, se = e.download()
    for k in GAS_FIELDS:
        assert relerr(getattr(be, k), getattr(bo, k)) < TOL, k
    for k in ("x", "y", "z", "vx", "vy", "vz", "m", "radius"):
        assert relerr(getattr(se, k), getattr(so, k)) < TOL, "sink " + k


@pytest.mark.gpu
def test_one_step_fixed_h(built_engine):
    """h ~ 1e-3 only: at h ~ 1e-7 the members' pair forces carry the ~1e-7 conditioning of planted_tolerance, which a
    step spreads into the state."""
    _one_step(case_of("fixed", "h1e-3"), built_engine)


@pytest.mark.gpu
def test_one_step_variable_h(built_engine):
    """The h iteration (k_density<true>) on the planted binaries: every member grows its h from the edge of its partner."""
    _one_step(case_of("variable", "h1e-3"), built_engine)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fixed", "variable"])
def test_interpolate_wide_point_runs(mode, built_engine):
    """sph_interpolate bounds its prefilter by the run's width already; points on a coarse grid over the whole cube mixed
    with points planted at 2 h_j (1 - eps) from binary members make the point runs wide."""
    from test_widen_interpolate import checker, assert_matches
    c = case_of(mode, "h1e-3")
    p, b, s = c["params"], c["bodies"], c["sinks"]
    rng = np.random.default_rng(5)
    g = np.linspace(-HALF, HALF, 12)
    grid = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    rows = c["pairs"].reshape(-1)
    hj = b.h[rows] if p.mode & MODE_VARIABLE_H else np.full(len(rows), p.h_fixed)
    eps = 10.0 ** rng.uniform(-9, -3, len(rows))
    planted = np.stack([b.x[rows], b.y[rows], b.z[rows]], 1) + (2.0 * hj * (1.0 - eps))[:, None] * _directions(rng, len(rows))
    pts = np.concatenate([grid, planted])
    pts = pts[rng.permutation(len(pts))]
    with _engine(p) as e:
        e.upload(b, s)
        got = e.interpolate(pts)
    ref = checker(pts, b, p)
    assert_matches(got, ref, mode)
    assert ref["count"].max() >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_domains_clustered_case(world, built_engine, tmp_path):
    """Variable h, h ~ 1e-3, under the Morton domains (host communicator, ranks sharing one GPU): the integers and the
    counters of one rank, the fields to 1e-12.  The worker's "tree" evaluation runs with the exact counters on, which
    bypasses the two walk screens: here only the gravity screens run as in the default mode (they have no exact-counter
    bypass).  The walk screens in the default mode are checked on one rank, by the tests above."""
    from test_multi_gpu import run_ranks
    from test_domains import compare
    c = case_of("variable", "h1e-3")
    p, b, s = c["params"], c["bodies"], c["sinks"]
    path = str(tmp_path / "case.npz")
    cols = {"in_" + k: getattr(b, k) for k in GAS_FIELDS}
    cols.update({"in_sink_" + k: getattr(s, k) for k in SINK_FIELDS})
    np.savez(path, params=np.frombuffer(bytes(p), np.uint8), **cols)
    ref = run_ranks(tmp_path, "one", 1, "host", int(p.mode), steps=0, n=len(b), extra="tree", case=path)[0]
    res = run_ranks(tmp_path, f"dd{world}", world, "host", int(p.mode), steps=0, n=len(b), domains=1, extra="tree", case=path)
    for r in range(world):
        compare(res[r], ref, f"world {world} rank {r}", 1e-12, 0.0)
