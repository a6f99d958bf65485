"""Tens of sinks against the oracle: every sink path of the engine is a loop over n_sink or a kernel with one thread per
sink (the sink terms of the gravity walks, k_sink_seg_fold / k_sink_reduce, k_sink_pairs, k_flags / k_accrete_apply with
sinks 32 and up in the second warp, k_kick_sinks, k_cull_sinks, k_create_apply, k_sink_merge, k_same_sinks, the sink
sums of sph_conserved and sph_gravity_at, the n_sink + 8 output of sph_step_host).  Uploads take up to
SPH_MAX_SINKS - 8 = 56 sinks; the variable-h program adds at most one per step, up to 64.

Each sink accretes on its own (F:484-556 | V:616-688): a particle inside several radii adds its mass to each of them, so
the accretion list can hold more (sink, particle) entries than there are particles; the cases below make it do so.

Sinks are compared one by one (a massive sink must not hide a 1e-11 one): x, v, m, radius relative to max(|value|, a
floor of the field); the sink accelerations to 1e-10 of their conditioning sum_j G m_j / r_js^2 + sum_b G m_b / r_bs^2."""
import numpy as np
import pytest

from summersph_b200 import (default_params, MODE_FIXED_H, MODE_VARIABLE_H, FLAG_SOFT_USES_HI, FLAG_SINK_MERGE_SPIN,
                            EVAL_TREE, ics, Bodies, Sinks)
from summersph_b200.state import GAS_FIELDS, SINK_FIELDS
from oracle.oracle import Oracle
from conftest import relerr

G = float(np.float32(39.47841760435743))          # the reference's real(4) G (F:7)
TOL = 1e-10
MAX_UPLOAD = 56                                    # SPH_MAX_SINKS - 8
FLOOR = {"x": 1.0, "y": 1.0, "z": 1.0, "vx": 1e-2, "vy": 1e-2, "vz": 1e-2, "m": 0.0, "radius": 0.0}


def list_cap(n):
    """The accretion list's first capacity: the particle capacity n + n/64 + 1024."""
    return n + n // 64 + 1024


def make_sinks(x, y, z, vx, vy, vz, m, radius):
    return Sinks(*[np.asarray(a, dtype=float) for a in (x, y, z, vx, vy, vz, m, radius)])


def join(*ss):
    return Sinks(*[np.concatenate([getattr(s, k) for s in ss]) for k in SINK_FIELDS])


def star(radius=1.0):
    return make_sinks([0.0], [0.0], [0.0], [0.0], [0.0], [0.0], [1.0], [radius])


def orbiting(r, phi, z, m, radius, frac=1.0):
    """Sinks on (a fraction of) circular orbits about the central star."""
    v = frac * np.sqrt(G / r)
    return make_sinks(r * np.cos(phi), r * np.sin(phi), z, -v * np.sin(phi), v * np.cos(phi), np.zeros(len(r)), m, radius)


def sink_table(n_sink, seed, radius=0.05, zeros=True):
    """The star, then sinks in turn inside the gas (10 < r < 100), in the central gap (r < 10) and outside the gas; masses
    from 1e-11 to 1e-2, zero for two sinks in the middle of the table (`zeros`).  A step turns a massless sink's position
    into (0 x + 0) / 0 = NaN (F:498-501): the variable-h program then culls it, the fixed-h one spreads the NaN, so the
    tables that are stepped have none."""
    if n_sink == 1:
        return star()
    rng = np.random.default_rng(seed)
    k = np.arange(1, n_sink)
    r = np.where(k % 3 == 0, rng.uniform(20.0, 90.0, len(k)), np.where(k % 3 == 1, rng.uniform(2.0, 8.0, len(k)), rng.uniform(120.0, 200.0, len(k))))
    z = np.where(k % 3 == 0, rng.normal(0.0, 1.0, len(k)), rng.normal(0.0, 5.0, len(k)))
    m = 10.0 ** rng.uniform(-11.0, -2.0, len(k))
    if zeros:
        m[[n_sink // 3 - 1, n_sink // 2 - 1]] = 0.0        # table rows n_sink // 3 and n_sink // 2
    return join(star(), orbiting(r, rng.uniform(0, 2 * np.pi, len(k)), z, m, np.full(len(k), radius), frac=0.9))


def positions(a):
    return np.stack([a.x, a.y, a.z], 1)


def accel_conditioning(b, s):
    """Per sink: sum_j G m_j / r_js^2 (gas) + sum_b G m_b / r_bs^2 (the other sinks)."""
    X, S = positions(b), positions(s)
    d2 = ((S[:, None, :] - X[None, :, :]) ** 2).sum(2)
    c = G * (b.m[None, :] / d2).sum(1)
    ds2 = ((S[:, None, :] - S[None, :, :]) ** 2).sum(2)
    np.fill_diagonal(ds2, np.inf)
    return c + G * (np.abs(s.m)[None, :] / ds2).sum(1)


def assert_sinks_match(se, so, what, tol=TOL):
    assert len(se) == len(so), what
    for k in SINK_FIELDS:
        a, r = getattr(se, k), getattr(so, k)
        scale = np.maximum(np.abs(r), FLOOR[k])
        err = np.where(scale > 0, np.abs(a - r) / np.where(scale > 0, scale, 1.0), np.where(a == r, 0.0, np.inf))
        assert np.all(err <= tol), (what, k, int(np.argmax(err)), float(np.max(err)))


def assert_sink_accels_match(de, do, cond, what, tol=TOL):
    for k in ("sink_ax", "sink_ay", "sink_az"):
        err = np.abs(de[k] - do[k]) / cond
        assert np.all(err <= tol), (what, k, int(np.argmax(err)), float(np.max(err)))


def l1_entries(b, s):
    """(sink, particle) pairs with |x_j - x_s|_1 < R_s: the variable-h program's accretion test (V:668-669; such a
    particle passes every ancestor-cell and leaf test), and the per-particle count of radii it lies in."""
    inside = np.abs(positions(b)[None, :, :] - positions(s)[:, None, :]).sum(2) < s.radius[:, None]
    return int(inside.sum()), inside.sum(0)


def f537_entries(b, s, tree):
    """Fixed h: a lower bound on the accretion entries - pairs with |x_j - x_s|_inf < R_s (every ancestor cell and the
    leaf pass F:529 / F:536) and F:537's dr = sum sqrt(c^2 - x_s^2) on the leaf centre c below R_s."""
    X, S = positions(b), positions(s)
    C = np.stack([tree["cx"], tree["cy"], tree["cz"]], 1)
    near = np.abs(X[None, :, :] - S[:, None, :]).max(2) < s.radius[:, None]
    with np.errstate(invalid="ignore"):
        dr = np.sqrt(C[None, :, :] ** 2 - S[:, None, :] ** 2).sum(2)
    inside = near & (dr < s.radius[:, None]) & (tree["n_in_leaf"] == 1)[None, :]
    return int(inside.sum()), inside.sum(0)


# ---- the planted inputs ---------------------------------------------------------------------------------------------
LEAVING = (10, 20, 21)          # table rows of the sinks that leave the bounding cube in the first step (variable h)


def overlap_case(mode):
    """4000-particle disc with 40 overlapping accreting sinks: the accretion list outgrows the particle count.
    Variable h: the star and 40 sinks of mass 1e-4, radius ~25 at r = 20-40 in the mid-plane (L1 balls), with three more
    in the middle of the table that cross the bounding cube in the first step.  Fixed h: F:537's sqrt(c^2 - x_s^2) is the
    L1 norm of the leaf centre only for sinks near the origin, so 40 sinks of mass ~1e-6, radius 35-45 in the unit cube
    around it (no star: it would fling them out before they accrete)."""
    b, _ = ics.keplerian_disc(4000, seed=5)
    rng = np.random.default_rng(3)
    if mode & MODE_VARIABLE_H:
        r = rng.uniform(20.0, 40.0, 40); ph = rng.uniform(0, 2 * np.pi, 40)
        s = join(star(), orbiting(r, ph, np.zeros(40), np.full(40, 1e-4), rng.uniform(24.5, 25.5, 40), frac=0.2))
        p = default_params(mode)
        out = make_sinks([1499.99, -1499.995, 3.0], [0.0, 7.0, 1499.99], [0.0, 0.0, 0.0], [5.0, -5.0, 0.0], [0.0, 0.0, 5.0],
                         [0.0, 0.0, 0.0], [2e-5, 3e-7, 0.0], [0.5, 0.5, 0.5])
        for q, k in enumerate(LEAVING):
            s = Sinks(*[np.insert(getattr(s, f), k, getattr(out, f)[q]) for f in SINK_FIELDS])
    else:
        S = rng.uniform(-1.0, 1.0, (40, 3))
        s = make_sinks(S[:, 0], S[:, 1], S[:, 2], *rng.normal(0.0, 0.05, (3, 40)), 1e-6 * rng.uniform(0.5, 2.0, 40), rng.uniform(35.0, 45.0, 40))
        p = default_params(mode)
    return p, b, s


def quiet_case(n=10_000, seed=23, n_sink=44):
    """Moving sinks that accrete nothing and stay in the cube: the star, then sinks in the gap, outside the gas and among
    the gas with radius 1e-4; masses that are not powers of two."""
    b, _ = ics.keplerian_disc(n, seed=seed)
    s = sink_table(n_sink, seed + 1, radius=1e-4, zeros=False)
    s.m[1:] *= 1.37
    return b, s


SEED_ROWS = (311, 777, 1234, 1500, 2020, 2500, 3001, 3333, 3900)


def creation_case(n_sink=MAX_UPLOAD, seeds=SEED_ROWS, seed=21):
    """test_gpu_parity.test_sink_creation's seeds (m = 5e-3, h = 0.2 with max_length = 0.21: over-dense, h kept), one per
    row of `seeds`, beside `n_sink` uploaded sinks of radius 1e-3 away from them."""
    p = default_params(MODE_VARIABLE_H, max_length=0.21)
    b, _ = ics.keplerian_disc(4000, seed=seed)
    for j in seeds:
        b.m[j] = 5e-3; b.h[j] = 0.2
    s = sink_table(n_sink, seed + 7, radius=1e-3, zeros=False)
    return p, b, s


def seed_clearance(b, s, seeds=SEED_ROWS):
    """Smallest gap |x_seed - x_other| - (R_other + 2 h_seed) to every sink and every other seed (radius 2 h)."""
    X = positions(b)[list(seeds)]; h = b.h[list(seeds)]
    ds = np.sqrt(((X[:, None, :] - positions(s)[None, :, :]) ** 2).sum(2)) - (s.radius[None, :] + 2 * h[:, None])
    dd = np.sqrt(((X[:, None, :] - X[None, :, :]) ** 2).sum(2)) - (2 * h[None, :] + 2 * h[:, None])
    np.fill_diagonal(dd, np.inf)
    return min(float(ds.min()), float(dd.min()))


def round_trip_case():
    """50 sinks, one seed, and sink 25 on its way out of the cube: the first step creates a sink and culls one."""
    p, b, s = creation_case(n_sink=50, seeds=(1234,))
    s.x[25], s.vx[25] = 1499.99, 5.0
    return p, b, s


def chain_case():
    """Eight chains of five sinks 0.8 apart with radius 1 in the disc (each overlaps the next only), mass 1e-5-1e-4."""
    b, _ = ics.keplerian_disc(4000, seed=12)
    rng = np.random.default_rng(8)
    rows = [star()]
    for c in range(8):
        r0, ph0 = rng.uniform(25.0, 80.0), rng.uniform(0, 2 * np.pi)
        r = r0 + 0.8 * np.arange(5)
        rows.append(orbiting(r, np.full(5, ph0), np.zeros(5), 10.0 ** rng.uniform(-5, -4, 5), np.full(5, 1.0)))
    return b, join(*rows)


# ---- CPU: the builders plant what they claim ----------------------------------------------------------------------
def test_builders_plant_what_they_claim():
    p, b, s = overlap_case(MODE_VARIABLE_H)
    assert len(s) == 44
    ent, per = l1_entries(b, s)
    assert ent > 1.1 * list_cap(len(b)) and np.max(per) >= 2 and np.sum(per >= 2) > 100, (ent, list_cap(len(b)))
    x1 = positions(s) + 0.01 * np.stack([s.vx, s.vy, s.vz], 1)          # one drift at the first dt
    gone = np.flatnonzero(np.abs(x1).max(1) > p.bounding_size)
    assert list(gone) == list(LEAVING) and np.all(np.abs(positions(s)).max(1) <= p.bounding_size)

    p, b, s = overlap_case(MODE_FIXED_H)
    o = Oracle(p); o.upload(b, s); o.evaluate(EVAL_TREE)
    ent, per = f537_entries(b, s, o.tree())
    assert ent > 1.5 * list_cap(len(b)) and np.sum(per >= 2) > 100, (ent, list_cap(len(b)))

    for n_sink in (1, 31, 32, 33, 56):
        s = sink_table(n_sink, 5)
        assert len(s) == n_sink and s.m[0] == 1.0
        if n_sink > 3:
            assert s.m[n_sink // 3] == 0.0 and s.m[n_sink // 2] == 0.0
            r = np.hypot(s.x, s.y)[1:]
            assert np.any(r < 10) and np.any(r > 110) and np.any((r > 10) & (r < 100))

    b, s = quiet_case()
    assert len(s) >= 40 and np.unique(s.m).size == len(s) and np.all(s.m > 0)
    assert l1_entries(b, s)[0] == 0

    p, b, s = creation_case()
    assert len(s) == MAX_UPLOAD and seed_clearance(b, s) > 0.5
    _, b1, s1 = round_trip_case()
    assert len(s1) == 50 and seed_clearance(b1, s1, (1234,)) > 0.5 and s1.x[25] + 0.01 * s1.vx[25] > p.bounding_size
    assert np.all(b.m[list(SEED_ROWS)] * (p.eta / b.h[list(SEED_ROWS)]) ** 3 > 0.5)
    others = np.setdiff1d(np.arange(len(b)), SEED_ROWS)
    assert np.all(b.m[others] * (p.eta / b.h[others]) ** 3 < 0.5)

    b, s = chain_case()
    ds = np.sqrt(((positions(s)[:, None, :] - positions(s)[None, :, :]) ** 2).sum(2))
    over = (ds < np.maximum(s.radius[:, None], s.radius[None, :])) & ~np.eye(len(s), dtype=bool)
    assert len(s) == 41 and over.sum() == 2 * 8 * 4                     # neighbours in a chain only


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def E(built_engine):
    from summersph_b200.engine import Engine
    return Engine


def compare_eval_sinks(o, e, b, s):
    from test_gpu_parity import compare_eval
    compare_eval(o, e)
    assert_sink_accels_match(e.diag(), o.diag(), accel_conditioning(b, s), "evaluation")


def step_both(o, e, dto, to, dte, te, what):
    dto, to = o.step(dto, to); dte, te = e.step(dte, te)
    assert (dto, to) == (dte, te), what
    assert o.sizes() == e.sizes(), what
    return dto, to, dte, te


def compare_states(o, e, what, rebuild=False):
    """Gas rows to TOL, sinks one by one, and the Morton order - of a tree built anew (`rebuild`) after a step that removed
    particles, which leaves none behind."""
    bo, so = o.download(); be, se = e.download()
    assert len(bo) == len(be), what
    for k in GAS_FIELDS:
        assert relerr(getattr(be, k), getattr(bo, k)) < TOL, (what, k, relerr(getattr(be, k), getattr(bo, k)))
    assert_sinks_match(se, so, what)
    if rebuild:
        o.evaluate(EVAL_TREE); e.evaluate(EVAL_TREE)
    assert np.array_equal(o.tree()["order"], e.tree()["order"]), what
    return bo, so


@pytest.mark.gpu
@pytest.mark.parametrize("n_sink", [1, 31, 32, 33, 56])
@pytest.mark.parametrize("mode", [MODE_FIXED_H, MODE_VARIABLE_H, MODE_VARIABLE_H | FLAG_SOFT_USES_HI])
def test_evaluation(mode, n_sink, E):
    """One evaluation of a 10k disc with sinks in the gas, in the gap and outside it, masses mixed and two zero."""
    p = default_params(mode)
    b, _ = ics.keplerian_disc(10_000, seed=61)
    s = sink_table(n_sink, 62)
    o = Oracle(p); o.record_neighbours(True); o.upload(b, s); o.evaluate()
    with E(p) as e:
        e.upload(b, s); e.evaluate()
        assert e.sizes() == (len(b), n_sink)
        compare_eval_sinks(o, e, b, s)


FAR_ENVS = {"lists": {}, "walk": {"SPH_B200_NO_FAR_LISTS": "1"}, "overflow": {"SPH_B200_FAR_SLOTS": "48"}}


@pytest.mark.gpu
@pytest.mark.parametrize("mode,far", [(MODE_FIXED_H, "lists"), (MODE_VARIABLE_H, "lists"), (MODE_VARIABLE_H, "walk"),
                                      (MODE_VARIABLE_H, "overflow")])
def test_moving_sinks_far_reuse(mode, far, E, monkeypatch):
    """44 moving sinks that remove nothing: evaluation A of steps 3 and 4 keeps the stored far sums and takes the sink
    terms anew (with the near-only walk `k_gravity<1>` adding them for the runs whose recorded pairs overflowed)."""
    for k in ("SPH_B200_NO_FAR_LISTS", "SPH_B200_FAR_SLOTS", "SPH_B200_NO_FAR_REUSE"):
        monkeypatch.delenv(k, raising=False)
    for k, v in FAR_ENVS[far].items():
        monkeypatch.setenv(k, v)
    p = default_params(mode)
    b, s = quiet_case()
    o = Oracle(p); o.upload(b, s)
    with E(p) as e:
        e.upload(b, s)
        dto = dte = 0.01; to = te = 0.0
        for k in range(4):
            dto, to, dte, te = step_both(o, e, dto, to, dte, te, k)
        assert e.sizes() == (len(b), len(s))
        assert e.far_reuse_count() == 2
        bo, so = compare_states(o, e, "after 4 steps")
        assert_sink_accels_match(e.diag(), o.diag(), accel_conditioning(bo, so), "after 4 steps")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [MODE_VARIABLE_H, MODE_FIXED_H])
def test_accretion_list_longer_than_the_particles(mode, E):
    """Overlapping sinks accrete one particle each (double counting included) with more (sink, particle) entries than the
    list's first capacity: the list grows, the step goes on, and the sinks gain what the oracle's sinks gain.  Variable h:
    three sinks from the middle of the table leave the cube in the first step (k_cull_sinks keeps the order)."""
    p, b, s = overlap_case(mode)
    if mode & MODE_VARIABLE_H:
        ent, per = l1_entries(b, s)
    else:
        t = Oracle(p); t.upload(b, s); t.evaluate(EVAL_TREE)
        ent, per = f537_entries(b, s, t.tree())
    assert ent > 1.1 * list_cap(len(b)) and np.max(per) >= 2, (ent, list_cap(len(b)))
    o = Oracle(p); o.upload(b, s)
    with E(p) as e:
        e.upload(b, s)
        dto = dte = 0.01; to = te = 0.0
        for k in range(3):
            dto, to, dte, te = step_both(o, e, dto, to, dte, te, k)
            bo, so = compare_states(o, e, f"step {k}", rebuild=True)
            if k == 0:
                assert len(bo) < len(b)
                gained, lost = float(np.sum(so.m) - np.sum(s.m)), float(np.sum(b.m) - np.sum(bo.m))
                assert gained > 2.0 * lost                     # each of the overlapping sinks took the particle's mass
                if mode & MODE_VARIABLE_H:
                    assert len(so) == len(s) - len(LEAVING)
                    keep = np.setdiff1d(np.arange(len(s)), LEAVING)
                    assert np.array_equal(so.radius, s.radius[keep])      # order kept


@pytest.mark.gpu
def test_creation_up_to_the_table_limit(E):
    """56 uploaded sinks and nine over-dense seeds: each of the first eight steps creates one sink (mass 1e-11, radius 2h)
    that accretes its seed; the ninth finds the table full and says so (the reference's table would grow to 65)."""
    from summersph_b200.engine import SphError
    p, b, s = creation_case()
    o = Oracle(p); o.upload(b, s)
    with E(p) as e:
        e.upload(b, s)
        dto = dte = 0.01; to = te = 0.0
        for k in range(8):
            dto, to, dte, te = step_both(o, e, dto, to, dte, te, k)
            assert e.sizes() == (len(b) - k - 1, MAX_UPLOAD + k + 1), k
        compare_states(o, e, "after 8 creations", rebuild=True)
        _, so = o.download()
        assert np.all(so.m[MAX_UPLOAD:] > 5e-3)              # each new sink holds its seed
        with pytest.raises(SphError) as ex:
            e.step(dte, te)
        assert ex.value.code == -5 and "sink table full" in str(ex.value)
    o.step(dto, to)
    assert o.sizes()[1] == 65


@pytest.mark.gpu
def test_upload_limits(E):
    """56 sinks are taken, 57 are an argument error - through sph_upload and sph_step_host."""
    from summersph_b200.engine import SphError
    p = default_params(MODE_VARIABLE_H)
    b, _ = ics.keplerian_disc(2000, seed=3)
    ok, bad = sink_table(MAX_UPLOAD, 4, zeros=False), sink_table(MAX_UPLOAD + 1, 4, zeros=False)
    with E(p) as e:
        e.upload(b, ok)
        assert e.sizes() == (len(b), MAX_UPLOAD)
        with pytest.raises(SphError) as ex:
            e.upload(b, bad)
        assert ex.value.code == -1
    with E(p) as e:
        dt, t, n, ns = e.step_host(b, ok, 0.01, 0.0)
        assert (n, ns) == (len(b), MAX_UPLOAD)
        with pytest.raises(SphError) as ex:
            e.step_host(b, bad, 0.01, 0.0)
        assert ex.value.code == -1


def _sinks_head(os_, ns):
    return Sinks(*[getattr(os_, k)[:ns].copy() for k in SINK_FIELDS])


@pytest.mark.gpu
def test_step_host_round_trip(E):
    """50 sinks through sph_step_host: bit-identical (state hash and rows) to upload + step + download over a step that
    creates a sink and culls one, and the steps after; a handed-back state out of a step that removed nothing is
    recognised; one ulp in sink 47 (the second warp of k_same_sinks) makes it a new state."""
    p, b, s = round_trip_case()
    with E(p) as e1, E(p) as e2:
        b1, s1, b2, s2 = b, s, b, s
        dt1 = dt2 = 0.01; t1 = t2 = 0.0
        sizes = []
        for k in range(4):
            e1.upload(b1, s1); dt1, t1 = e1.step(dt1, t1); b1, s1 = e1.download()
            ob, os_ = Bodies.empty(len(b2)), Sinks.empty(len(s2) + 8)
            h0 = e2.resident_hits()
            dt2, t2, n2, ns2 = e2.step_host(b2, s2, dt2, t2, into=(ob, os_))
            if k >= 2:                                          # step 1 created a sink and removed its seed, step 2 removed nothing
                assert e2.resident_hits() == h0 + 1, k
            b2, s2 = Bodies(*[getattr(ob, f)[:n2].copy() for f in GAS_FIELDS]), _sinks_head(os_, ns2)
            assert (dt1, t1, len(b1), len(s1)) == (dt2, t2, n2, ns2), k
            assert e1.state_hash()[0] == e2.state_hash()[0], k
            for f in GAS_FIELDS:
                assert np.array_equal(getattr(b1, f), getattr(b2, f)), (k, f)
            for f in SINK_FIELDS:
                assert np.array_equal(getattr(s1, f), getattr(s2, f)), (k, f)
            sizes.append((n2, ns2))
        assert sizes[0] == (len(b) - 1, len(s)) and sizes[-1][1] == len(s)       # +1 created, -1 culled
        assert len(s2) > 47
        for field in ("m", "x", "radius"):
            s3 = _sinks_head(s2, len(s2))
            getattr(s3, field)[47] = np.nextafter(getattr(s3, field)[47], np.inf)
            h0 = e2.resident_hits()
            e2.upload(b2, s3); dta, ta = e2.step(dt2, t2); ba, sa = e2.download()
            assert e2.resident_hits() == h0, field
            with E(p) as cold:
                cold.set_resident_check(False)
                cold.upload(b2, s3); dtc, tc = cold.step(dt2, t2); bc, sc_ = cold.download()
            assert (dta, ta) == (dtc, tc), field
            for f in GAS_FIELDS:
                assert np.array_equal(getattr(ba, f), getattr(bc, f)), (field, f)
            for f in SINK_FIELDS:
                assert np.array_equal(getattr(sa, f), getattr(sc_, f)), (field, f)
            b2, s2, dt2, t2 = ba, sa, dta, ta


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [MODE_FIXED_H, MODE_VARIABLE_H])
def test_diagnostics(mode, E):
    """sph_conserved and sph_gravity_at with 56 sinks (two of them massless), at points on every sink too."""
    from test_widen_conserved import assert_same_sums
    from test_widen_gravity_at import checker, probe_points, assert_matches
    p = default_params(mode)
    b, _ = ics.keplerian_disc(10_000, seed=31)
    s = sink_table(MAX_UPLOAD, 32)
    pts = probe_points(b, s, 33)
    hp = np.random.default_rng(34).uniform(0.3, 5.0, len(pts))
    o = checker(p); o.upload(b, s)
    go = o.conserved()
    o.evaluate(EVAL_TREE)
    with E(p) as e:
        e.upload(b, s)
        assert_same_sums(e.conserved(), go)
        got, goth = e.gravity_at(pts), e.gravity_at(pts, h=hp)
    ref, refh = o.gravity_at(pts), o.gravity_at(pts, h=hp)
    assert_matches(got, ref, "many sinks")
    assert_matches(goth, refh, "many sinks with h")
    on = slice(len(pts) - len(s), len(pts))
    for k in ("phi_sink", "gx_sink", "gy_sink", "gz_sink"):
        assert np.all(np.isfinite(got[k][on])), k          # a point on a sink leaves that sink out


@pytest.mark.gpu
def test_merger_chains(E):
    """41 sinks in eight chains of overlaps (FLAG_SINK_MERGE_SPIN): the merger scans again after every merge, so a
    chain can end as one sink; three steps against the oracle."""
    from test_widen_sink_merger import compare_sinks, orbital_L, sinks_L
    p = default_params(MODE_VARIABLE_H | FLAG_SINK_MERGE_SPIN)
    b, s = chain_case()
    L_scale = np.linalg.norm(orbital_L(b.m, b.x, b.y, b.z, b.vx, b.vy, b.vz)) + np.linalg.norm(sinks_L(s))
    o = Oracle(p); o.upload(b, s)
    with E(p) as e:
        e.upload(b, s)
        dto = dte = 0.01; to = te = 0.0
        for k in range(3):
            dto, to, dte, te = step_both(o, e, dto, to, dte, te, k)
            compare_sinks(e, o, L_scale)
            _, so = o.download(); _, se = e.download()
            assert_sinks_match(se, so, k)
    assert o.sizes()[1] < 41
