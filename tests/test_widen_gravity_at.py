"""The gravitational field at arbitrary points (`sph_gravity_at`, include/sph_b200.h) and rotation curves.

The checker is the CPU oracle itself with one entry point added beside it (tests/_gravat_oracle.py): each point becomes
a Particle of smoothing length h_k that is not in the tree, walked by the oracle's particle_gravforce_one and
potential_one (self = -1), plus the unsoftened sink terms.  CPU tests pin the checker to the oracle's gravity pass and
its conserved sums; GPU tests compare the CUDA call with it (accepted counts exact, the values to 1e-12).
The domain forms run in tests/_dd_gravat_rank.py, one process per rank."""
import json
import os
import subprocess
import sys
import uuid

import numpy as np
import pytest

from conftest import relerr
from summersph_b200 import (default_params, MODE_FIXED_H, MODE_VARIABLE_H, FLAG_SOFT_USES_HI, EVAL_TREE, EVAL_DENSITY,
                            EVAL_GRAVITY, EVAL_SINKS, EVAL_ALL, ics, Bodies, Sinks)

HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "_dd_gravat_rank.py")
MODES = {"fixed": MODE_FIXED_H, "variable": MODE_VARIABLE_H, "variable_soft_hi": MODE_VARIABLE_H | FLAG_SOFT_USES_HI}
COLS = ("phi_gas", "gx_gas", "gy_gas", "gz_gas", "phi_sink", "gx_sink", "gy_sink", "gz_sink", "accepted")
G = float(np.float32(39.47841760435743))          # the reference's real(4) G (F:7)


def checker(params):
    from _gravat_oracle import GravAtOracle
    return GravAtOracle(params)


def soft_potential(q):
    """sph_conserved's phi(q) (-1/q beyond 2), vectorised."""
    q = np.asarray(q, dtype=float)
    q2 = q * q
    inner = -1.4 + q2 * (2.0 / 3.0 + q2 * (-0.3 + 0.1 * q))
    with np.errstate(divide="ignore"):
        mid = -1.6 + 1.0 / (15.0 * q) + q2 * (4.0 / 3.0 - q + 0.3 * q2 - (1.0 / 30.0) * q2 * q)
        out = -1.0 / q
    return np.where(q < 1.0, inner, np.where(q < 2.0, mid, out))


def probe_points(b, s, seed, n_in=600):
    """Points inside the disc, on particles, near the outer and inner edges, outside the root cube, far away, on the sinks."""
    rng = np.random.default_rng(seed)
    r = np.sqrt(rng.uniform(5.0 ** 2, 105.0 ** 2, n_in)); phi = rng.uniform(0, 2 * np.pi, n_in)
    inside = np.stack([r * np.cos(phi), r * np.sin(phi), rng.normal(0.0, 3.0, n_in)], 1)
    on = np.stack([b.x, b.y, b.z], 1)[rng.choice(len(b), 200, replace=False)]
    pe = rng.uniform(0, 2 * np.pi, 200); re_ = np.where(np.arange(200) % 2 == 0, 100.0, 10.0) + rng.normal(0.0, 2.0, 200)
    edge = np.stack([re_ * np.cos(pe), re_ * np.sin(pe), rng.normal(0.0, 2.0, 200)], 1)
    outside = rng.uniform(-1.0, 1.0, (60, 3)) * 40.0 + np.array([180.0, -150.0, 60.0])
    far = rng.normal(0.0, 1.0, (20, 3)) * 1e4
    sinks = np.stack([s.x, s.y, s.z], 1)
    return np.concatenate([inside, on, edge, outside, far, sinks])


def assert_matches(got, ref, what, tol=1e-12):
    for k in COLS:
        if k not in got:
            continue
        if k == "accepted":
            assert np.array_equal(got[k], ref[k]), (what, k, np.flatnonzero(got[k] != ref[k])[:5])
        else:
            assert relerr(got[k], ref[k]) <= tol, (what, k, relerr(got[k], ref[k]))


def two_sinks():
    return Sinks([0.0, 60.0], [0.0, 0.0], [0.0, 0.0], [0.0, 0.0], [0.0, 8.0], [0.0, 0.0], [1.0, 0.01], [1.0, 1.0])


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the checker against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(MODES))
def test_checker_at_the_particles_is_the_gravity_pass(name):
    """At x_i with h_i, the checker's gas columns are the oracle's gravity-pass acceleration bit for bit, and with the
    one sink added its gravity + sinks acceleration; the accepted counts add up to its grav_accepted."""
    p = default_params(MODES[name])
    b, s = ics.keplerian_disc(1500, seed=5)
    o = checker(p)
    o.upload(b, s); o.evaluate(EVAL_ALL)
    parts, ctr = o.accel_parts(), o.counters()
    got = o.gravity_at(np.stack([b.x, b.y, b.z], 1), h=b.h if name != "fixed" else None)
    g = np.stack([got["gx_gas"], got["gy_gas"], got["gz_gas"]], 1)
    gs = np.stack([got["gx_sink"], got["gy_sink"], got["gz_sink"]], 1)
    assert np.array_equal(g, parts["grav"])
    assert np.array_equal(g + gs, parts["grav_sink"])            # one sink: a - m w == a + (0 - m w)
    assert int(got["accepted"].sum()) == ctr["grav_accepted"]


@pytest.mark.parametrize("name", list(MODES))
def test_checker_potential_is_the_conserved_gas_energy(name):
    """Leaves of one particle each: 1/2 sum m_i (phi_gas(x_i) - G m_i phi(sqrt(soft) / h'_i) / h'_i) = E_gg of the oracle's
    conserved sums, which leaves each particle's own leaf out."""
    p = default_params(MODES[name])
    b, s = ics.keplerian_disc(1200, seed=6)
    o = checker(p)
    o.upload(b, s)
    e_gg = o.conserved()["e_pot_gas"]
    o.evaluate(EVAL_TREE)
    t = o.tree()
    assert np.all(t["n_in_leaf"] == 1)
    variable = bool(p.mode & MODE_VARIABLE_H)
    h = b.h if variable else np.full(len(b), p.h_fixed)
    soft = 0.001 * (b.h if p.mode & FLAG_SOFT_USES_HI else np.full(len(b), p.h_fixed))
    got = o.gravity_at(np.stack([b.x, b.y, b.z], 1), h=b.h)
    own = G * b.m * soft_potential(np.sqrt(soft) / h) / h
    assert abs(0.5 * np.sum(b.m * (got["phi_gas"] - own)) - e_gg) <= 1e-13 * abs(e_gg)


def test_checker_far_point_is_the_softened_monopole():
    p = default_params(MODE_VARIABLE_H)
    b, s = ics.keplerian_disc(1000, seed=7)
    o = checker(p)
    o.upload(b, s); o.evaluate(EVAL_TREE)
    size = o.tree()["root_size"]
    M = b.m.sum()
    com = np.array([np.sum(b.m * b.x), np.sum(b.m * b.y), np.sum(b.m * b.z)]) / M
    x = com + np.array([3.0, -2.0, 2.5]) * size            # |x - COM| = 4.5 root sizes
    got = o.gravity_at(x[None, :], h=np.array([1.7]))
    d = x - com
    dist = np.sqrt(d @ d + 0.001 * p.h_fixed)
    assert got["accepted"][0] == 1.0
    assert got["phi_gas"][0] == pytest.approx(G * M * soft_potential(dist / 1.7) / 1.7, rel=1e-12)
    for k, c in zip(("gx_gas", "gy_gas", "gz_gas"), d):
        assert got[k][0] == pytest.approx(-G * M * c / dist ** 3, rel=1e-12)
    r = np.sqrt(x @ x)
    assert got["phi_sink"][0] == pytest.approx(-G * 1.0 / r, rel=1e-14)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def lib(built_engine):
    return built_engine


def engine(p):
    from summersph_b200.engine import Engine
    return Engine(p, device=0)


@pytest.mark.gpu
@pytest.mark.parametrize("sinks", ["one", "two"])
@pytest.mark.parametrize("name", list(MODES))
def test_columns_match_the_oracle(name, sinks, lib):
    p = default_params(MODES[name])
    b, s = ics.keplerian_disc(10_000, seed=31)
    if sinks == "two":
        s = two_sinks()
    pts = probe_points(b, s, 32)
    hp = np.random.default_rng(33).uniform(0.3, 5.0, len(pts))
    o = checker(p)
    o.upload(b, s); o.evaluate(EVAL_TREE)
    with engine(p) as e:
        e.upload(b, s)
        got = e.gravity_at(pts)
        goth = e.gravity_at(pts, h=hp)
        part = e.gravity_at(pts, n_out=3)
    assert_matches(got, o.gravity_at(pts), name)
    assert_matches(goth, o.gravity_at(pts, h=hp), name + " with h")
    assert set(part) == set(COLS[:3]) and all(np.array_equal(part[k], got[k]) for k in part)
    assert np.all(got["accepted"][-len(s) - 20:-len(s)] == 1.0), "far away: the root alone"
    on_star = -G * 0.01 / 60.0 if sinks == "two" else 0.0          # the point on the star feels only the other sink
    assert got["phi_sink"][-len(s)] == on_star


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fixed", "variable"])
def test_depth_limited_leaves(name, lib):
    p = default_params(MODES[name], max_depth=5)
    b, s = ics.keplerian_disc(3000, seed=51)
    pts = probe_points(b, s, 52, 300)
    o = checker(p)
    o.upload(b, s); o.evaluate(EVAL_TREE)
    assert o.tree()["n_in_leaf"].max() > 1
    with engine(p) as e:
        e.upload(b, s)
        got = e.gravity_at(pts, h=b.h[:len(pts)])
    assert_matches(got, o.gravity_at(pts, h=b.h[:len(pts)]), name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODES))
def test_at_the_particles_is_the_engines_gravity(name, lib):
    """x_i with h_i: the gas columns are sph_evaluate(TREE|DENSITY|GRAVITY)'s acceleration; + SINKS adds the sink columns."""
    p = default_params(MODES[name])
    b, s = ics.keplerian_disc(10_000, seed=61)
    with engine(p) as e:
        e.upload(b, s)
        e.evaluate(EVAL_TREE | EVAL_DENSITY | EVAL_GRAVITY)
        bb, _ = e.download()
        a = e.diag()
        got = e.gravity_at(np.stack([bb.x, bb.y, bb.z], 1), h=bb.h)
        e.evaluate(EVAL_TREE | EVAL_DENSITY | EVAL_GRAVITY | EVAL_SINKS)
        a2 = e.diag()
    for k in ("x", "y", "z"):
        assert relerr(got[f"g{k}_gas"], a[f"a{k}"]) <= 1e-12, k
        assert relerr(got[f"g{k}_gas"] + got[f"g{k}_sink"], a2[f"a{k}"]) <= 1e-12, k


@pytest.mark.gpu
def test_repeatable_and_permutable(lib):
    p = default_params(MODE_VARIABLE_H)
    b, s = ics.keplerian_disc(6000, seed=71)
    pts = probe_points(b, s, 72, 3000)
    hp = np.random.default_rng(73).uniform(0.3, 5.0, len(pts))
    perm = np.random.default_rng(74).permutation(len(pts))
    with engine(p) as e:
        e.upload(b, s)
        e.step(0.01, 0.0)
        a = e.gravity_at(pts, h=hp)
        a2 = e.gravity_at(pts, h=hp)
        ap = e.gravity_at(pts[perm], h=hp[perm])
    for k in COLS:
        assert np.array_equal(a[k], a2[k]), k
        assert np.array_equal(ap[k], a[k][perm]), k


@pytest.mark.gpu
def test_errors(lib):
    from summersph_b200.engine import load_library, SphError, _p
    ARG, STATE = -1, -5                     # SPH_ERR_ARG, SPH_ERR_STATE
    L = load_library()
    p = default_params(MODE_VARIABLE_H)
    b, s = ics.keplerian_disc(500, seed=91)
    pts = np.ones((4, 3))
    with engine(p) as e:
        with pytest.raises(SphError) as ei:
            e.gravity_at(pts)
        assert ei.value.code == STATE, "no upload"
        e.upload(b, s)
        for n_out in (0, 10):
            with pytest.raises(SphError) as ei:
                e.gravity_at(pts, n_out=n_out)
            assert ei.value.code == ARG, n_out
        bad = pts.copy(); bad[2, 1] = np.inf
        with pytest.raises(SphError) as ei:
            e.gravity_at(bad)
        assert ei.value.code == ARG
        for hv in (0.0, -1.0, np.nan, np.inf):
            with pytest.raises(SphError) as ei:
                e.gravity_at(pts, h=np.array([1.0, 1.0, hv, 1.0]))
            assert ei.value.code == ARG, hv
        z = np.zeros(1)
        assert L.sph_gravity_at(e._c, 0, _p(z), _p(z), _p(z), None, _p(z), 9) == 0
        assert L.sph_gravity_at(e._c, -1, _p(z), _p(z), _p(z), None, _p(z), 9) == ARG
        for k in range(4):
            args = [_p(z)] * 4
            args[3 if k == 3 else k] = None
            assert L.sph_gravity_at(e._c, 1, args[0], args[1], args[2], None, args[3], 9) == ARG, k
        got = e.gravity_at(np.zeros((0, 3)))
        assert set(got) == set(COLS) and all(len(v) == 0 for v in got.values())
        assert e.gravity_at(pts)["phi_gas"].shape == (4,)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fixed", "variable"])
def test_the_call_does_not_change_the_run(name, lib):
    """Calls before and between the steps leave the run where the same run without them ends (state fingerprint, dt, t,
    far-field reuses); counters, stage times and the accelerations of the last evaluation are untouched by a call."""
    p = default_params(MODES[name])
    b, s = ics.keplerian_disc(6000, seed=81)
    pts = probe_points(b, s, 82, 500)
    res = []
    for ask in (0, 1):
        with engine(p) as e:
            e.upload(b, s)
            if ask:
                e.gravity_at(pts)
            dt, t = 0.01, 0.0
            for _ in range(3):
                dt, t = e.step(dt, t)
                if ask:
                    st, ctr, d = e.stage_times(), e.counters(), e.diag()
                    e.gravity_at(pts, h=np.full(len(pts), 1.5))
                    assert e.stage_times() == st and e.counters() == ctr
                    d2 = e.diag()
                    assert all(np.array_equal(d[k], d2[k]) for k in d)
            res.append((e.state_hash()[0], dt, t, e.far_reuse_count()))
    assert res[1] == res[0], res


@pytest.mark.gpu
def test_uniform_sphere_is_newtonian(lib):
    p = default_params(MODE_FIXED_H)
    R = 100.0
    b, s = ics.uniform_sphere(20_000, radius=R)
    rng = np.random.default_rng(3)
    u = rng.normal(size=(64, 3)); u /= np.linalg.norm(u, axis=1)[:, None]
    r_out, r_in = np.array([150.0, 200.0, 400.0]), np.array([50.0, 60.0, 70.0, 80.0, 90.0])
    rr = np.concatenate([r_out, r_in])
    pts = (rr[:, None, None] * u[None, :, :]).reshape(-1, 3)
    with engine(p) as e:
        e.upload(b, s)
        got = e.gravity_at(pts)
    g = np.stack([got["gx_gas"], got["gy_gas"], got["gz_gas"]], 1).reshape(len(rr), 64, 3)
    gr = -(g * u[None, :, :]).sum(2)                       # inward radial component
    M = b.m.sum()
    # outside: the 64-direction mean within 1 % of the point mass; single directions keep the sphere's shot noise and
    # the monopole error of the accepted cells (a few per mille, up to ~1 % at 1.5 R)
    out = gr[:len(r_out)] / (G * M / r_out[:, None] ** 2)
    assert np.all(np.abs(out.mean(1) - 1.0) <= 0.01) and np.all(np.abs(out - 1.0) <= 0.05), out
    rad = np.sqrt(b.x ** 2 + b.y ** 2 + b.z ** 2)
    m_in = np.array([b.m[rad < r].sum() for r in r_in])
    assert np.all(np.abs(gr[len(r_out):].mean(1) / (G * m_in / r_in ** 2) - 1.0) <= 0.05)


@pytest.mark.gpu
def test_rotation_curve_of_the_keplerian_disc(tmp_path, lib):
    from summersph_b200 import rotation_curve as rcm
    from summersph_b200.textio import make_save
    p = default_params(MODE_VARIABLE_H)
    b, s = ics.keplerian_disc(20_000, seed=101)
    radii = np.linspace(20.0, 90.0, 15)
    pts, phi = rcm.ring_points(radii, 256)
    with engine(p) as e:
        e.upload(b, s)
        rc = rcm.rotation_curve(e, radii, per_ring=256)
        g = e.gravity_at(pts)
    kep = np.sqrt(G * 1.0 / radii)
    assert np.max(np.abs(rc["v_c_sink"] / kep - 1.0)) <= 1e-12
    # the signed inward pull of the gas: in the inner disc the gas outside R pulls outward (a disc is not a sphere), so
    # v_c_gas is 0 there and v_c falls below the Keplerian speed; farther out the enclosed gas wins
    inward = -(g["gx_gas"].reshape(len(radii), -1) * np.cos(phi) + g["gy_gas"].reshape(len(radii), -1) * np.sin(phi)).mean(1)
    assert np.max(np.abs(rc["v_c_gas"] - np.sqrt(np.maximum(0.0, radii * inward)))) <= 1e-14 * kep.max()
    assert np.max(np.abs(rc["v_c"] ** 2 - (kep ** 2 + radii * inward))) <= 1e-12 * np.max(kep ** 2)
    assert np.all(inward[radii >= 40.0] > 0.0) and np.all(rc["v_c"][radii >= 40.0] > rc["v_c_sink"][radii >= 40.0])
    assert np.max(np.abs(rc["v_phi"] / rc["v_c"] - 1.0)) <= 0.03, rc["v_phi"] / rc["v_c"]
    s.radius[:] = p.sink_radius
    path = make_save(b, s, 3, p, directory=str(tmp_path))
    out = str(tmp_path / "rc.txt")
    rcm.main([path, "--variable", "--rmin", "20", "--rmax", "90", "--rings", "8", "--per-ring", "64", "--out", out])
    tab = np.loadtxt(out)
    assert tab.shape == (8, 5)
    assert np.max(np.abs(tab[:, 3] / np.sqrt(G / tab[:, 0]) - 1.0)) <= 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# GPU, domains: one process per rank (tests/_dd_gravat_rank.py)
# ---------------------------------------------------------------------------------------------------------------------
def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def run_ranks(tmp_path, tag, world, spec, comm="host"):
    token = "-"
    if world > 1:
        if comm == "nccl":
            import ctypes as C
            from summersph_b200.engine import load_library
            buf = (C.c_char * 128)()
            assert load_library().sph_comm_unique_id(buf) == 0
            token = bytes(buf).hex()
        else:
            token = "/sphgravat_" + uuid.uuid4().hex[:16]
    procs, outs = [], []
    for r in range(world):
        out = str(tmp_path / f"{tag}_r{r}.npz")
        outs.append(out)
        procs.append(subprocess.Popen([sys.executable, WORKER, str(r), str(world), comm, str(r if comm == "nccl" else 0), token, out,
                                       json.dumps(spec)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    logs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=float(os.environ.get("SPH_TEST_RANK_TIMEOUT", "900")))
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        logs.append(o)
    for r, p in enumerate(procs):
        assert p.returncode == 0, f"rank {r} failed:\n{logs[r][-4000:]}"
    return [dict(np.load(o)) for o in outs]


def assert_ranks_equal_one(res, one, exact=False):
    keys = [k for k in one if k.startswith(("up_", "st_"))]
    for k in keys:
        for r in range(1, len(res)):
            assert np.array_equal(res[r][k], res[0][k]), (k, r)
        if exact or k.endswith("accepted"):
            assert np.array_equal(res[0][k], one[k]), k
        else:
            assert relerr(res[0][k], one[k]) <= 1e-12, (k, relerr(res[0][k], one[k]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fixed", "variable"])
@pytest.mark.parametrize("world", [2, 3])
def test_domains_equal_one_rank(world, name, tmp_path, lib):
    spec = {"scenario": "values", "mode": MODES[name], "decomposition": 1}
    one = run_ranks(tmp_path, f"one_{name}", 1, spec)[0]
    assert_ranks_equal_one(run_ranks(tmp_path, f"w{world}_{name}", world, spec), one)


@pytest.mark.gpu
def test_domains_mismatch_is_an_argument_error(tmp_path, lib):
    res = run_ranks(tmp_path, "mismatch", 3, {"scenario": "mismatch", "mode": MODE_VARIABLE_H, "decomposition": 1})
    for r in res:
        assert list(r["codes"]) == [1, 1, 1, 0], r["codes"]      # other points, one rank's NaN, other h; then agreed


@pytest.mark.gpu
def test_domains_call_does_not_change_the_run(tmp_path, lib):
    res = run_ranks(tmp_path, "ask", 2, {"scenario": "ask", "mode": MODE_VARIABLE_H, "decomposition": 1, "steps": 3})
    for r in range(2):
        assert np.array_equal(res[r]["run1"], res[r]["run0"]), (r, res[r]["run0"], res[r]["run1"])


@pytest.mark.gpu
def test_replicated_two_ranks_is_one_rank(tmp_path, lib):
    spec = {"scenario": "values", "mode": MODE_VARIABLE_H, "decomposition": 0}
    one = run_ranks(tmp_path, "rep1", 1, spec)[0]
    assert_ranks_equal_one(run_ranks(tmp_path, "rep2", 2, spec), one, exact=True)


@pytest.mark.gpu
@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_domains_nccl_two_gpus(tmp_path, lib):
    spec = {"scenario": "values", "mode": MODE_VARIABLE_H, "decomposition": 1}
    one = run_ranks(tmp_path, "nccl1", 1, spec)[0]
    assert_ranks_equal_one(run_ranks(tmp_path, "nccl2", 2, spec, comm="nccl"), one)
