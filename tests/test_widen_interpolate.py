"""SPH interpolation at arbitrary points (`sph_interpolate`, include/sph_b200.h) and density slices.

The checker is a dense numpy statement of the definition (O(N M)): W = w_table(q) / (pi h^3) with the oracle's own
table, lerp and the mode's normalisation (fixed h: h = h_fixed for every particle, pi = 3.14159265359; variable h:
h = h_j, pi in single precision), members = { j : |x - x_j| / h_j <= 2, h_j finite and > 0 }, rho = sum m_j W, the
means sum m_j f_j W / rho (0 where rho = 0), the member count.  CPU tests pin the checker to the oracle (its kernel
samples and its fixed-h density at the particles); GPU tests compare the CUDA call with it (1e-12, counts exact).
The domain forms run in tests/_dd_interp_rank.py, one process per rank."""
import json
import os
import subprocess
import sys
import uuid

import numpy as np
import pytest

from conftest import relerr
from summersph_b200 import default_params, MODE_FIXED_H, MODE_VARIABLE_H, ics, Bodies, Sinks

HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "_dd_interp_rank.py")
MODES = {"fixed": MODE_FIXED_H, "variable": MODE_VARIABLE_H}
COLS = ("rho", "vx", "vy", "vz", "u", "alpha", "count")
PI_F, PI_V = 3.14159265359, float(np.float32(np.pi))


# ---------------------------------------------------------------------------------------------------------------------
# checker
# ---------------------------------------------------------------------------------------------------------------------
_TABLES = {}


def w_table(params):
    key = int(params.nq)
    if key not in _TABLES:
        from oracle.oracle import Oracle
        _TABLES[key] = Oracle(params).tables()[0]
    return _TABLES[key]


def kernel_W(r, h, params):
    """The oracle's lookup_kernel W, vectorised (F:113-126 | V:139-140); r, h arrays of one shape."""
    wt = w_table(params)
    nq = int(params.nq); dq = 2.0 / nq
    variable = bool(params.mode & MODE_VARIABLE_H)
    q = r / h
    inside = (q >= 0.0) & (q <= 2.0)
    qq = np.where(inside, q, 0.0)
    i = np.minimum((qq / dq).astype(np.int64), nq - 1)
    a = (qq - i * dq) / dq
    w = np.where(inside, (1.0 - a) * wt[i] + a * wt[i + 1], 0.0)
    hn = h if variable else np.full_like(h, params.h_fixed)
    return w / ((PI_V if variable else PI_F) * ((hn * hn) * hn))


def checker(points, b, params, block=2_000_000):
    """dict of the 7 columns at `points` (M, 3) for the gas rows `b`."""
    pts = np.asarray(points, dtype=float).reshape(-1, 3)
    variable = bool(params.mode & MODE_VARIABLE_H)
    h = np.asarray(b.h, dtype=float) if variable else np.full(len(b), float(params.h_fixed))
    ok = np.isfinite(h) & (h > 0.0)
    hs = np.where(ok, h, 1.0)
    f = np.stack([b.vx, b.vy, b.vz, b.u, b.alpha], 1)
    out = {k: np.zeros(len(pts)) for k in COLS}
    step = max(1, block // max(len(b), 1))
    for s in range(0, len(pts), step):
        p = pts[s:s + step]
        dx = p[:, 0:1] - b.x[None, :]; dy = p[:, 1:2] - b.y[None, :]; dz = p[:, 2:3] - b.z[None, :]
        r = np.sqrt((dx * dx + dy * dy) + dz * dz)
        hh = np.broadcast_to(hs, r.shape)
        mem = ok[None, :] & (r / hh <= 2.0)
        mw = np.where(mem, b.m[None, :] * kernel_W(np.where(mem, r, 0.0), hh, params), 0.0)
        rho = mw.sum(1)
        num = mw @ f
        out["rho"][s:s + step] = rho
        with np.errstate(divide="ignore", invalid="ignore"):
            means = np.where(rho[:, None] != 0.0, num / rho[:, None], 0.0)
        for k, name in enumerate(("vx", "vy", "vz", "u", "alpha")):
            out[name][s:s + step] = means[:, k]
        out["count"][s:s + step] = mem.sum(1)
    return out


def assert_matches(got, ref, what, tol=1e-12):
    for k in COLS:
        if k not in got:
            continue
        if k == "count":
            assert np.array_equal(got[k], ref[k]), (what, k, np.flatnonzero(got[k] != ref[k])[:5])
        else:
            assert relerr(got[k], ref[k]) <= tol, (what, k, relerr(got[k], ref[k]))


def probe_points(b, seed, n_in=600):
    """Points inside the disc, on particles, near the outer and inner edges, and outside the root cube."""
    rng = np.random.default_rng(seed)
    r = np.sqrt(rng.uniform(5.0 ** 2, 105.0 ** 2, n_in)); phi = rng.uniform(0, 2 * np.pi, n_in)
    inside = np.stack([r * np.cos(phi), r * np.sin(phi), rng.normal(0.0, 3.0, n_in)], 1)
    on = np.stack([b.x, b.y, b.z], 1)[rng.choice(len(b), 200, replace=False)]
    pe = rng.uniform(0, 2 * np.pi, 200); re_ = np.where(np.arange(200) % 2 == 0, 100.0, 10.0) + rng.normal(0.0, 2.0, 200)
    edge = np.stack([re_ * np.cos(pe), re_ * np.sin(pe), rng.normal(0.0, 2.0, 200)], 1)
    outside = rng.uniform(-1.0, 1.0, (60, 3)) * 40.0 + np.array([180.0, -150.0, 60.0])
    return np.concatenate([inside, on, edge, outside])


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the checker against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(MODES))
def test_checker_kernel_is_the_oracles(name):
    from oracle.oracle import Oracle
    p = default_params(MODES[name])
    o = Oracle(p)
    rng = np.random.default_rng(3)
    h = rng.uniform(0.5, 4.0, 40) if name == "variable" else np.full(40, p.h_fixed)
    r = h * rng.uniform(0.0, 2.2, 40)
    r[:3] = 0.0, h[1], 2.0 * h[2]
    got = kernel_W(r, h, p)
    ref = np.array([o.lookup_kernel(float(ri), float(hi))[0] for ri, hi in zip(r, h)])
    assert np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)) <= 1e-14
    assert np.all(got[r / h > 2.0] == 0.0)


def test_checker_at_particles_is_the_oracle_density_fixed_h():
    """Fixed h: the membership ball lies inside the reference's leaf box (F:443), so at x = x_i the checker's rho is the
    reference's rho_i up to summation order (no coincident particles here)."""
    from oracle.oracle import Oracle
    p = default_params(MODE_FIXED_H)
    b, s = ics.keplerian_disc(1500, seed=5)
    o = Oracle(p); o.upload(b, s); o.evaluate()
    ref = o.diag()["rho"]
    got = checker(np.stack([b.x, b.y, b.z], 1), b, p)["rho"]
    assert relerr(got, ref) <= 1e-12


def test_checker_means_of_a_constant_field_and_an_empty_region():
    p = default_params(MODE_VARIABLE_H)
    b, _ = ics.keplerian_disc(800, seed=9)
    b.vx[:] = 3.25; b.vy[:] = -1.5; b.vz[:] = 0.125; b.u[:] = 0.7; b.alpha[:] = 0.3
    pts = np.concatenate([np.stack([b.x[:50], b.y[:50], b.z[:50]], 1), [[500.0, 500.0, 500.0], [0.0, 0.0, 80.0]]])
    out = checker(pts, b, p)
    for k, v in (("vx", 3.25), ("vy", -1.5), ("vz", 0.125), ("u", 0.7), ("alpha", 0.3)):
        assert np.max(np.abs(out[k][:50] - v)) <= 1e-14 * abs(v), k
    assert np.all(out["count"][:50] >= 1) and np.all(out["rho"][:50] > 0.0)
    for k in COLS:
        assert np.all(out[k][50:] == 0.0), k


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
def test_fixed_h_rho_at_particles_is_the_density_pass(lib):
    p = default_params(MODE_FIXED_H)
    b, s = ics.keplerian_disc(20_000, seed=21)
    s = Sinks([0.0, 60.0], [0.0, 0.0], [0.0, 0.0], [0.0, 0.0], [0.0, 8.0], [0.0, 0.0], [1.0, 0.01], [1.0, 1.0])
    with engine(p) as e:
        e.upload(b, s); e.evaluate()
        ref = e.diag()["rho"]
        bb, _ = e.download()
        got = e.interpolate(np.stack([bb.x, bb.y, bb.z], 1))
    assert relerr(got["rho"], ref) <= 1e-12
    assert np.all(got["count"] >= 1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODES))
def test_columns_match_the_checker(name, lib):
    p = default_params(MODES[name])
    b, s = ics.keplerian_disc(2000, seed=31)
    pts = probe_points(b, 32)
    with engine(p) as e:
        e.upload(b, s)
        got = e.interpolate(pts)
        part = e.interpolate(pts, n_out=3)
    ref = checker(pts, b, p)
    assert_matches(got, ref, name)
    assert set(part) == {"rho", "vx", "vy"} and all(np.array_equal(part[k], got[k]) for k in part)
    assert np.all(got["count"][-60:] == 0) and np.all(got["rho"][-60:] == 0.0), "outside the root cube"
    assert got["count"].max() > 10


@pytest.mark.gpu
def test_variable_h_after_steps_with_accretion(lib):
    """h changed by calc_smoothing, the tree of evaluation B reused, particles accreted: the call sees the resident state."""
    p = default_params(MODE_VARIABLE_H, bounding_size=95.0)
    b, s = ics.keplerian_disc(3000, seed=41)
    s.radius[:] = 12.0
    with engine(p) as e:
        e.upload(b, s)
        dt, t = 0.01, 0.0
        for _ in range(3):
            dt, t = e.step(dt, t)
        bb, _ = e.download()
        assert len(bb) < 3000, "the set-up is meant to remove particles"
        pts = probe_points(bb, 42)
        got = e.interpolate(pts)
    assert not np.array_equal(bb.h, b.h[:len(bb)])
    assert_matches(got, checker(pts, bb, p), "after steps")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODES))
def test_depth_limited_leaves_are_members(name, lib):
    """Coincident particles under a small max_depth share a depth-limited leaf that the density walk skips; here they
    are ordinary members."""
    p = default_params(MODES[name], max_depth=5)
    b, s = ics.keplerian_disc(1500, seed=51)
    k = np.arange(0, 1500, 7)
    for f in ("x", "y", "z", "h"):
        getattr(b, f)[k + 1] = getattr(b, f)[k]          # 215 coincident pairs
    pts = np.concatenate([np.stack([b.x[k], b.y[k], b.z[k]], 1), probe_points(b, 52, 200)])
    with engine(p) as e:
        e.upload(b, s)
        got = e.interpolate(pts)
    ref = checker(pts, b, p)
    assert_matches(got, ref, name)
    assert np.all(got["count"][:len(k)] >= 2)


@pytest.mark.gpu
def test_repeatable_permutable_and_batch_independent(lib):
    p = default_params(MODE_VARIABLE_H)
    b, s = ics.keplerian_disc(4000, seed=61)
    pts = probe_points(b, 62, 3000)
    rng = np.random.default_rng(63)
    perm = rng.permutation(len(pts))
    alone = rng.choice(len(pts), 12, replace=False)
    with engine(p) as e:
        e.upload(b, s)
        dt, t = e.step(0.01, 0.0)            # velocities and h vary from their initial values
        a = e.interpolate(pts)
        a2 = e.interpolate(pts)
        ap = e.interpolate(pts[perm])
        single = [e.interpolate(pts[i:i + 1]) for i in alone]
    for k in COLS:
        assert np.array_equal(a[k], a2[k]), k
        assert np.array_equal(ap[k], a[k][perm]), k
        one = np.array([d[k][0] for d in single])
        # the walk visits a run's source groups in an order that depends on the run's box (DESIGN.md §5a): equal up to
        # the order of the sum, on the scale of the column
        scale = max(np.sqrt(np.mean(a[k] ** 2)), 1e-300)
        assert np.max(np.abs(one - a[k][alone])) <= 1e-14 * scale, k


@pytest.mark.gpu
def test_z_integral_is_the_column_density(lib):
    """sum_k rho(x, y, z_k) dz over a fine z column = sph_column_density at the same pixel centres (pixels < h)."""
    p = default_params(MODE_FIXED_H, h_fixed=2.5)
    b, s = ics.keplerian_disc(3000, seed=71, r_out=40.0, r_in=5.0)
    n_px, half = 24, 30.0
    zmax = float(np.max(np.abs(b.z))) + 2.0 * p.h_fixed + 0.1
    nz = 1600
    dz = 2.0 * zmax / nz
    zc = -zmax + (np.arange(nz) + 0.5) * dz
    c = -half + (np.arange(n_px) + 0.5) * (2.0 * half / n_px)
    X, Y, Z = np.meshgrid(c, c, zc, indexing="ij")          # x = u (column), y = v (row)
    pts = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1)
    with engine(p) as e:
        e.upload(b, s)
        rho = e.interpolate(pts, n_out=1)["rho"].reshape(n_px, n_px, nz)
        img = e.column_density("z", (-half, half, -half, half), (n_px, n_px))
    col = rho.sum(2).T * dz                                   # [iv, iu]
    assert img.max() > 0.0
    assert np.max(np.abs(col - img)) <= 1e-4 * img.max(), np.max(np.abs(col - img)) / img.max()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODES))
def test_the_call_does_not_change_the_run(name, lib):
    """Interpolation before and between the steps (device-resident steps and host round trips) leaves the run where the
    same run without the calls ends: state fingerprint, far-field reuses, recognised uploads; the stage times stay the
    last step's."""
    p = default_params(MODES[name])
    b, s = ics.keplerian_disc(6000, seed=81)
    pts = probe_points(b, 82, 500)
    res = []
    for ask in (0, 1):
        with engine(p) as e:
            e.upload(b, s)
            if ask:
                e.interpolate(pts)
            dt, t = 0.01, 0.0
            for _ in range(2):
                dt, t = e.step(dt, t)
                if ask:
                    e.interpolate(pts)
            be, se = e.download()
            for _ in range(3):
                ob, os_ = Bodies.empty(len(be)), Sinks.empty(len(se) + 8)
                dt, t, n2, ns2 = e.step_host(be, se, dt, t, into=(ob, os_))
                be = ob; se = Sinks(*[getattr(os_, k)[:ns2].copy() for k in ("x", "y", "z", "vx", "vy", "vz", "m", "radius")])
                if ask:
                    st = e.stage_times()
                    e.interpolate(pts)
                    assert e.stage_times() == st
            res.append((e.state_hash()[0], dt, t, e.far_reuse_count(), e.resident_hits()))
    assert res[1] == res[0], res


@pytest.mark.gpu
def test_errors(lib):
    from summersph_b200.engine import load_library, SphError, _p
    ARG, STATE = -1, -5                     # SPH_ERR_ARG, SPH_ERR_STATE
    L = load_library()
    p = default_params(MODE_VARIABLE_H)
    b, s = ics.keplerian_disc(500, seed=91)
    pts = np.zeros((4, 3))
    with engine(p) as e:
        with pytest.raises(SphError) as ei:
            e.interpolate(pts)
        assert ei.value.code == STATE, "no upload"
        e.upload(b, s)
        for n_out in (0, 8):
            with pytest.raises(SphError) as ei:
                e.interpolate(pts, n_out=n_out)
            assert ei.value.code == ARG, n_out
        bad = pts.copy(); bad[2, 1] = np.nan
        with pytest.raises(SphError) as ei:
            e.interpolate(bad)
        assert ei.value.code == ARG
        z = np.zeros(1)
        assert L.sph_interpolate(e._c, 0, _p(z), _p(z), _p(z), _p(z), 7) == 0
        assert L.sph_interpolate(e._c, 1, None, _p(z), _p(z), _p(z), 7) == ARG
        got = e.interpolate(np.zeros((0, 3)))
        assert set(got) == set(COLS) and all(len(v) == 0 for v in got.values())
        assert e.interpolate(pts)["rho"].shape == (4,)


@pytest.mark.gpu
def test_more_points_than_one_chunk(lib):
    """A 170^3 grid (4.9M points: two device chunks of 2^22) over a small disc, checked on a seeded sample."""
    p = default_params(MODE_VARIABLE_H)
    b, s = ics.keplerian_disc(2000, seed=101)
    g = np.linspace(-110.0, 110.0, 170)
    X, Y, Z = np.meshgrid(g, g, np.linspace(-12.0, 12.0, 170), indexing="ij")
    pts = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1)
    assert len(pts) > 1 << 22
    with engine(p) as e:
        e.upload(b, s)
        got = e.interpolate(pts)
    sel = np.random.default_rng(102).choice(len(pts), 2000, replace=False)
    sel = np.concatenate([sel, np.arange((1 << 22) - 20, (1 << 22) + 20)])      # both sides of the chunk boundary
    ref = checker(pts[sel], b, p)
    assert_matches({k: v[sel] for k, v in got.items()}, ref, "chunks")
    assert got["count"].max() > 0


@pytest.mark.gpu
def test_density_image_slice_cli(tmp_path, lib):
    from summersph_b200 import density_image
    from summersph_b200.textio import make_save, read_data_from_file
    p = default_params(MODE_VARIABLE_H)
    b, s = ics.keplerian_disc(3000, seed=111)
    s.radius[:] = p.sink_radius
    path = make_save(b, s, 7, p, directory=str(tmp_path))
    out, npy = str(tmp_path / "slice.pgm"), str(tmp_path / "slice.npy")
    density_image.main([path, "--variable", "--slice", "0.5", "--axis", "x", "--size", "110", "--pixels", "64", "--out", out, "--npy", npy])
    img = np.load(npy)
    bb, ss = read_data_from_file(path, p, log=None)
    with engine(p) as e:
        e.upload(bb, ss)
        ref = density_image.density_slice(e, "x", 0.5, 110.0, 64)
        px = 220.0 / 64
        one = e.interpolate(np.array([[0.5, -110.0 + 11.5 * px, -110.0 + 31.5 * px]]), n_out=1)["rho"][0]
    assert img.shape == (64, 64) and np.array_equal(img, ref) and img.max() > 0.0
    assert one == pytest.approx(img[31, 11], rel=1e-13, abs=0.0)      # axis x: u = y (column), v = z (row)
    head = b"P5\n64 64\n255\n"
    with open(out, "rb") as f:
        assert f.read(len(head)) == head
    assert os.path.getsize(out) == len(head) + 64 * 64


# ---------------------------------------------------------------------------------------------------------------------
# GPU, domains: one process per rank (tests/_dd_interp_rank.py)
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
            token = "/sphinterp_" + uuid.uuid4().hex[:16]
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


def assert_ranks_identical(res, keys):
    for k in keys:
        for r in range(1, len(res)):
            assert np.array_equal(res[r][k], res[0][k]), (k, r)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODES))
@pytest.mark.parametrize("world", [2, 3, 4])
def test_domains_equal_one_rank(world, name, tmp_path, lib):
    """After the upload (the call builds migration, halo and LET) and after steps: every rank returns the same bits,
    equal to the single-rank result up to the grouping of the sums."""
    spec = {"scenario": "values", "mode": MODES[name], "decomposition": 1}
    one = run_ranks(tmp_path, f"one_{name}", 1, spec)[0]
    res = run_ranks(tmp_path, f"w{world}_{name}", world, spec)
    keys = [k for k in one if k.startswith(("up_", "st_"))]
    assert_ranks_identical(res, keys)
    for k in keys:
        tol = 0 if k.endswith("count") else 1e-12
        if tol == 0:
            assert np.array_equal(res[0][k], one[k]), k
        else:
            assert relerr(res[0][k], one[k]) <= tol, (k, relerr(res[0][k], one[k]))
    assert sum(int(r["halo"][0]) for r in res) > 0


@pytest.mark.gpu
def test_domains_different_points_is_an_argument_error(tmp_path, lib):
    res = run_ranks(tmp_path, "mismatch", 3, {"scenario": "mismatch", "mode": MODE_VARIABLE_H, "decomposition": 1})
    for r in res:
        assert list(r["codes"]) == [1, 1, 0], r["codes"]      # mismatched points, one rank's NaN; then an agreed call succeeds


@pytest.mark.gpu
def test_domains_call_does_not_change_the_run(tmp_path, lib):
    res = run_ranks(tmp_path, "ask", 2, {"scenario": "ask", "mode": MODE_VARIABLE_H, "decomposition": 1, "steps": 3})
    for r in range(2):
        assert np.array_equal(res[r]["run1"], res[r]["run0"]), (r, res[r]["run0"], res[r]["run1"])


@pytest.mark.gpu
def test_replicated_two_ranks_is_one_rank(tmp_path, lib):
    spec = {"scenario": "values", "mode": MODE_VARIABLE_H, "decomposition": 0}
    one = run_ranks(tmp_path, "rep1", 1, spec)[0]
    res = run_ranks(tmp_path, "rep2", 2, spec)
    keys = [k for k in one if k.startswith(("up_", "st_"))]
    assert_ranks_identical(res, keys)
    for k in keys:
        assert np.array_equal(res[0][k], one[k]), k


@pytest.mark.gpu
@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_domains_nccl_two_gpus(tmp_path, lib):
    spec = {"scenario": "values", "mode": MODE_VARIABLE_H, "decomposition": 1}
    one = run_ranks(tmp_path, "nccl1", 1, spec)[0]
    res = run_ranks(tmp_path, "nccl2", 2, spec, comm="nccl")
    keys = [k for k in one if k.startswith(("up_", "st_"))]
    assert_ranks_identical(res, keys)
    for k in keys:
        assert relerr(res[0][k], one[k]) <= 1e-12, k
