"""ctypes binding of the C-ABI engine (include/sph_b200.h -> libsph_b200.so).

This is the reference-facing call path a Python host uses; tests and bench go through it, so every
number they report crosses the same `extern "C"` boundary a Fortran ISO_C_BINDING host would.
No CPU fallback: a missing library or CUDA device raises.
"""
import ctypes as C
import os
import numpy as np

from ._abi import SphParams, SphCounts, EVAL_ALL, ERRORS, CONSERVED, conserved_dict
from .state import Bodies, Sinks, GAS_FIELDS

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPH_B200_LIB") or os.path.join(_HERE, "libsph_b200.so")   # override: developer experiments only
_LIB = None

INTERP = ("rho", "vx", "vy", "vz", "u", "alpha", "count")      # the SPH_INTERP_COUNT output columns of sph_interpolate
GRAVAT = ("phi_gas", "gx_gas", "gy_gas", "gz_gas", "phi_sink", "gx_sink", "gy_sink", "gz_sink", "accepted")   # SPH_GRAVAT_COUNT columns of sph_gravity_at
STAGES = ("keys", "sort", "tree", "density", "gravity", "sph", "integrate", "h_iter", "cull", "comm", "halo", "let", "migrate", "gravity_near")


class SphError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"sph_b200 error {code} ({ERRORS.get(code, '?')}): {msg}")
        self.code = code


def load_library(path=None):
    """Load libsph_b200.so (built in-tree by summersph_b200.build). Fails loudly if it is missing."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FileNotFoundError(f"{p} not found: build it with `python -m summersph_b200.build` "
                                "(there is no CPU fallback for the SPH step)")
    lib = C.CDLL(p)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    lib.sph_last_error.restype = C.c_char_p
    lib.sph_last_error.argtypes = [vp]
    lib.sph_default_params.argtypes = [i32, C.POINTER(SphParams)]
    lib.sph_create.argtypes = [C.POINTER(SphParams), i32, C.POINTER(vp)]
    lib.sph_destroy.argtypes = [vp]
    lib.sph_comm_unique_id.argtypes = [vp]
    lib.sph_comm_init.argtypes = [vp, i32, i32, vp]
    lib.sph_slice_bounds.argtypes = [i32, i32, vp]
    lib.sph_comm_init_host.argtypes = [vp, i32, i32, C.c_char_p]
    lib.sph_upload.argtypes = [vp, i64] + [vp] * 10 + [i32] + [vp] * 8
    lib.sph_upload_local.argtypes = [vp, i64, i64, vp, i64] + [vp] * 10 + [i32] + [vp] * 8
    lib.sph_state_hash.argtypes = [vp, C.POINTER(C.c_uint64), vp]
    lib.sph_domain_stats.argtypes = [vp, vp]
    lib.sph_local_size.argtypes = [vp, C.POINTER(i64)]
    lib.sph_download_local.argtypes = [vp] + [vp] * 11
    lib.sph_ics_disc.argtypes = [vp, i64, C.c_uint64] + [dbl] * 8
    lib.sph_evaluate.argtypes = [vp, i32]
    lib.sph_step.argtypes = [vp, C.POINTER(dbl), C.POINTER(dbl), C.POINTER(i64), C.POINTER(i32)]
    lib.sph_step_host.argtypes = [vp, i64, vp, i32, vp, C.POINTER(dbl), C.POINTER(dbl), vp, vp, C.POINTER(i64), C.POINTER(i32)]
    lib.sph_run_until.argtypes = [vp, dbl, i64, C.POINTER(dbl), C.POINTER(dbl), C.POINTER(i64), C.POINTER(i64), C.POINTER(i32)]
    lib.sph_sizes.argtypes = [vp, C.POINTER(i64), C.POINTER(i32)]
    lib.sph_download.argtypes = [vp] + [vp] * 18
    lib.sph_download_diag.argtypes = [vp] + [vp] * 12
    lib.sph_download_tree.argtypes = [vp] + [vp] * 7
    lib.sph_download_neighbours.argtypes = [vp, vp, vp, vp, vp, i64]
    lib.sph_counters.argtypes = [vp, C.POINTER(SphCounts)]
    lib.sph_set_exact_counters.argtypes = [vp, i32]
    lib.sph_stage_times.argtypes = [vp, vp, i32]
    lib.sph_launch_count.argtypes = [vp]
    lib.sph_launch_count.restype = i64
    lib.sph_group_count.argtypes = [vp]
    lib.sph_group_count.restype = i64
    lib.sph_far_reuse_count.argtypes = [vp]
    lib.sph_far_reuse_count.restype = i64
    lib.sph_far_overflow_runs.argtypes = [vp]
    lib.sph_far_overflow_runs.restype = i64
    lib.sph_resident_hits.argtypes = [vp]
    lib.sph_resident_hits.restype = i64
    lib.sph_set_resident_check.argtypes = [vp, i32]
    lib.sph_timer_start.argtypes = [vp]
    lib.sph_timer_stop.argtypes = [vp, C.POINTER(dbl)]
    lib.sph_fp64_peak.argtypes = [vp, C.POINTER(dbl)]
    lib.sph_conserved.argtypes = [vp, vp, i32]
    lib.sph_download_sink_spin.argtypes = [vp, vp, vp, vp]
    lib.sph_column_density.argtypes = [vp, i32, dbl, dbl, dbl, dbl, i32, i32, vp]
    lib.sph_interpolate.argtypes = [vp, i64, vp, vp, vp, vp, i32]
    lib.sph_gravity_at.argtypes = [vp, i64, vp, vp, vp, vp, vp, i32]
    if path is None:
        _LIB = lib
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Engine:
    """One engine context on one CUDA device (`sph_ctx`)."""

    def __init__(self, params: SphParams, device=0, exact_counters=False, lib_path=None):
        """`lib_path`: developer experiments only (a variant build under summersph_b200/variants/)."""
        self._l = load_library(lib_path)
        self.params = params
        self._c = C.c_void_p()
        rc = self._l.sph_create(C.byref(params), int(device), C.byref(self._c))
        if rc != 0:
            msg = self._l.sph_last_error(None)
            self._c = None
            raise SphError(rc, (msg or b"").decode())
        if exact_counters:
            self.set_exact_counters(True)

    def set_exact_counters(self, on=True):
        """Count every leaf-box candidate like the reference (slower); default: cull exact-zero pairs early."""
        self._ck(self._l.sph_set_exact_counters(self._c, 1 if on else 0))

    def close(self):
        if getattr(self, "_c", None):
            self._l.sph_destroy(self._c)
            self._c = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise SphError(rc, (self._l.sph_last_error(self._c) or b"").decode())

    # -- multi-GPU ---------------------------------------------------------------------------------
    def unique_id(self):
        buf = (C.c_char * 128)()
        rc = self._l.sph_comm_unique_id(buf)
        if rc != 0:
            raise SphError(rc, (self._l.sph_last_error(None) or b"").decode())
        return bytes(buf)

    def comm_init(self, rank, n_ranks, unique_id: bytes):
        buf = (C.c_char * 128).from_buffer_copy(unique_id)
        self._ck(self._l.sph_comm_init(self._c, int(rank), int(n_ranks), buf))

    def comm_init_host(self, rank, n_ranks, name: str):
        """Small collectives through a host shared-memory segment instead of NCCL (several ranks may share a GPU)."""
        self._ck(self._l.sph_comm_init_host(self._c, int(rank), int(n_ranks), name.encode()))

    # -- state -------------------------------------------------------------------------------------
    def upload(self, b: Bodies, s: Sinks):
        rad = s.radius
        self._ck(self._l.sph_upload(self._c, len(b), _p(b.x), _p(b.y), _p(b.z), _p(b.vx), _p(b.vy), _p(b.vz),
                                    _p(b.u), _p(b.m), _p(b.alpha), _p(b.h), len(s),
                                    _p(s.x), _p(s.y), _p(s.z), _p(s.vx), _p(s.vy), _p(s.vz), _p(s.m), _p(rad)))

    def state_hash(self):
        """(fingerprint, sums): `sph_state_hash` - equal fingerprints <=> bit-identical states."""
        h = C.c_uint64(); sums = np.zeros(5)
        self._ck(self._l.sph_state_hash(self._c, C.byref(h), _p(sums)))
        return int(h.value), dict(zip(("mass", "m_x2", "m_v2", "m_u", "count"), sums.tolist()))

    def domain_stats(self):
        out = np.zeros(8, np.int64)
        self._ck(self._l.sph_domain_stats(self._c, _p(out)))
        return dict(zip(("domains", "own", "halo", "own_groups", "halo_groups", "let_nodes", "top_slots", "global"), out.tolist()))

    def upload_local(self, n_global, b: Bodies, s: Sinks, id_first=0, numbers=None):
        """Domain decomposition: hand over rows [id_first, id_first + len(b)) - or the rows `numbers` - of the
        n_global gas rows (`sph_upload_local`)."""
        num = None if numbers is None else np.ascontiguousarray(numbers, dtype=np.int32)
        self._ck(self._l.sph_upload_local(self._c, int(n_global), int(id_first), _p(num), len(b), _p(b.x), _p(b.y), _p(b.z), _p(b.vx), _p(b.vy), _p(b.vz),
                                          _p(b.u), _p(b.m), _p(b.alpha), _p(b.h), len(s),
                                          _p(s.x), _p(s.y), _p(s.z), _p(s.vx), _p(s.vy), _p(s.vz), _p(s.m), _p(s.radius)))

    def ics_disc(self, n, seed=20251018, r_in=10.0, r_out=100.0, aspect=0.05, m_star=1.0, m_disc=0.01, u=0.25, alpha=0.1, eta=1.2):
        """Keplerian disc + central sink generated on the device (`sph_ics_disc`); same parameters as ics.keplerian_disc."""
        self._ck(self._l.sph_ics_disc(self._c, int(n), int(seed), r_in, r_out, aspect, m_star, m_disc, u, alpha, eta))

    def local_size(self):
        n = C.c_int64()
        self._ck(self._l.sph_local_size(self._c, C.byref(n)))
        return n.value

    def download_local(self, into=None):
        """The rows this rank owns: (numbers, Bodies) in the rank's Morton order (`sph_download_local`)."""
        n = self.local_size()
        b = into if into is not None else Bodies.empty(n)
        num = np.zeros(n, np.int32)
        self._ck(self._l.sph_download_local(self._c, _p(num), _p(b.x), _p(b.y), _p(b.z), _p(b.vx), _p(b.vy), _p(b.vz), _p(b.u), _p(b.m),
                                            _p(b.alpha), _p(b.h)))
        return num, b

    def sizes(self):
        n, ns = C.c_int64(), C.c_int32()
        self._ck(self._l.sph_sizes(self._c, C.byref(n), C.byref(ns)))
        return n.value, ns.value

    def evaluate(self, mask=EVAL_ALL):
        self._ck(self._l.sph_evaluate(self._c, int(mask)))

    def step(self, dt, t):
        cdt, ct, n, ns = C.c_double(dt), C.c_double(t), C.c_int64(), C.c_int32()
        self._ck(self._l.sph_step(self._c, C.byref(cdt), C.byref(ct), C.byref(n), C.byref(ns)))
        return cdt.value, ct.value

    def step_host(self, b: Bodies, s: Sinks, dt, t, into=None):
        """`sph_step_host`: upload (b, s), one loop body, download - one call, the copies run under the compute (pinned
        host arrays for the overlap).  `into` = (Bodies, Sinks) with room for len(b) rows and len(s) + 8 sinks (may be
        the input arrays); returns (dt, t, n_gas, n_sink): the first n_gas / n_sink rows of `into` hold the result."""
        if into is None:
            into = (Bodies.empty(len(b)), Sinks.empty(len(s) + 8))
        ob, os_ = into
        gin = (C.c_void_p * 10)(*[_p(getattr(b, k)) for k in GAS_FIELDS])
        sin = (C.c_void_p * 8)(*[_p(getattr(s, k)) for k in ("x", "y", "z", "vx", "vy", "vz", "m", "radius")])
        gout = (C.c_void_p * 10)(*[_p(getattr(ob, k)) for k in GAS_FIELDS])
        sout = (C.c_void_p * 8)(*[_p(getattr(os_, k)) for k in ("x", "y", "z", "vx", "vy", "vz", "m", "radius")])
        cdt, ct, n, ns = C.c_double(dt), C.c_double(t), C.c_int64(), C.c_int32()
        self._ck(self._l.sph_step_host(self._c, len(b), gin, len(s), sin, C.byref(cdt), C.byref(ct), gout, sout, C.byref(n), C.byref(ns)))
        return cdt.value, ct.value, n.value, ns.value

    def run_until(self, t_stop, dt, t, max_steps=0):
        cdt, ct, steps, n, ns = C.c_double(dt), C.c_double(t), C.c_int64(), C.c_int64(), C.c_int32()
        self._ck(self._l.sph_run_until(self._c, float(t_stop), int(max_steps), C.byref(cdt), C.byref(ct),
                                       C.byref(steps), C.byref(n), C.byref(ns)))
        return cdt.value, ct.value, steps.value

    def download(self, into=None):
        n, ns = self.sizes()
        b, s = (into if into is not None else (Bodies.empty(n), Sinks.empty(ns)))
        self._ck(self._l.sph_download(self._c, _p(b.x), _p(b.y), _p(b.z), _p(b.vx), _p(b.vy), _p(b.vz), _p(b.u), _p(b.m),
                                      _p(b.alpha), _p(b.h), _p(s.x), _p(s.y), _p(s.z), _p(s.vx), _p(s.vy), _p(s.vz),
                                      _p(s.m), _p(s.radius)))
        return b, s

    def sinks_only(self):
        """The (replicated) sinks without touching the gas rows."""
        _, ns = self.sizes()
        s = Sinks.empty(ns)
        self._ck(self._l.sph_download(self._c, *([None] * 10), _p(s.x), _p(s.y), _p(s.z), _p(s.vx), _p(s.vy), _p(s.vz), _p(s.m), _p(s.radius)))
        return s

    def diag(self):
        n, ns = self.sizes()
        keys = ("rho", "omega", "P", "c", "ax", "ay", "az", "udot", "alphadot")
        d = {k: np.zeros(n) for k in keys}
        d.update({k: np.zeros(ns) for k in ("sink_ax", "sink_ay", "sink_az")})
        self._ck(self._l.sph_download_diag(self._c, *[_p(d[k]) for k in keys + ("sink_ax", "sink_ay", "sink_az")]))
        return d

    def tree(self):
        n, _ = self.sizes()
        t = {"order": np.zeros(n, np.int32), "key": np.zeros(n, np.uint64), "level": np.zeros(n, np.int32),
             "cx": np.zeros(n), "cy": np.zeros(n), "cz": np.zeros(n), "size": np.zeros(n)}
        self._ck(self._l.sph_download_tree(self._c, *[_p(t[k]) for k in ("order", "key", "level", "cx", "cy", "cz", "size")]))
        return t

    def neighbours(self, with_list=True):
        n, _ = self.sizes()
        count = np.zeros(n, np.int32); hsh = np.zeros(n, np.uint64); off = np.zeros(n + 1, np.int64)
        self._ck(self._l.sph_download_neighbours(self._c, _p(count), _p(hsh), _p(off), None, 0))
        lst = None
        if with_list:
            tot = int(off[-1])
            lst = np.zeros(max(tot, 1), np.int32)
            self._ck(self._l.sph_download_neighbours(self._c, _p(count), _p(hsh), _p(off), _p(lst), tot))
            lst = lst[:tot]
        return count, hsh, off, lst

    def counters(self):
        c = SphCounts()
        self._ck(self._l.sph_counters(self._c, C.byref(c)))
        return c.as_dict()

    def stage_times(self):
        ms = np.zeros(16)
        self._ck(self._l.sph_stage_times(self._c, _p(ms), 16))
        return dict(zip(STAGES, ms[:len(STAGES)].tolist()))

    def launch_count(self):
        return int(self._l.sph_launch_count(self._c))

    def timer_start(self):
        self._ck(self._l.sph_timer_start(self._c))

    def timer_stop(self):
        ms = C.c_double()
        self._ck(self._l.sph_timer_stop(self._c, C.byref(ms)))
        return ms.value

    def fp64_peak(self):
        v = C.c_double()
        self._ck(self._l.sph_fp64_peak(self._c, C.byref(v)))
        return v.value

    def conserved(self):
        """Energy / momentum / angular-momentum sums of the resident state (`sph_conserved`)."""
        out = np.zeros(len(CONSERVED))
        self._ck(self._l.sph_conserved(self._c, _p(out), len(out)))
        return conserved_dict(out)

    def sink_spin(self):
        """(n_sink, 3) array of sink spins (`sph_download_sink_spin`): zero unless FLAG_SINK_MERGE_SPIN is set."""
        _, ns = self.sizes()
        sp = [np.zeros(ns) for _ in range(3)]
        self._ck(self._l.sph_download_sink_spin(self._c, *[_p(v) for v in sp]))
        return np.stack(sp, 1)

    def column_density(self, axis="z", extent=(-100.0, 100.0, -100.0, 100.0), shape=(512, 512)):
        """Column density of the resident gas projected along `axis` (`sph_column_density`): array of shape
        (nv, nu) = `shape`, rows along the image ordinate; extent = (u0, u1, v0, v1) like matplotlib's imshow
        with origin='lower'.  Image axes: x -> (y, z), y -> (z, x), z -> (x, y)."""
        ax = {"x": 0, "y": 1, "z": 2}.get(axis, axis)
        nv, nu = int(shape[0]), int(shape[1])
        img = np.zeros((nv, nu))
        u0, u1, v0, v1 = (float(e) for e in extent)
        self._ck(self._l.sph_column_density(self._c, int(ax), u0, u1, v0, v1, nu, nv, _p(img)))
        return img

    def interpolate(self, points, n_out=len(INTERP)):
        """The SPH interpolant of the resident gas at the rows of `points` ((M, 3): x, y, z), computed on the device
        (`sph_interpolate`): dict of length-M arrays {rho, vx, vy, vz, u, alpha, count} truncated to the first `n_out`.
        rho = sum m_j W(|x - x_j|, h_j), the means are mass-weighted (sum m_j f_j W / rho, 0 where rho = 0), count = the
        number of particles with |x - x_j| <= 2 h_j.  Collective under the Morton domains: every rank passes the same points."""
        pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
        m = len(pts)
        cols = [np.ascontiguousarray(pts[:, k]) for k in range(3)]
        out = np.zeros(max(int(n_out), 0) * m)
        self._ck(self._l.sph_interpolate(self._c, m, *[_p(c) for c in cols], _p(out), int(n_out)))
        return {k: out[i * m:(i + 1) * m] for i, k in enumerate(INTERP[:n_out])}

    def gravity_at(self, points, h=None, n_out=len(GRAVAT)):
        """The gravitational potential and acceleration at the rows of `points` ((M, 3): x, y, z), computed on the device
        (`sph_gravity_at`): dict of length-M arrays {phi_gas, gx_gas, gy_gas, gz_gas, phi_sink, gx_sink, gy_sink, gz_sink,
        accepted} truncated to the first `n_out`.  Each point is treated as a gas particle of smoothing length `h` (length-M
        array; None: h_fixed) that adds nothing to the tree: the gas part is the reference's Barnes-Hut sum over the nodes
        it would accept, the sink part the unsoftened direct sum.  Collective under the Morton domains: every rank passes
        the same points and h."""
        pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
        m = len(pts)
        cols = [np.ascontiguousarray(pts[:, k]) for k in range(3)]
        hh = None if h is None else np.ascontiguousarray(np.broadcast_to(np.asarray(h, dtype=np.float64), (m,)))
        out = np.zeros(max(int(n_out), 0) * m)
        self._ck(self._l.sph_gravity_at(self._c, m, *[_p(c) for c in cols], _p(hh), _p(out), int(n_out)))
        return {k: out[i * m:(i + 1) * m] for i, k in enumerate(GRAVAT[:n_out])}

    def group_count(self):
        return int(self._l.sph_group_count(self._c))

    def resident_hits(self):
        """Uploads so far that were recognised as the state the context already holds (`sph_resident_hits`)."""
        return int(self._l.sph_resident_hits(self._c))

    def set_resident_check(self, on=True):
        self._ck(self._l.sph_set_resident_check(self._c, 1 if on else 0))

    def far_reuse_count(self):
        """Gravity evaluations so far that walked only the near field on top of the stored far sums."""
        return int(self._l.sph_far_reuse_count(self._c))

    def far_overflow_runs(self):
        """Walk runs the last far-sum-storing gravity walk flagged for the near-only walk: some particle had more
        near terms than the recorded slots (`sph_far_overflow_runs`)."""
        return int(self._l.sph_far_overflow_runs(self._c))
