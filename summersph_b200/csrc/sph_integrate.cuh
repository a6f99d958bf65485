// sph_integrate.cuh — kick / drift / timestep ladder / sink creation / accretion / bounds cull.
//
// Replaces kick, drift (SUMMER_SPH.f90:742-776), zero_rates (F:779-793), get_next_timestep
// (F:831-860 | Variable.f90:1035-1065), check_sink_creation (V:549-597), initiate_sink_accretion +
// sink2gasdists + pack_sinks (F:484-556 | V:616-688) and check_bounds (F:471-482 | V:599-614).
#pragma once
#include "sph_common.cuh"
#include "sph_gravity.cuh"

// device-resident loop scalars
struct SimScalars {
  double dt, t;
  double dt_min;          // minval of the 4N candidates (before scaling)
  int    n_sink;
  int    n_removed;       // gas particles flagged by accretion or bounds this step
  int    n_accreted;      // entries in the accretion list
  int    err;             // sticky error flag (key depth)
  int    any_sink_mass;   // any(sinks%mass > 0) F:919
  unsigned long long create_cand;   // (id << 32) | sorted index of the first over-dense particle, ~0 if none
  int    far_bad;         // end of step: the stored far-field gravity may not be kept (k_far_check)
  int    far_ovf;         // runs of the last full gravity walk whose recorded near pairs did not fit their slots
};

struct StateArrays { double *x, *y, *z, *vx, *vy, *vz, *u, *m, *alpha, *h; int* id; };
struct RateArrays { double *ax, *ay, *az, *udot, *adot; };

// half kick: F:749-758. DRIFT fuses the following full drift F:769-771.
template <bool DRIFT>
__global__ void k_kick(int n, StateArrays s, RateArrays r, const SimScalars* sc) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double dt = sc->dt;
  double vx = s.vx[i] + 0.5 * r.ax[i] * dt;
  double vy = s.vy[i] + 0.5 * r.ay[i] * dt;
  double vz = s.vz[i] + 0.5 * r.az[i] * dt;
  s.vx[i] = vx; s.vy[i] = vy; s.vz[i] = vz;
  s.u[i] = s.u[i] + 0.5 * r.udot[i] * dt;
  s.alpha[i] = s.alpha[i] + r.adot[i] * dt * 0.5;
  if (DRIFT) {
    s.x[i] = s.x[i] + vx * dt; s.y[i] = s.y[i] + vy * dt; s.z[i] = s.z[i] + vz * dt;
  }
}

template <bool DRIFT>
__global__ void k_kick_sinks(SinkArrays S, const SimScalars* sc) {
  int s = threadIdx.x;
  if (s >= sc->n_sink) return;
  const double dt = sc->dt;
  S.vx[s] = S.vx[s] + 0.5 * S.ax[s] * dt; S.vy[s] = S.vy[s] + 0.5 * S.ay[s] * dt; S.vz[s] = S.vz[s] + 0.5 * S.az[s] * dt;   // F:753-755
  if (DRIFT) { S.x[s] = S.x[s] + S.vx[s] * dt; S.y[s] = S.y[s] + S.vy[s] * dt; S.z[s] = S.z[s] + S.vz[s] * dt; }          // F:773-775
}

// timestep candidates: F:845-851. fmin drops NaNs like gfortran's MINVAL.
__global__ void k_dt_partial(int p_begin, int p_end, DevParams P, StateArrays s, RateArrays r, const double* __restrict__ cs,
                             double* __restrict__ partial) {
  double mn = INFINITY;
  for (int i = p_begin + blockIdx.x * blockDim.x + threadIdx.x; i < p_end; i += gridDim.x * blockDim.x) {
    const double vx = s.vx[i], vy = s.vy[i], vz = s.vz[i];
    const double ax = r.ax[i], ay = r.ay[i], az = r.az[i];
    const double vv = __dadd_rn(__dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy)), __dmul_rn(vz, vz));
    const double aa = __dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az));
    const double hh = P.variable_h ? s.h[i] : P.h_fixed;
    const double c = cs[i];
    mn = fmin(mn, sqrt(vv / aa));
    mn = fmin(mn, s.u[i] / fabs(r.udot[i]));
    mn = fmin(mn, hh / sqrt(vv));
    mn = fmin(mn, hh / __dadd_rn(c, __dmul_rn(1.2, c)));
  }
  mn = warp_min(mn);
  __shared__ double sm[32];
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) sm[w] = mn;
  __syncthreads();
  if (w == 0) {
    mn = (l < (blockDim.x >> 5)) ? sm[l] : INFINITY;
    mn = warp_min(mn);
    if (l == 0) partial[blockIdx.x] = mn;
  }
}

// fold the block minima of this rank's slice. One warp.
__global__ void k_dt_fold(int nblocks, const double* __restrict__ partial, SimScalars* sc) {
  double mn = INFINITY;
  for (int b = threadIdx.x; b < nblocks; b += 32) mn = fmin(mn, partial[b]);
  mn = warp_min(mn);
  if (threadIdx.x == 0) sc->dt_min = mn;
}
// the x1.5 / x0.5 ladder F:855-859 on the global minimum; also t = t + dt (F:914)
__global__ void k_dt_ladder(DevParams P, SimScalars* sc, int advance_time) {
  double dt = sc->dt;
  if (advance_time) sc->t = sc->t + dt;
  const double cand = sc->dt_min * P.tscale;
  if (cand > 2.0 * dt && 1.5 * dt < P.lit_01) dt = 1.5 * dt;
  else if (cand < 0.5 * dt && dt * 0.5 > P.lit_1em4) dt = 0.5 * dt;
  sc->dt = dt;
}

// V:559-560 first (lowest number) particle with m (eta/h)^3 > 0.5
__global__ void k_create_scan(int n, DevParams P, StateArrays s, SimScalars* sc) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double e = P.eta / s.h[i];
  if (s.m[i] * ((e * e) * e) > 0.5)
    atomicMin(&sc->create_cand, ((unsigned long long)(unsigned)s.id[i] << 32) | (unsigned)i);
}
__global__ void k_create_apply(StateArrays s, SinkArrays S, SimScalars* sc, double* __restrict__ spin) {
  if (threadIdx.x != 0) return;
  const unsigned long long c = sc->create_cand;
  sc->create_cand = ~0ull;
  if (c == ~0ull) return;
  const int i = (int)(c & 0xffffffffu);
  const int ns = sc->n_sink;
  for (int j = 0; j < ns; ++j) {
    const double dx = S.x[j] - s.x[i], dy = S.y[j] - s.y[i], dz = S.z[j] - s.z[i];
    const double dr = sqrt(dx * dx + dy * dy + dz * dz);
    if (dr < S.radius[j] + 2.0 * s.h[i]) return;                                   // V:563-565
  }
  if (ns >= SPH_MAX_SINKS) { sc->err = 3; return; }      // loud: the reference grows sinks(:) without bound (V:568-586)
  S.x[ns] = s.x[i]; S.y[ns] = s.y[i]; S.z[ns] = s.z[i];
  S.vx[ns] = s.vx[i]; S.vy[ns] = s.vy[i]; S.vz[ns] = s.vz[i];
  S.ax[ns] = S.ay[ns] = S.az[ns] = 0.0;
  S.m[ns] = 0.00000000001; S.radius[ns] = 2.0 * s.h[i];                            // V:581-582
  if (spin) spin[ns] = spin[SPH_MAX_SINKS + ns] = spin[2 * SPH_MAX_SINKS + ns] = 0.0;  // V:580
  sc->n_sink = ns + 1;
}

// accretion + bounds flags. keep[i] = 1 unless accreted by some sink (F:538-540 | V:670-672) or outside
// the bounding cube (F:478).  Accreted (sink, id, index) triples are appended to `acc_key/acc_val`.
// The tree walk of sink2gasdists is replayed per particle along its own root-to-leaf path: every ancestor
// cell must pass `all |c - x_s| < R_s + size/2` (F:529), the leaf `< 2 R_s + size/2` (F:536) | `< R_s + size/2`
// (V:668), then dr = sum sqrt(c^2 - x_s^2) on the leaf cell centre (F:537) | sum sqrt((x - x_s)^2) (V:669).
__global__ void k_flags(int n, DevParams P, StateArrays s, const uint64_t* __restrict__ key, const uint64_t* __restrict__ key_lo, const int* __restrict__ level,
                        const double* __restrict__ lcx, const double* __restrict__ lcy, const double* __restrict__ lcz,
                        const double* __restrict__ reach, const RootBox* __restrict__ rb, SinkArrays S, SimScalars* sc,
                        unsigned char* __restrict__ keep, unsigned long long* __restrict__ acc_key,
                        int* __restrict__ acc_val, int acc_cap) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double px = s.x[i], py = s.y[i], pz = s.z[i];
  bool kp = true;
  if (sc->any_sink_mass && reach[i] > 0.0) {
    const int ns = sc->n_sink;
    const int lev = level[i];
    double lsize = rb->size;
    for (int q = 0; q < lev; ++q) lsize = lsize * 0.5;
    const double cx = lcx[i], cy = lcy[i], cz = lcz[i];
    for (int j = 0; j < ns; ++j) {
      const double sx = S.x[j], sy = S.y[j], sz = S.z[j], R = S.radius[j];
      const double lim = (P.variable_h ? R : 2.0 * R) + lsize / 2.0;
      if (!(fabs(cx - sx) < lim && fabs(cy - sy) < lim && fabs(cz - sz) < lim)) continue;
      double dr;
      if (P.variable_h) {
        const double a = px - sx, b = py - sy, c = pz - sz;
        dr = __dadd_rn(__dadd_rn(__dsqrt_rn(__dmul_rn(a, a)), __dsqrt_rn(__dmul_rn(b, b))), __dsqrt_rn(__dmul_rn(c, c)));
      } else {
        dr = __dadd_rn(__dadd_rn(__dsqrt_rn(__dsub_rn(__dmul_rn(cx, cx), __dmul_rn(sx, sx))),
                                 __dsqrt_rn(__dsub_rn(__dmul_rn(cy, cy), __dmul_rn(sy, sy)))),
                       __dsqrt_rn(__dsub_rn(__dmul_rn(cz, cz), __dmul_rn(sz, sz))));
      }
      if (!(dr < R)) continue;
      // ancestors along the path (levels 0 .. lev-1)
      double ax = rb->cx, ay = rb->cy, az = rb->cz, as = rb->size;
      const uint64_t k = key[i], k2 = key_lo ? key_lo[i] : 0;
      bool pass = true;
      for (int l = 0; l < lev; ++l) {
        const double al = R + as / 2.0;
        if (!(fabs(ax - sx) < al && fabs(ay - sy) < al && fabs(az - sz) < al)) { pass = false; break; }
        const int dg = key_digit(k, k2, l);
        const double q = 0.25 * as;
        ax = __dadd_rn(ax, (dg & 1) ? q : -q); ay = __dadd_rn(ay, (dg & 2) ? q : -q); az = __dadd_rn(az, (dg & 4) ? q : -q);
        as = as * 0.5;
      }
      if (!pass) continue;
      kp = false;
      const int slot = atomicAdd(&sc->n_accreted, 1);
      if (slot < acc_cap) { acc_key[slot] = ((unsigned long long)j << 32) | (unsigned)s.id[i]; acc_val[slot] = i; }
    }
  }
  if (kp) kp = (fabs(px) <= P.bounding) && (fabs(py) <= P.bounding) && (fabs(pz) <= P.bounding);   // F:478
  keep[i] = kp ? 1 : 0;
  if (!kp) atomicAdd(&sc->n_removed, 1);
}

// sink update from the (sink, number)-sorted accretion list: sums in ascending number like sum(pack(...)) F:497-508
// `spin` (null unless SPH_FLAG_SINK_MERGE_SPIN): what the orbit loses goes into the sink's spin, so that the summed
// angular momentum of sink + accreted gas about the origin is unchanged (not in the reference, F:509 asks for it).
__global__ void k_accrete_apply(int n_acc, const unsigned long long* __restrict__ acc_key, const int* __restrict__ acc_val,
                                StateArrays s, SinkArrays S, SimScalars* sc, double* __restrict__ spin) {
  const int j = threadIdx.x;
  if (j >= sc->n_sink || !sc->any_sink_mass) return;
  double sm = 0.0, sp[3] = {0.0, 0.0, 0.0}, sv[3] = {0.0, 0.0, 0.0}, lb[3] = {0.0, 0.0, 0.0};
  int n_mine = 0;
  // the list is sorted by (sink, number): this sink's entries are one contiguous range, summed in ascending number
  int lo = 0, hi = n_acc;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if ((int)(acc_key[mid] >> 32) < j) lo = mid + 1; else hi = mid; }
  int e1 = lo; hi = n_acc;
  while (e1 < hi) { const int mid = (e1 + hi) >> 1; if ((int)(acc_key[mid] >> 32) <= j) e1 = mid + 1; else hi = mid; }
  for (int e = lo; e < e1; ++e) {
    const int i = acc_val[e];
    const double mi = s.m[i];
    if (spin) {
      const double x = s.x[i], y = s.y[i], z = s.z[i], vx = s.vx[i], vy = s.vy[i], vz = s.vz[i];
      lb[0] = lb[0] + mi * (y * vz - z * vy); lb[1] = lb[1] + mi * (z * vx - x * vz); lb[2] = lb[2] + mi * (x * vy - y * vx);
      ++n_mine;
    }
    sm = __dadd_rn(sm, mi);
    sp[0] = __dadd_rn(sp[0], __dmul_rn(mi, s.x[i])); sp[1] = __dadd_rn(sp[1], __dmul_rn(mi, s.y[i])); sp[2] = __dadd_rn(sp[2], __dmul_rn(mi, s.z[i]));
    sv[0] = __dadd_rn(sv[0], __dmul_rn(mi, s.vx[i])); sv[1] = __dadd_rn(sv[1], __dmul_rn(mi, s.vy[i])); sv[2] = __dadd_rn(sv[2], __dmul_rn(mi, s.vz[i]));
  }
  const double ms = S.m[j];
  if (spin && n_mine > 0) {
    const double x = S.x[j], y = S.y[j], z = S.z[j], vx = S.vx[j], vy = S.vy[j], vz = S.vz[j];
    lb[0] = lb[0] + ms * (y * vz - z * vy); lb[1] = lb[1] + ms * (z * vx - x * vz); lb[2] = lb[2] + ms * (x * vy - y * vx);
  }
  const double nm = __dadd_rn(ms, sm);                                                          // F:497
  S.x[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.x[j]), sp[0]), nm);                              // F:498-501
  S.y[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.y[j]), sp[1]), nm);
  S.z[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.z[j]), sp[2]), nm);
  S.vx[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.vx[j]), sv[0]), nm);                            // F:503-506
  S.vy[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.vy[j]), sv[1]), nm);
  S.vz[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.vz[j]), sv[2]), nm);
  S.m[j] = __dadd_rn(ms, sm);                                                                   // F:508
  if (spin && n_mine > 0) {
    const double x = S.x[j], y = S.y[j], z = S.z[j], vx = S.vx[j], vy = S.vy[j], vz = S.vz[j], m2 = S.m[j];
    spin[j] = spin[j] + (lb[0] - (0.0 + m2 * (y * vz - z * vy)));
    spin[SPH_MAX_SINKS + j] = spin[SPH_MAX_SINKS + j] + (lb[1] - (0.0 + m2 * (z * vx - x * vz)));
    spin[2 * SPH_MAX_SINKS + j] = spin[2 * SPH_MAX_SINKS + j] + (lb[2] - (0.0 + m2 * (x * vy - y * vx)));
  }
}

__global__ void k_any_sink_mass(SinkArrays S, SimScalars* sc) {
  if (threadIdx.x != 0) return;
  int any = 0;
  for (int j = 0; j < sc->n_sink; ++j) if (S.m[j] > 0.0) any = 1;                               // F:919
  sc->any_sink_mass = any;
}

// V:610,613 cull sinks outside the bounding cube (order preserving)
__global__ void k_cull_sinks(DevParams P, SinkArrays S, SimScalars* sc, double* __restrict__ spin) {
  if (threadIdx.x != 0) return;
  const int ns = sc->n_sink; int w = 0;
  for (int j = 0; j < ns; ++j) {
    if (fabs(S.x[j]) <= P.bounding && fabs(S.y[j]) <= P.bounding && fabs(S.z[j]) <= P.bounding) {
      if (w != j) {
        S.x[w] = S.x[j]; S.y[w] = S.y[j]; S.z[w] = S.z[j]; S.vx[w] = S.vx[j]; S.vy[w] = S.vy[j]; S.vz[w] = S.vz[j];
        S.m[w] = S.m[j]; S.radius[w] = S.radius[j]; S.ax[w] = S.ax[j]; S.ay[w] = S.ay[j]; S.az[w] = S.az[j];
        if (spin) for (int k = 0; k < 3; ++k) spin[k * SPH_MAX_SINKS + w] = spin[k * SPH_MAX_SINKS + j];
      }
      ++w;
    }
  }
  sc->n_sink = w;
}

// Sink merger: NOT in the reference (check_sink_merger is an empty stub, V:1067-1073; its call is commented out at
// V:1159).  Opt-in (SPH_FLAG_SINK_MERGE_SPIN), run where that call sits.  Two sinks with mass merge when one centre lies
// inside the other's accretion radius, |x_a - x_b| < max(R_a, R_b): the lower index survives with the summed mass, the
// mass-weighted position / velocity / acceleration, the larger radius and spin = S_a + S_b + (orbital L of the two -
// orbital L of the merged sink); the higher index is removed, order preserved.  Pairs (a, b > a) are scanned ascending
// and the scan restarts after every merge.  One thread: at most SPH_MAX_SINKS sinks.
__global__ void k_sink_merge(SinkArrays S, SimScalars* sc, double* __restrict__ spin) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int M = SPH_MAX_SINKS;
  int ns = sc->n_sink;
  bool merged = true;
  while (merged) {
    merged = false;
    for (int a = 0; a < ns && !merged; ++a)
      for (int b = a + 1; b < ns && !merged; ++b) {
        const double ma = S.m[a], mb = S.m[b];
        if (!(ma > 0.0 && mb > 0.0)) continue;
        const double dx = S.x[a] - S.x[b], dy = S.y[a] - S.y[b], dz = S.z[a] - S.z[b];
        const double dr = sqrt(dx * dx + dy * dy + dz * dz);
        const double R = fmax(S.radius[a], S.radius[b]);
        if (!(dr < R)) continue;
        double lb[3];
        lb[0] = 0.0 + ma * (S.y[a] * S.vz[a] - S.z[a] * S.vy[a]); lb[1] = 0.0 + ma * (S.z[a] * S.vx[a] - S.x[a] * S.vz[a]); lb[2] = 0.0 + ma * (S.x[a] * S.vy[a] - S.y[a] * S.vx[a]);
        lb[0] = lb[0] + mb * (S.y[b] * S.vz[b] - S.z[b] * S.vy[b]); lb[1] = lb[1] + mb * (S.z[b] * S.vx[b] - S.x[b] * S.vz[b]); lb[2] = lb[2] + mb * (S.x[b] * S.vy[b] - S.y[b] * S.vx[b]);
        const double Mt = ma + mb;
        double* f[9] = {S.x, S.y, S.z, S.vx, S.vy, S.vz, S.ax, S.ay, S.az};
        for (int k = 0; k < 9; ++k) f[k][a] = (ma * f[k][a] + mb * f[k][b]) / Mt;
        S.m[a] = Mt; S.radius[a] = R;
        const double l0 = 0.0 + Mt * (S.y[a] * S.vz[a] - S.z[a] * S.vy[a]), l1 = 0.0 + Mt * (S.z[a] * S.vx[a] - S.x[a] * S.vz[a]), l2 = 0.0 + Mt * (S.x[a] * S.vy[a] - S.y[a] * S.vx[a]);
        spin[a] = spin[a] + spin[b] + (lb[0] - l0);
        spin[M + a] = spin[M + a] + spin[M + b] + (lb[1] - l1);
        spin[2 * M + a] = spin[2 * M + a] + spin[2 * M + b] + (lb[2] - l2);
        for (int j = b; j + 1 < ns; ++j) {
          for (int k = 0; k < 9; ++k) f[k][j] = f[k][j + 1];
          S.m[j] = S.m[j + 1]; S.radius[j] = S.radius[j + 1];
          for (int k = 0; k < 3; ++k) spin[k * M + j] = spin[k * M + j + 1];
        }
        --ns;
        merged = true;
      }
  }
  sc->n_sink = ns;
}

__global__ void k_iota(int n, int* a) { int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) a[i] = i; }

// scatter by id for downloads in ascending number order: out[rank(id)] ; ids are persistent upload indices,
// so the ascending-number position of a particle is its rank among surviving ids (computed on the host side
// from the id array, see sph_engine.cu).
template <class T> __global__ void k_scatter(int n, const int* __restrict__ pos, const T* __restrict__ src, T* __restrict__ dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) dst[pos[i]] = src[i];
}

// FP64 FMA throughput probe (roofline denominator for the walk kernels; MEASURED_PEAKS.json has no FP64 figure)
__global__ void k_fp64_peak(int iters, double mul, double* out) {
  double a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double b = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, mul, b); a1 = fma(a1, mul, b); a2 = fma(a2, mul, b); a3 = fma(a3, mul, b);
    a4 = fma(a4, mul, b); a5 = fma(a5, mul, b); a6 = fma(a6, mul, b); a7 = fma(a7, mul, b);
  }
  double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 123.456) *out = s;
}
