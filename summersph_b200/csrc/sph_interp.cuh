// sph_interp.cuh — the SPH interpolant at caller-given points (sph_interpolate, include/sph_b200.h).
//
// For a point x and the resident gas particles j (sinks are not SPH particles and take no part):
//   W(r, h) = w_table(r / h) / (pi h^3)   (the density pass's table lerp and normalisation: F:125-126 with h = h_fixed
//                                          for every j | V:139-140 with h = h_j and the single-precision pi)
//   members of x = { j : |x - x_j| / h_j <= 2 }   (scatter form: each source's own h; a source whose h is not finite
//                                          and positive is never a member)
//   raw[0] = sum m_j W,  raw[1..3] = sum m_j v_j W,  raw[4] = sum m_j u_j W,  raw[5] = sum m_j alpha_j W,  raw[6] = #members
// The means are raw[k] / raw[0] (0 where raw[0] == 0), taken after the ranks' raw sums are added (k_interp_finish).
//
// Sources: the walk groups of the current tree under a PRIVATE implicit 8-ary BVH whose reach boxes bound the balls
// |x - x_j| <= 2 h_j of the current h (k_interp_reach + k_bvh_leaf / k_bvh_up of sph_tree.cuh with the positions as the
// "leaf centres"); the tree's own BVH (reach 2h + size/2 of the build) is neither read nor written.
// Targets: the points, sorted by a Morton key over their own bounding box (ties broken by a hash of the coordinate
// bits, so the sorted sequence does not depend on the caller's order), cut into runs of 32 (one warp, lane = point).
// A run walks the private BVH with its outward-rounded FP32 box as the target box (neighbour_walk of sph_walk.cuh).
#pragma once
#include "sph_walk.cuh"

#define SPH_INTERP_CHUNK (1 << 22)     // points per device pass: bounds the scratch whatever the call's n_points
#define INTERP_WARPS 8                 // warps per block of k_interpolate
#define INTERP_FIELDS 11               // staged doubles per source: x y z h pi*h^3 m vx vy vz u alpha
#define INTERP_WARP_DOUBLES (INTERP_FIELDS * WALK_TILE + 2 * WALK_TILE)   // tile + float4 prefilter tile

struct InterpArrays { const double *x, *y, *z, *vx, *vy, *vz, *u, *m, *alpha, *h; const double* reach2; };

// 2 h_j (h_j = h_fixed in fixed-h mode) when h_j is finite and positive, else -1: k_bvh_leaf leaves such a source out
// of the reach boxes and InterpOp::source_filter never stages it.
__global__ void k_interp_reach(int n, const double* __restrict__ h, int variable_h, double h_fixed, double* __restrict__ reach2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double hj = variable_h ? h[i] : h_fixed;
  reach2[i] = (hj > 0.0 && hj < INFINITY) ? 2.0 * hj : -1.0;
}

// Sort keys of the points: key = 63-bit Morton code of the point in the points' bounding box (21 bits per axis),
// tie = a hash of the coordinate bits (sorted first, stably, so that equal Morton codes fall in a caller-independent order).
__global__ void k_interp_keys(int n, const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ z,
                              const RootBox* __restrict__ rb, uint64_t* __restrict__ key, uint64_t* __restrict__ tie, int* __restrict__ idx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double p[3] = {x[i], y[i], z[i]};
  uint64_t k = 0, t = 0;
  unsigned c[3];
  for (int a = 0; a < 3; ++a) {
    const double ext = rb->mx[a] - rb->mn[a];
    double s = ext > 0.0 ? (p[a] - rb->mn[a]) / ext * 2097152.0 : 0.0;
    s = fmin(fmax(s, 0.0), 2097151.0);
    c[a] = (unsigned)s;
    t = mix64(t ^ (uint64_t)__double_as_longlong(p[a]));
  }
  for (int b = 20; b >= 0; --b)
    k = (k << 3) | (uint64_t)(((c[0] >> b) & 1u) | (((c[1] >> b) & 1u) << 1) | (((c[2] >> b) & 1u) << 2));
  key[i] = k; tie[i] = t; idx[i] = i;
}

struct InterpOp {
  static const bool SYMMETRIC = false;
  static const bool LISTS = false;
  static const bool FUSED = false;
  const InterpArrays& A;
  double* t;                       // tile: INTERP_FIELDS arrays of WALK_TILE doubles
  float4* ft;                      // float copy for the prefilter: position relative to the run's origin, bound on r^2
  const double* wt; int nq; double dq, inv_dq;
  int variable_h; double h_fixed, pi_norm;
  float gplo[3], gphi[3];          // the run's box
  double g0x, g0y, g0z, gd;        // its centre and largest half-extent
  // lane state
  bool live;
  double px, py, pz; float pxf, pyf, pzf;
  double a0, a1, a2, a3, a4, a5, a6;

  __device__ InterpOp(const InterpArrays& a) : A(a) {}

  // could the ball |x - x_j| <= 2 h_j reach the run's box?  (FP64, the run's box is already rounded outward)
  __device__ __forceinline__ bool source_filter(int j) const {
    const double R = A.reach2[j], x = A.x[j], y = A.y[j], z = A.z[j];
    return (R > 0.0) & (x - R <= (double)gphi[0]) & (x + R >= (double)gplo[0]) & (y - R <= (double)gphi[1]) & (y + R >= (double)gplo[1]) &
           (z - R <= (double)gphi[2]) & (z + R >= (double)gplo[2]);
  }
  __device__ __forceinline__ void stage(int s, int j) {
    const double hj = variable_h ? A.h[j] : h_fixed;
    const double x = A.x[j], y = A.y[j], z = A.z[j];
    t[0 * WALK_TILE + s] = x; t[1 * WALK_TILE + s] = y; t[2 * WALK_TILE + s] = z;
    t[3 * WALK_TILE + s] = hj; t[4 * WALK_TILE + s] = pi_norm * ((hj * hj) * hj);      // the density pass's n3 (F:125 | V:139)
    t[5 * WALK_TILE + s] = A.m[j];
    t[6 * WALK_TILE + s] = A.vx[j]; t[7 * WALK_TILE + s] = A.vy[j]; t[8 * WALK_TILE + s] = A.vz[j];
    t[9 * WALK_TILE + s] = A.u[j]; t[10 * WALK_TILE + s] = A.alpha[j];
    // Prefilter bound.  The run-relative float coordinates of a point and of a member are within gd and gd + 2h of the
    // origin, so each carries at most 2^-24 of that, and the float difference 2^-24 of at most 2h: the float distance
    // exceeds the exact one by at most sqrt(3) 2^-24 (2 gd + 4 h) < 4e-7 (gd + 2h).  A member therefore has
    // r_float <= b = 2h + 4e-7 (gd + 2h), and the fmaf sum of squares adds < 1e-6 relative: b^2 (1 + 1e-4) rounded up
    // never drops one.  (Infinite or NaN float coordinates compare false and pass to the exact test.)
    const double b = 2.0 * hj + 4e-7 * (gd + 2.0 * hj);
    ft[s] = make_float4((float)(x - g0x), (float)(y - g0y), (float)(z - g0z), __double2float_ru(b * b * 1.0001));
  }
  __device__ __forceinline__ void consume(int count) {
    unsigned mask = 0;
    if (live) {
#pragma unroll 4
      for (int k = 0; k < count; ++k) {
        const float4 sj = ft[k];
        const float dx = pxf - sj.x, dy = pyf - sj.y, dz = pzf - sj.z;
        mask |= (fmaf(dx, dx, fmaf(dy, dy, dz * dz)) > sj.w ? 0u : 1u) << k;
      }
    }
    // survivors in tile order, one accumulator per column: a point's sums follow the walk's source order
    while (mask) {
      const int k = __ffs(mask) - 1; mask &= mask - 1;
      term(k);
    }
  }
  __device__ __forceinline__ void term(int k) {
    // |x - x_j| / h_j with correctly rounded operations and no contraction: membership is the definition's, bit for bit
    const double dx = __dsub_rn(px, t[0 * WALK_TILE + k]), dy = __dsub_rn(py, t[1 * WALK_TILE + k]), dz = __dsub_rn(pz, t[2 * WALK_TILE + k]);
    const double r2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    const double q = __ddiv_rn(__dsqrt_rn(r2), t[3 * WALK_TILE + k]);
    if (q <= 2.0) {
      const double w = table_lerp1(wt, nq, dq, inv_dq, q);
      const double mw = t[5 * WALK_TILE + k] * (w / t[4 * WALK_TILE + k]);
      a0 += mw;
      a1 += mw * t[6 * WALK_TILE + k]; a2 += mw * t[7 * WALK_TILE + k]; a3 += mw * t[8 * WALK_TILE + k];
      a4 += mw * t[9 * WALK_TILE + k]; a5 += mw * t[10 * WALK_TILE + k];
      a6 += 1.0;
    }
  }
};

// One warp per run of 32 sorted points (lane = point).  perm[i] = the point's index in the chunk; raw[k * n + perm[i]].
// dynamic shared memory: [table: nq + 1 doubles, padded to even][per warp: tile][per warp: walk state]
__global__ void __launch_bounds__(INTERP_WARPS * 32)
k_interpolate(int n, const double* __restrict__ qx, const double* __restrict__ qy, const double* __restrict__ qz, const int* __restrict__ perm,
              const int2* __restrict__ groups, InterpArrays A, const BvhBox* __restrict__ box, const __grid_constant__ BvhInfo bi,
              const double* __restrict__ g_wt, DevParams P, double* __restrict__ raw) {
  extern __shared__ double smem[];
  const int nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* wt = smem;
  double* tiles = wt + (P.nq + 1) + ((P.nq + 1) & 1);
  unsigned* ws = reinterpret_cast<unsigned*>(tiles + (size_t)nwarp * INTERP_WARP_DOUBLES);
  for (int i = threadIdx.x; i <= P.nq; i += blockDim.x) wt[i] = g_wt[i];
  __syncthreads();
  const int run = blockIdx.x * nwarp + warp;
  if (run * 32 >= n) return;
  double* tile = tiles + (size_t)warp * INTERP_WARP_DOUBLES;
  unsigned* stack = ws + (size_t)warp * WALK_WS;
  unsigned* cq = stack + WALK_STACK;
  const int i = run * 32 + lane;
  const bool live = i < n;
  const int o = live ? perm[i] : 0;
  InterpOp op(A);
  op.t = tile; op.ft = reinterpret_cast<float4*>(tile + INTERP_FIELDS * WALK_TILE);
  op.wt = wt; op.nq = P.nq; op.dq = P.dq; op.inv_dq = P.inv_dq;
  op.variable_h = P.variable_h; op.h_fixed = P.h_fixed; op.pi_norm = P.pi_norm;
  op.live = live;
  op.px = live ? qx[o] : 0.0; op.py = live ? qy[o] : 0.0; op.pz = live ? qz[o] : 0.0;
  BvhBox g;
  {
    const double p[3] = {op.px, op.py, op.pz};
    for (int k = 0; k < 3; ++k) {
      g.plo[k] = warp_minf(live ? __double2float_rd(p[k]) : INFINITY);
      g.phi[k] = warp_maxf(live ? __double2float_ru(p[k]) : -INFINITY);
      g.rlo[k] = g.plo[k]; g.rhi[k] = g.phi[k];
      op.gplo[k] = g.plo[k]; op.gphi[k] = g.phi[k];
    }
  }
  op.g0x = 0.5 * ((double)g.plo[0] + (double)g.phi[0]); op.g0y = 0.5 * ((double)g.plo[1] + (double)g.phi[1]); op.g0z = 0.5 * ((double)g.plo[2] + (double)g.phi[2]);
  op.gd = 0.5 * fmax(fmax((double)g.phi[0] - (double)g.plo[0], (double)g.phi[1] - (double)g.plo[1]), (double)g.phi[2] - (double)g.plo[2]);
  op.pxf = (float)(op.px - op.g0x); op.pyf = (float)(op.py - op.g0y); op.pzf = (float)(op.pz - op.g0z);
  op.a0 = op.a1 = op.a2 = op.a3 = op.a4 = op.a5 = op.a6 = 0.0;
  neighbour_walk(op, g, groups, box, bi, stack, cq);
  if (live) {
    raw[0 * (size_t)n + o] = op.a0; raw[1 * (size_t)n + o] = op.a1; raw[2 * (size_t)n + o] = op.a2; raw[3 * (size_t)n + o] = op.a3;
    raw[4 * (size_t)n + o] = op.a4; raw[5 * (size_t)n + o] = op.a5; raw[6 * (size_t)n + o] = op.a6;
  }
}

// raw sums -> the output columns: the means divide by rho after the ranks' sums are added (the same bits on every rank)
__global__ void k_interp_finish(int n, double* __restrict__ raw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double rho = raw[i];
  for (int k = 1; k <= 5; ++k) raw[(size_t)k * n + i] = rho != 0.0 ? raw[(size_t)k * n + i] / rho : 0.0;
}
