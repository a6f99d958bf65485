// sph_gravat.cuh — the gravitational potential and acceleration at caller-given points (sph_gravity_at, include/sph_b200.h).
//
// Point k is a gas particle of smoothing length h_k at x_k that adds nothing to the tree: the reference's Barnes-Hut walk
// (particle_gravforce_one, F:264-290 | V:285-311) with the opening test `size/dist < theta .or. no children`,
// dist = sqrt(|x - COM|^2 + soft), soft = 0.001 h_fixed (0.001 h_k under SPH_FLAG_SOFT_USES_HI), kernel length
// h' = h_fixed (F:280) | h_k (V:301).  Over the accepted nodes:
//   phi = G sum M phi(dist / h') / h'      (phi = soft_potential of sph_conserved.cuh; no node is left out)
//   g   = -G sum M g(dist / h') (x - COM) / dist^3      (the reference's term, g = the gravity table, 1 beyond q = 2)
// and the number of accepted nodes.  The sinks' direct terms (unsoftened, F:572) are added per point after the walk.
//
// One thread per point over the gravity walk layout (WNode), as k_conserved_partial walks it: the opening test is the
// reference's arithmetic without contraction, so the accepted node set is the reference's own.  The points are sorted
// by k_interp_keys' Morton order first, so the threads of a warp walk neighbouring points.
//
// Under the Morton domains the layout is [top | local | LET]; the LET covers this rank's own domain only, so the walk
// never enters it.  owner[v] of a top slot is the rank that holds the complete node, -1 for a cell straddling ranks.
// An accepted top node is added only on its owner (a straddling cell on rank 0); an opened one is descended only on its
// owner (a straddling cell on every rank).  Local slots belong to this rank.  Summed over the ranks this is the
// single-rank node set: top slots and local nodes are bit copies of the single-rank nodes.
#pragma once
#include "sph_common.cuh"
#include "sph_walk.cuh"
#include "sph_conserved.cuh"

#define GRAVAT_COLS 9              // SPH_GRAVAT_COUNT output columns
#define GRAVAT_RAW 5               // columns the walk writes (summed over the ranks): phi, gx, gy, gz, accepted
#define GRAVAT_THREADS 128

// raw[c * n + perm[t]], c < GRAVAT_RAW; q: the points (x, y, z, h) at q + k * cap; h column unused without qh
__global__ void __launch_bounds__(GRAVAT_THREADS)
k_gravity_at(int n, const double* __restrict__ q, size_t cap, int with_h, const int* __restrict__ perm, DevParams P,
             const WNode* __restrict__ wn, const double* __restrict__ gt, int n_top, const int* __restrict__ owner, int rank,
             double* __restrict__ raw) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int o = perm[t];
  const double xi = q[o], yi = q[cap + o], zi = q[2 * cap + o];
  const double hk = with_h ? q[3 * cap + o] : P.h_fixed;
  const double hp = P.variable_h ? hk : P.h_fixed;                            // F:280 | V:301
  const double inv_h = 1.0 / hp;
  const double soft = P.soft_hi ? 0.001 * hk : 0.001 * P.h_fixed;            // F:275 | V:296 | T:298
  double phi = 0.0, gx = 0.0, gy = 0.0, gz = 0.0, acc = 0.0;
  int2 stk[SPH_KEY_LEVELS2];
  int sp = 0, cur = 0, end = 1;                                               // the root block: slot 0 alone
  for (;;) {
    const int v = cur++;
    const int own = v < n_top ? owner[v] : rank;
    if (own < 0 || own == rank) {                                             // another rank's complete node: its owner adds it
      const WNode g = wn[v];
      const double dx = xi - g.cx, dy = yi - g.cy, dz = zi - g.cz;
      const double d2 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)), soft);   // F:275
      const double dist = __dsqrt_rn(d2);
      if (g.nchild == 0 || __ddiv_rn(g.size, dist) < P.theta) {               // F:278
        if (own == rank || rank == 0) {                                       // a straddling cell is added once, on rank 0
          acc += 1.0;
          if (g.m > 0.0 && dist > 0.0) {                                      // F:279
            const double qq = dist * inv_h;
            const double w = qq <= 2.0 ? table_lerp1(gt, P.nq, P.dq, P.inv_dq, qq) : 1.0;        // F:129-146
            phi += g.m * (soft_potential(qq) * inv_h);
            const double f = P.G * g.m * w / (d2 * dist);                     // F:281
            gx -= f * dx; gy -= f * dy; gz -= f * dz;
          }
        }
      } else {
        if (cur < end) stk[sp++] = make_int2(cur, end);
        cur = g.child; end = g.child + g.nchild;
      }
    }
    if (cur == end) {                                                          // block done: a stacked level always has siblings left
      if (sp == 0) break;
      --sp; cur = stk[sp].x; end = stk[sp].y;
    }
  }
  raw[o] = P.G * phi; raw[(size_t)n + o] = gx; raw[2 * (size_t)n + o] = gy; raw[3 * (size_t)n + o] = gz; raw[4 * (size_t)n + o] = acc;
}

// after the ranks' sums: accepted moves to column 8, the sink columns 4..7 are taken (the same bits on every rank).
// Sinks with m_s > 0 and |x - x_s| > 0 only: the dummy zero-mass sink and a point on a sink add nothing.
__global__ void k_gravity_at_sinks(int n, const double* __restrict__ q, size_t cap, DevParams P, int n_sink, SinkArrays S,
                                   double* __restrict__ raw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double xi = q[i], yi = q[cap + i], zi = q[2 * cap + i];
  double phi = 0.0, gx = 0.0, gy = 0.0, gz = 0.0;
  for (int s = 0; s < n_sink; ++s) {
    const double ms = S.m[s];
    const double vx = xi - S.x[s], vy = yi - S.y[s], vz = zi - S.z[s];
    const double dr = sqrt(vx * vx + vy * vy + vz * vz);
    if (!(ms > 0.0) || !(dr > 0.0)) continue;
    const double d3 = dr * dr * dr;
    phi -= P.G * ms / dr;
    gx -= ms * (P.G * vx / d3); gy -= ms * (P.G * vy / d3); gz -= ms * (P.G * vz / d3);      // F:572-574
  }
  raw[8 * (size_t)n + i] = raw[4 * (size_t)n + i];
  raw[4 * (size_t)n + i] = phi; raw[5 * (size_t)n + i] = gx; raw[6 * (size_t)n + i] = gy; raw[7 * (size_t)n + i] = gz;
}
