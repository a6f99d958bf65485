// sph_conserved.cuh — energy / momentum / angular-momentum sums of the resident state (on demand, not per step).
//
// The reference computes none of these (no energy or momentum bookkeeping anywhere in SUMMER_SPH.f90); the
// definitions are this build's own (SURVEY.md §8(c): "E = sum 1/2 m v^2 + sum m u + E_grav and L"), chosen to
// match the forces the reference applies:
//   E_kin   = sum_gas 1/2 m v.v + sum_sinks 1/2 m v.v
//   E_int   = sum_gas m u
//   E_gg    = 1/2 sum_i m_i Phi_i,  Phi_i = G sum over the nodes the reference's Barnes-Hut walk accepts for
//             particle i (same opening test, same softened distance: SUMMER_SPH.f90:273-279 | Variable.f90:294-300)
//             of M_node phi(dist / h) / h, h = `smoothing` (F) | h_i (V); i's own single-particle leaf is left out.
//             phi is the cubic-spline softened point-mass potential whose radial derivative is the reference's
//             g(q) / q^2 (the polynomials of init_grav_kernel_table, F:91,94), -1/q beyond q = 2.
//   E_sink  = -G sum_sinks sum_gas m_s m_j / r  -  G sum_{sink pairs} m_a m_b / r     (unsoftened, F:559-591)
//   P, L    = sum m v, sum m x cross v over gas and sinks (+ the sinks' spin when SPH_FLAG_SINK_MERGE_SPIN keeps it); M = total mass.
// The walk is one thread per particle over the gravity walk layout (WNode): a diagnostic called a few times per run,
// not a hot kernel.
#pragma once
#include "sph_common.cuh"
#include "sph_integrate.cuh"

#define CONS_FIELDS 12             // sph_conserved() output slots (include/sph_b200.h)
#define CONS_SUMS 11               // per-thread sums: ekin eint px py pz lx ly lz mass egg esg
#define CONS_THREADS 128
#define CONS_MAX_BLOCKS 2368       // 148 SMs x 16 resident blocks of 128 threads

// phi(q): d phi / d q = g(q) / q^2 with g from F:91 (q <= 1), F:94 (1 < q <= 2), 1 beyond; phi -> -1/q.
__host__ __device__ inline double soft_potential(double q) {
  if (q < 1.0) {
    const double q2 = q * q;
    return -1.4 + q2 * (2.0 / 3.0 + q2 * (-0.3 + 0.1 * q));
  }
  if (q < 2.0) {
    const double q2 = q * q;
    return -1.6 + 1.0 / (15.0 * q) + q2 * (4.0 / 3.0 - q + 0.3 * q2 - (1.0 / 30.0) * q2 * q);
  }
  return -1.0 / q;
}

// Row of the particle of every single-particle leaf of the local tree in the walk layout, -1 for every other slot
// (internal and depth-limited childless nodes).  Rows, not numbers: what the walk leaves out is the particle itself,
// whatever numbers the host gave the rows.  wbase: first slot of the local tree (0; DD_TOP_CAP under domains).
__global__ void k_conserved_wpart(int n_nodes, const int* __restrict__ node_part, const int* __restrict__ widx, int wbase,
                                  int* __restrict__ wpart) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_nodes) return;
  const int w = widx[v];
  if (w >= 0) wpart[wbase + w] = node_part[v] >= 0 ? node_part[v] : -1;
}

// Walk layout: root at slot 0, the children of a node at [child, child + nchild), nchild == 0 accepted whole (leaves and
// depth-limited childless nodes, F:182).  Children are visited in block order, which is the octree's preorder
// (k_oct_widx assigns each block in child-chain order), so every particle sums the nodes of the preorder walk with skip
// pointers in the same order and with the same bits.  Under domains the layout is [top | local | LET]: top nodes are
// assembled in k_oct_up's order and LET nodes are bit copies, so each particle's term equals its single-rank term.  A
// LET node whose children were not pulled still holds the owner's child index; it is never opened here, because the
// LET pulls the children of every node that passes dd_may_open (soft = 0 plus a margin against the domain's position
// boxes), a superset of the nodes this test (soft > 0) opens.
// wpart: k_conserved_wpart under the layout (plus the top slots that copy one of this rank's single-particle leaves;
// -1 on the LET slots: a remote particle is never i).
// Stack: one (cursor, end) pair per opened level; the pair being walked stays in registers and a level is pushed only
// when siblings remain (so one pop always yields a node: every trip of the loop visits one).  A node is opened only
// above lmax <= SPH_KEY_LEVELS2, so at most 42 pairs are stacked.  The walk is bound by the latency of its dependent node
// loads: 8 resident blocks (64 registers, a few accumulator spills) walk as fast as the preorder walk did; at the
// 80 registers the compiler picks by itself (6 blocks) the 16M call is 1.27x slower on a B200.
__global__ void __launch_bounds__(CONS_THREADS, 8)
k_conserved_partial(int n, DevParams P, StateArrays s, const WNode* __restrict__ wn, const int* __restrict__ wpart,
                    int n_sink, SinkArrays S, double* __restrict__ partial) {
  double acc[CONS_SUMS];
#pragma unroll
  for (int k = 0; k < CONS_SUMS; ++k) acc[k] = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double xi = s.x[i], yi = s.y[i], zi = s.z[i];
    const double vx = s.vx[i], vy = s.vy[i], vz = s.vz[i];
    const double mi = s.m[i];
    acc[0] += 0.5 * mi * (vx * vx + vy * vy + vz * vz);
    acc[1] += mi * s.u[i];
    acc[2] += mi * vx; acc[3] += mi * vy; acc[4] += mi * vz;
    acc[5] += mi * (yi * vz - zi * vy); acc[6] += mi * (zi * vx - xi * vz); acc[7] += mi * (xi * vy - yi * vx);
    acc[8] += mi;
    // gas-gas potential over the reference's accepted node set
    const double hi = P.variable_h ? s.h[i] : P.h_fixed;
    const double inv_h = 1.0 / hi;
    const double soft = P.soft_hi ? 0.001 * hi : 0.001 * P.h_fixed;          // F:275 | V:296 | T:298
    double phi = 0.0;
    int2 stk[SPH_KEY_LEVELS2];
    int sp = 0, cur = 0, end = 1;                                              // the root block: slot 0 alone
    for (;;) {
      const int v = cur++;
      const WNode g = wn[v];
      const double dx = xi - g.cx, dy = yi - g.cy, dz = zi - g.cz;
      const double d2 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)), soft);   // F:275
      const double dist = __dsqrt_rn(d2);
      if (g.nchild == 0 || __ddiv_rn(g.size, dist) < P.theta) {                // F:278
        if (g.m > 0.0 && dist > 0.0 && wpart[v] != i) phi += g.m * (soft_potential(dist * inv_h) * inv_h);
      } else {
        if (cur < end) stk[sp++] = make_int2(cur, end);
        cur = g.child; end = g.child + g.nchild;
      }
      if (cur == end) {                                                        // block done: a stacked level always has siblings left
        if (sp == 0) break;
        --sp; cur = stk[sp].x; end = stk[sp].y;
      }
    }
    acc[9] += 0.5 * mi * (P.G * phi);
    double es = 0.0;
    for (int j = 0; j < n_sink; ++j) {
      const double ms = S.m[j];
      if (!(ms > 0.0)) continue;                                               // the dummy sink of F:698-707 carries no mass
      const double ax = xi - S.x[j], ay = yi - S.y[j], az = zi - S.z[j];
      es -= ms / sqrt(ax * ax + ay * ay + az * az);
    }
    acc[10] += P.G * mi * es;
  }
  __shared__ double sm[CONS_THREADS / 32][CONS_SUMS];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < CONS_SUMS; ++k) {
    const double t = warp_sum(acc[k]);
    if (l == 0) sm[w][k] = t;
  }
  __syncthreads();
  if (threadIdx.x < CONS_SUMS) {
    double t = 0.0;
    for (int q = 0; q < CONS_THREADS / 32; ++q) t += sm[q][threadIdx.x];
    partial[(size_t)blockIdx.x * CONS_SUMS + threadIdx.x] = t;
  }
}

// one warp: the CONS_SUMS totals of `nblocks` partials (lane-strided, then a warp sum: a fixed order); lane 0 writes tot
__device__ __forceinline__ void cons_fold(int nblocks, const double* __restrict__ partial, double* tot) {
  const int l = threadIdx.x;
  for (int k = 0; k < CONS_SUMS; ++k) {
    double t = 0.0;
    for (int b = l; b < nblocks; b += 32) t += partial[(size_t)b * CONS_SUMS + k];
    t = warp_sum(t);
    if (l == 0) tot[k] = t;
  }
}

// domains: one rank's CONS_SUMS totals (all-gathered, then folded by k_conserved_final like block partials)
__global__ void k_conserved_fold(int nblocks, const double* __restrict__ partial, double* __restrict__ out) { cons_fold(nblocks, partial, out); }

// one warp: fold the block partials (or, under domains, the ranks' totals), add the sinks' own terms once, write the
// CONS_FIELDS outputs
__global__ void k_conserved_final(int nblocks, const double* __restrict__ partial, DevParams P, int n_sink, SinkArrays S,
                                  const double* __restrict__ spin, double* __restrict__ out) {
  __shared__ double tot[CONS_SUMS];
  const int l = threadIdx.x;
  cons_fold(nblocks, partial, tot);
  __syncwarp();
  if (l != 0) return;
  double ekin = tot[0], px = tot[2], py = tot[3], pz = tot[4], lx = tot[5], ly = tot[6], lz = tot[7], mass = tot[8];
  double ess = 0.0;
  for (int a = 0; a < n_sink; ++a) {
    const double ma = S.m[a];
    if (!(ma > 0.0)) continue;
    const double x = S.x[a], y = S.y[a], z = S.z[a], vx = S.vx[a], vy = S.vy[a], vz = S.vz[a];
    ekin += 0.5 * ma * (vx * vx + vy * vy + vz * vz);
    px += ma * vx; py += ma * vy; pz += ma * vz;
    lx += ma * (y * vz - z * vy); ly += ma * (z * vx - x * vz); lz += ma * (x * vy - y * vx);
    if (spin) { lx += spin[a]; ly += spin[SPH_MAX_SINKS + a]; lz += spin[2 * SPH_MAX_SINKS + a]; }   // SPH_FLAG_SINK_MERGE_SPIN
    mass += ma;
    for (int b = 0; b < a; ++b) {
      const double mb = S.m[b];
      if (!(mb > 0.0)) continue;
      const double dx = x - S.x[b], dy = y - S.y[b], dz = z - S.z[b];
      ess -= P.G * ma * mb / sqrt(dx * dx + dy * dy + dz * dz);
    }
  }
  const double esink = tot[10] + ess;
  out[0] = ekin; out[1] = tot[1]; out[2] = tot[9] + esink;
  out[3] = px; out[4] = py; out[5] = pz; out[6] = lx; out[7] = ly; out[8] = lz;
  out[9] = mass; out[10] = tot[9]; out[11] = esink;
}
