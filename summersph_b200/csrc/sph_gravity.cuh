// sph_gravity.cuh — Barnes-Hut gravity walk + direct sink gravity.
//
// Replaces particle_gravforces / particle_gravforce_one (SUMMER_SPH.f90:249-290 | Variable.f90:270-311)
// and sink_gravforces (F:559-591 | V:691-726).
//
// The reference's opening decision is per particle: `size/dist < theta .or. no children` with
// dist = sqrt(|x - COM|^2 + 0.001*smoothing) (F:275-278), and every accepted-node set stays identical to it.
// What changes is who decides.  One warp owns a run of 32 Morton-consecutive particles (lane = particle; the runs
// restart at every 64th walk group, see k_seg_chunks) and keeps a stack of (node, lane mask) entries in shared
// memory.  Each trip pops up to 32 entries and classifies them lane-parallel against the run's bounding box
// (lane = node, one coalesced 48-byte load each, child blocks are contiguous in the walk layout) - in FP32 on
// box-relative coordinates with 3e-5 margins, since anything uncertain is simply "mixed":
//   * every particle of the run accepts (even the closest point of the box passes the test, or the node is
//     childless)                                   -> interaction list, mask unchanged;
//   * every particle opens (even the farthest point fails it)  -> push the child block, mask unchanged;
//   * otherwise the node is mixed: each particle in the mask runs the reference's own test (FP32 screen, then
//     the FP64 form with a 2e-12 guard band, then the exact uncontracted arithmetic inside the band); the node's
//     lane collects the two ballots: the accepting lanes become the list entry's mask, the opening lanes the
//     mask of the pushed children.  One list insert and one child push per trip serve all three classes.
// The interaction list (COM, G*M, mask) is evaluated in batches with lane = particle (18 FP64 instructions per
// entry, two entries in flight per lane), node data read once per run instead of once per particle.  The
// accumulation order differs from the reference's recursion order (rounding-level only).
#pragma once
#include "sph_common.cuh"
#include "sph_walk.cuh"

struct SinkArrays { double *x, *y, *z, *vx, *vy, *vz, *m, *radius, *ax, *ay, *az; };

#ifndef GW_WARPS
#define GW_WARPS 20         // warps per block
#endif
#ifndef GW_ILP
#define GW_ILP 2            // interaction-list entries in flight per lane
#endif
#define GW_STACK 384        // (node, mask) entries per warp in shared memory
#ifndef GW_LIST
#define GW_LIST  64         // interaction-list entries per warp (evaluated when fewer than 32 slots are left)
#endif
#define GW_SPILL 8192       // per-warp overflow entries in global memory (never reached in practice; loud if it is)


#ifdef GW_STATS       // developer build: what the walk does per launch (scripts/build_variant.sh stats -DGW_STATS)
__device__ unsigned long long gw_stats[16];
#define GWS(slot, v) do { const unsigned long long v_ = (unsigned long long)(v); if (lane == 0) gws[slot] += v_; } while (0)      // v may hold a warp vote: evaluated by every lane
#else
#define GWS(slot, v) do {} while (0)
#endif

struct GravWarpSmem {
  int2     stack[GW_STACK];
  double2  lxy[GW_LIST], lzg[GW_LIST];     // (cx, cy), (cz, G*M)
  unsigned lmask[GW_LIST];
  double   mcx[32], mcy[32], mcz[32], msize[32], mlo[32], mhi[32];   // mixed nodes of the current trip: COM, size, d2 band of the cheap FP64 test
  float4   mf[32];                                                   // the same nodes for the FP32 screen: COM relative to the run's origin, size^2 / theta^2
                                                                     //   (NaN: the screen cannot decide for this run, every particle takes the FP64 test)
  unsigned mmask[32];
  double   nacc[3][32];                                              // full walk: the near sums of the lanes between list evaluations (registers are short there)
  double   hpar[3][32];                                              // full walk: 1/h, 4 h^2, hc2 of the lanes (only the near entries need them)
  int      lidx[GW_LIST];                                            // node index of every list entry (recorded with the near pairs)
  int      ncnt[32];                                                 // full walk: near pairs recorded so far, per lane
};

// 1/sqrt(x): MUFU seed (~2^-20) + one Halley step (cubic: ~2^-58), x > 0
__device__ __forceinline__ double fast_rsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double e = fma(-(x * y), y, 1.0);
  const double t = fma(0.375, e, 0.5);
  return fma(y * e, t, y);
}

// one list entry against one particle: a -= G M g(dist/h) dir / dist^3                  F:279-281 | F:129-146
// h2x4 = 4 h^2: dist/h <= 2 is decided on the squares (g(2) = 1 and the table is continuous there, so which side
// of the branch a borderline pair takes changes the term by rounding only); W = 1 beyond it needs no multiply.
// KIND 0: far-list entry (d2 > hc2 for every particle of the run, decided at listing): W = 1, far sum.
// KIND 1: near-list entry of the full walk: the term joins the near sum when d2 <= hc2, else the far sum.
// KIND 2: near-only walk: only the terms with d2 <= hc2 (the far sum is the stored one).
// KIND 3: a recorded near pair (d2 <= hc2 held when the full walk recorded it): near sum, no test.
// KIND 4: near-list entry of a full walk that stores nothing: one sum, like KIND 0 but with the softening test.
template <int KIND>
__device__ __forceinline__ bool grav_term(const double2 a, const double2 b, const bool on, const double xi, const double yi,
                                          const double zi, const double inv_h, const double h2x4, const double hc2, const double soft, const double* __restrict__ gt,
                                          const int nq, const double dq, const double inv_dq, double& gx, double& gy, double& gz,
                                          double& nx, double& ny, double& nz) {
  const double dx = xi - a.x, dy = yi - a.y, dz = zi - b.x;                  // F:274
  const double d2 = fma(dx, dx, fma(dy, dy, fma(dz, dz, soft)));
  const double rs = fast_rsqrt(d2);                                          // F:279: M > 0 is checked when the entry is listed; d2 >= soft > 0
  double gm = b.y;
  if (KIND != 0) { if (d2 <= h2x4) gm *= table_lerp1(gt, nq, dq, inv_dq, (d2 * rs) * inv_h); }      // far entries: d2 > 4 h^2 for every particle of the run (decided at listing)
  const double f = gm * (rs * rs * rs);
  if (KIND == 0 || KIND == 4) { if (on) { gx = fma(-f, dx, gx); gy = fma(-f, dy, gy); gz = fma(-f, dz, gz); } return false; }
  else {
    const bool nr = on && (KIND == 3 || d2 <= hc2);
    if (nr) { nx = fma(-f, dx, nx); ny = fma(-f, dy, ny); nz = fma(-f, dz, nz); }
    if (KIND == 1) { if (on && !nr) { gx = fma(-f, dx, gx); gy = fma(-f, dy, gy); gz = fma(-f, dz, gz); } }
    return nr;
  }
}

// Far-field reuse.  Evaluation A of a loop body sees the positions, masses, sinks and tree of the previous body's
// evaluation B (F:894 after F:905-912: the second kick moves nothing), and the reference's opening test does not
// involve h (soft = 0.001 x the fixed smoothing, F:275), so every accepted (node, particle) pair and its distance are
// the same; only h changed (calc_smoothing, V:1152), and h enters a term only through g(dist/h) for dist < 2 h
// (F:138-141).  The full walk (MODE 0) therefore adds the terms with d2 <= hc2 = 4 (GW_HCUT h)^2 and all the others
// apart, and stores the far sum of the tree terms (the direct sink terms are taken anew in every evaluation: sinks move,
// grow and, with a mass that is not a power of two, shift by an ulp in every accretion pass, F:497-501); while the tree and
// "4 h^2 <= hc2 for every particle" stand (checked on the device at the end of every step), the next evaluation is the near-only walk
// (MODE 1): subtrees whose cell cannot hold a centre of mass within sqrt(max hc2) of the run's box are dropped at
// classification, the opening decisions on the others are the full walk's own, the near terms are evaluated with the
// new h and added to the stored far sum.  Same terms as a full walk, summed in another order (rounding level).
// Only ~10 % of the lane slots of the near entries hold such a term (an entry is near for the run's box, a term for one
// particle), so the full walk also records, per particle, the node of every term it added to the near sum
// (list[run][slot][lane], `slots` per lane; ~70 per particle), and the next evaluation is k_gravity_near: lane =
// particle, one gathered node per trip, every lane slot a needed term, no walk.  A run in which some lane needs more
// slots is flagged (ovf) and served by the near-only walk instead.
#ifndef GW_HCUT
#define GW_HCUT 1.1
#endif
struct FarField { double *fx, *fy, *fz; const double* hc2; int store; int* list; int* cnt; unsigned char* ovf; int slots; int* n_ovf; };
__global__ void k_far_hcut(int n, DevParams P, const double* __restrict__ h, double factor, double* __restrict__ hc2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double hc = factor * (P.variable_h ? h[i] : P.h_fixed);
  hc2[i] = 4.0 * hc * hc;
}
// end of a step: may the next evaluation keep the stored far sums?  Not when some h grew beyond its cutoff (or is NaN)
__global__ void k_far_check(int n, DevParams P, const double* __restrict__ h, const double* __restrict__ hc2, int* __restrict__ far_bad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool bad = false;
  if (i < n && P.variable_h) { const double hi = h[i]; bad = !(4.0 * hi * hi <= hc2[i]); }
  if (__any_sync(FULL_MASK, bad) && (threadIdx.x & 31) == 0) atomicOr(far_bad, 1);
}

// direct sink <-> gas (unsoftened) F:567-576 for the 32 particles of one run: the gas side goes into (gx, gy, gz), the
// sink side into the run's slot of sink_partial (one warp sum per sink, no block barrier)
__device__ __forceinline__ void sink_terms(const DevParams& P, const SinkArrays& S, int n_sink, bool live, double xi, double yi, double zi, double mi,
                                           double& gx, double& gy, double& gz, double* __restrict__ run_partial) {
  const int lane = threadIdx.x & 31;
  for (int s = 0; s < n_sink; ++s) {
    const double vx_ = xi - S.x[s], vy_ = yi - S.y[s], vz_ = zi - S.z[s];
    const double dr = sqrt(vx_ * vx_ + vy_ * vy_ + vz_ * vz_);
    const double d3 = dr * dr * dr;
    double wx = P.G * vx_ / d3, wy = P.G * vy_ / d3, wz = P.G * vz_ / d3;    // F:572
    const double ms = S.m[s];
    double px = 0.0, py = 0.0, pz = 0.0;
    if (live) {
      gx -= ms * wx; gy -= ms * wy; gz -= ms * wz;                             // F:574
      px = mi * wx; py = mi * wy; pz = mi * wz;                               // F:573
    }
    px = warp_sum(px); py = warp_sum(py); pz = warp_sum(pz);
    if (lane == 0) { double* o = run_partial + (size_t)s * 3; o[0] = px; o[1] = py; o[2] = pz; }
  }
}

#ifdef SCREEN_AUDIT
// the reference's opening test, F:274-278, without contraction: accept the node
__device__ __forceinline__ bool audit_mac_accept(double dx, double dy, double dz, double soft, double size, double theta) {
  const double e2 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)), soft);
  return __ddiv_rn(size, __dsqrt_rn(e2)) < theta;
}
#endif

// dynamic smem: grav table (nq+1 doubles, padded to even) then one GravWarpSmem per warp
// MODE 0: full walk that stores the far sums and records the near pairs; MODE 1: near-only walk on top of the stored far
// sums (see "Far-field reuse" above); MODE 2: full walk that stores nothing (no near / far split: one sum per particle)
template <int MODE>
__global__ void __launch_bounds__(GW_WARPS * 32, 1)
k_gravity(int g_begin, int g_end, const int2* __restrict__ groups, const BvhBox* __restrict__ gbox, DevParams P,
          const WNode* __restrict__ wn, const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ z,
          const double* __restrict__ h, const double* __restrict__ m, const double* __restrict__ g_gt,
          double* __restrict__ ax, double* __restrict__ ay, double* __restrict__ az,
          int do_grav, int n_sink, SinkArrays S, double* __restrict__ sink_partial, WalkCounters* ctr, int* work,
          int2* __restrict__ spill, int* err_flag, FarField F) {
  extern __shared__ __align__(16) double gsm[];
  double* gt = gsm;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  GravWarpSmem& W = reinterpret_cast<GravWarpSmem*>(gsm + (P.nq + 1) + ((P.nq + 1) & 1))[warp];
  for (int i = threadIdx.x; i <= P.nq; i += blockDim.x) gt[i] = g_gt[i];
  __syncthreads();
  int2* myspill = spill + (size_t)(blockIdx.x * (blockDim.x >> 5) + warp) * GW_SPILL;
  const unsigned lt_mask = (1u << lane) - 1u;
  const double theta = P.theta, theta2 = theta * theta, inv_theta2 = 1.0 / theta2;
  unsigned long long n_open = 0, n_acc = 0;
#ifdef GW_STATS
  unsigned long long gws[16] = {};
#endif

  for (;;) {
    int chunk = 0;
    if (lane == 0) chunk = atomicAdd(work, 1);
    chunk = __shfl_sync(FULL_MASK, chunk, 0);
    if (chunk >= g_end) break;
    const int2 tg = groups[chunk];
    const int i = tg.x + lane;
    const bool live = lane < tg.y;
    const double xi = live ? x[i] : 0.0, yi = live ? y[i] : 0.0, zi = live ? z[i] : 0.0;
    const double hi = live ? (P.variable_h ? h[i] : P.h_fixed) : 1.0;
    const double inv_h = 1.0 / hi, h2x4 = 4.0 * hi * hi;
    constexpr bool FULL = MODE != 1, SPLIT = MODE == 0;
    const double hc2 = MODE == 2 ? (live ? h2x4 : 0.0) : (live ? F.hc2[i] : 0.0);      // >= h2x4: the near / far split of the sums
    const double soft = P.soft_hi ? 0.001 * hi : 0.001 * P.h_fixed;          // F:275 | V:296 | T:298
    double gx[GW_ILP], gy[GW_ILP], gz[GW_ILP];
#pragma unroll
    for (int u = 0; u < GW_ILP; ++u) gx[u] = gy[u] = gz[u] = 0.0;
    double nx = 0.0, ny = 0.0, nz = 0.0;                                     // terms with d2 <= hc2
    if (FULL) { W.hpar[0][lane] = inv_h; W.hpar[1][lane] = h2x4; }
    if (SPLIT) { W.nacc[0][lane] = 0.0; W.nacc[1][lane] = 0.0; W.nacc[2][lane] = 0.0; W.hpar[2][lane] = hc2; W.ncnt[lane] = 0; }
    if (MODE == 1 && F.list && !F.ovf[chunk]) continue;                      // near-only walk behind k_gravity_near: only the runs whose lists overflowed

    // The list is filled from both ends: far entries (no particle of the run lies within 2 h of the node: W = 1, F:138-141,
    // no softening test at all) from slot 0 upwards, the others from the last slot downwards.
    auto evaluate_list = [&](int nfar, int nnear) {
      int k = 0;
      if (FULL) {
        for (; k + GW_ILP <= nfar; k += GW_ILP) {          // GW_ILP independent chains per trip
#pragma unroll
          for (int u = 0; u < GW_ILP; ++u)
            grav_term<0>(W.lxy[k + u], W.lzg[k + u], (W.lmask[k + u] >> lane) & 1u, xi, yi, zi, 0.0, 0.0, 0.0, soft, gt, P.nq, P.dq, P.inv_dq, gx[u], gy[u], gz[u], nx, ny, nz);
        }
        for (; k < nfar; ++k) grav_term<0>(W.lxy[k], W.lzg[k], (W.lmask[k] >> lane) & 1u, xi, yi, zi, 0.0, 0.0, 0.0, soft, gt, P.nq, P.dq, P.inv_dq, gx[0], gy[0], gz[0], nx, ny, nz);
        if (nnear == 0) return;
      }
      constexpr int NK = MODE == 0 ? 1 : MODE == 1 ? 2 : 4;
      const double e_inv_h = FULL ? W.hpar[0][lane] : inv_h, e_h2x4 = FULL ? W.hpar[1][lane] : h2x4, e_hc2 = SPLIT ? W.hpar[2][lane] : hc2;
      if (SPLIT) { nx = W.nacc[0][lane]; ny = W.nacc[1][lane]; nz = W.nacc[2][lane]; }
      const bool rec = SPLIT && F.list != nullptr;                           // record the node of every term that joins the near sum
      int nc = rec ? W.ncnt[lane] : 0;
      int* const lst = rec ? F.list + ((size_t)chunk * F.slots) * 32 + lane : nullptr;
      k = GW_LIST - nnear;
      for (; k + GW_ILP <= GW_LIST; k += GW_ILP) {
        bool hit[GW_ILP];
#pragma unroll
        for (int u = 0; u < GW_ILP; ++u)
          hit[u] = grav_term<NK>(W.lxy[k + u], W.lzg[k + u], (W.lmask[k + u] >> lane) & 1u, xi, yi, zi, e_inv_h, e_h2x4, e_hc2, soft, gt, P.nq, P.dq, P.inv_dq, gx[u], gy[u], gz[u], nx, ny, nz);
        if (rec) {
#pragma unroll
          for (int u = 0; u < GW_ILP; ++u) if (hit[u]) { if (nc < F.slots) lst[(size_t)nc * 32] = W.lidx[k + u]; ++nc; }
        }
      }
      for (; k < GW_LIST; ++k) {
        const bool hit = grav_term<NK>(W.lxy[k], W.lzg[k], (W.lmask[k] >> lane) & 1u, xi, yi, zi, e_inv_h, e_h2x4, e_hc2, soft, gt, P.nq, P.dq, P.inv_dq, gx[0], gy[0], gz[0], nx, ny, nz);
        if (rec && hit) { if (nc < F.slots) lst[(size_t)nc * 32] = W.lidx[k]; ++nc; }
      }
      if (SPLIT) { W.nacc[0][lane] = nx; W.nacc[1][lane] = ny; W.nacc[2][lane] = nz; if (rec) W.ncnt[lane] = nc; }
    };

    GWS(0, 1);
    if (do_grav && tg.y > 0) {               // tg.y == 0: an unused tail entry of the run table
      const BvhBox gb = gbox[chunk];
      const double lo0 = gb.plo[0], lo1 = gb.plo[1], lo2 = gb.plo[2], hi0 = gb.phi[0], hi1 = gb.phi[1], hi2 = gb.phi[2];
      const double soft_min = warp_min(live ? soft : INFINITY), soft_max = warp_max(live ? soft : 0.0);
      const unsigned livemask = __ballot_sync(FULL_MASK, live);
      // FP32 screens (classification against the run's box, and the per-particle test on mixed nodes): coordinates
      // relative to the box centre g0.  A particle is within hw = max(hxf, hyf, hzf) of g0 per axis and a node's COM
      // within rho = max |r| of it; each float coordinate carries 2^-24 of its magnitude and the float difference
      // 2^-24 of at most hw + rho, so the float distance from a particle to a node is off by at most
      // sqrt(3) 2^-23 (hw + rho) < delta = 4e-7 (hw + rho), and each per-axis distance by less than delta (the code
      // takes the sums of the three half-widths and of the three |r| components, which bound hw and rho).  The run
      // can be far wider than the distances decided on (runs straddle coarse cells), so delta is an absolute band:
      // the classification shrinks the per-axis distances to the box by delta and grows the far ones by delta (3e-5
      // relative margins on top for the float arithmetic).  A mixed node's per-particle test keeps its 3e-5 margins
      // on W = size^2 / theta^2 where delta <= 1e-5 sqrt(W): the float distance d_f is within delta of d, so
      // d_f^2 + soft moves by less than (1 +- 1e-5)^2 - 1 ~ 2e-5 of W around the decision, the margins' remaining 1e-5
      // covers the float arithmetic of d^2 and W.  Where delta is larger the node's W is stored as NaN: both float
      // comparisons fail and every particle takes the FP64 test.  Whatever falls inside a margin is decided by the
      // FP64 tests below, so no decision changes.
      const double g0x = 0.5 * (lo0 + hi0), g0y = 0.5 * (lo1 + hi1), g0z = 0.5 * (lo2 + hi2);
      const float hxf = __double2float_ru(0.5 * (hi0 - lo0)) * 1.00001f, hyf = __double2float_ru(0.5 * (hi1 - lo1)) * 1.00001f, hzf = __double2float_ru(0.5 * (hi2 - lo2)) * 1.00001f;
      const float xif = (float)(xi - g0x), yif = (float)(yi - g0y), zif = (float)(zi - g0z);
      const float softf = (float)soft, softf_min = __double2float_rd(soft_min), softf_max = __double2float_ru(soft_max);
      const float th2f = (float)theta2, inv_th2f = (float)inv_theta2;
      const float nearf = __double2float_ru(warp_max(hc2)) * 1.0001f;      // d2 above it: beyond the near / far split (hence farther than 2 h) for every particle of the run
      int sn = 1, gsp = 0, ln = 0, nn = 0;
      if (lane == 0) W.stack[0] = make_int2(0, (int)livemask);
      __syncwarp();

      auto make_room = [&](int need) {       // keep the pushes inside the shared-memory stack
        if (sn + need <= GW_STACK) return;
        __syncwarp();
        if (gsp + sn > GW_SPILL) { if (lane == 0) atomicExch(err_flag, 2); sn = 0; }     // loud: the host returns an error
        for (int e = lane; e < sn; e += 32) myspill[gsp + e] = W.stack[e];
        gsp += sn; sn = 0;
        __syncwarp();
      };

      for (;;) {
        if (sn == 0) {
          if (gsp == 0) break;
          const int take = gsp < GW_STACK / 2 ? gsp : GW_STACK / 2;
          for (int e = lane; e < take; e += 32) W.stack[e] = myspill[gsp - take + e];
          gsp -= take; sn = take;
          __syncwarp();
        }
        const int npop = sn < 32 ? sn : 32;
        const bool valid = lane < npop;
        const int2 e = valid ? W.stack[sn - 1 - lane] : make_int2(0, 0);
        __syncwarp();
        sn -= npop;
        // ---- lane = node: classify against the group box
        int cls = 0;                           // 1 all accept, 2 all open, 3 mixed
        double ncx = 0.0, ncy = 0.0, ncz = 0.0, nm = 0.0, nsize = 0.0; int nchild = 0, nnch = 0;
        float rxf = 0.f, ryf = 0.f, rzf = 0.f, s2f = 0.f, dmin2 = 0.f, dlt = 0.f;
        if (valid) {
          const double2* p = reinterpret_cast<const double2*>(wn + e.x);
          const double2 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
          ncx = a.x; ncy = a.y; ncz = b.x; nm = b.y; nsize = c.x;
          nchild = __double2loint(c.y); nnch = __double2hiint(c.y);
          rxf = (float)(ncx - g0x); ryf = (float)(ncy - g0y); rzf = (float)(ncz - g0z);
          const float axf = fabsf(rxf), ayf = fabsf(ryf), azf = fabsf(rzf);
          dlt = 4e-7f * ((hxf + hyf + hzf) + (axf + ayf + azf));
          const float nx = fmaxf(axf - hxf - dlt, 0.f), ny = fmaxf(ayf - hyf - dlt, 0.f), nz = fmaxf(azf - hzf - dlt, 0.f);
          const float fx = axf + hxf + dlt, fy = ayf + hyf + dlt, fz = azf + hzf + dlt;
          dmin2 = fmaf(nx, nx, fmaf(ny, ny, fmaf(nz, nz, softf_min)));
          const float dmax2 = fmaf(fx, fx, fmaf(fy, fy, fmaf(fz, fz, softf_max)));
          const float szf = (float)nsize;
          s2f = szf * szf;
          if (nnch == 0 || s2f < th2f * dmin2 * (1.f - 3e-5f)) cls = 1;
          else if (s2f > th2f * dmax2 * (1.f + 3e-5f)) cls = 2;
          else cls = 3;
          if (MODE == 1) {       // every centre of mass of the subtree lies in the node's cell, i.e. within `size` of the node's own per axis
            const float px = fmaxf(axf - hxf - szf - 2e-6f * (axf + hxf + szf), 0.f), py = fmaxf(ayf - hyf - szf - 2e-6f * (ayf + hyf + szf), 0.f),
                        pz = fmaxf(azf - hzf - szf - 2e-6f * (azf + hzf + szf), 0.f);
            if (fmaf(px, px, fmaf(py, py, pz * pz)) > nearf) cls = 0;       // no term of the subtree can be near for any particle of the run
          }
        }
        const unsigned emask = (unsigned)e.y;
#ifdef SCREEN_AUDIT
        {   // the nodes classified for the whole run: the exact test of every particle of the node's lane set
          unsigned bc = __ballot_sync(FULL_MASK, (cls == 1 || cls == 2) && nnch != 0), bad = 0;
          while (bc) {
            const int L = __ffs(bc) - 1; bc &= bc - 1;
            const double cx = __shfl_sync(FULL_MASK, ncx, L), cy = __shfl_sync(FULL_MASK, ncy, L), cz = __shfl_sync(FULL_MASK, ncz, L), sz = __shfl_sync(FULL_MASK, nsize, L);
            const int cl = __shfl_sync(FULL_MASK, cls, L);
            const unsigned em = __shfl_sync(FULL_MASK, emask, L);
            if ((em >> lane) & 1u) bad += audit_mac_accept(xi - cx, yi - cy, zi - cz, soft, sz, theta) != (cl == 1) ? 1u : 0u;
          }
          if (bad) atomicAdd(&screen_audit[2], (unsigned long long)bad);
        }
#endif
        const unsigned balM = __ballot_sync(FULL_MASK, cls == 3);
        const int nmix = __popc(balM);
        GWS(1, npop); GWS(2, __popc(__ballot_sync(FULL_MASK, valid && cls == 0))); GWS(3, __popc(__ballot_sync(FULL_MASK, cls == 1)));
        GWS(4, __popc(__ballot_sync(FULL_MASK, cls == 2))); GWS(5, nmix); GWS(10, 1);
        if (cls == 3) {
          const int pos = __popc(balM & lt_mask);
          W.mcx[pos] = ncx; W.mcy[pos] = ncy; W.mcz[pos] = ncz; W.msize[pos] = nsize; W.mmask[pos] = emask;
          // size^2 < theta^2 d2 (1 - 1e-12)  <=>  d2 > size^2 / (theta^2 (1 - 1e-12)); the band in between gets the exact test
          const double s2t = nsize * nsize * inv_theta2;
          W.mhi[pos] = s2t * (1.0 + 2e-12); W.mlo[pos] = s2t * (1.0 - 2e-12);
          const float wf = s2f * inv_th2f;
          W.mf[pos] = make_float4(rxf, ryf, rzf, dlt * dlt <= 1e-10f * wf ? wf : __int_as_float(0x7fffffff));
        }
        __syncwarp();
        // ---- lane = particle: the reference's own test on the mixed nodes; the node's lane keeps the two ballots
        unsigned acc_mask = (cls == 1) ? emask : 0u, open_mask = (cls == 2) ? emask : 0u;
        unsigned bm = balM;
#pragma unroll 2
        for (int q = 0; q < nmix; ++q) {
          const int L = __ffs(bm) - 1; bm &= bm - 1;
          const unsigned mm = W.mmask[q];
          const bool in = (mm >> lane) & 1u;
          const float4 mq = W.mf[q];
          const float dxf = xif - mq.x, dyf = yif - mq.y, dzf = zif - mq.z;
          const float d2f = fmaf(dxf, dxf, fmaf(dyf, dyf, fmaf(dzf, dzf, softf)));
          bool accept = d2f > mq.w * (1.f + 3e-5f);
#ifdef SCREEN_AUDIT
          if (in && (accept || d2f < mq.w * (1.f - 3e-5f)) && audit_mac_accept(xi - W.mcx[q], yi - W.mcy[q], zi - W.mcz[q], soft, W.msize[q], theta) != accept)
            atomicAdd(&screen_audit[2], 1ull);
#endif
          if (!accept && !(d2f < mq.w * (1.f - 3e-5f))) {       // inside the float margin: the FP64 test
            const double dx = xi - W.mcx[q], dy = yi - W.mcy[q], dz = zi - W.mcz[q];          // F:274
            const double d2 = fma(dx, dx, fma(dy, dy, fma(dz, dz, soft)));
            accept = d2 > W.mhi[q];
            if (!accept && !(d2 < W.mlo[q])) {   // borderline: redo the reference's arithmetic exactly (no contraction)       F:275-278
              const double size = W.msize[q];
              const double e2 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)), soft);
              accept = __ddiv_rn(size, __dsqrt_rn(e2)) < theta;
            }
          }
          const unsigned balAcc = __ballot_sync(FULL_MASK, in && accept), balOpen = __ballot_sync(FULL_MASK, in && !accept);
          if (lane == L) { acc_mask = balAcc; open_mask = balOpen; }
        }
        // ---- lane = node again: accepted (node, lane set) pairs join the interaction list, opened ones push their child block
        if (FULL) { n_acc += __popc(acc_mask); n_open += __popc(open_mask); }
        const bool ins0 = acc_mask != 0u && nm > 0.0;                               // F:279: massless nodes add nothing
        const bool insn = ins0 && !(dmin2 > nearf);                                 // some particle of the run may be within the near / far split of it
        const bool ins = FULL ? ins0 : insn;
        const unsigned balL = FULL ? __ballot_sync(FULL_MASK, ins && !insn) : 0u, balN = __ballot_sync(FULL_MASK, insn);
        if (ins) {
          const int pos = insn ? GW_LIST - 1 - (nn + __popc(balN & lt_mask)) : ln + __popc(balL & lt_mask);
          W.lxy[pos] = make_double2(ncx, ncy); W.lzg[pos] = make_double2(ncz, P.G * nm); W.lmask[pos] = acc_mask;
          if (SPLIT) W.lidx[pos] = e.x;
        }
#ifdef SCREEN_AUDIT
        {   // far entries: no particle they are accepted for may lie within its near / far split
          unsigned bf = balL, bad = 0;
          while (bf) {
            const int L = __ffs(bf) - 1; bf &= bf - 1;
            const double cx = __shfl_sync(FULL_MASK, ncx, L), cy = __shfl_sync(FULL_MASK, ncy, L), cz = __shfl_sync(FULL_MASK, ncz, L);
            const unsigned am = __shfl_sync(FULL_MASK, acc_mask, L);
            const double dx = xi - cx, dy = yi - cy, dz = zi - cz;
            if ((am >> lane) & 1u) bad += fma(dx, dx, fma(dy, dy, fma(dz, dz, soft))) <= hc2 ? 1u : 0u;
          }
          if (bad) atomicAdd(&screen_audit[2], (unsigned long long)bad);
        }
#endif
        nn += __popc(balN);
        ln += __popc(balL);
        GWS(6, __popc(balL)); GWS(7, __popc(balN));
#ifdef GW_STATS
        { int a = (ins && !insn) ? __popc(acc_mask) : 0, b = insn ? __popc(acc_mask) : 0;
          for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(FULL_MASK, a, o); b += __shfl_xor_sync(FULL_MASK, b, o); }
          GWS(8, a); GWS(9, b); }
#endif
        const int nch = open_mask ? nnch : 0;
        int incl = nch;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += t; }
        const int total = __shfl_sync(FULL_MASK, incl, 31);
        make_room(total);
        for (int k = 0; k < nch; ++k) W.stack[sn + incl - nch + k] = make_int2(nchild + k, (int)open_mask);
        sn += total;
        __syncwarp();
        if (ln + nn > GW_LIST - 32) { GWS(12, 1); evaluate_list(ln, nn); ln = nn = 0; __syncwarp(); }
      }
      if (ln + nn > 0) evaluate_list(ln, nn);
      __syncwarp();
    }
#pragma unroll
    for (int u = 1; u < GW_ILP; ++u) { gx[0] += gx[u]; gy[0] += gy[u]; gz[0] += gz[u]; }
    if (MODE == 1) { gx[0] = live ? F.fx[i] : 0.0; gy[0] = live ? F.fy[i] : 0.0; gz[0] = live ? F.fz[i] : 0.0; }      // the stored far sum of the tree terms
    else if (SPLIT && F.store && live) { F.fx[i] = gx[0]; F.fy[i] = gy[0]; F.fz[i] = gz[0]; }
    // the sinks are not part of the stored sums: their terms are taken with the sinks as they are now, in every evaluation
    sink_terms(P, S, n_sink, live, xi, yi, zi, live ? m[i] : 0.0, gx[0], gy[0], gz[0], sink_partial + (size_t)(chunk - g_begin) * n_sink * 3);
    if (MODE == 1) {
      if (live) { ax[i] = gx[0] + nx; ay[i] = gy[0] + ny; az[i] = gz[0] + nz; }
      continue;
    }
    if (SPLIT && F.list) {          // near pairs recorded per lane; a lane that needed more slots sends its run to the near-only walk
      const int nc = W.ncnt[lane];
      F.cnt[(size_t)chunk * 32 + lane] = nc;
      const bool over = __any_sync(FULL_MASK, nc > F.slots);
      if (lane == 0) { F.ovf[chunk] = over ? 1 : 0; if (over) atomicAdd(F.n_ovf, 1); }
    }
    if (live) {
      if (SPLIT) { ax[i] = gx[0] + W.nacc[0][lane]; ay[i] = gy[0] + W.nacc[1][lane]; az[i] = gz[0] + W.nacc[2][lane]; }
      else { ax[i] = gx[0]; ay[i] = gy[0]; az[i] = gz[0]; }
    }
  }
  n_open = (unsigned long long)warp_sum_ll((long long)n_open); n_acc = (unsigned long long)warp_sum_ll((long long)n_acc);
  if (MODE != 1 && lane == 0 && do_grav) { atomicAdd(&ctr->grav_opened, n_open); atomicAdd(&ctr->grav_accepted, n_acc); }
#ifdef GW_STATS
  if (lane == 0) for (int k = 0; k < 16; ++k) if (gws[k]) atomicAdd(&gw_stats[k], gws[k]);
#endif
}

// The near field from the recorded pairs (see "Far-field reuse"): one warp per run, lane = particle, trip k evaluates
// the k-th recorded node of every lane (coalesced index load, gathered 32-byte node read) with the current h and adds
// it in the order the full walk did; the stored far sum completes the acceleration.  dynamic smem: the kernel table.
#define GN_WARPS 8
__global__ void __launch_bounds__(GN_WARPS * 32)
k_gravity_near(int n_runs, const int2* __restrict__ groups, DevParams P, const WNode* __restrict__ wn, const double* __restrict__ x,
               const double* __restrict__ y, const double* __restrict__ z, const double* __restrict__ h, const double* __restrict__ m, const double* __restrict__ g_gt,
               double* __restrict__ ax, double* __restrict__ ay, double* __restrict__ az, int n_sink, SinkArrays S, double* __restrict__ sink_partial, FarField F) {
  extern __shared__ __align__(16) double gsm[];
  double* gt = gsm;
  for (int i = threadIdx.x; i <= P.nq; i += blockDim.x) gt[i] = g_gt[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  for (int run = blockIdx.x * GN_WARPS + (threadIdx.x >> 5); run < n_runs; run += gridDim.x * GN_WARPS) {
    const int2 tg = groups[run];
    if (tg.y == 0 || F.ovf[run]) continue;
    const int i = tg.x + lane;
    const bool live = lane < tg.y;
    const double xi = live ? x[i] : 0.0, yi = live ? y[i] : 0.0, zi = live ? z[i] : 0.0;
    const double hi = live ? (P.variable_h ? h[i] : P.h_fixed) : 1.0;
    const double inv_h = 1.0 / hi, h2x4 = 4.0 * hi * hi, soft = 0.001 * P.h_fixed;          // F:275 (the reuse is off under the (test new) softening)
    const int cnt = live ? F.cnt[(size_t)run * 32 + lane] : 0;
    int cmax = cnt;
    for (int o = 16; o > 0; o >>= 1) cmax = max(cmax, __shfl_xor_sync(FULL_MASK, cmax, o));
    const int* lst = F.list + ((size_t)run * F.slots) * 32 + lane;
    double nx = 0.0, ny = 0.0, nz = 0.0, dum = 0.0;
    int k = 0;
    for (; k + 2 <= cmax; k += 2) {             // two gathers in flight per lane; the sums stay in recorded order
      const bool on0 = k < cnt, on1 = k + 1 < cnt;
      const int j0 = on0 ? lst[(size_t)k * 32] : 0, j1 = on1 ? lst[(size_t)(k + 1) * 32] : 0;
      const double2* p0 = reinterpret_cast<const double2*>(wn + j0); const double2* p1 = reinterpret_cast<const double2*>(wn + j1);
      const double2 a0 = __ldg(p0), b0 = __ldg(p0 + 1), a1 = __ldg(p1), b1 = __ldg(p1 + 1);
      grav_term<3>(a0, make_double2(b0.x, P.G * b0.y), on0, xi, yi, zi, inv_h, h2x4, 0.0, soft, gt, P.nq, P.dq, P.inv_dq, dum, dum, dum, nx, ny, nz);
      grav_term<3>(a1, make_double2(b1.x, P.G * b1.y), on1, xi, yi, zi, inv_h, h2x4, 0.0, soft, gt, P.nq, P.dq, P.inv_dq, dum, dum, dum, nx, ny, nz);
    }
    if (k < cmax) {
      const bool on0 = k < cnt;
      const int j0 = on0 ? lst[(size_t)k * 32] : 0;
      const double2* p0 = reinterpret_cast<const double2*>(wn + j0);
      const double2 a0 = __ldg(p0), b0 = __ldg(p0 + 1);
      grav_term<3>(a0, make_double2(b0.x, P.G * b0.y), on0, xi, yi, zi, inv_h, h2x4, 0.0, soft, gt, P.nq, P.dq, P.inv_dq, dum, dum, dum, nx, ny, nz);
    }
    double gx = live ? F.fx[i] : 0.0, gy = live ? F.fy[i] : 0.0, gz = live ? F.fz[i] : 0.0;      // far tree terms, then the sinks as they are now, then the near terms: the full walk's order
    sink_terms(P, S, n_sink, live, xi, yi, zi, live ? m[i] : 0.0, gx, gy, gz, sink_partial + (size_t)run * n_sink * 3);
    if (live) { ax[i] = gx + nx; ay[i] = gy + ny; az[i] = gz + nz; }
  }
}

// Gravity walk groups: runs of GRAV_CHUNK_WIDTH Morton-consecutive particles.  The gravity walk tolerates a run that
// straddles a coarse cell boundary (more mixed nodes, decided per particle), and full warps matter more to it than
// tight boxes.  Runs restart at every GRAV_SEG-th SPH walk group, and rank slices are cut only at those boundaries,
// so the set of runs - hence every particle's accumulation order - does not depend on the number of ranks.
#define GRAV_SEG 64
// Run formation inside one segment (SPH groups [s * GRAV_SEG, (s + 1) * GRAV_SEG), particles [pa, pb)): walk groups
// are appended to the current run; when the next group does not fit, the run is closed at that (cell) boundary if it
// already holds GRAV_MINFILL particles, else it is filled up with the head of the group.  One thread per segment.
#ifndef GRAV_MINFILL
#define GRAV_MINFILL 33          // > width: never close early (fixed runs)
#endif
template <bool WRITE>
__device__ __forceinline__ int seg_runs(int ga, int gb, int width, const int2* __restrict__ sg, int2* __restrict__ out) {
  int n_runs = 0, first = sg[ga].x, cur = 0;
  for (int g = ga; g < gb; ++g) {
    int sz = sg[g].y;
    while (sz > 0) {
      const int space = width - cur;
      if (sz <= space) { cur += sz; sz = 0; }
      else if (cur >= GRAV_MINFILL) { if (WRITE) out[n_runs] = make_int2(first, cur); ++n_runs; first += cur; cur = 0; continue; }
      else { cur += space; sz -= space; }
      if (cur == width) { if (WRITE) out[n_runs] = make_int2(first, cur); ++n_runs; first += cur; cur = 0; }
    }
  }
  if (cur > 0) { if (WRITE) out[n_runs] = make_int2(first, cur); ++n_runs; }
  return n_runs;
}
__global__ void k_seg_count(int seg0, int nseg, int n_groups, int width, const int2* __restrict__ sg, int* __restrict__ cnt) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s > nseg) return;
  if (s == nseg) { cnt[s] = 0; return; }
  const int ga = (seg0 + s) * GRAV_SEG, gb = min(ga + GRAV_SEG, n_groups);
  cnt[s] = seg_runs<false>(ga, gb, width, sg, nullptr);
}
__global__ void k_seg_chunks(int seg0, int nseg, int n_groups, int width, const int2* __restrict__ sg, const int* __restrict__ off,
                             int2* __restrict__ groups) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  const int ga = (seg0 + s) * GRAV_SEG, gb = min(ga + GRAV_SEG, n_groups);
  seg_runs<true>(ga, gb, width, sg, groups + off[s]);
}
// one warp per run: its position box
__global__ void k_grav_boxes(int n_chunks, const int2* __restrict__ groups, const double* __restrict__ x, const double* __restrict__ y,
                             const double* __restrict__ z, BvhBox* __restrict__ box) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_chunks) return;
  const int2 g = groups[warp];
  float plo[3] = {INFINITY, INFINITY, INFINITY}, phi[3] = {-INFINITY, -INFINITY, -INFINITY};
  if (lane < g.y) {
    const int i = g.x + lane;
    const double p[3] = {x[i], y[i], z[i]};
    for (int k = 0; k < 3; ++k) { plo[k] = __double2float_rd(p[k]); phi[k] = __double2float_ru(p[k]); }
  }
  for (int k = 0; k < 3; ++k) { plo[k] = warp_minf(plo[k]); phi[k] = warp_maxf(phi[k]); }
  if (lane == 0) {
    BvhBox b;
    for (int k = 0; k < 3; ++k) { b.plo[k] = plo[k]; b.phi[k] = phi[k]; b.rlo[k] = 0.f; b.rhi[k] = 0.f; }
    box[warp] = b;
  }
}

// Sink-side sums of the gas terms, in an order that does not depend on the number of ranks: the per-run partials
// (one warp sum per 32-particle run, written by k_gravity) are folded serially per GRAV_SEG segment - segments and
// their runs are the same for any rank count, rank slices are cut at segment boundaries - into the global segment
// table seg[global segment][sink][3]; the ranks exchange their rows; k_sink_reduce then folds ALL segments of the
// tree with one fixed pattern on every rank.  (Per-rank totals added by an all-reduce would group the FP64 sum by
// rank: the sinks start at v = 0, so an ulp there reaches every gas acceleration within a step.)
__global__ void k_sink_seg_fold(int nseg, int seg0, int n_sink, const int* __restrict__ seg_off, const double* __restrict__ partial,
                                double* __restrict__ seg) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nseg * n_sink * 3) return;
  const int s = t / (n_sink * 3), r = t % (n_sink * 3);
  double v = 0.0;
  for (int b = seg_off[s]; b < seg_off[s + 1]; ++b) v += partial[(size_t)b * n_sink * 3 + r];
  seg[(size_t)(seg0 + s) * n_sink * 3 + r] = v;
}
__global__ void k_sink_reduce(int n_parts, int n_sink, const double* __restrict__ partial, SinkArrays S, int do_sinks) {
  __shared__ double red[256];
  const int t = threadIdx.x;
  for (int s = 0; s < n_sink; ++s)
    for (int k = 0; k < 3; ++k) {
      double v = 0.0;
      if (do_sinks) for (int b = t; b < n_parts; b += 256) v += partial[((size_t)b * n_sink + s) * 3 + k];
      red[t] = v;
      __syncthreads();
      for (int o = 128; o > 0; o >>= 1) { if (t < o) red[t] += red[t + o]; __syncthreads(); }
      if (t == 0) { double* a = (k == 0) ? S.ax : (k == 1) ? S.ay : S.az; a[s] = red[0]; }
      __syncthreads();
    }
}
// sink-sink pairs F:578-590 (after the cross-rank sum of the gas contributions)
__global__ void k_sink_pairs(int n_sink, SinkArrays S, double G, int do_sinks) {
  if (threadIdx.x != 0 || !do_sinks || n_sink < 2) return;
  for (int i = 0; i < n_sink; ++i)
    for (int j = 0; j < i; ++j) {
      double v[3] = {S.x[j] - S.x[i], S.y[j] - S.y[i], S.z[j] - S.z[i]};
      double dr = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
      double d3 = dr * dr * dr;
      double* A[3] = {S.ax, S.ay, S.az};
      for (int k = 0; k < 3; ++k) {
        double w = G * v[k] / d3;
        A[k][i] += S.m[j] * w;
        A[k][j] -= S.m[i] * w;
      }
    }
}
