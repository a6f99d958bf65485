// sph_walk.cuh — neighbour walks: density(+Omega)+EOS, h Newton-Raphson, SPH pair forces, diagnostics.
//
// Replaces density_tree_search / get_density (SUMMER_SPH.f90:398-457 | Variable.f90:440-496),
// get_pressure_and_sound_speed (F:459-468 | V:502-512), calc_smoothing (V:515-546) and
// SPH_tree_search / get_SPH (F:295-395 | V:324-432).
//
// Membership is the reference's, bit for bit: j is a candidate of i iff the leaf box test
//     all_k |x_i,k - c_leaf(j),k| < 2 h_j + size_leaf(j)/2          (F:443 | V:479)
// passes (h_j = the value in the tree = at build time; F: the global smoothing), evaluated in FP64 with
// the same operations.  HOW candidates are found is free: one warp owns a walk group of <= 32 Morton-adjacent
// targets (lane = target), walks the implicit 8-ary BVH of group boxes with a shared-memory stack (8 child
// boxes per popped node tested by 8 lanes, coalesced), filters the source particles of each hit group
// (lane = source) into a shared-memory tile, and consumes the tile: an FP32 prefilter (could any term be
// non-zero?) followed by the exact FP64 leaf-box test and the kernel arithmetic on the survivors.  The density
// pass also saves, per group, the candidate list the pair loop needs (NeighbourListSink), so the pair loop of
// the same evaluation streams that list instead of walking again; it evaluates its hits with lane = pair
// (compacted hit list) and in gather form (SURVEY.md Appendix B): each particle sums its own side, no
// atomics, every term equal to the reference's term, per-target sums in a fixed order.
#pragma once
#include "sph_common.cuh"

struct BvhInfo { int nlev; int off[12]; int cnt[12]; };

#ifndef DENS_WARPS
#define DENS_WARPS 16        // warps per block of the density kernels
#endif
#define WALK_STACK 224      // node stack entries per warp
#define WALK_CQ    96       // chunk queue entries per warp
#define WALK_TILE  32       // staged source particles per warp
#define WALK_WS    (WALK_STACK + WALK_CQ + WALK_TILE)   // unsigned words of walk state per warp
#define PAIR_WIN   64       // compacted (target, source) hits evaluated per window, lane = pair
#define DENS_SLOTS (2 * WALK_TILE)                                 // tile slots: WALK_TILE consumed at a time + one chunk of overflow
#define DENS_WARP_DOUBLES (8 * DENS_SLOTS + 2 * DENS_SLOTS + 32)    // tile + float4 tile + saved-list buffer (64 ints)

#ifdef WALK_DEBUG
__device__ unsigned long long wk_dbg[16];
#define WKD(i, v) do { if ((threadIdx.x & 31) == 0) atomicAdd(&wk_dbg[i], (unsigned long long)(v)); } while (0)
#else
#define WKD(i, v)
#endif

struct WalkCounters { unsigned long long dens_cand, dens_contrib, sph_pairs, grav_opened, grav_accepted, h_iters; };

__device__ __forceinline__ bool box_overlap(const float* alo, const float* ahi, const float* blo, const float* bhi) {
  return alo[0] <= bhi[0] && ahi[0] >= blo[0] && alo[1] <= bhi[1] && ahi[1] >= blo[1] && alo[2] <= bhi[2] && ahi[2] >= blo[2];
}

// Generic warp walk. OP interface:
//   static const bool SYMMETRIC;                     // also accept sources lying inside the group's reach box
//   static const bool LISTS;                         // the op also saves a candidate list for a later pass (list_append)
//   static const bool FUSED;                         // filter_stage() instead of source_filter() + stage()
//   int    source_filter(int j)                      // per-source prefilter against the group (lane = source):
//                                                    // bit 0 = stage into the tile, bit 1 = append to the saved list
//   void   stage(int slot, int j)                    // copy source j into tile slot
//   int    filter_stage(int j, bool in_range, int tn), void shift(int rest)    // FUSED: both at once, 2-tile slots
//   void   consume(int count)                        // all lanes process tile[0..count)
// The target box `tgt` is the warp's own: a walk group's level-0 box (the overload below), or the box of any other 32
// targets (sph_interp.cuh: a run of interpolation points).
template <class OP>
__device__ void neighbour_walk(OP& op, const BvhBox& tgt, const int2* __restrict__ groups, const BvhBox* __restrict__ box, const BvhInfo& bi,
                               unsigned* stack, unsigned* cq) {
  unsigned* tix = cq + WALK_CQ;          // particle indices of the tile being collected
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  const BvhBox g = tgt;
  int sn = 0, qn = 0, qpos = 0, tn = 0;

  auto hit = [&](const BvhBox& b) -> bool {
    bool r = box_overlap(g.plo, g.phi, b.rlo, b.rhi);
    if (OP::SYMMETRIC) r = r || box_overlap(g.rlo, g.rhi, b.plo, b.phi);
    return r;
  };
  const int top = bi.nlev - 1;
  {
    bool ok = lane < bi.cnt[top];
    if (ok) ok = hit(box[bi.off[top] + lane]);
    unsigned bal = __ballot_sync(FULL_MASK, ok);
    int pos = __popc(bal & lt);
    if (ok) { if (top == 0) cq[pos] = (unsigned)lane; else stack[pos] = ((unsigned)top << 28) | (unsigned)lane; }
    if (top == 0) qn = __popc(bal); else sn = __popc(bal);
    __syncwarp();
  }
  // One loop iteration = one tile.  The walk is written as a producer with its state in registers so that the
  // source filter, the staging and the consumer are each instantiated ONCE in the kernel (three inlined copies of
  // the consumer made the kernel instruction-fetch bound).  Hit chunks -> passing sources: the descriptors of up
  // to 32 queued chunks come in with one lane-parallel load; each chunk costs one round of filter loads
  // (lane = source) that appends the passing particle indices to the tile's index list; a chunk that does not
  // fit stays pending (ballot + index in registers) and opens the next tile.
  int2 mysg = make_int2(0, 0);
  int pend_cnt = 0, pend_j = 0; unsigned pend_bal = 0; bool pend_ok = false;
  for (;;) {
    if (pend_cnt) { if (pend_ok) tix[__popc(pend_bal & lt)] = (unsigned)pend_j; tn = pend_cnt; pend_cnt = 0; }
    bool exhausted = false;
    for (;;) {
      if (qpos < qn) {
        if ((qpos & 31) == 0) mysg = (qpos + lane < qn) ? groups[cq[qpos + lane]] : make_int2(0, 0);
        const int sgx = __shfl_sync(FULL_MASK, mysg.x, qpos & 31), sgy = __shfl_sync(FULL_MASK, mysg.y, qpos & 31);
        ++qpos;
        const int j = sgx + lane;
        if constexpr (OP::FUSED) {
          tn += op.filter_stage(j, lane < sgy, tn);
          if (tn >= WALK_TILE) break;
          continue;
        } else {
          const int fl = (lane < sgy) ? op.source_filter(j) : 0;
          if constexpr (OP::LISTS) op.list_append((fl & 2) != 0, j);
          const bool ok = (fl & 1) != 0;
          const unsigned bal = __ballot_sync(FULL_MASK, ok);
          const int cntc = __popc(bal);
          if (cntc == 0) continue;
          if (tn + cntc > WALK_TILE) { pend_cnt = cntc; pend_bal = bal; pend_j = j; pend_ok = ok; break; }
          if (ok) tix[tn + __popc(bal & lt)] = (unsigned)j;
          tn += cntc;
          continue;
        }
      }
      // chunk queue drained: refill it from the node stack (4 nodes x 8 child boxes per trip, coalesced)
      qn = 0; qpos = 0;
      if (sn == 0) { exhausted = true; break; }
      __syncwarp();
      while (sn > 0 && qn <= WALK_CQ - 32) {
        const int npop = sn < 4 ? sn : 4;
        const int grp = lane >> 3;
        const bool valid = grp < npop;
        const unsigned e = valid ? stack[sn - 1 - grp] : 0u;
        __syncwarp();
        sn -= npop;
        const int lev = (int)(e >> 28), idx = (int)(e & 0x0fffffffu);
        const int clev = lev - 1;
        const int child = idx * SPH_BVH_FAN + (lane & 7);
        bool ok = valid && child < bi.cnt[clev > 0 ? clev : 0];
        if (ok) ok = hit(box[bi.off[clev] + child]);
        const bool ok0 = ok && clev == 0, okn = ok && clev > 0;
        const unsigned b0 = __ballot_sync(FULL_MASK, ok0), bn = __ballot_sync(FULL_MASK, okn);
        if (ok0) cq[qn + __popc(b0 & lt)] = (unsigned)child;
        if (okn) stack[sn + __popc(bn & lt)] = ((unsigned)clev << 28) | (unsigned)child;
        qn += __popc(b0); sn += __popc(bn);
        __syncwarp();
      }
    }
    if constexpr (OP::FUSED) {
      if (tn > 0) {
        const int cnt = tn < WALK_TILE ? tn : WALK_TILE;
        __syncwarp();
        op.consume(cnt);
        __syncwarp();
        op.shift(tn - cnt);
        tn -= cnt;
        __syncwarp();
      }
      if (exhausted && tn == 0) break;
    } else {
      if (tn > 0) {
        __syncwarp();
        if (lane < tn) op.stage(lane, (int)tix[lane]);
        __syncwarp();
        op.consume(tn);
        tn = 0;
        __syncwarp();
      }
      if (exhausted && !pend_cnt) break;
    }
  }
}
// targets = walk group `chunk`
template <class OP>
__device__ __forceinline__ void neighbour_walk(OP& op, const int2* __restrict__ groups, int chunk, const BvhBox* __restrict__ box, const BvhInfo& bi,
                                               unsigned* stack, unsigned* cq) {
  neighbour_walk(op, box[bi.off[0] + chunk], groups, box, bi, stack, cq);
}

// Saved candidate lists.  The density pass walks the BVH with the symmetric (pair-loop) criterion and writes,
// per walk group, the indices of every source the pair loop will need into a chain of 32-int blocks taken from
// a global pool: ints [0, NL_PER_BLOCK) = sorted particle indices, [30] = how many, [31] = next block (-1: end).
// The pair loop of the same evaluation then streams its group's chain instead of walking and filtering again.
// ctl[0] = block cursor, ctl[2] = pool overflowed (the host grows it), ctl[1] = "lists unusable" (pool overflow, or a non-finite P/(Omega rho^2) + c somewhere:
// the reference lets such a particle poison every box partner through 0 * NaN, which the distance cull applied
// to the list would hide) -> the walking pair kernel runs instead.
#define NL_PER_BLOCK 30
#define NL_BATCH 16
struct NeighbourListSink { int* pool; int* head; int* ctl; int pool_blocks; };

// shared kernel-table lookup: returns table-space (w, dw) at q (<= 2 assumed), F:113-118
__device__ __forceinline__ void table_lerp(const double* __restrict__ wt, const double* __restrict__ dwt,
                                           int nq, double dq, double inv_dq, double q, double& w, double& dw) {
  int i = (int)(q * inv_dq); i = i < nq - 1 ? i : nq - 1;
  double a = (q - i * dq) * inv_dq;
  double b = 1.0 - a;
  w = b * wt[i] + a * wt[i + 1];
  dw = b * dwt[i] + a * dwt[i + 1];
}
__device__ __forceinline__ double table_lerp1(const double* __restrict__ t, int nq, double dq, double inv_dq, double q) {
  int i = (int)(q * inv_dq); i = i < nq - 1 ? i : nq - 1;
  double a = (q - i * dq) * inv_dq;
  return (1.0 - a) * t[i] + a * t[i + 1];
}

// ------------------------------------------------------------------------------------------------------
// density (+ Omega) operator, also used by the h iteration
// ------------------------------------------------------------------------------------------------------
struct DensityArrays {
  const double *x, *y, *z, *m, *lcx, *lcy, *lcz, *reach;
};

template <bool PRODUCE>
struct DensityOp {
  static const bool SYMMETRIC = PRODUCE;
  static const bool LISTS = PRODUCE;
  static const bool FUSED = true;          // filter_stage() instead of source_filter() + stage()
  // saved-list state (PRODUCE): lbuf = 64 ints of shared memory per warp
  NeighbourListSink nl; int* lbuf; int ln, cur_blk, res_next, res_end; float grlo[3], grhi[3]; const double* hsrc; int variable_h; double h_fixed;
  // tile (per warp, shared memory): 8 arrays of WALK_TILE doubles
  double *sx, *sy, *sz, *sm, *scx, *scy, *scz, *sR;
  float4* ft;                        // float copy of the tile positions, relative to the group's origin (prefilter)
  double g0x, g0y, g0z; float xif, yif, zif, r2maxif;
  const DensityArrays& A;
  const double *wt, *dwt;            // shared-memory tables
  int nq; double dq, inv_dq;
  float gplo[3], gphi[3];            // group position box (for the per-source prefilter)
  // lane state
  double xi, yi, zi, inv_h;
  double r2max;                      // 4 h_i^2 (1 + 1e-9): beyond it q > 2 for certain and the term is an exact zero
  double g_r2max;                    // the same for the largest h of the group's active targets
  bool count_all;                    // keep every box candidate (exact candidate counter) instead of culling exact zeros early
  bool active;
  double accW, accB;                 // sum m_j w(q), sum m_j r dw(q)
  unsigned cand, contrib;

  __device__ DensityOp(const DensityArrays& a) : A(a) {}

  // Fused filter + stage (lane = source of one chunk): the values that decide the filter are the values the tile
  // needs, so the passing lanes write them straight from registers into the tile slots [tn, tn + count) - no index
  // list, no second (gathered) read.  The tile has 2 * WALK_TILE slots: the walk consumes the first WALK_TILE when
  // they are full and shifts the rest down.  Returns how many sources were staged.
  __device__ __forceinline__ int filter_stage(int j, bool in_range, int tn) {
    const int lane = threadIdx.x & 31;
    double R = -1.0, cx = 0.0, cy = 0.0, cz = 0.0, px = 0.0, py = 0.0, pz = 0.0, mj = 0.0, hj = h_fixed;
    if (in_range) {
      R = A.reach[j]; cx = A.lcx[j]; cy = A.lcy[j]; cz = A.lcz[j]; px = A.x[j]; py = A.y[j]; pz = A.z[j]; mj = A.m[j];
      if (PRODUCE && variable_h) hj = hsrc[j];
    }
    const bool box = (R > 0.0) & (cx - R <= (double)gphi[0]) & (cx + R >= (double)gplo[0]) &
                     (cy - R <= (double)gphi[1]) & (cy + R >= (double)gplo[1]) &
                     (cz - R <= (double)gphi[2]) & (cz + R >= (double)gplo[2]);
    const double ex = fmax(fmax((double)gplo[0] - px, px - (double)gphi[0]), 0.0), ey = fmax(fmax((double)gplo[1] - py, py - (double)gphi[1]), 0.0),
                 ez = fmax(fmax((double)gplo[2] - pz, pz - (double)gphi[2]), 0.0);
    const double e2 = ex * ex + ey * ey + ez * ez;
    const bool ok = in_range & box & (!(e2 > g_r2max) | count_all);      // farther than 2 h_i from every target: W = 0 exactly
    if (PRODUCE) {
      const bool b = (px >= (double)grlo[0]) & (px <= (double)grhi[0]) & (py >= (double)grlo[1]) & (py <= (double)grhi[1]) &
                     (pz >= (double)grlo[2]) & (pz <= (double)grhi[2]);
      const bool nz = !(e2 > fmax(g_r2max, 4.0 * hj * hj * (1.0 + 1e-9)));
      list_append(in_range & (box | b) & (nz | count_all), j);            // the pair loop's criterion (ForceOp::source_filter)
    }
    const unsigned bal = __ballot_sync(FULL_MASK, ok);
    if (ok) {
      const int s = tn + __popc(bal & ((1u << lane) - 1u));
      sx[s] = px; sy[s] = py; sz[s] = pz; sm[s] = mj; scx[s] = cx; scy[s] = cy; scz[s] = cz; sR[s] = R;
      ft[s] = make_float4((float)(px - g0x), (float)(py - g0y), (float)(pz - g0z), 0.f);
    }
    return __popc(bal);
  }
  // move the slots [WALK_TILE, WALK_TILE + rest) down to [0, rest)
  __device__ __forceinline__ void shift(int rest) {
    const int lane = threadIdx.x & 31;
    const bool mv = lane < rest;
    const int s = WALK_TILE + lane;
    double v0 = 0, v1 = 0, v2 = 0, v3 = 0, v4 = 0, v5 = 0, v6 = 0, v7 = 0; float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
    if (mv) { v0 = sx[s]; v1 = sy[s]; v2 = sz[s]; v3 = sm[s]; v4 = scx[s]; v5 = scy[s]; v6 = scz[s]; v7 = sR[s]; f = ft[s]; }
    __syncwarp();
    if (mv) { sx[lane] = v0; sy[lane] = v1; sz[lane] = v2; sm[lane] = v3; scx[lane] = v4; scy[lane] = v5; scz[lane] = v6; sR[lane] = v7; ft[lane] = f; }
  }
  // ---- saved list: append the flagged sources of one chunk (lane = source), flushing full blocks to the pool
  // blocks are taken from the pool NL_BATCH at a time per warp (one returning atomic per batch, not per block)
  __device__ __forceinline__ int take_block() {
    const int lane = threadIdx.x & 31;
    if (res_next == res_end) {
      int b = 0;
      if (lane == 0) b = atomicAdd(&nl.ctl[0], NL_BATCH);
      res_next = __shfl_sync(FULL_MASK, b, 0); res_end = res_next + NL_BATCH;
    }
    int r = res_next++;
    if (r >= nl.pool_blocks) { if (lane == 0) { nl.ctl[1] = 1; nl.ctl[2] = 1; } r = -2; }   // pool exhausted: this evaluation's lists are void
    return r;
  }
  __device__ __forceinline__ void list_flush(int cnt, bool last) {
    const int lane = threadIdx.x & 31;
    const int nxt = last ? -1 : take_block();
    if (cur_blk >= 0) {
      const int v = lane < cnt ? lbuf[lane] : (lane == 30 ? cnt : (lane == 31 ? (nxt < 0 ? -1 : nxt) : 0));
      nl.pool[(size_t)cur_blk * 32 + lane] = v;
    }
    cur_blk = nxt;
  }
  __device__ __forceinline__ void list_begin(int chunk) {
    cur_blk = take_block(); ln = 0;
    if ((threadIdx.x & 31) == 0) nl.head[chunk] = cur_blk;
  }
  __device__ __forceinline__ void list_append(bool want, int j) {
    const int lane = threadIdx.x & 31;
    const unsigned bal = __ballot_sync(FULL_MASK, want);
    const int cnt = __popc(bal);
    if (cnt == 0) return;
    const int pos = ln + __popc(bal & ((1u << lane) - 1u));
    if (want) lbuf[pos] = j;                                                     // ln <= 29, cnt <= 32: fits the 64-int buffer
    ln += cnt;
    while (ln >= NL_PER_BLOCK) {
      __syncwarp();
      list_flush(NL_PER_BLOCK, false);
      __syncwarp();
      const int rest = ln - NL_PER_BLOCK;
      const int v = lane < rest ? lbuf[NL_PER_BLOCK + lane] : 0;
      __syncwarp();
      if (lane < rest) lbuf[lane] = v;
      ln = rest;
    }
  }
  __device__ __forceinline__ void list_end() { __syncwarp(); list_flush(ln, true); __syncwarp(); }
  __device__ __forceinline__ void consume(int count) {
    // Prefilter, lane = target, FP32 on group-relative coordinates: |x_i - x_j|^2 against r2maxif, the square of
    // b_i = 2 h_i + 4e-7 (gd + 2 h_i) (density_bound).  Beyond it W(q > 2) = 0 exactly (F:112), so it only drops
    // exact zeros; the reference's leaf-box test (F:443 | V:479) and q <= 2 are evaluated in FP64 on the survivors.
    // With the exact candidate counter on, every staged source goes through the FP64 tests.
    unsigned mask = 0;
    if (active) {
      if (count_all) mask = count >= 32 ? 0xffffffffu : ((1u << count) - 1u);
      else {
#pragma unroll 4
        for (int k = 0; k < count; ++k) {
          const float4 sj = ft[k];
          const float dx = xif - sj.x, dy = yif - sj.y, dz = zif - sj.z;
          const bool far = fmaf(dx, dx, fmaf(dy, dy, dz * dz)) > r2maxif;
          mask |= (far ? 0u : 1u) << k;
        }
      }
    }
#ifdef SCREEN_AUDIT
    if (active && !count_all) {          // every staged source the screen dropped: would the FP64 test have summed it?
      unsigned bad = 0;
      for (int k = 0; k < count; ++k) {
        if ((mask >> k) & 1u) continue;
        const double R = sR[k], dx = xi - sx[k], dy = yi - sy[k], dz = zi - sz[k];
        const bool box = (fabs(xi - scx[k]) < R) & (fabs(yi - scy[k]) < R) & (fabs(zi - scz[k]) < R);
        const double r2 = dx * dx + dy * dy + dz * dz;
        double r, rs; fast_sqrt_rsqrt(r2, r, rs);
        r = (r2 == 0.0) ? 0.0 : r;
        bad += (box & (r * inv_h <= 2.0)) ? 1u : 0u;
      }
      if (bad) atomicAdd(&screen_audit[0], (unsigned long long)bad);
    }
#endif
#ifdef WALK_DEBUG
    { int hc = __popc(mask); int mx = hc, sm = hc; for (int o = 16; o > 0; o >>= 1) { mx = max(mx, __shfl_xor_sync(FULL_MASK, mx, o)); sm += __shfl_xor_sync(FULL_MASK, sm, o); }
      WKD(8, 1); WKD(9, count); WKD(10, mx); WKD(11, sm); }
#endif
    // two survivors per trip, branch-free, so two independent dependency chains are in flight per lane
    double w2 = 0.0, b2 = 0.0;
    while (mask) {
      const int k0 = __ffs(mask) - 1; mask &= mask - 1;
      const bool v1 = mask != 0;
      const int k1 = v1 ? __ffs(mask) - 1 : k0; mask &= mask - 1;
      term(k0, true, accW, accB);
      term(k1, v1, w2, b2);
    }
    accW += w2; accB += b2;
  }
  __device__ __forceinline__ void term(int k, bool valid, double& aW, double& aB) {
    const double R = sR[k];
    const double dx = xi - sx[k], dy = yi - sy[k], dz = zi - sz[k];
    const bool box = valid & (fabs(xi - scx[k]) < R) & (fabs(yi - scy[k]) < R) & (fabs(zi - scz[k]) < R);   // F:443 | V:479
    const double r2 = dx * dx + dy * dy + dz * dz;
    double r, rs; fast_sqrt_rsqrt(r2, r, rs);
    r = (r2 == 0.0) ? 0.0 : r;                                           // self term, W(0)
    const double q = r * inv_h;
    const bool in = box & (q <= 2.0);
    double w, dw; table_lerp(wt, dwt, nq, dq, inv_dq, in ? q : 0.0, w, dw);
    const double mj = in ? sm[k] : 0.0;
    aW += mj * w;
    aB += mj * (r * dw);
    cand += box ? 1u : 0u;
    contrib += in ? 1u : 0u;
  }
};

// Rounding bound of the walks' FP32 prefilters.  Coordinates are taken relative to g0, the centre of the group's
// position box of half-width gd (largest axis).  A target is within gd of g0 per axis, and a source that can be a
// member at distance r <= 2h within gd + 2h.  Each float coordinate carries at most 2^-24 of its magnitude and the float
// difference 2^-24 of at most 2h: per axis the float difference is off by at most 2^-24 (2 gd + 4h), the float distance
// by at most sqrt(3) 2^-24 (2 gd + 4h) < 4e-7 (gd + 2h).  So a member has r_float <= b = 2h + 4e-7 (gd + 2h); the fmaf
// sum of squares adds < 1e-6 relative, which the caller's 1e-4 covers.  A fixed relative margin would not do: gd is
// the group's width, unrelated to h (a sparse cell's bucket can be 1e4 h wide or more).
__device__ __forceinline__ double group_half_width(const float* lo, const float* hi) {
  return 0.5 * fmax(fmax((double)hi[0] - (double)lo[0], (double)hi[1] - (double)lo[1]), (double)hi[2] - (double)lo[2]);
}
__device__ __forceinline__ double walk_bound(double h, double gd) { return 2.0 * h + 4e-7 * (gd + 2.0 * h); }
// The pair loop's limit for one side is r2max 1.00012 + pad, r2max = 4 h^2 (1 + 1e-9) (INFINITY: keep every partner),
// rounded up: with c = 4e-7 gd, b^2 = (2h (1 + 4e-7) + c)^2 <= r2max (1 + 4e-7)^2 (1 + t) + c^2 (1 + 1/t) for any t > 0;
// t = 1e-5 and the 1e-4 of the fmaf sum give r2max 1.00012 + 1.0001e5 c^2 (4.1e-7: the float arithmetic of c), and the
// larger of the two sides' limits is that of H = max(h_i, h_j).  Where the group is a few h wide, c^2 1e5 is ~1e-8 h^2
// and the limit is the old r2max 1.0001 to 2e-5 of r^2; the pad grows only with the group's width.
__device__ __forceinline__ float pair_pad(const float* lo, const float* hi) {
  const float c = 4.1e-7f * 0.5f * fmaxf(fmaxf(hi[0] - lo[0], hi[1] - lo[1]), hi[2] - lo[2]);
  return __fmul_ru(1.0001e5f, c * c);
}
// r2maxif of the density prefilter: b^2 (1 + 1e-9) (the FP64 limit's margin) rounded up, then the 1e-4 for the fmaf sum
__device__ __forceinline__ float density_bound(double h, double gd) {
  const double b = walk_bound(h, gd);
  return __double2float_ru(b * b * (1.0 + 1e-9)) * 1.0001f;
}

// dynamic shared memory layout: [tables: 2*(nq+1) doubles][per warp: tile 8*WALK_TILE doubles][per warp: stack+cq]
template <bool HITER>
__global__ void __launch_bounds__(DENS_WARPS * 32, 1)
k_density(int n_groups, const int2* __restrict__ groups, DevParams P, DensityArrays A, const BvhBox* __restrict__ box, const __grid_constant__ BvhInfo bi,
          const double* __restrict__ g_wt, const double* __restrict__ g_dwt,
          const double* __restrict__ u, double* __restrict__ h,
          double* __restrict__ rho, double* __restrict__ omega, double* __restrict__ prs, double* __restrict__ cs,
          double* __restrict__ por2, WalkCounters* ctr, int* work, int count_all, NeighbourListSink nl) {
  extern __shared__ double smem[];
  const int nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* wt = smem; double* dwt = smem + (P.nq + 1);
  double* tiles = dwt + (P.nq + 1);
  unsigned* ws = reinterpret_cast<unsigned*>(tiles + (size_t)nwarp * DENS_WARP_DOUBLES);
  for (int i = threadIdx.x; i <= P.nq; i += blockDim.x) { wt[i] = g_wt[i]; dwt[i] = g_dwt[i]; }
  __syncthreads();
  double* tile = tiles + (size_t)warp * DENS_WARP_DOUBLES;
  unsigned* stack = ws + (size_t)warp * WALK_WS;
  unsigned* cq = stack + WALK_STACK;
  const int nchunk = n_groups;
  unsigned long long tot_cand = 0, tot_contrib = 0, tot_iter = 0;
  int res_next = 0, res_end = 0;         // this warp's reserve of list-pool blocks

  for (;;) {
    int chunk = 0;
    if (lane == 0) chunk = atomicAdd(work, 1);
    chunk = __shfl_sync(FULL_MASK, chunk, 0);
    if (chunk >= nchunk) break;
    const int2 tg = groups[chunk];
    const int i = tg.x + lane;
    const bool live = lane < tg.y;
    DensityOp<!HITER> op(A);
    op.sx = tile; op.sy = tile + DENS_SLOTS; op.sz = tile + 2 * DENS_SLOTS; op.sm = tile + 3 * DENS_SLOTS;
    op.scx = tile + 4 * DENS_SLOTS; op.scy = tile + 5 * DENS_SLOTS; op.scz = tile + 6 * DENS_SLOTS; op.sR = tile + 7 * DENS_SLOTS;
    op.ft = reinterpret_cast<float4*>(tile + 8 * DENS_SLOTS);
    op.lbuf = reinterpret_cast<int*>(tile + 10 * DENS_SLOTS);
    op.nl = nl; op.hsrc = h; op.variable_h = P.variable_h; op.h_fixed = P.h_fixed; op.res_next = res_next; op.res_end = res_end;
    op.wt = wt; op.dwt = dwt; op.nq = P.nq; op.dq = P.dq; op.inv_dq = P.inv_dq;
    const BvhBox g = box[bi.off[0] + chunk];
    for (int k = 0; k < 3; ++k) { op.gplo[k] = g.plo[k]; op.gphi[k] = g.phi[k]; op.grlo[k] = g.rlo[k]; op.grhi[k] = g.rhi[k]; }
    op.xi = live ? A.x[i] : 0.0; op.yi = live ? A.y[i] : 0.0; op.zi = live ? A.z[i] : 0.0;
    op.cand = 0; op.contrib = 0; op.count_all = count_all != 0;
    op.g0x = 0.5 * ((double)g.plo[0] + (double)g.phi[0]); op.g0y = 0.5 * ((double)g.plo[1] + (double)g.phi[1]); op.g0z = 0.5 * ((double)g.plo[2] + (double)g.phi[2]);
    op.xif = (float)(op.xi - op.g0x); op.yif = (float)(op.yi - op.g0y); op.zif = (float)(op.zi - op.g0z);
    double hi = live ? (P.variable_h ? h[i] : P.h_fixed) : 1.0;
    const double mi = live ? A.m[i] : 0.0;

    if (!HITER) {
      op.active = live; op.inv_h = 1.0 / hi; op.r2max = 4.0 * hi * hi * (1.0 + 1e-9); op.accW = 0.0; op.accB = 0.0;
      op.g_r2max = warp_max(live ? op.r2max : 0.0);
      op.r2maxif = density_bound(hi, group_half_width(op.gplo, op.gphi));
      op.list_begin(chunk);
      neighbour_walk(op, groups, chunk, box, bi, stack, cq);
      op.list_end();
      res_next = op.res_next; res_end = op.res_end;
      if (live) {
        // W/(pi h^3), dW/(pi h^4): F:125-126 (global smoothing) | V:139-140
        const double hn = P.variable_h ? hi : P.h_fixed;
        const double n3 = P.pi_norm * ((hn * hn) * hn), n4 = P.pi_norm * ((hn * hn) * (hn * hn));
        const double r = op.accW / n3;
        double om = 1.0;
        if (P.variable_h) {
          // Omega = 1 + h/(3 rho) * sum m_j (3W - r dW)/h                                   V:455,487
          const double s = (3.0 * op.accW / n3 - op.accB / n4) / hi;
          om = 1.0 + (hi / (3.0 * r)) * s;
        }
        const double p = P.gm1 * u[i] * r;                               // F:465 | V:509
        const double c = sqrt(P.gamma * p / r);                          // F:466 | V:510
        rho[i] = r; omega[i] = om; prs[i] = p; cs[i] = c;
        const double po = P.variable_h ? p / ((om * r) * r) : p / (r * r);     // V:413 | F:381
        por2[i] = po;
        if (!(fabs(po + c) < INFINITY)) nl.ctl[1] = 1;                        // the pair loop must see every box partner of this particle
      }
      tot_cand += op.cand; tot_contrib += op.contrib;
    } else {
      // calc_smoothing V:515-546 for the 32 targets of this chunk; lanes iterate while growing by > conv
      double r = live ? rho[i] : 1.0, om = live ? omega[i] : 1.0;
      double old_len = hi;
      bool iter = false;
      if (live) {
        const double e3 = P.eta / hi;
        hi = hi * (1.0 + ((mi * ((e3 * e3) * e3) / r) - 1.0) / (3.0 * om));                   // V:527
        if (hi < P.max_length && hi > P.lit_001) iter = (((hi - old_len) / old_len) > P.conv) && (hi < 10.0);   // V:528-529
        else hi = old_len;                                                                   // V:541
      }
      while (__any_sync(FULL_MASK, iter)) {
        op.active = iter; op.inv_h = 1.0 / hi; op.r2max = 4.0 * hi * hi * (1.0 + 1e-9); op.accW = 0.0; op.accB = 0.0;
        op.g_r2max = warp_max(iter ? op.r2max : 0.0);
        if (iter) old_len = hi;
        op.r2maxif = density_bound(hi, group_half_width(op.gplo, op.gphi));
        neighbour_walk(op, groups, chunk, box, bi, stack, cq);
        if (iter) {
          const double n3 = P.pi_norm * ((hi * hi) * hi), n4 = P.pi_norm * ((hi * hi) * (hi * hi));
          r = op.accW / n3;
          const double s = (3.0 * op.accW / n3 - op.accB / n4) / hi;
          om = 1.0 + (hi / (3.0 * r)) * s;                                                   // V:535
          const double e3 = P.eta / hi;
          hi = hi * (1.0 + ((mi * ((e3 * e3) * e3)) / r - 1.0) / (3.0 * om));                 // V:538
          ++tot_iter;
          iter = (((hi - old_len) / old_len) > P.conv) && (hi < 10.0);
        }
      }
      if (live) { h[i] = hi; rho[i] = r; omega[i] = om; }
    }
  }
  if (!HITER) {
    tot_cand = (unsigned long long)warp_sum_ll((long long)tot_cand);
    tot_contrib = (unsigned long long)warp_sum_ll((long long)tot_contrib);
    if (lane == 0) { atomicAdd(&ctr->dens_cand, tot_cand); atomicAdd(&ctr->dens_contrib, tot_contrib); }
  } else {
    tot_iter = (unsigned long long)warp_sum_ll((long long)tot_iter);
    if (lane == 0) atomicAdd(&ctr->h_iters, tot_iter);
  }
}

// ------------------------------------------------------------------------------------------------------
// SPH pair force operator (gather form)
// ------------------------------------------------------------------------------------------------------
struct ForceArrays {
  const double *x, *y, *z, *vx, *vy, *vz, *m, *h, *rho, *c, *alpha, *por2, *lcx, *lcy, *lcz, *reach;
  const int* id;
};
#define FORCE_FIELDS 18
#define FORCE_TG_FIELDS 19
#define FORCE_WARP_DOUBLES (FORCE_FIELDS * WALK_TILE + FORCE_TG_FIELDS * 32 + 5 * PAIR_WIN + PAIR_WIN / 4 + 2 * WALK_TILE + 2)   // tile + targets + results + hit list + float4 tile + the group's pair_pad

struct ForceOp {
  static const bool SYMMETRIC = true;
  static const bool LISTS = false;
  static const bool FUSED = false;
  double* t;             // tile: FORCE_FIELDS arrays of WALK_TILE doubles
  int* tid;              // tile ids
  double* tg;            // the group's targets: FORCE_TG_FIELDS arrays of 32 doubles (x y z vx vy vz h 1/h 1/(pi h^4) rho c alpha P/(Omega rho^2)
                         //   leaf centre (3) reach r2max id)
  float4* ft;            // float copy of the tile for the prefilter: position relative to the group's origin, r2max rounded up
  double g0x, g0y, g0z;  // the group's origin (centre of its position box)
  float xif, yif, zif, r2maxif;
  double* res;           // pair results of the current window: f dx, f dy, f dz, u, a
  unsigned short* plist; // compacted hit list of the current window: (target lane << 5) | tile slot
  const ForceArrays& A;
  const double* dwt; int nq; double dq, inv_dq;
  float gplo[3], gphi[3], grlo[3], grhi[3];
  int variable_h; double h_fixed, pi_norm, lit_001;
  // lane state
  bool live;
  double xi, yi, zi;
  double g_r2max; bool count_all;   // group maximum of r2max; exact pair counter wanted (no early cull)
  double ax, ay, az, ud, ad;
  unsigned pairs;

  __device__ ForceOp(const ForceArrays& a) : A(a) {}

  __device__ __forceinline__ bool source_filter(int j) const {
    // all loads first (independent, one latency), then a branch-free decision
    const double R = A.reach[j], cx = A.lcx[j], cy = A.lcy[j], cz = A.lcz[j], px = A.x[j], py = A.y[j], pz = A.z[j];
    const double hj = variable_h ? A.h[j] : h_fixed;
    const double fj = A.por2[j] + A.c[j];          // NaN / inf here spreads through 0 * NaN in the reference: never cull it
    const bool a = (cx - R <= (double)gphi[0]) & (cx + R >= (double)gplo[0]) &
                   (cy - R <= (double)gphi[1]) & (cy + R >= (double)gplo[1]) &
                   (cz - R <= (double)gphi[2]) & (cz + R >= (double)gplo[2]);
    const bool b = (px >= (double)grlo[0]) & (px <= (double)grhi[0]) & (py >= (double)grlo[1]) & (py <= (double)grhi[1]) &
                   (pz >= (double)grlo[2]) & (pz <= (double)grhi[2]);
    // farther than 2 max(h_i, h_j) from every target of the group: both kernel gradients are exact zeros
    const double ex = fmax(fmax((double)gplo[0] - px, px - (double)gphi[0]), 0.0), ey = fmax(fmax((double)gplo[1] - py, py - (double)gphi[1]), 0.0),
                 ez = fmax(fmax((double)gplo[2] - pz, pz - (double)gphi[2]), 0.0);
    const bool nz = !(ex * ex + ey * ey + ez * ez > fmax(g_r2max, 4.0 * hj * hj * (1.0 + 1e-9))) | !(fabs(fj) < INFINITY);
    // R <= 0: j sits in a depth-limited multi-particle node - nobody finds it (a), but it still visits others (b)
    return (((R > 0.0) & a) | b) & (nz | count_all);
  }
  __device__ __forceinline__ void stage(int s, int j) {
    const double hj = variable_h ? A.h[j] : h_fixed;
    t[0 * WALK_TILE + s] = A.x[j];  t[1 * WALK_TILE + s] = A.y[j];  t[2 * WALK_TILE + s] = A.z[j];
    t[3 * WALK_TILE + s] = A.vx[j]; t[4 * WALK_TILE + s] = A.vy[j]; t[5 * WALK_TILE + s] = A.vz[j];
    t[6 * WALK_TILE + s] = A.m[j];  t[7 * WALK_TILE + s] = hj;
    t[8 * WALK_TILE + s] = 1.0 / (pi_norm * ((hj * hj) * (hj * hj)));
    t[17 * WALK_TILE + s] = 1.0 / hj;
    t[9 * WALK_TILE + s] = A.rho[j]; t[10 * WALK_TILE + s] = A.c[j]; t[11 * WALK_TILE + s] = A.alpha[j];
    t[12 * WALK_TILE + s] = A.por2[j];
    t[13 * WALK_TILE + s] = A.lcx[j]; t[14 * WALK_TILE + s] = A.lcy[j]; t[15 * WALK_TILE + s] = A.lcz[j];
    t[16 * WALK_TILE + s] = A.reach[j];
    tid[s] = A.id[j];
    const double r2max_j = (fabs(A.por2[j] + A.c[j]) < INFINITY) ? 4.0 * hj * hj * (1.0 + 1e-9) : INFINITY;
    ft[s] = make_float4((float)(t[0 * WALK_TILE + s] - g0x), (float)(t[1 * WALK_TILE + s] - g0y), (float)(t[2 * WALK_TILE + s] - g0z),
                        __fmaf_ru(__double2float_ru(r2max_j), 1.00012f, reinterpret_cast<const float*>(ft + WALK_TILE)[0]));
  }
  __device__ __forceinline__ void consume(int count) {
    // Prefilter, lane = target, FP32: |x_i - x_j|^2 against the larger of the two sides' limits (pair_pad), which
    // bounds the square of b = 2H + 4e-7 (gd + 2H), H = max(h_i, h_j) (walk_bound), the float distance of any pair
    // with a non-zero term (r <= 2H).  It only ever drops pairs whose every term is an exact zero; the reference's own membership test (FP64, F:351-354 |
    // V:380-383) and the exact distance cull run in the lane = pair phase on the survivors.  With the exact pair
    // counter on, every staged source is a candidate.
    unsigned mask = 0;
    if (live) {
      if (count_all) mask = count >= 32 ? 0xffffffffu : ((1u << count) - 1u);
      else {
#pragma unroll 4
        for (int k = 0; k < count; ++k) {
          const float4 sj = ft[k];
          const float dx = xif - sj.x, dy = yif - sj.y, dz = zif - sj.z;
          const float r2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
          const bool far = r2 > fmaxf(r2maxif, sj.w);
          mask |= (far ? 0u : 1u) << k;
        }
      }
    }
#ifdef SCREEN_AUDIT
    if (live && !count_all) {            // every staged source the screen dropped: the lane = pair phase's FP64 decision
      const double* g = tg + (threadIdx.x & 31);
      const int idi_ = (int)g[18 * 32];
      unsigned bad = 0;
      for (int k = 0; k < count; ++k) {
        if ((mask >> k) & 1u) continue;
        const int idj = tid[k];
        const bool lt = idj < idi_;
        const double xj = t[0 * WALK_TILE + k], yj = t[1 * WALK_TILE + k], zj = t[2 * WALK_TILE + k];
        const double px = lt ? g[0 * 32] : xj, py = lt ? g[1 * 32] : yj, pz = lt ? g[2 * 32] : zj;
        const double cx = lt ? t[13 * WALK_TILE + k] : g[13 * 32], cy = lt ? t[14 * WALK_TILE + k] : g[14 * 32], cz = lt ? t[15 * WALK_TILE + k] : g[15 * 32];
        const double R = lt ? t[16 * WALK_TILE + k] : g[16 * 32];
        const bool in = (idj != idi_) & (fabs(px - cx) < R) & (fabs(py - cy) < R) & (fabs(pz - cz) < R);
        const double dx = g[0 * 32] - xj, dy = g[1 * 32] - yj, dz = g[2 * 32] - zj;
        const double hj_ = t[7 * WALK_TILE + k];
        const double r2max_j = (fabs(t[12 * WALK_TILE + k] + t[10 * WALK_TILE + k]) < INFINITY) ? 4.0 * hj_ * hj_ * (1.0 + 1e-9) : INFINITY;
        bad += (in & !(dx * dx + dy * dy + dz * dz > fmax(g[17 * 32], r2max_j))) ? 1u : 0u;
      }
      if (bad) atomicAdd(&screen_audit[1], (unsigned long long)bad);
    }
#endif
    // Compact the hits (target lane, tile slot) of the whole warp and evaluate them with lane = pair: the
    // ~95 FP64 instructions of a pair run with every lane busy however unevenly a tile's sources fall among
    // the targets.  Each target then adds its own terms in tile order (F:383-391, own side; deterministic).
    const int lane = threadIdx.x & 31;
    const int c = __popc(mask);
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += v; }
    const int total = __shfl_sync(FULL_MASK, incl, 31);
    unsigned mw = mask, ms = mask;
    int gw = incl - c, gs = gw;
    for (int base = 0; base < total; base += PAIR_WIN) {
      const int lim = base + PAIR_WIN;
      while (mw && gw < lim) { const int k = __ffs(mw) - 1; mw &= mw - 1; plist[gw - base] = (unsigned short)((lane << 5) | k); ++gw; }
      __syncwarp();
      const int nwin = total - base < PAIR_WIN ? total - base : PAIR_WIN;
      for (int p = lane; p < nwin; p += 32) {
        const int e = plist[p], tl = e >> 5, k = e & 31;
        // idj < idi: i is the higher-numbered `body`: is x_i inside Box(j)?   F:351-354 | V:380-383
        // idj > idi: j is the `body` that visits i: is x_j inside Box(i)?   (Box(i) is empty when R_i = -1)
        const double* g = tg + tl;
        const int idj = tid[k], idi_ = (int)g[18 * 32];
        const bool lt = idj < idi_;
        const double xi_ = g[0 * 32], yi_ = g[1 * 32], zi_ = g[2 * 32];
        const double xj = t[0 * WALK_TILE + k], yj = t[1 * WALK_TILE + k], zj = t[2 * WALK_TILE + k];
        const double px = lt ? xi_ : xj, py = lt ? yi_ : yj, pz = lt ? zi_ : zj;
        const double cx = lt ? t[13 * WALK_TILE + k] : g[13 * 32], cy = lt ? t[14 * WALK_TILE + k] : g[14 * 32], cz = lt ? t[15 * WALK_TILE + k] : g[15 * 32];
        const double R = lt ? t[16 * WALK_TILE + k] : g[16 * 32];
        const bool in = (idj != idi_) & (fabs(px - cx) < R) & (fabs(py - cy) < R) & (fabs(pz - cz) < R);
        const double dx = xi_ - xj, dy = yi_ - yj, dz = zi_ - zj;
        const double hj_ = t[7 * WALK_TILE + k];
        const double r2max_j = (fabs(t[12 * WALK_TILE + k] + t[10 * WALK_TILE + k]) < INFINITY) ? 4.0 * hj_ * hj_ * (1.0 + 1e-9) : INFINITY;
        const bool nz = !(dx * dx + dy * dy + dz * dz > fmax(g[17 * 32], r2max_j));
        pairs += in ? 1u : 0u;
        double f = 0.0, u = 0.0, a = 0.0;
        if (in & nz) pair(tl, k, f, u, a);
        res[p] = f * dx; res[PAIR_WIN + p] = f * dy; res[2 * PAIR_WIN + p] = f * dz;      // F:383 (own side)
        res[3 * PAIR_WIN + p] = u; res[4 * PAIR_WIN + p] = a;
      }
      __syncwarp();
      const int ge = gs + __popc(ms) < lim ? gs + __popc(ms) : lim;       // this lane's hits are contiguous in the list
      for (; gs < ge; ++gs) {
        const int q = gs - base;
        ax -= res[q]; ay -= res[PAIR_WIN + q]; az -= res[2 * PAIR_WIN + q];
        ud += res[3 * PAIR_WIN + q]; ad += res[4 * PAIR_WIN + q];
        ms &= ms - 1;
      }
      __syncwarp();
    }
  }
  // one pair (target lane tl, tile slot k): f = m_j * A / dr  (a_i -= f * (x_i - x_j)), u = du/dt term, a = alpha-rate term
  __device__ __forceinline__ void pair(int tl, int k, double& f, double& u, double& a) const {
    const double* g = tg + tl;
    const double nx = g[0 * 32] - t[0 * WALK_TILE + k], ny = g[1 * 32] - t[1 * WALK_TILE + k], nz = g[2 * 32] - t[2 * WALK_TILE + k];   // F:356
    const double wx = g[3 * 32] - t[3 * WALK_TILE + k], wy = g[4 * 32] - t[4 * WALK_TILE + k], wz = g[5 * 32] - t[5 * WALK_TILE + k];   // F:358
    const double hi_ = g[6 * 32], inv_hi_ = g[7 * 32], inv_n4i_ = g[8 * 32], rhoi_ = g[9 * 32], ci_ = g[10 * 32], alphai_ = g[11 * 32], por2i_ = g[12 * 32];
    const double r2 = nx * nx + ny * ny + nz * nz;
    double dr, inv_dr; fast_sqrt_rsqrt(r2, dr, inv_dr);                 // dr == 0 -> NaN like F:363
    const double rv = wx * nx + wy * ny + wz * nz;
    const double vdotr = rv >= 0.0 ? 0.0 : rv;                          // F:361
    const double mj = t[6 * WALK_TILE + k], hj = t[7 * WALK_TILE + k];
    // kernel gradient magnitudes dW/dr at h_i and h_j                                   F:366 | V:395-396
    const double qi = dr * inv_hi_;
    const bool ini = qi <= 2.0;
    const double dWi = ini ? table_lerp1(dwt, nq, dq, inv_dq, qi) * inv_n4i_ : ((qi != qi) ? qi : 0.0);
    double dWj = dWi;
    if (variable_h) {
      const double qj = dr * t[17 * WALK_TILE + k];
      const bool inj = qj <= 2.0;
      dWj = inj ? table_lerp1(dwt, nq, dq, inv_dq, qj) * t[8 * WALK_TILE + k] : 0.0;
    }
    const double hbar = variable_h ? (hi_ + hj) / 2.0 : hi_;            // V:402
    const double nu = (hbar * vdotr) * fast_rcp(r2 + lit_001 * hbar * hbar);   // F:373 | V:405
    const double cbar = 0.5 * (ci_ + t[10 * WALK_TILE + k]);
    const double abar = 0.5 * (alphai_ + t[11 * WALK_TILE + k]);
    const double visc = (-abar * cbar * nu + 2.0 * abar * nu * nu) * fast_rcp(0.5 * (rhoi_ + t[9 * WALK_TILE + k]));   // F:378 | V:410
    const double por2j = t[12 * WALK_TILE + k];
    const double rvn = rv * inv_dr;                                     // n_hat . v_ij
    double scal, vdg;
    if (variable_h) {
      vdg = (dWi * rvn + dWj * rvn) / 2.0;                              // V:401
      scal = (por2i_ * dWi + por2j * dWj) + visc * (dWi + dWj) / 2.0;   // V:413-414
    } else {
      vdg = dWi * rvn;                                                  // F:370
      scal = ((por2i_ + por2j) + visc) * dWi;                           // F:381-382
    }
    f = mj * scal * inv_dr;
    u = mj * vdg * (por2i_ + 0.5 * visc);                               // F:387 | V:419-421
    a = mj * vdg;                                                       // F:390
  }
};

// Multi-GPU: the pair kernel is the last writer of a, du/dt and d(alpha)/dt, and every rank needs them for all
// particles (replicated integration).  Instead of copying the finished slice afterwards, the kernel stores each value
// into every peer's copy of the arrays as it is produced (peer-mapped pointers, NVLink stores), so the exchange
// overlaps the walk and only a barrier remains after the kernel.
#define SPH_MAX_PEERS 7
struct PeerOut { int n; double* p[SPH_MAX_PEERS][5]; };

// LISTED: stream the group's saved candidate chain (written by the density pass of this evaluation) instead of
// walking the BVH and filtering the sources again; runs only while the lists are usable (nl.ctl[1] == 0).
// !LISTED: the walking form; with only_if_void it runs only when the lists were declared void on the device.
template <bool LISTED>
__global__ void __launch_bounds__(512, 1)
k_force(int n_groups, const int2* __restrict__ groups, DevParams P, ForceArrays A, const BvhBox* __restrict__ box, const __grid_constant__ BvhInfo bi, const double* __restrict__ g_dwt,
        double* __restrict__ ax, double* __restrict__ ay, double* __restrict__ az, double* __restrict__ udot,
        double* __restrict__ adot, WalkCounters* ctr, int* work, int count_all, NeighbourListSink nl, int only_if_void, const __grid_constant__ PeerOut po) {
  if (LISTED) { if (nl.ctl[1] != 0) return; }
  else if (only_if_void && nl.ctl[1] == 0) return;
  extern __shared__ double smem[];
  const int nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* dwt = smem;
  double* tiles = dwt + (P.nq + 1) + ((P.nq + 1) & 1);
  int* tids = reinterpret_cast<int*>(tiles + (size_t)nwarp * FORCE_WARP_DOUBLES);
  unsigned* ws = reinterpret_cast<unsigned*>(tids + (size_t)nwarp * WALK_TILE);     // only the walking form uses (and sizes) it
  for (int i = threadIdx.x; i <= P.nq; i += blockDim.x) dwt[i] = g_dwt[i];
  __syncthreads();
  double* tile = tiles + (size_t)warp * FORCE_WARP_DOUBLES;
  unsigned* stack = ws + (size_t)warp * WALK_WS;
  unsigned* cq = stack + WALK_STACK;
  const int nchunk = n_groups;
  unsigned long long tot_pairs = 0;
  for (;;) {
    int chunk = 0;
    if (lane == 0) chunk = atomicAdd(work, 1);
    chunk = __shfl_sync(FULL_MASK, chunk, 0);
    if (chunk >= nchunk) break;
    const int2 tg = groups[chunk];
    const int i = tg.x + lane;
    const bool live = lane < tg.y;
    ForceOp op(A);
    op.t = tile; op.tid = tids + warp * WALK_TILE;
    op.tg = tile + FORCE_FIELDS * WALK_TILE; op.res = op.tg + FORCE_TG_FIELDS * 32;
    op.plist = reinterpret_cast<unsigned short*>(op.res + 5 * PAIR_WIN);
    op.ft = reinterpret_cast<float4*>(op.res + 5 * PAIR_WIN + PAIR_WIN / 4);
    op.dwt = dwt; op.nq = P.nq; op.dq = P.dq; op.inv_dq = P.inv_dq;
    op.variable_h = P.variable_h; op.h_fixed = P.h_fixed; op.pi_norm = P.pi_norm; op.lit_001 = P.lit_001;
    const BvhBox g = box[bi.off[0] + chunk];
    for (int k = 0; k < 3; ++k) { op.gplo[k] = g.plo[k]; op.gphi[k] = g.phi[k]; op.grlo[k] = g.rlo[k]; op.grhi[k] = g.rhi[k]; }
    op.live = live;
    const int ii = live ? i : 0;
    op.xi = A.x[ii]; op.yi = A.y[ii]; op.zi = A.z[ii];
    const double hi = P.variable_h ? A.h[ii] : P.h_fixed, rhoi = A.rho[ii], ci = A.c[ii], alphai = A.alpha[ii], por2i = A.por2[ii];
    {
      double* g = op.tg + lane;
      g[0 * 32] = op.xi; g[1 * 32] = op.yi; g[2 * 32] = op.zi; g[3 * 32] = A.vx[ii]; g[4 * 32] = A.vy[ii]; g[5 * 32] = A.vz[ii];
      g[6 * 32] = hi; g[7 * 32] = 1.0 / hi; g[8 * 32] = 1.0 / (P.pi_norm * ((hi * hi) * (hi * hi)));
      g[9 * 32] = rhoi; g[10 * 32] = ci; g[11 * 32] = alphai; g[12 * 32] = por2i;
    }
    const double r2max = (fabs(por2i + ci) < INFINITY) ? 4.0 * hi * hi * (1.0 + 1e-9) : INFINITY;   // own NaN: keep every partner
    {
      double* g = op.tg + lane;
      g[13 * 32] = A.lcx[ii]; g[14 * 32] = A.lcy[ii]; g[15 * 32] = A.lcz[ii]; g[16 * 32] = A.reach[ii]; g[17 * 32] = r2max; g[18 * 32] = (double)A.id[ii];
    }
    op.g0x = 0.5 * ((double)g.plo[0] + (double)g.phi[0]); op.g0y = 0.5 * ((double)g.plo[1] + (double)g.phi[1]); op.g0z = 0.5 * ((double)g.plo[2] + (double)g.phi[2]);
    op.xif = (float)(op.xi - op.g0x); op.yif = (float)(op.yi - op.g0y); op.zif = (float)(op.zi - op.g0z);
    {
      const float pad = pair_pad(op.gplo, op.gphi);          // kept in shared memory (after the float tile) for stage()
      if (lane == 0) reinterpret_cast<float*>(op.ft + WALK_TILE)[0] = pad;
      op.r2maxif = __fmaf_ru(__double2float_ru(r2max), 1.00012f, pad);
    }
    op.g_r2max = warp_max(live ? r2max : 0.0); op.count_all = count_all != 0;
    op.ax = op.ay = op.az = op.ud = op.ad = 0.0; op.pairs = 0;
    __syncwarp();
    if (LISTED) {
      // one block = one tile; the next block's words are requested before the current tile is consumed
      int blk = nl.head[chunk];
      int v = nl.pool[(size_t)blk * 32 + lane];
      for (;;) {
        const int cnt = __shfl_sync(FULL_MASK, v, 30), nxt = __shfl_sync(FULL_MASK, v, 31);
        int vn = 0;
        if (nxt >= 0) vn = nl.pool[(size_t)nxt * 32 + lane];
        if (cnt > 0) {
          if (lane < cnt) op.stage(lane, v);
          __syncwarp();
          op.consume(cnt);
          __syncwarp();
        }
        if (nxt < 0) break;
        v = vn;
      }
    } else {
      neighbour_walk(op, groups, chunk, box, bi, stack, cq);
    }
    if (live) {
      const double vax = ax[i] + op.ax, vay = ay[i] + op.ay, vaz = az[i] + op.az, vud = udot[i] + op.ud;
      // alpha-rate clean-up F:316-318 | V:345-347
      const double vad = fmax(op.ad / rhoi, 0.0) + P.lit_015 * ((0.1 - alphai) * ci / hi);
      ax[i] = vax; ay[i] = vay; az[i] = vaz; udot[i] = vud; adot[i] = vad;
      for (int r = 0; r < po.n; ++r) {
        po.p[r][0][i] = vax; po.p[r][1][i] = vay; po.p[r][2][i] = vaz; po.p[r][3][i] = vud; po.p[r][4][i] = vad;
      }
    }
    tot_pairs += op.pairs;
  }
  tot_pairs = (unsigned long long)warp_sum_ll((long long)tot_pairs);
  if (lane == 0) atomicAdd(&ctr->sph_pairs, tot_pairs);    // each unordered pair is seen from both sides
}

// ------------------------------------------------------------------------------------------------------
// neighbour diagnostics: per-target candidate count + order-independent hash, optional CSR list
// ------------------------------------------------------------------------------------------------------
struct NgbOp {
  static const bool SYMMETRIC = false;
  static const bool LISTS = false;
  static const bool FUSED = false;
  double *scx, *scy, *scz, *sR; int* sid;
  const DensityArrays& A; const int* id;
  float gplo[3], gphi[3];
  double xi, yi, zi; bool live;
  unsigned count; unsigned long long hash;
  int* out;              // CSR row start for this lane or nullptr
  __device__ NgbOp(const DensityArrays& a) : A(a) {}
  __device__ __forceinline__ bool source_filter(int j) const {
    double R = A.reach[j];
    if (!(R > 0.0)) return false;
    double cx = A.lcx[j], cy = A.lcy[j], cz = A.lcz[j];
    return (cx - R <= (double)gphi[0]) && (cx + R >= (double)gplo[0]) && (cy - R <= (double)gphi[1]) && (cy + R >= (double)gplo[1]) &&
           (cz - R <= (double)gphi[2]) && (cz + R >= (double)gplo[2]);
  }
  __device__ __forceinline__ void stage(int s, int j) {
    scx[s] = A.lcx[j]; scy[s] = A.lcy[j]; scz[s] = A.lcz[j]; sR[s] = A.reach[j]; sid[s] = id[j];
  }
  __device__ __forceinline__ void consume(int cnt) {
    if (!live) return;
    for (int k = 0; k < cnt; ++k) {
      double R = sR[k];
      bool in = (fabs(xi - scx[k]) < R) && (fabs(yi - scy[k]) < R) && (fabs(zi - scz[k]) < R);
      if (in) { if (out) out[count] = sid[k]; ++count; hash += mix64((unsigned long long)sid[k]); }
    }
  }
};

__global__ void __launch_bounds__(256)
k_neighbours(int n_groups, const int2* __restrict__ groups, DensityArrays A, const int* __restrict__ id, const BvhBox* __restrict__ box, const __grid_constant__ BvhInfo bi,
             int* __restrict__ count, unsigned long long* __restrict__ hash, const long long* __restrict__ offsets,
             int* __restrict__ list) {
  extern __shared__ double smem[];
  const int nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* tile = smem + (size_t)warp * 4 * WALK_TILE;
  int* sid = reinterpret_cast<int*>(smem + (size_t)nwarp * 4 * WALK_TILE) + warp * WALK_TILE;
  unsigned* ws = reinterpret_cast<unsigned*>(reinterpret_cast<int*>(smem + (size_t)nwarp * 4 * WALK_TILE) + nwarp * WALK_TILE);
  unsigned* stack = ws + (size_t)warp * WALK_WS;
  unsigned* cq = stack + WALK_STACK;
  const int nchunk = n_groups;
  for (int chunk = blockIdx.x * nwarp + warp; chunk < nchunk; chunk += gridDim.x * nwarp) {
    const int2 tg = groups[chunk];
    const int i = tg.x + lane;
    NgbOp op(A);
    op.scx = tile; op.scy = tile + WALK_TILE; op.scz = tile + 2 * WALK_TILE; op.sR = tile + 3 * WALK_TILE; op.sid = sid; op.id = id;
    const BvhBox g = box[bi.off[0] + chunk];
    for (int k = 0; k < 3; ++k) { op.gplo[k] = g.plo[k]; op.gphi[k] = g.phi[k]; }
    op.live = lane < tg.y;
    op.xi = op.live ? A.x[i] : 0.0; op.yi = op.live ? A.y[i] : 0.0; op.zi = op.live ? A.z[i] : 0.0;
    op.count = 0; op.hash = 0;
    op.out = (list && op.live) ? list + offsets[i] : nullptr;
    neighbour_walk(op, groups, chunk, box, bi, stack, cq);
    if (op.live) { count[i] = (int)op.count; hash[i] = op.hash; }
  }
}
