// sph_domain.cuh — kernels of the Morton-domain decomposition (multi-GPU form of north_star / SURVEY.md §8(e)).
//
// Rank r owns one contiguous range of the global descent-key order (the order create_tree / build_tree give the
// leaves, SUMMER_SPH.f90:795-816, 149-246).  Keys are taken in the all-reduced root cube, so a rank's sorted slice IS
// the global order restricted to it and every leaf cell equals the single-rank tree's.  Per tree build:
//   samples -> splitters -> particles migrate to their owners (pulled over peer-mapped memory)
//   local octree; the few cells that straddle a domain boundary form the TOP TREE, assembled on every rank from an
//     all-gather of their locally complete children (k_dd_top_contrib) with the single-rank summation order
//   locally essential tree: nodes of the peers' subtrees that some particle of this domain may open are pulled
//     breadth-first straight out of the peers' node arrays (k_dd_let_level)
//   halo: walk groups of the peers whose reach / position box touches this domain are pulled behind the own
//     particles (k_dd_halo_mark, k_dd_pull); the density / pair / gravity kernels then run unchanged on
//     [own | halo] with the own groups as targets.
#pragma once
#include "sph_common.cuh"
#include "sph_walk.cuh"

#define DD_MAX_RANKS 8
#define DD_SAMPLES 2048            // key samples per rank for the splitter search
#define DD_TOP_CAP 4096            // walk-layout slots reserved for the top tree (straddling cells x children)
#define DD_MAX_CELLS 512           // straddling cells (<= (ranks - 1) x 22 levels)
#define DD_PULL_FIELDS 16

// per-rank facts the others need after a tree build (all-gathered on the host)
struct DDInfo { long long n_own; int ng_own, cur, key_slot, perm_slot; unsigned long long first_key, last_key; int n_acc, pad; };

// ---- splitters ------------------------------------------------------------------------------------------------------
__global__ void k_dd_samples(int n, const uint64_t* __restrict__ key, int S, uint64_t* __restrict__ out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  out[s] = n > 0 ? key[(long long)s * n / S] : ~0ull;
}
// samples: R rows of S sorted keys; counts[q] = particles of rank q.  Block k finds splitter k + 1: the smallest key x
// with  sum_q (counts[q] / S) * #{samples of q < x}  >=  (k + 1) N / R  (every rank runs the same arithmetic on the same
// all-gathered input).  The samples are staged in shared memory and one warp narrows [lo, hi] with 32 probes per round
// (13 rounds instead of 63 dependent bisection steps through global memory: this kernel was most of the migration stage).
// split[0] = 0.  Dynamic shared memory: R * S keys.
__global__ void k_dd_splitters(int R, int S, const uint64_t* __restrict__ samples, const long long* __restrict__ counts,
                               uint64_t* __restrict__ split) {
  extern __shared__ uint64_t dd_sm[];
  for (int i = threadIdx.x; i < R * S; i += blockDim.x) dd_sm[i] = samples[i];
  __syncthreads();
  const int k = blockIdx.x, lane = threadIdx.x;
  if (k == 0 && lane == 0) split[0] = 0ull;
  if (lane >= 32) return;
  long long N = 0;
  for (int q = 0; q < R; ++q) N += counts[q];
  const double target = (double)(k + 1) * (double)N / (double)R;
  auto pass = [&](uint64_t x) {                  // estimated number of particles with key < x reaches the target
    double f = 0.0;
    for (int q = 0; q < R; ++q) {
      const uint64_t* sq = dd_sm + (size_t)q * S;
      int lo = 0, hi = S;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (sq[mid] < x) lo = mid + 1; else hi = mid; }
      f += (double)counts[q] * (double)lo / (double)S;
    }
    return f >= target;
  };
  uint64_t lo = 0ull, hi = 1ull << 63;           // smallest x in [lo, hi] that passes (hi itself if none below it does); keys are 63-bit
  while (lo < hi) {
    const uint64_t width = hi - lo, step = width / 32 + 1;
    const uint64_t p = lo + (uint64_t)lane * step;
    const bool in = p < hi;
    const bool ok = in ? pass(p) : true;
    const unsigned bal = __ballot_sync(FULL_MASK, ok);
    if (bal == 0u) { lo = lo + 31ull * step + 1ull; continue; }   // all 32 probes lie below hi and fail
    const int f = __ffs(bal) - 1;
    if (f == 0) { hi = lo; break; }
    hi = min(hi, lo + (uint64_t)f * step);       // first passing probe (or hi when it lies beyond)
    lo = lo + (uint64_t)(f - 1) * step + 1;      // one past the last failing probe
  }
  if (lane == 0) split[k + 1] = lo;
}
// first sorted index of every destination rank's segment: send_off[r] = #{keys < split[r]}, send_off[R] = n; and the
// first / last key of every segment (segkeys[r], segkeys[DD_MAX_RANKS + r]; 0 when empty): with all ranks' tables every
// rank knows every domain's boundary keys and size after the migration without asking again.  One warp.
__global__ void k_dd_segments(int R, int n, const uint64_t* __restrict__ key, const uint64_t* __restrict__ split, int* __restrict__ send_off,
                              uint64_t* __restrict__ segkeys) {
  const int r = threadIdx.x;
  int lo = n;
  if (r < R) {
    const uint64_t x = split[r];
    int hi = n; lo = 0;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (key[mid] < x) lo = mid + 1; else hi = mid; }
  }
  const int next = __shfl_down_sync(FULL_MASK, lo, 1);
  if (r <= R) send_off[r] = lo;
  if (r < R) { segkeys[r] = next > lo ? key[lo] : 0ull; segkeys[DD_MAX_RANKS + r] = next > lo ? key[next - 1] : 0ull; }
}

// ---- migration: every rank pulls what it now owns out of the peers' (unsorted) state through their sort permutation
struct DDMigrate {
  int R; int dst_off[DD_MAX_RANKS + 1];         // destination offsets (prefix of the incoming counts)
  int src_off[DD_MAX_RANKS];                    // first sorted index of my segment on rank q
  const double* st[DD_MAX_RANKS][10]; const int* id[DD_MAX_RANKS]; const uint64_t* key[DD_MAX_RANKS]; const int* perm[DD_MAX_RANKS];
  double* dst[10]; int* dst_id; uint64_t* dst_key;
};
__global__ void k_dd_migrate(const __grid_constant__ DDMigrate a) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.dst_off[a.R]) return;
  int q = 0;
  while (q + 1 < a.R && t >= a.dst_off[q + 1]) ++q;
  const int k = a.src_off[q] + (t - a.dst_off[q]);
  const int j = a.perm[q][k];
  a.dst_key[t] = a.key[q][k];
  a.dst_id[t] = a.id[q][j];
#pragma unroll
  for (int f = 0; f < 10; ++f) a.dst[f][t] = a.st[q][f][j];
}

// ---- top tree: locally complete children of the cells that straddle a domain boundary ---------------------------------
struct DDCell { uint64_t prefix; int level; int child_top; };    // child_top bit c: child octant c straddles too (is a top cell itself)
struct DDContrib { double m, sx, sy, sz, size; int count, nchild, child, row; };      // row: the particle's local row when count == 1, else -1
// one thread per (cell, octant): if the child cell is not a top cell and holds particles of THIS rank, the rank owns all
// of it: report its node (pre-finalize sums, so the top nodes add children exactly like k_oct_up does)
__global__ void k_dd_top_contrib(int ncell, const DDCell* __restrict__ cells, int n, const uint64_t* __restrict__ key,
                                 const int* __restrict__ off, const int* __restrict__ cnt, const int* __restrict__ node_count,
                                 const GNode* __restrict__ nodes, const int* __restrict__ wcount, const int* __restrict__ wstart,
                                 DDContrib* __restrict__ out, int* err_flag) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ncell * 8) return;
  DDContrib rec; rec.m = rec.sx = rec.sy = rec.sz = rec.size = 0.0; rec.count = rec.nchild = rec.child = 0; rec.row = -1;
  const DDCell C = cells[t >> 3]; const int c = t & 7;
  if (!((C.child_top >> c) & 1) && n > 0 && C.level < SPH_KEY_LEVELS) {
    const int shift = 3 * (SPH_KEY_LEVELS - 1 - C.level);
    const uint64_t kmin = C.prefix | ((uint64_t)c << shift), kmax = kmin | ((1ull << shift) - 1ull);
    int lo = 0, hi = n;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (key[mid] < kmin) lo = mid + 1; else hi = mid; }
    const int a = lo; hi = n;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (key[mid] <= kmax) lo = mid + 1; else hi = mid; }
    const int b = lo - 1;
    if (b >= a) {
      int v = -1;
      if (a == b) v = a + off[a] + cnt[a];
      else for (int k = 0; k < cnt[a]; ++k) if (node_count[a + off[a] + k] == b - a + 1) { v = a + off[a] + k; break; }
      if (v < 0) { atomicExch(err_flag, 4); }
      else {
        const GNode g = nodes[v];
        rec.m = g.m; rec.sx = g.cx; rec.sy = g.cy; rec.sz = g.cz; rec.size = g.size;
        rec.count = b - a + 1; rec.nchild = wcount[v]; rec.child = 1 + wstart[v]; rec.row = a == b ? a : -1;
      }
    }
  }
  out[t] = rec;
}

// ---- what decides "near this domain": the 8-ary BVH over the OWN walk groups (level 0 = the exported group boxes in
// c->bvh, upper levels in a private array that bi.off[l >= 1] indexes), walked per query with early exit.  A chunk of a Morton range can span a whole
// parent cell, so a fixed handful of chunk boxes selected most of the other domain; the group boxes themselves are tight.
template <class PRED>
__device__ __forceinline__ bool dd_bvh_any(const BvhBox* __restrict__ lvl0, const BvhBox* __restrict__ upper, const BvhInfo& bi, PRED pred) {
  int stack[112]; int sn = 0;                                    // <= 32 top boxes + 7 net pushes per level
  const int top = bi.nlev - 1;
  const BvhBox* tb = top == 0 ? lvl0 : upper + bi.off[top];
  for (int i = 0; i < bi.cnt[top]; ++i) if (pred(tb[i])) { if (top == 0) return true; stack[sn++] = (top << 27) | i; }
  while (sn > 0) {
    const int e = stack[--sn]; const int cl = (e >> 27) - 1, idx = e & 0x7ffffff;
    const BvhBox* cb = cl == 0 ? lvl0 : upper + bi.off[cl];
    const int c0 = idx * SPH_BVH_FAN, c1 = min(c0 + SPH_BVH_FAN, bi.cnt[cl]);
    for (int ch = c0; ch < c1; ++ch) if (pred(cb[ch])) { if (cl == 0) return true; if (sn < 112) stack[sn++] = (cl << 27) | ch; else return true; }
  }
  return false;
}

// ---- locally essential tree -------------------------------------------------------------------------------------------
// A remote node must have its children here iff some particle of this domain may open it (the reference's test,
// F:275-278: size / sqrt(d^2 + soft) >= theta).  Conservative form against the position boxes of this domain's walk
// groups, with soft = 0 and a 1e-4 margin (the walk's own float screens use 3e-5): a node that fails it is accepted by
// every run of this rank whatever path the classification takes, so its children are never read.
struct DDLetEntry { int slot, owner, rchild, nchild; };    // patch wnodes[slot].child; children live at peer `owner`, index rchild
struct DDPeerNodes { const WNode* wn[DD_MAX_RANKS]; };
__device__ __forceinline__ bool dd_may_open(const WNode& w, const BvhBox* __restrict__ lvl0, const BvhBox* __restrict__ upper, const BvhInfo& bi, double theta2) {
  const double s2 = w.size * w.size * (1.0 + 1e-4);
  const double cx = w.cx, cy = w.cy, cz = w.cz;
  return dd_bvh_any(lvl0, upper, bi, [&](const BvhBox& q) {
    const double ex = fmax(fmax((double)q.plo[0] - cx, cx - (double)q.phi[0]), 0.0);
    const double ey = fmax(fmax((double)q.plo[1] - cy, cy - (double)q.phi[1]), 0.0);
    const double ez = fmax(fmax((double)q.plo[2] - cz, cz - (double)q.phi[2]), 0.0);
    return s2 >= theta2 * (ex * ex + ey * ey + ez * ez);          // empty boxes (plo = +inf) never pass
  });
}
// one BFS level: every frontier entry copies its children block from the owner's node array into a fresh block of the
// LET area (atomic cursor: the block positions are arbitrary, the child ORDER inside a block is the owner's) and queues
// the children that may be opened in turn.  Eight lanes per entry, one child each: the (remote) node loads of a block
// are in flight together.  ctl: [0] cursor, [1] overflow flag, [2 + level] frontier counts.
__global__ void k_dd_let_level(const DDLetEntry* __restrict__ fin, const int* __restrict__ n_in, DDLetEntry* __restrict__ fout, int* n_out,
                               int fcap, int* cursor, int let_end, int* overflow, const __grid_constant__ DDPeerNodes peers,
                               WNode* __restrict__ wn, const BvhBox* __restrict__ lvl0, const BvhBox* __restrict__ upper, const __grid_constant__ BvhInfo bi, double theta2) {
  const int n = *n_in < fcap ? *n_in : fcap;
  const int k = threadIdx.x & 7, lane = threadIdx.x & 31;
  const unsigned gmask = 0xffu << (lane & 24);
  const int nsub = (gridDim.x * blockDim.x) >> 3;
  for (int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 3; t < n; t += nsub) {
    const DDLetEntry e = fin[t];
    int d = 0;
    if (k == 0) d = atomicAdd(cursor, e.nchild);
    d = __shfl_sync(gmask, d, lane & 24);
    if (d + e.nchild > let_end) { if (k == 0) atomicExch(overflow, 1); continue; }
    if (k < e.nchild) {
      const double2* src = reinterpret_cast<const double2*>(peers.wn[e.owner] + e.rchild + k);
      const double2 a = src[0], b = src[1], c2 = src[2];
      double2* dst = reinterpret_cast<double2*>(wn + d + k);
      dst[0] = a; dst[1] = b; dst[2] = c2;                         // child index still the owner's: patched when (if) it is opened
      WNode w; w.cx = a.x; w.cy = a.y; w.cz = b.x; w.m = b.y; w.size = c2.x; w.child = __double2loint(c2.y); w.nchild = __double2hiint(c2.y);
      if (w.nchild > 0 && dd_may_open(w, lvl0, upper, bi, theta2)) {
        const int o = atomicAdd(n_out, 1);
        if (o < fcap) fout[o] = DDLetEntry{d + k, e.owner, w.child, w.nchild}; else atomicExch(overflow, 2);
      }
    }
    __syncwarp(gmask);
    if (k == 0) wn[e.slot].child = d;
  }
}
// top-region entries whose children live on a peer: decide whether this domain may open them (frontier of level 0)
__global__ void k_dd_let_seed(int n_cand, const DDLetEntry* __restrict__ cand, DDLetEntry* __restrict__ fout, int* n_out,
                              const WNode* __restrict__ wn, const BvhBox* __restrict__ lvl0, const BvhBox* __restrict__ upper, const __grid_constant__ BvhInfo bi, double theta2) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cand) return;
  const DDLetEntry e = cand[t];
  if (dd_may_open(wn[e.slot], lvl0, upper, bi, theta2)) fout[atomicAdd(n_out, 1)] = e;
}

// ---- halo ---------------------------------------------------------------------------------------------------------------
struct DDPeerGroups { int ng[DD_MAX_RANKS]; int goff[DD_MAX_RANKS + 1]; const int2* groups[DD_MAX_RANKS]; const BvhBox* box[DD_MAX_RANKS]; };
// flag[G] = 1 iff the peer group G (virtual index over all peers' own groups, this rank's own groups excluded by
// ng[self] = 0) can hold a source or a partner of some own particle: its reach box meets a position box of this
// domain (x_i inside Box(j), F:443 | V:479) or its position box meets a reach box (x_j inside Box(i), the pair loop's
// other direction).  A superset is harmless: the walks keep their exact tests.
__global__ void k_dd_halo_mark(const __grid_constant__ DDPeerGroups pg, const BvhBox* __restrict__ lvl0, const BvhBox* __restrict__ upper,
                               const __grid_constant__ BvhInfo bi, unsigned char* __restrict__ flag, int* __restrict__ hsize) {
  const int G = blockIdx.x * blockDim.x + threadIdx.x;
  if (G == pg.goff[DD_MAX_RANKS]) hsize[G] = 0;                  // the scan's total lands here
  if (G >= pg.goff[DD_MAX_RANKS]) return;
  int q = 0;
  while (q + 1 < DD_MAX_RANKS && G >= pg.goff[q + 1]) ++q;
  const BvhBox b = pg.box[q][G - pg.goff[q]];
  const bool hit = dd_bvh_any(lvl0, upper, bi, [&](const BvhBox& d) {
    return box_overlap(d.plo, d.phi, b.rlo, b.rhi) || box_overlap(d.rlo, d.rhi, b.plo, b.phi); });
  flag[G] = hit ? 1 : 0;
  hsize[G] = hit ? pg.groups[q][G - pg.goff[q]].y : 0;           // particles this group adds behind the own ones
}
// [0] selected groups, [1] their particles, [2] 1 when own + halo exceed the rank's capacity (all-reduced afterwards)
__global__ void k_dd_halo_check(const int* __restrict__ nsel, const int* __restrict__ total, int n_own, int ng_own, long long cap, int* __restrict__ out3) {
  out3[0] = *nsel; out3[1] = *total;
  out3[2] = ((long long)n_own + *total > cap || (long long)ng_own + *nsel > cap) ? 1 : 0;
}
// one warp per halo group: copy `nf` double fields (+ optionally the ids) of its particles from the owner's arrays;
// with write_groups the group table entry [ng_own + k] = (local first, size) is written as well
struct DDPull {
  int nf; int with_id; int write_groups; int ng_own; int n_own;
  const double* src[DD_MAX_RANKS][DD_PULL_FIELDS]; const int* src_id[DD_MAX_RANKS];
  double* dst[DD_PULL_FIELDS]; int* dst_id;
};
__global__ void k_dd_pull(int nh, const int* __restrict__ list, const int* __restrict__ poff, const __grid_constant__ DDPeerGroups pg,
                          const __grid_constant__ DDPull a, int2* __restrict__ groups) {
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (k >= nh) return;
  const int G = list[k];
  int q = 0;
  while (q + 1 < DD_MAX_RANKS && G >= pg.goff[q + 1]) ++q;
  const int2 sg = pg.groups[q][G - pg.goff[q]];
  const int first = a.n_own + poff[G];
  if (a.write_groups && lane == 0) groups[a.ng_own + k] = make_int2(first, sg.y);
  if (lane < sg.y) {
    double v[DD_PULL_FIELDS]; int vid = 0;                       // all (remote) loads first: they are in flight together
#pragma unroll
    for (int f = 0; f < DD_PULL_FIELDS; ++f) if (f < a.nf) v[f] = a.src[q][f][sg.x + lane];
    if (a.with_id) vid = a.src_id[q][sg.x + lane];
#pragma unroll
    for (int f = 0; f < DD_PULL_FIELDS; ++f) if (f < a.nf) a.dst[f][first + lane] = v[f];
    if (a.with_id) a.dst_id[first + lane] = vid;
  }
}

// ---- accretion across ranks: (sink, number)-keyed records instead of local indices --------------------------------------
struct DDAccRec { double m, x, y, z, vx, vy, vz; };
__global__ void k_dd_acc_records(int n_acc, const unsigned long long* __restrict__ acc_key, const int* __restrict__ acc_val,
                                 const double* __restrict__ m, const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ z,
                                 const double* __restrict__ vx, const double* __restrict__ vy, const double* __restrict__ vz,
                                 unsigned long long* __restrict__ out_key, DDAccRec* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_acc) return;
  const int i = acc_val[e];
  out_key[e] = acc_key[e];
  out[e] = DDAccRec{m[i], x[i], y[i], z[i], vx[i], vy[i], vz[i]};
}

// sink update from ALL ranks' accretion records, sorted by (sink, number): the same sums in the same order as
// k_accrete_apply (sum(pack(...)) in ascending number, F:497-508), on every rank.  idx = sort permutation of the records.
__global__ void k_dd_accrete_apply(int n_acc, const unsigned long long* __restrict__ key, const int* __restrict__ idx,
                                   const DDAccRec* __restrict__ rec, SinkArrays S, SimScalars* sc, double* __restrict__ spin) {
  const int j = threadIdx.x;
  if (j >= sc->n_sink || !sc->any_sink_mass) return;
  int lo = 0, hi = n_acc;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if ((int)(key[mid] >> 32) < j) lo = mid + 1; else hi = mid; }
  int e1 = lo; hi = n_acc;
  while (e1 < hi) { const int mid = (e1 + hi) >> 1; if ((int)(key[mid] >> 32) <= j) e1 = mid + 1; else hi = mid; }
  double sm = 0.0, sp[3] = {0.0, 0.0, 0.0}, sv[3] = {0.0, 0.0, 0.0}, lb[3] = {0.0, 0.0, 0.0};
  for (int e = lo; e < e1; ++e) {
    const DDAccRec r = rec[idx[e]];
    if (spin) { lb[0] = lb[0] + r.m * (r.y * r.vz - r.z * r.vy); lb[1] = lb[1] + r.m * (r.z * r.vx - r.x * r.vz); lb[2] = lb[2] + r.m * (r.x * r.vy - r.y * r.vx); }
    sm = __dadd_rn(sm, r.m);
    sp[0] = __dadd_rn(sp[0], __dmul_rn(r.m, r.x)); sp[1] = __dadd_rn(sp[1], __dmul_rn(r.m, r.y)); sp[2] = __dadd_rn(sp[2], __dmul_rn(r.m, r.z));
    sv[0] = __dadd_rn(sv[0], __dmul_rn(r.m, r.vx)); sv[1] = __dadd_rn(sv[1], __dmul_rn(r.m, r.vy)); sv[2] = __dadd_rn(sv[2], __dmul_rn(r.m, r.vz));
  }
  const int n_mine = e1 - lo;
  const double ms = S.m[j];
  if (spin && n_mine > 0) {
    const double x = S.x[j], y = S.y[j], z = S.z[j], vx = S.vx[j], vy = S.vy[j], vz = S.vz[j];
    lb[0] = lb[0] + ms * (y * vz - z * vy); lb[1] = lb[1] + ms * (z * vx - x * vz); lb[2] = lb[2] + ms * (x * vy - y * vx);
  }
  const double nm = __dadd_rn(ms, sm);
  S.x[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.x[j]), sp[0]), nm);
  S.y[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.y[j]), sp[1]), nm);
  S.z[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.z[j]), sp[2]), nm);
  S.vx[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.vx[j]), sv[0]), nm);
  S.vy[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.vy[j]), sv[1]), nm);
  S.vz[j] = __ddiv_rn(__dadd_rn(__dmul_rn(ms, S.vz[j]), sv[2]), nm);
  S.m[j] = __dadd_rn(ms, sm);
  if (spin && n_mine > 0) {
    const double x = S.x[j], y = S.y[j], z = S.z[j], vx = S.vx[j], vy = S.vy[j], vz = S.vz[j], m2 = S.m[j];
    spin[j] = spin[j] + (lb[0] - (0.0 + m2 * (y * vz - z * vy)));
    spin[SPH_MAX_SINKS + j] = spin[SPH_MAX_SINKS + j] + (lb[1] - (0.0 + m2 * (z * vx - x * vz)));
    spin[2 * SPH_MAX_SINKS + j] = spin[2 * SPH_MAX_SINKS + j] + (lb[2] - (0.0 + m2 * (x * vy - y * vx)));
  }
}
// check_sink_creation across ranks (V:549-597): the winning candidate's owner publishes x v h (others add zeros)
// the candidate word is (number << 32) | local index: ranks compare the numbers only
__global__ void k_dd_cand_id(unsigned long long* cand) { if (*cand != ~0ull) *cand = (*cand >> 32) << 32; }
__global__ void k_dd_create_publish(const unsigned long long* __restrict__ local_cand, const unsigned long long* __restrict__ global_cand,
                                    StateArrays s, double* __restrict__ out8) {
  if (threadIdx.x != 0) return;
  for (int k = 0; k < 8; ++k) out8[k] = 0.0;
  const unsigned long long g = *global_cand, l = *local_cand;
  if (g == ~0ull || l == ~0ull || ((l >> 32) << 32) != g) return;
  const int i = (int)(l & 0xffffffffu);
  out8[0] = s.x[i]; out8[1] = s.y[i]; out8[2] = s.z[i]; out8[3] = s.vx[i]; out8[4] = s.vy[i]; out8[5] = s.vz[i]; out8[6] = s.h[i]; out8[7] = 1.0;
}
__global__ void k_dd_create_apply(const double* __restrict__ in8, SinkArrays S, SimScalars* sc, double* __restrict__ spin) {
  if (threadIdx.x != 0) return;
  sc->create_cand = ~0ull;
  if (!(in8[7] > 0.5)) return;
  const int ns = sc->n_sink;
  const double h = in8[6];
  for (int j = 0; j < ns; ++j) {
    const double dx = S.x[j] - in8[0], dy = S.y[j] - in8[1], dz = S.z[j] - in8[2];
    const double dr = sqrt(dx * dx + dy * dy + dz * dz);
    if (dr < S.radius[j] + 2.0 * h) return;                                       // V:563-565
  }
  if (ns >= SPH_MAX_SINKS) { sc->err = 3; return; }
  S.x[ns] = in8[0]; S.y[ns] = in8[1]; S.z[ns] = in8[2]; S.vx[ns] = in8[3]; S.vy[ns] = in8[4]; S.vz[ns] = in8[5];
  S.ax[ns] = S.ay[ns] = S.az[ns] = 0.0;
  S.m[ns] = 0.00000000001; S.radius[ns] = 2.0 * h;                                // V:581-582
  if (spin) spin[ns] = spin[SPH_MAX_SINKS + ns] = spin[2 * SPH_MAX_SINKS + ns] = 0.0;
  sc->n_sink = ns + 1;
}

// ---- state fingerprint -----------------------------------------------------------------------------------------------------
// Order-independent 64-bit fingerprint of the gas state: sum over particles of a hash chain over (number, the bit
// patterns of x y z vx vy vz u m alpha h), so that two runs hold bit-identical states iff (up to hash collisions) their
// fingerprints agree - whatever the storage order and however the particles are spread over ranks.  sums[0..4] =
// sum m, sum m |x|^2, sum m |v|^2, sum m u, count (plain FP64 atomics: compare with a tolerance, not bit for bit).
__global__ void k_state_hash(int n, StateArrays s, unsigned long long* hash, double* sums) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long hv = 0ull; double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, a4 = 0.0;
  if (i < n) {
    const double f[10] = {s.x[i], s.y[i], s.z[i], s.vx[i], s.vy[i], s.vz[i], s.u[i], s.m[i], s.alpha[i], s.h[i]};
    hv = mix64((unsigned long long)(unsigned)s.id[i]);
    for (int k = 0; k < 10; ++k) hv = mix64(hv ^ (unsigned long long)__double_as_longlong(f[k]));
    a0 = f[7]; a1 = f[7] * (f[0] * f[0] + f[1] * f[1] + f[2] * f[2]); a2 = f[7] * (f[3] * f[3] + f[4] * f[4] + f[5] * f[5]); a3 = f[7] * f[6]; a4 = 1.0;
  }
  for (int o = 16; o > 0; o >>= 1) { hv += __shfl_xor_sync(FULL_MASK, hv, o); }
  a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2); a3 = warp_sum(a3); a4 = warp_sum(a4);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(hash, hv);
    atomicAdd(sums, a0); atomicAdd(sums + 1, a1); atomicAdd(sums + 2, a2); atomicAdd(sums + 3, a3); atomicAdd(sums + 4, a4);
  }
}
