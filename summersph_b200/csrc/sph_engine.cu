// sph_engine.cu — context, step orchestration and the C-ABI of include/sph_b200.h.
//
// One context = one CUDA device + one stream.  All particle data live in HBM between calls; the host
// sees them only through sph_upload / sph_download.  There is no CPU code path for any stage.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <ctime>
#include <string>
#include <vector>
#include <algorithm>
#include <functional>
#include <dlfcn.h>
#include <cub/cub.cuh>
#include <cub/device/device_merge.cuh>
#include <cuda/std/functional>

#include "../../include/sph_b200.h"
#include "sph_common.cuh"
#include "sph_hostcomm.h"
#include "sph_tree.cuh"
#include "sph_walk.cuh"
#define GRAV_CHUNK_WIDTH 32        // gravity walk groups: fixed runs of this many Morton-consecutive particles
#include "sph_gravity.cuh"
#include "sph_integrate.cuh"
#include "sph_conserved.cuh"
#include "sph_image.cuh"
#include "sph_interp.cuh"
#include "sph_gravat.cuh"
#include "sph_domain.cuh"
#include "sph_ics.cuh"

namespace {

thread_local std::string g_create_error;

enum Stage { ST_KEYS = 0, ST_SORT, ST_TREE, ST_DENSITY, ST_GRAVITY, ST_SPH, ST_INTEGRATE, ST_HITER, ST_CULL, ST_COMM, ST_HALO, ST_LET, ST_MIGRATE, ST_GRAV_NEAR, ST_COUNT };   // halo / let / migrate: domain decomposition only; grav_near: gravity evaluations on the stored far sums

// x**n in libgcc __powidf2 order (kernel tables, SUMMER_SPH.f90:63-100)
inline double powi(double x, int n) { double y = (n % 2) ? x : 1.0; while (n >>= 1) { x = x * x; if (n % 2) y *= x; } return y; }

struct NcclUid { char b[128]; };
struct NcclApi {   // resolved at run time from the already-loaded (torch-bundled) or system libnccl
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, NcclUid /*ncclUniqueId by value*/, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
};
enum { NC_INT8 = 0, NC_INT32 = 2, NC_UINT64 = 5, NC_FLOAT64 = 8, NC_SUM = 0, NC_MAX = 2, NC_MIN = 3 };

}  // namespace

struct sph_ctx {
  sph_params p; DevParams dp; int device = 0; int n_sm = 148; int max_smem = 0; cudaStream_t stream = nullptr;
  std::string err;
  int64_t n = 0, cap = 0, n_upload = 0; int n_sink = 0;
  // particle state, double buffered for the Morton re-order / compaction; between calls the spare buffer is scratch (sph_download_neighbours)
  double* st[2][10] = {}; int* id[2] = {}; int cur = 0;
  double *rho = nullptr, *omega = nullptr, *prs = nullptr, *cs = nullptr, *por2 = nullptr;
  double *ax = nullptr, *ay = nullptr, *az = nullptr, *udot = nullptr, *adot = nullptr;
  // tree
  uint64_t* key[2] = {}; uint64_t* key_lo[2] = {}; bool two_word = false; int* perm[2] = {}; int* level = nullptr;
  double *lcx = nullptr, *lcy = nullptr, *lcz = nullptr, *reach = nullptr;
  BvhBox* bvh = nullptr; size_t bvh_cap = 0; BvhInfo bi;
  int *node_count = nullptr, *gsize = nullptr, *gfirst = nullptr; int2* groups = nullptr; int n_groups = 0;
  GNode* nodes = nullptr; int *node_part = nullptr, *parent = nullptr, *nchild = nullptr, *arrive = nullptr, *cnt = nullptr, *off = nullptr;
  int* nl_pool = nullptr; size_t nl_pool_blocks = 0; int* nl_head = nullptr; size_t nl_head_cap = 0; int* nl_ctl = nullptr; bool nl_valid = false;   // saved candidate lists (density pass -> pair loop)
  int2* ggroups = nullptr; BvhBox* gbvh = nullptr; size_t ggroups_cap = 0; int *seg_cnt = nullptr, *seg_off = nullptr; size_t seg_cap = 0; bool grav_groups_valid = false;   // gravity walk groups (fixed runs of the rank's slice)
  WNode* wnodes = nullptr; int *wcount = nullptr, *wstart = nullptr, *widx = nullptr; int2* grav_spill = nullptr;   // gravity walk layout
  RootBox* root = nullptr; double* partial = nullptr; int n_partial = 0;
  void* cub_tmp = nullptr; size_t cub_bytes = 0;
  double *d_wt = nullptr, *d_dwt = nullptr, *d_gt = nullptr;
  SinkArrays S = {}; double* sink_buf = nullptr; double* sink_partial = nullptr; size_t sink_partial_cap = 0;
  double* sink_seg = nullptr; size_t sink_seg_cap = 0;     // [global GRAV_SEG segment][sink][3]: gas terms of the sink accelerations (exchanged between ranks)
  SimScalars* sc = nullptr; SimScalars* h_sc = nullptr;     // device + pinned host mirror
  int* h_rb = nullptr;                                      // pinned scratch for readback(): 16 ints
  int resident_check = 1; int64_t resident_hits = 0; int* d_same = nullptr; double* sink_land = nullptr;      // upload_impl: "is this the state I hold?"
  WalkCounters* ctr = nullptr; WalkCounters* h_ctr = nullptr; int* work = nullptr;
  unsigned char* keep = nullptr; unsigned long long* acc_key[2] = {}; int* acc_val[2] = {}; int64_t acc_cap = 0; int* d_nsel = nullptr;   // accretion list (ensure_acc_capacity)
  int* pos = nullptr;           // ascending-number position of each sorted particle (downloads)
  double* stage_d = nullptr; double* stage_d2 = nullptr; int stage_flip = 0;   // device staging for ordered downloads
  bool tree_valid = false; bool pos_moved = true; int tree_reuse = 1; int use_lists = 1; int fused_push = 1; int nl_exact = 0; int exact_counters = 0;   // pos_moved: positions / particle set changed since the last build
  sph_counts counts; double stage_ms[ST_COUNT] = {};
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> ev_used; std::vector<cudaEvent_t> ev_pool;
  int64_t launches = 0;
  cudaEvent_t tm0 = nullptr, tm1 = nullptr;
  // multi-GPU
  NcclApi nccl; void* comm = nullptr; int rank = 0, n_ranks = 1;
  HostComm* hc = nullptr;            // sph_comm_init_host: small collectives through host shared memory instead of NCCL (sph_hostcomm.h)
  std::vector<int> rank_g, rank_p;   // per-rank first group / first particle of its target slice (size n_ranks + 1)
  // peer-memory exchange: every exchanged array of every rank mapped here (CUDA IPC, or the raw pointer when the peer
  // lives in this process); slices are pushed with copy-engine transfers on their own stream
  cudaStream_t xstream = nullptr; cudaEvent_t x_ready = nullptr, x_done = nullptr;
  std::vector<cudaStream_t> pstream; std::vector<cudaEvent_t> pevent;   // one copy stream per peer: the pushes to different peers run on different copy engines
  bool p2p_stale = true, p2p_ok = false, x_pending = false;
  std::vector<std::vector<double*>> peer;      // [array slot][rank]
  std::vector<void*> ipc_opened; int* d_flag = nullptr; void* d_blob = nullptr; size_t blob_cap = 0;
  int g0 = 0, g1 = 0, p0 = 0, p1 = 0;
  double* cons_partial = nullptr; double* cons_out = nullptr;   // sph_conserved: block partials (+ the ranks' totals under domains), result slots
  int* cons_wpart = nullptr; size_t cons_wpart_n = 0;            // sph_conserved: per walk-layout slot, the row of a single-particle leaf (else -1)
  // far-field reuse of the gravity walk (sph_gravity.cuh): stored far sums of the tree terms, per-particle near / far split, the walk's counters
  double *far_fx = nullptr, *far_fy = nullptr, *far_fz = nullptr, *far_hc2 = nullptr; unsigned long long* far_ctr = nullptr;
  bool far_valid = false; int far_reuse = 1; int64_t far_count = 0; bool far_want_store = false; int steps_since_upload = 0; double far_hcut = GW_HCUT;
  int* far_list = nullptr; int* far_cnt = nullptr; unsigned char* far_ovf = nullptr; size_t far_list_runs = 0; int far_slots = 128; bool far_lists = true; int far_n_ovf = 0;   // recorded near pairs: [run][slot][lane]
  // sph_step_host: copies under the compute.  Late fields = gas columns still on their way from the host when the tree build starts
  // (they land in st[0] on io_stream; the state re-order permutes them when their first reader is due); early results leave
  // through staging buffers on io_stream while the step goes on
  cudaStream_t io_stream = nullptr; cudaEvent_t io_ev_xyz = nullptr, io_ev_out = nullptr, io_ev_done = nullptr, io_ev_field[10] = {};
  unsigned late_pending = 0; const double* late_src[10] = {}; double* late_dst[10] = {}; const int* late_perm = nullptr; bool late_permuted = false; int late_order[10] = {}; int late_n = 0;
  double* io_stage[5] = {}; size_t io_stage_cap = 0; bool io_active = false; double* io_out[10] = {}; unsigned io_fetched = 0; bool io_busy = false;
  double* sink_spin = nullptr; int sink_extras = 0;               // SPH_FLAG_SINK_MERGE_SPIN: spin[3][SPH_MAX_SINKS]; null pointer into the kernels when off
  double* img_table = nullptr;
  // sph_interpolate: the private BVH of the source balls (2 h_j of the current h) and the per-chunk query scratch, grown on demand
  double* ip_reach = nullptr; size_t ip_reach_cap = 0; BvhBox* ip_bvh = nullptr; size_t ip_bvh_cap = 0; BvhInfo ip_bi;
  double *ip_pts = nullptr, *ip_raw = nullptr, *ip_bpart = nullptr; uint64_t *ip_key[2] = {}, *ip_tie[2] = {}; int* ip_idx[2] = {}; RootBox* ip_rb = nullptr;
  void* ip_cub = nullptr; size_t ip_cub_bytes = 0; size_t ip_cap = 0;
  // sph_gravity_at: the points (x, y, z, h) and the output columns of one chunk (sorted by the sph_interpolate scratch), the top-slot owners
  double *ga_q = nullptr, *ga_raw = nullptr; size_t ga_cap = 0; int* ga_owner = nullptr;
  // ---- Morton-domain decomposition (sph_domain.cuh / sph_domain_host.inl); in this mode n = own particles, cap = own + halo capacity
  bool dd = false; int64_t n_global = 0; int n_halo = 0, ng_own = 0, ng_halo = 0;
  uint64_t* key_alloc[2] = {}; int* perm_alloc[2] = {};          // the allocations behind key[] / perm[] (which swap)
  uint64_t *dd_samples = nullptr, *dd_split = nullptr; long long* dd_counts = nullptr; int* dd_sendoff = nullptr; uint64_t* dd_segkeys = nullptr; std::vector<WNode> dd_top_host; std::vector<int> dd_top_part;
  std::vector<int> dd_top_owner;      // per top slot: the rank holding the complete node, -1 for a cell straddling ranks (sph_gravity_at)
  DDCell* dd_cells = nullptr; DDContrib* dd_contrib = nullptr; BvhBox* dd_obvh = nullptr; size_t dd_obvh_cap = 0; BvhInfo dd_ob; int* dd_let_ctl = nullptr; double* dd_create8 = nullptr; unsigned long long* dd_cand = nullptr;
  bool dd_fields_pending = false; cudaEvent_t let_done = nullptr; bool let_pending = false; double* let_flag = nullptr; std::vector<DDLetEntry> dd_cand_host;
  DDLetEntry* dd_let_f[2] = {}; int dd_let_fcap = 0, dd_let_begin = 0, dd_let_end = 0, dd_let_used = 0, dd_top_n = 0;
  unsigned char* dd_halo_flag = nullptr; int *dd_halo_list = nullptr, *dd_halo_size = nullptr, *dd_halo_poff = nullptr; size_t dd_halo_cap = 0;
  unsigned long long* dd_acc_key = nullptr; DDAccRec* dd_acc_rec = nullptr;                      // exported: this rank's accretion records
  unsigned long long* dd_accg_key[2] = {}; int* dd_accg_idx[2] = {}; DDAccRec* dd_accg_rec = nullptr; size_t dd_accg_cap = 0;   // all ranks' records
  std::vector<DDInfo> dd_info; DDPeerGroups dd_pg; std::vector<DDContrib> dd_top_recs;
  int *dd_gid = nullptr, *dd_gpos = nullptr, *dd_gcnt = nullptr, *dd_goff = nullptr; double* dd_gstage = nullptr; size_t dd_g_cap = 0;   // gathers for the host-facing downloads                                    // sph_column_density: line-of-sight integral of the M4 shape
};

namespace {

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { c->err = std::string(#call) + ": " + cudaGetErrorString(e_); return SPH_ERR_CUDA; } } while (0)
#define LAUNCH(kern, grid, block, smem, ...) do { kern<<<(grid), (block), (smem), c->stream>>>(__VA_ARGS__); ++c->launches; } while (0)

inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
// boxes of the levels above n0 level-0 boxes of the 8-ary BVH (bvh_levels): below n0 / 7, plus one partial box per level
inline size_t bvh_upper_boxes(int64_t n0) { return (size_t)(n0 / 7 + 64); }

StateArrays state_of(sph_ctx* c, int which) {
  double** s = c->st[which];
  return StateArrays{s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7], s[8], s[9], c->id[which]};
}
RateArrays rates_of(sph_ctx* c) { return RateArrays{c->ax, c->ay, c->az, c->udot, c->adot}; }

void stage_begin(sph_ctx* c, int st) {
  cudaEvent_t a, b;
  auto get = [&]() { cudaEvent_t e; if (!c->ev_pool.empty()) { e = c->ev_pool.back(); c->ev_pool.pop_back(); } else cudaEventCreate(&e); return e; };
  a = get(); b = get();
  cudaEventRecord(a, c->stream);
  c->ev_used.push_back({st, {a, b}});
}
void stage_end(sph_ctx* c) { cudaEventRecord(c->ev_used.back().second.second, c->stream); }
void stage_collect(sph_ctx* c, bool reset) {   // call after a stream sync
  if (reset) for (int i = 0; i < ST_COUNT; ++i) c->stage_ms[i] = 0.0;
  for (auto& e : c->ev_used) {
    float ms = 0.f; cudaEventElapsedTime(&ms, e.second.first, e.second.second);
    c->stage_ms[e.first] += ms;
    c->ev_pool.push_back(e.second.first); c->ev_pool.push_back(e.second.second);
  }
  c->ev_used.clear();
}

template <class T> int dalloc(sph_ctx* c, T** p, size_t count) {
  if (*p) { cudaFree(*p); *p = nullptr; }
  if (count == 0) count = 1;
  cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
  if (e != cudaSuccess) { c->err = std::string("cudaMalloc: ") + cudaGetErrorString(e); cudaGetLastError(); return SPH_ERR_OOM; }
  return SPH_OK;
}
#define DA(ptr, count) do { int r_ = dalloc(c, &(ptr), (size_t)(count)); if (r_) return r_; } while (0)

int cub_reserve(sph_ctx* c, size_t bytes);

// The accretion list of k_flags: one (sink, particle) entry for every sink whose radius holds the particle (each sink
// accretes on its own, F:484-556 | V:616-688), so with overlapping sinks it can hold more entries than there are
// particles.  Grown to at least `want` entries, never below `cap` (the domain re-order borrows acc_key[0] / acc_val[0]
// as merge scratch); under domains the exported records (dd_acc_key / dd_acc_rec, k_dd_acc_records) are as long.  The CUB
// temp storage is checked every time: ensure_capacity re-sizes it for the particle count alone.
int ensure_acc_capacity(sph_ctx* c, int64_t want) {
  if (want > c->acc_cap || (c->dd && !c->dd_acc_key)) {
    const int64_t cap = std::max(want, c->acc_cap);
    c->acc_cap = 0;
    for (int b = 0; b < 2; ++b) { DA(c->acc_key[b], cap); DA(c->acc_val[b], cap); }
    if (c->dd) { DA(c->dd_acc_key, cap); DA(c->dd_acc_rec, cap); c->p2p_stale = true; }
    c->acc_cap = cap;
  }
  size_t b1 = 0;
  cub::DoubleBuffer<unsigned long long> dk(c->acc_key[0], c->acc_key[1]); cub::DoubleBuffer<int> dv(c->acc_val[0], c->acc_val[1]);
  cub::DeviceRadixSort::SortPairs(nullptr, b1, dk, dv, (int)c->acc_cap, 0, 64, c->stream);
  return cub_reserve(c, b1);
}

int ensure_capacity(sph_ctx* c, int64_t n) {
  if (n <= c->cap) return SPH_OK;
  const int64_t cap = n + n / 64 + 1024;
  c->cap = 0; c->tree_valid = false; c->pos_moved = true; c->p2p_stale = true;      // a failed grow must not leave the old capacity standing over freed arrays
  for (int b = 0; b < 2; ++b) if (c->key_lo[b]) { cudaFree(c->key_lo[b]); c->key_lo[b] = nullptr; }
  for (int b = 0; b < 2; ++b) { for (int f = 0; f < 10; ++f) DA(c->st[b][f], cap); DA(c->id[b], cap); DA(c->key[b], cap); DA(c->perm[b], cap); }
  for (int b = 0; b < 2; ++b) { c->key_alloc[b] = c->key[b]; c->perm_alloc[b] = c->perm[b]; }
  DA(c->rho, cap); DA(c->omega, cap); DA(c->prs, cap); DA(c->cs, cap); DA(c->por2, cap);
  DA(c->ax, cap); DA(c->ay, cap); DA(c->az, cap); DA(c->udot, cap); DA(c->adot, cap);
  DA(c->far_fx, cap); DA(c->far_fy, cap); DA(c->far_fz, cap); DA(c->far_hc2, cap); c->far_valid = false;
  DA(c->level, cap); DA(c->lcx, cap); DA(c->lcy, cap); DA(c->lcz, cap); DA(c->reach, cap);
  DA(c->node_count, 2 * cap); DA(c->gsize, cap); DA(c->gfirst, cap); DA(c->groups, cap);
  DA(c->nodes, 2 * cap); DA(c->node_part, 2 * cap); DA(c->parent, 2 * cap); DA(c->nchild, 2 * cap); DA(c->arrive, 2 * cap);
  DA(c->cnt, cap + 1); DA(c->off, cap + 1);
  if (c->dd) {      // walk layout: [top tree | local tree | locally essential nodes of the peers]; LET frontier; fixed BVH capacity (exported)
    c->dd_let_begin = DD_TOP_CAP + (int)(2 * cap); c->dd_let_end = c->dd_let_begin + (int)cap; c->dd_let_fcap = (int)std::max<int64_t>(cap / 4, 65536);
    DA(c->wnodes, (size_t)c->dd_let_end);
    DA(c->dd_let_f[0], c->dd_let_fcap); DA(c->dd_let_f[1], c->dd_let_fcap);
    c->bvh_cap = (cap + bvh_upper_boxes(cap)) * 5 / 4; DA(c->bvh, c->bvh_cap);
  } else DA(c->wnodes, 2 * cap);
  DA(c->wcount, 2 * cap); DA(c->wstart, 2 * cap); DA(c->widx, 2 * cap);
  DA(c->keep, cap); DA(c->pos, cap); DA(c->stage_d, cap); DA(c->stage_d2, cap);
  // CUB temp: radix sort pairs (u64,int), exclusive scan, select
  size_t b1 = 0, b2 = 0, b3 = 0, b4 = 0, b5 = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, b5, c->wcount, c->wstart, (int)(2 * cap), c->stream);
  cub::DeviceSelect::Flagged(nullptr, b4, cub::CountingInputIterator<int>(0), c->gsize, c->gfirst, c->d_nsel, (int)cap, c->stream);
  cub::DoubleBuffer<uint64_t> dk(c->key[0], c->key[1]); cub::DoubleBuffer<int> dv(c->perm[0], c->perm[1]);
  cub::DeviceRadixSort::SortPairs(nullptr, b1, dk, dv, (int)cap, 0, 64, c->stream);
  cub::DeviceScan::ExclusiveSum(nullptr, b2, c->cnt, c->off, (int)cap + 1, c->stream);
  cub::DeviceSelect::Flagged(nullptr, b3, c->perm[0], c->keep, c->perm[1], c->d_nsel, (int)cap, c->stream);
  c->cub_bytes = std::max(std::max(std::max(b1, b4), std::max(b2, b3)), b5) + 256;
  if (c->cub_tmp) { cudaFree(c->cub_tmp); c->cub_tmp = nullptr; }
  if (cudaMalloc(&c->cub_tmp, c->cub_bytes) != cudaSuccess) { c->err = "cudaMalloc(cub temp)"; cudaGetLastError(); return SPH_ERR_OOM; }
  { int r_ = ensure_acc_capacity(c, cap); if (r_) return r_; }
  c->cap = cap;
  c->p2p_stale = true;
  return SPH_OK;
}

// grow the CUB temp storage to at least `bytes`
int cub_reserve(sph_ctx* c, size_t bytes) {
  if (bytes + 256 <= c->cub_bytes) return SPH_OK;
  c->cub_bytes = bytes + 256; if (c->cub_tmp) cudaFree(c->cub_tmp); c->cub_tmp = nullptr;
  if (cudaMalloc(&c->cub_tmp, c->cub_bytes) != cudaSuccess) { c->err = "cudaMalloc(cub temp)"; return SPH_ERR_OOM; }
  return SPH_OK;
}

void make_dev_params(sph_ctx* c) {
  const sph_params& p = c->p; DevParams& d = c->dp;
  d.variable_h = (p.mode & SPH_MODE_VARIABLE_H) ? 1 : 0;
  d.soft_hi = (p.mode & SPH_FLAG_SOFT_USES_HI) ? 1 : 0;
  d.nq = p.nq;
  const int key_cap = c->two_word ? SPH_KEY_LEVELS2 : SPH_KEY_LEVELS;
  d.lmax = p.max_depth < key_cap ? p.max_depth : key_cap;
  d.depth_unbounded = p.max_depth > key_cap;
  d.dq = 2.0 / p.nq; d.inv_dq = 1.0 / d.dq;
  d.h_fixed = p.h_fixed;
  d.pi_norm = d.variable_h ? (double)3.1415926535897932f : 3.14159265359;      // V:7 | F:125
  d.gamma = d.variable_h ? p.gamma : 1.4;                                      // F:466
  d.gm1 = d.variable_h ? (p.gamma - 1.0) : 0.4;                                // F:465
  d.theta = p.theta_override ? p.theta : 0.5;                                  // F:825
  d.G = (double)39.47841760435743f;                                            // F:7
  d.eta = p.eta; d.conv = p.convergence_criteria; d.max_length = p.max_length;
  d.tscale = d.variable_h ? p.timestep_scale : 0.25;                           // F:851
  d.bounding = p.bounding_size;
  d.lit_001 = (double)0.01f; d.lit_015 = (double)0.15f; d.lit_01 = (double)0.1f; d.lit_1em4 = (double)0.0001f;
}

int upload_tables(sph_ctx* c) {
  const int nq = c->p.nq; const double dq = 2.0 / nq;
  std::vector<double> w(nq + 1), dw(nq + 1), g(nq + 1);
  for (int i = 0; i <= nq; ++i) {
    volatile double q = i * dq;
    if (q >= 0.0 && q <= 1.0) {
      w[i] = 1.0 - 1.5 * powi(q, 2) + 0.75 * powi(q, 3);
      dw[i] = -3.0 * q + 2.25 * powi(q, 2);
      g[i] = ((40.0 * powi(q, 3)) - (36.0 * powi(q, 5)) + (15.0 * powi(q, 6))) / 30.0;
    } else if (q > 1.0 && q <= 2.0) {
      w[i] = 0.25 * powi(2.0 - q, 3);
      dw[i] = -0.75 * powi(2.0 - q, 2);
      g[i] = ((80.0 * powi(q, 3)) - (90.0 * powi(q, 4)) + (36.0 * powi(q, 5)) - (5.0 * powi(q, 6)) - 2.0) / 30.0;
    } else { w[i] = 0.0; dw[i] = 0.0; g[i] = 1.0; }
  }
  DA(c->d_wt, nq + 2); DA(c->d_dwt, nq + 2); DA(c->d_gt, nq + 2);
  CK(cudaMemcpy(c->d_wt, w.data(), (nq + 1) * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c->d_dwt, dw.data(), (nq + 1) * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c->d_gt, g.data(), (nq + 1) * 8, cudaMemcpyHostToDevice));
  return SPH_OK;
}

// ---------------------------------------------------------------------------------------------------
// multi-GPU: particles are replicated on every rank, target work is sharded by contiguous group slices;
// results travel with an all-gather-v (one in-place ncclBroadcast per owner inside a group call).
// ---------------------------------------------------------------------------------------------------
#define NC(call) do { int r_ = (call); if (r_ != 0) { c->err = std::string(#call) + ": " + (c->nccl.GetErrorString ? c->nccl.GetErrorString(r_) : "nccl error"); return SPH_ERR_COMM; } } while (0)

// ---- small collectives: NCCL on the given stream, or (sph_comm_init_host) through the host segment ----------------
size_t nc_size(int dtype) { return dtype == NC_INT8 ? 1 : dtype == NC_INT32 ? 4 : 8; }
template <class T> void host_fold(T* acc, const T* v, size_t count, int op) {
  for (size_t i = 0; i < count; ++i) acc[i] = op == NC_SUM ? (T)(acc[i] + v[i]) : op == NC_MAX ? (v[i] > acc[i] ? v[i] : acc[i]) : (v[i] < acc[i] ? v[i] : acc[i]);
}
int coll_allreduce(sph_ctx* c, cudaStream_t st, void* buf, size_t count, int dtype, int op) {
  if (c->n_ranks <= 1) return SPH_OK;
  if (!c->hc) { NC(c->nccl.AllReduce(buf, buf, count, dtype, op, c->comm, st)); return SPH_OK; }
  const size_t bytes = count * nc_size(dtype);
  std::vector<char> mine(bytes), all(bytes * c->n_ranks);
  CK(cudaMemcpyAsync(mine.data(), buf, bytes, cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st));
  if (!c->hc->allgather(mine.data(), bytes, all.data())) { c->err = "host communicator: all-gather failed (payload too large or a peer timed out)"; return SPH_ERR_COMM; }
  std::memcpy(mine.data(), all.data(), bytes);                       // rank order 0..R-1: the same fold on every rank
  for (int r = 1; r < c->n_ranks; ++r) {
    const char* v = all.data() + bytes * r;
    if (dtype == NC_FLOAT64) host_fold((double*)mine.data(), (const double*)v, count, op);
    else if (dtype == NC_UINT64) host_fold((unsigned long long*)mine.data(), (const unsigned long long*)v, count, op);
    else if (dtype == NC_INT32) host_fold((int*)mine.data(), (const int*)v, count, op);
    else host_fold((signed char*)mine.data(), (const signed char*)v, count, op);
  }
  CK(cudaMemcpyAsync(buf, mine.data(), bytes, cudaMemcpyHostToDevice, st)); CK(cudaStreamSynchronize(st));
  return SPH_OK;
}
// recv[r * bytes ...] = rank r's send block (device buffers; send may alias its own block of recv)
int coll_allgather(sph_ctx* c, cudaStream_t st, const void* send, void* recv, size_t bytes) {
  if (c->n_ranks <= 1) { if (send != recv) CK(cudaMemcpyAsync(recv, send, bytes, cudaMemcpyDeviceToDevice, st)); return SPH_OK; }
  if (!c->hc) { NC(c->nccl.AllGather(send, recv, bytes, NC_INT8, c->comm, st)); return SPH_OK; }
  std::vector<char> mine(bytes), all(bytes * c->n_ranks);
  CK(cudaMemcpyAsync(mine.data(), send, bytes, cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st));
  if (!c->hc->allgather(mine.data(), bytes, all.data())) { c->err = "host communicator: all-gather failed (payload too large or a peer timed out)"; return SPH_ERR_COMM; }
  CK(cudaMemcpyAsync(recv, all.data(), all.size(), cudaMemcpyHostToDevice, st)); CK(cudaStreamSynchronize(st));
  return SPH_OK;
}
bool have_comm(const sph_ctx* c) { return c->hc != nullptr || c->comm != nullptr; }

// ---- peer-memory all-gather-v -------------------------------------------------------------------------
struct PeerRec { int pid; int device; unsigned long long hosthash; void* ptr; cudaIpcMemHandle_t h; };
#include <unistd.h>

std::vector<double*> exchanged_arrays(sph_ctx* c) {
  return {c->rho, c->cs, c->por2, c->ax, c->ay, c->az, c->udot, c->adot, c->omega, c->prs, c->st[0][9], c->st[1][9], c->sink_seg};
}

std::vector<void*> dd_exported(sph_ctx* c);      // sph_domain_host.inl

void p2p_close(sph_ctx* c) {
  for (void* p : c->ipc_opened) cudaIpcCloseMemHandle(p);
  c->ipc_opened.clear(); c->peer.clear(); c->p2p_ok = false;
}

// (Re)map the peers' arrays after an allocation changed. Collective. Falls back to NCCL broadcasts when any
// rank cannot map a peer (no NVLink/PCIe peer access, IPC disabled): all ranks agree through an all-reduce.
int p2p_setup(sph_ctx* c) {
  c->p2p_stale = false;
  p2p_close(c);
  if (c->n_ranks <= 1 || !have_comm(c) || (!c->hc && !c->nccl.AllGather) || getenv("SPH_B200_NO_P2P")) return SPH_OK;
  if (!c->xstream) { CK(cudaStreamCreateWithFlags(&c->xstream, cudaStreamNonBlocking)); CK(cudaEventCreateWithFlags(&c->x_ready, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&c->x_done, cudaEventDisableTiming)); }
  if (!c->d_flag) DA(c->d_flag, 4);
  std::vector<void*> arr;
  if (c->dd) arr = dd_exported(c); else for (double* q : exchanged_arrays(c)) arr.push_back(q);
  const int na = (int)arr.size(), R = c->n_ranks;
  char host[256] = {0}; gethostname(host, 255);
  unsigned long long hh = 1469598103934665603ull; for (char* q = host; *q; ++q) hh = (hh ^ (unsigned char)*q) * 1099511628211ull;
  std::vector<PeerRec> mine(na), all((size_t)na * R);
  int ok = 1;
  for (int a = 0; a < na; ++a) {
    mine[a].pid = (int)getpid(); mine[a].device = c->device; mine[a].hosthash = hh; mine[a].ptr = arr[a];
    std::memset(&mine[a].h, 0, sizeof(mine[a].h));
    if (cudaIpcGetMemHandle(&mine[a].h, arr[a]) != cudaSuccess) { cudaGetLastError(); ok = 0; }
  }
  const size_t bytes = sizeof(PeerRec) * na;
  if (c->blob_cap < bytes * R) { if (c->d_blob) cudaFree(c->d_blob); CK(cudaMalloc(&c->d_blob, bytes * R)); c->blob_cap = bytes * R; }
  CK(cudaMemcpyAsync((char*)c->d_blob + bytes * c->rank, mine.data(), bytes, cudaMemcpyHostToDevice, c->stream));
  { int r_ = coll_allgather(c, c->stream, (char*)c->d_blob + bytes * c->rank, c->d_blob, bytes); if (r_) return r_; }
  CK(cudaMemcpyAsync(all.data(), c->d_blob, bytes * R, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->peer.assign(na, std::vector<double*>(R, nullptr));
  for (int r = 0; r < R && ok; ++r) {
    for (int a = 0; a < na && ok; ++a) {
      const PeerRec& pr = all[(size_t)r * na + a];
      if (r == c->rank) { c->peer[a][r] = (double*)arr[a]; continue; }
      if (pr.hosthash != hh) { ok = 0; break; }
      if (pr.pid == (int)getpid()) {            // peer context lives in this process (threads): plain peer access
        if (pr.device != c->device) {
          int can = 0; cudaDeviceCanAccessPeer(&can, c->device, pr.device);
          if (!can) { ok = 0; break; }
          cudaError_t e = cudaDeviceEnablePeerAccess(pr.device, 0);
          if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); ok = 0; break; }
          cudaGetLastError();
        }
        c->peer[a][r] = (double*)pr.ptr;
      } else {
        void* q = nullptr;
        if (cudaIpcOpenMemHandle(&q, pr.h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = 0; break; }
        c->ipc_opened.push_back(q); c->peer[a][r] = (double*)q;
      }
    }
  }
  // every rank must have mapped every peer
  CK(cudaMemcpyAsync(c->d_flag, &ok, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  { int r_ = coll_allreduce(c, c->stream, c->d_flag, 1, NC_INT32, NC_MIN); if (r_) return r_; }
  int all_ok = 0;
  CK(cudaMemcpyAsync(&all_ok, c->d_flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (!all_ok) { p2p_close(c); return SPH_OK; }
  c->p2p_ok = true;
  return SPH_OK;
}

// Start the exchange of this rank's slice [p0, p1) of each array: push it into every peer's copy with
// copy-engine transfers on the exchange stream (no SMs: it runs under whatever kernel follows on the main
// stream), then a 4-byte all-reduce as the cross-rank "all pushes have landed" barrier.  allgatherv_end makes
// the main stream wait for it.  Without peer mapping: one in-place ncclBroadcast per owner on the main stream.
// `roff` (n_ranks + 1 element offsets) replaces the particle slices [rank_p[r], rank_p[r + 1]) when given.
int allgatherv_begin(sph_ctx* c, double* const* bufs, int nbufs, const size_t* roff = nullptr) {
  if (c->n_ranks <= 1) return SPH_OK;
  if (c->p2p_stale) { int r_ = p2p_setup(c); if (r_) return r_; }
  if (!c->p2p_ok) {
    if (c->hc) { c->err = "the host communicator moves bulk data over peer-mapped device memory only (peer mapping failed or SPH_B200_NO_P2P is set)"; return SPH_ERR_COMM; }
    NC(c->nccl.GroupStart());
    for (int b = 0; b < nbufs; ++b)
      for (int r = 0; r < c->n_ranks; ++r) {
        const long long cnt = roff ? (long long)(roff[r + 1] - roff[r]) : (long long)(c->rank_p[r + 1] - c->rank_p[r]);
        if (cnt <= 0) continue;
        double* p = bufs[b] + (roff ? roff[r] : (size_t)c->rank_p[r]);
        NC(c->nccl.Broadcast(p, p, (size_t)cnt, NC_FLOAT64, r, c->comm, c->stream));
      }
    NC(c->nccl.GroupEnd());
    return SPH_OK;
  }
  const std::vector<double*> arr = exchanged_arrays(c);
  CK(cudaEventRecord(c->x_ready, c->stream));
  CK(cudaStreamWaitEvent(c->xstream, c->x_ready, 0));
  while ((int)c->pstream.size() < c->n_ranks - 1) {
    cudaStream_t st; cudaEvent_t ev;
    CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)); CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    c->pstream.push_back(st); c->pevent.push_back(ev);
  }
  const size_t off = roff ? roff[c->rank] : (size_t)c->p0, cnt = roff ? roff[c->rank + 1] - roff[c->rank] : (size_t)(c->p1 - c->p0);
  std::vector<int> slot(nbufs, -1);
  for (int b = 0; b < nbufs; ++b) {
    for (int k = 0; k < (int)arr.size(); ++k) if (arr[k] == bufs[b]) slot[b] = k;
    if (slot[b] < 0) { c->err = "allgatherv: array is not registered for the peer exchange"; return SPH_ERR_STATE; }
  }
  for (int k = 1; k < c->n_ranks; ++k) {        // staggered peer order spreads the traffic over the switch
    const int r = (c->rank + k) % c->n_ranks;
    cudaStream_t st = c->pstream[k - 1];
    CK(cudaStreamWaitEvent(st, c->x_ready, 0));
    if (cnt > 0)
      for (int b = 0; b < nbufs; ++b)
        CK(cudaMemcpyAsync(c->peer[slot[b]][r] + off, bufs[b] + off, cnt * 8, cudaMemcpyDefault, st));
    CK(cudaEventRecord(c->pevent[k - 1], st));
    CK(cudaStreamWaitEvent(c->xstream, c->pevent[k - 1], 0));
  }
  { int r_ = coll_allreduce(c, c->xstream, c->d_flag + 1, 1, NC_INT32, NC_SUM); if (r_) return r_; }
  CK(cudaEventRecord(c->x_done, c->xstream));
  c->x_pending = true;
  return SPH_OK;
}
int allgatherv_end(sph_ctx* c) {
  if (!c->x_pending) return SPH_OK;
  CK(cudaStreamWaitEvent(c->stream, c->x_done, 0));
  c->x_pending = false;
  return SPH_OK;
}
int allgatherv(sph_ctx* c, double* const* bufs, int nbufs, const size_t* roff = nullptr) {
  int r = allgatherv_begin(c, bufs, nbufs, roff);
  return r ? r : allgatherv_end(c);
}
int allreduce(sph_ctx* c, void* buf, size_t count, int dtype, int op) {
  if (c->n_ranks <= 1) return SPH_OK;
  return coll_allreduce(c, c->stream, buf, count, dtype, op);
}

__global__ void k_set_int(int* p, int v) { *p = v; }
// A few control words back to the host by a kernel store into page-locked host memory (device-visible under unified
// addressing): a copy-engine transfer would queue behind the bulk columns sph_step_host has in flight on its own stream
// (measured: 10 ms per step-end read-back at 16M).  Valid on the host after the stream synchronises.
__global__ void k_readback(const int* __restrict__ src, int* __restrict__ dst, int nwords) { for (int i = threadIdx.x; i < nwords; i += blockDim.x) dst[i] = src[i]; }
void readback(sph_ctx* c, void* pinned_dst, const void* dev_src, size_t bytes);
__global__ void k_iota_from(int n, int first, int* a) { int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) a[i] = first + i; }

// first walk group of every rank's target slice (n_ranks + 1 entries): contiguous, cut only at multiples of GRAV_SEG
// groups (the gravity runs restart there, sph_gravity.cuh), so runs and segments are the same for any rank count
void slice_first_groups(int ng, int R, int* first) {
  for (int r = 0; r <= R; ++r) first[r] = r == R ? ng : (int)(((int64_t)ng * r / R) / GRAV_SEG * GRAV_SEG);
}
int compute_slices(sph_ctx* c) {
  const int R = c->n_ranks, ng = c->n_groups, n = (int)c->n;
  c->rank_g.assign(R + 1, 0); c->rank_p.assign(R + 1, 0);
  slice_first_groups(ng, R, c->rank_g.data());
  c->rank_p[R] = n;
  if (R > 1) {
    for (int r = 1; r < R; ++r)
      CK(cudaMemcpyAsync(&c->rank_p[r], c->gfirst + c->rank_g[r], sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  c->g0 = c->rank_g[c->rank]; c->g1 = c->rank_g[c->rank + 1];
  c->p0 = c->rank_p[c->rank]; c->p1 = c->rank_p[c->rank + 1];
  return SPH_OK;
}

// ---------------------------------------------------------------------------------------------------
// tree
// ---------------------------------------------------------------------------------------------------
void readback(sph_ctx* c, void* pinned_dst, const void* dev_src, size_t bytes) { LAUNCH(k_readback, 1, 64, 0, (const int*)dev_src, (int*)pinned_dst, (int)(bytes / 4)); }
int build_tree_impl(sph_ctx* c, bool* retry_two_word);

// sph_step_host: gas columns that were still in flight when the state was re-ordered.  They arrive in late_order; when a
// reader of some of them is due, everything queued up to the last one it needs is waited for and re-ordered (one launch).
int flush_late(sph_ctx* c, unsigned need) {
  const unsigned m = c->late_pending & need;
  if (!m) return SPH_OK;
  int last = -1;
  for (int k = 0; k < c->late_n; ++k) if ((m >> c->late_order[k]) & 1u) last = k;
  PermuteArgs pa; std::memset(&pa, 0, sizeof(pa));
  unsigned done = 0;
  for (int k = 0; k <= last; ++k) {
    const int f = c->late_order[k];
    if (!((c->late_pending >> f) & 1u)) continue;
    done |= 1u << f; pa.src[f] = c->late_src[f]; pa.dst[f] = c->late_dst[f];
  }
  CK(cudaStreamWaitEvent(c->stream, c->io_ev_field[c->late_order[last]], 0));
  if (c->late_permuted) LAUNCH(k_permute, cdiv(c->n, 4 * 256), 256, 0, (int)c->n, c->late_perm, pa);      // before any re-order they are in place already
  c->late_pending &= ~done;
  return SPH_OK;
}
enum { LF_H = 1u << 9, LF_M = 1u << 7, LF_U = 1u << 6, LF_ALL = 0x3ffu };

// ascending-number position of every listed particle: the rank of its id among the ids present (all on device)
__global__ void k_mark_present(int n, const int* __restrict__ id, int* __restrict__ present) {
  int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) present[id[i]] = 1;
}
__global__ void k_rank_of(int n, const int* __restrict__ id, const int* __restrict__ rank, int* __restrict__ pos) {
  int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) pos[i] = rank[id[i]];
}
// pos[i] = rank of id[i] among id[0 .. n); cnt / off: n_upload + 1 ints of scratch, off keeps the rank of every id
int id_ranks(sph_ctx* c, int n, const int* id, int* cnt, int* off, int* pos) {
  const int nu = (int)c->n_upload, T = 256;
  CK(cudaMemsetAsync(cnt, 0, sizeof(int) * (size_t)(nu + 1), c->stream));
  LAUNCH(k_mark_present, cdiv(n, T), T, 0, n, id, cnt);
  size_t bytes = c->cub_bytes;
  CK(cub::DeviceScan::ExclusiveSum(c->cub_tmp, bytes, cnt, off, nu + 1, c->stream));
  LAUNCH(k_rank_of, cdiv(n, T), T, 0, n, id, off, pos);
  return SPH_OK;
}

// Root cube (F:803-808) and descent keys of the n current particles.  The replicated form's ranks all hold every particle
// and find the same cube alone; under domains the extrema are all-reduced (min / max are exact: the same cube as one rank's).
int root_and_keys(sph_ctx* c, int n, uint64_t* key_lo) {
  const int T = 256;
  StateArrays s = state_of(c, c->cur);
  const int nb = std::max(1, std::min(cdiv(n, T), c->n_partial));
  LAUNCH(k_bbox_partial, nb, T, 0, n, s.x, s.y, s.z, c->partial);
  LAUNCH(k_bbox_final, 1, 32, 0, nb, c->partial, c->root);
  if (c->dd) {
    LAUNCH(k_dd_box_pack, 1, 32, 0, c->root, c->partial);            // [mn, -mx] so that one MIN all-reduce merges both
    { int r_ = coll_allreduce(c, c->stream, c->partial, 6, NC_FLOAT64, NC_MIN); if (r_) return r_; }
    LAUNCH(k_dd_box_unpack, 1, 32, 0, c->partial);
    LAUNCH(k_bbox_final, 1, 32, 0, 1, c->partial, c->root);
  }
  LAUNCH(k_keys, cdiv(std::max(n, 1), T), T, 0, n, s.x, s.y, s.z, c->root, c->dp.lmax, c->key[0], key_lo, c->perm[0]);
  return SPH_OK;
}

// stable radix sort of (key[0], perm[0]) by the single-word key; the sorted pair ends up in key[0] / perm[0]
int sort_keys(sph_ctx* c, int n) {
  size_t bytes = c->cub_bytes;
  cub::DoubleBuffer<uint64_t> dk(c->key[0], c->key[1]); cub::DoubleBuffer<int> dv(c->perm[0], c->perm[1]);
  CK(cub::DeviceRadixSort::SortPairs(c->cub_tmp, bytes, dk, dv, n, 0, 63, c->stream));
  if (dk.Current() != c->key[0]) std::swap(c->key[0], c->key[1]);
  if (dv.Current() != c->perm[0]) std::swap(c->perm[0], c->perm[1]);
  return SPH_OK;
}

// The local octree over the n sorted particles, in two halves so that a caller can act on a key collision in between.
// Leaf cells, then the internal-node count and the key-collision flag on the host.  has_prev / kprev, has_next / knext:
// under domains, the boundary keys of the neighbouring domains (k_leaf); zeros otherwise.
int octree_leaves(sph_ctx* c, int n, const uint64_t* klo, int has_prev, uint64_t kprev, int has_next, uint64_t knext, int* nn, int* key_err) {
  const int T = 256;
  StateArrays s = state_of(c, c->cur);
  { int r_ = flush_late(c, LF_H); if (r_) return r_; }
  LAUNCH(k_leaf, cdiv(n, T), T, 0, n, c->key[0], klo, s.h, c->root, c->dp, c->level, c->lcx, c->lcy, c->lcz, c->reach, &c->sc->err, has_prev, kprev, has_next, knext);
  LAUNCH(k_oct_nodes<false>, cdiv(n, T), T, 0, n, c->key[0], klo, c->dp.lmax, c->root, c->cnt, c->off, 0, c->nodes, c->node_part, c->node_count);
  CK(cudaMemsetAsync(c->cnt + n, 0, sizeof(int), c->stream));
  size_t bytes = c->cub_bytes;
  CK(cub::DeviceScan::ExclusiveSum(c->cub_tmp, bytes, c->cnt, c->off, n + 1, c->stream));
  // node count is needed on the host for launch sizes of the per-node passes
  readback(c, c->h_rb, c->off + n, sizeof(int));
  readback(c, c->h_rb + 1, &c->sc->err, sizeof(int));
  CK(cudaStreamSynchronize(c->stream));
  *nn = n + c->h_rb[0]; *key_err = c->h_rb[1];
  return SPH_OK;
}
// The nn nodes (preorder), their links, walk-layout slots and sums (k_oct_finalize is left to the caller), then the walk
// groups: cell-aligned buckets, their sizes in gsize, their first particles in gfirst and their count in d_nsel (device).
int octree_nodes(sph_ctx* c, int n, int nn, const uint64_t* klo) {
  const int T = 256;
  StateArrays s = state_of(c, c->cur);
  c->counts.n_nodes = nn;
  LAUNCH(k_oct_nodes<true>, cdiv(n, T), T, 0, n, c->key[0], klo, c->dp.lmax, c->root, c->cnt, c->off, nn, c->nodes, c->node_part, c->node_count);
  LAUNCH(k_oct_link, cdiv(nn, T), T, 0, nn, c->nodes, c->node_part, c->parent, c->nchild, c->wcount);
  size_t bytes = c->cub_bytes;
  CK(cub::DeviceScan::ExclusiveSum(c->cub_tmp, bytes, c->wcount, c->wstart, nn, c->stream));
  CK(cudaMemsetAsync(c->widx, 0xff, sizeof(int) * (size_t)nn, c->stream));
  LAUNCH(k_oct_widx, cdiv(nn, T), T, 0, nn, c->nodes, c->wcount, c->wstart, c->widx);
  CK(cudaMemsetAsync(c->arrive, 0, sizeof(int) * (size_t)nn, c->stream));
  { int r_ = flush_late(c, LF_M | LF_H); if (r_) return r_; }
  LAUNCH(k_oct_up, cdiv(n, T), T, 0, n, c->off, c->cnt, s.x, s.y, s.z, s.m, s.h, c->level, c->root, c->nodes, c->parent, c->nchild, c->arrive);
  CK(cudaMemsetAsync(c->gsize, 0, sizeof(int) * (size_t)n, c->stream));
  LAUNCH(k_group_mark, cdiv(nn, T), T, 0, nn, c->nodes, c->node_part, c->node_count, c->gsize);
  bytes = c->cub_bytes;
  CK(cub::DeviceSelect::Flagged(c->cub_tmp, bytes, cub::CountingInputIterator<int>(0), c->gsize, c->gfirst, c->d_nsel, n, c->stream));
  return SPH_OK;
}

// The implicit 8-ary BVH above n0 level-0 boxes at lvl0: every level boxes SPH_BVH_FAN boxes of the one below, up to a
// level of at most 32.  Level l >= 1 is written at upper + bi.off[l], the first of them at upper + off1.
void bvh_levels(sph_ctx* c, const BvhBox* lvl0, int n0, BvhBox* upper, int off1, BvhInfo& bi) {
  const int T = 256;
  bi.off[0] = 0; bi.cnt[0] = n0;
  int l = 0;
  for (int off = off1; bi.cnt[l] > 32; ++l) {
    const int np = cdiv(bi.cnt[l], SPH_BVH_FAN);
    bi.off[l + 1] = off; bi.cnt[l + 1] = np;
    LAUNCH(k_bvh_up, cdiv(np, T), T, 0, bi.cnt[l], l == 0 ? lvl0 : upper + bi.off[l], upper + off);
    off += np;
  }
  bi.nlev = l + 1;
}

// global segment table of the sink sums, nst segments: [segment][sink][3].  Outside the domain form it is peer-mapped,
// so a new allocation voids the mapping (the first exchange after a build maps it again)
int sink_seg_reserve(sph_ctx* c, int nst) {
  const int nsk = std::max(c->n_sink, 1);
  if ((size_t)nst * nsk * 3 > c->sink_seg_cap) {
    c->sink_seg_cap = (size_t)(nst + nst / 8 + 64) * (nsk + 1) * 3;
    DA(c->sink_seg, c->sink_seg_cap); if (!c->dd) c->p2p_stale = true;
  }
  return SPH_OK;
}

#include "sph_domain_host.inl"

// Single-word (63-bit, 21-level) keys are the fast path.  If two particles share a full key while the
// reference's max_depth is deeper, the build is repeated (and stays) on the two-word path: 42 levels,
// sorted with two stable radix passes (low word, then high word).
int refresh_tree(sph_ctx* c) {
  const int n = (int)c->n, T = 256;
  c->nl_valid = false;
  stage_begin(c, ST_TREE);
  if (c->dp.variable_h) {
    StateArrays s = state_of(c, c->cur);
    LAUNCH(k_refresh_reach, cdiv(n, T), T, 0, n, s.h, c->level, c->root, c->dp, c->reach);
    const int ng = c->n_groups;
    LAUNCH(k_bvh_leaf, cdiv((int64_t)ng * 32, T), T, 0, ng, c->groups, s.x, s.y, s.z, c->lcx, c->lcy, c->lcz, c->reach, c->bvh);
    bvh_levels(c, c->bvh, ng, c->bvh, ng, c->bi);
  }
  stage_end(c);
  return SPH_OK;
}

int build_tree(sph_ctx* c) {
  const bool reuse = c->tree_valid && !c->pos_moved && c->tree_reuse;
  if (!reuse) c->far_valid = false;          // the stored far sums belong to the tree they were taken on
  if (c->dd) return reuse ? dd_refresh_tree(c) : dd_build_tree(c);
  if (reuse) return refresh_tree(c);
  bool retry = false;
  int r = build_tree_impl(c, &retry);
  if (r == SPH_OK && retry) {
    c->two_word = true;
    make_dev_params(c);
    for (int b = 0; b < 2; ++b) DA(c->key_lo[b], c->cap);
    r = build_tree_impl(c, &retry);
  }
  return r;
}

int build_tree_impl(sph_ctx* c, bool* retry_two_word) {
  const int n = (int)c->n;
  c->nl_valid = false; c->grav_groups_valid = false;
  const int T = 256;
  *retry_two_word = false;
  if (c->two_word && !c->key_lo[0]) { for (int b = 0; b < 2; ++b) DA(c->key_lo[b], c->cap); }
  if (c->late_pending && c->late_permuted) { int r_ = flush_late(c, LF_ALL); if (r_) return r_; }      // a second re-order (two-word retry) takes complete columns
  stage_begin(c, ST_KEYS);
  { int r_ = root_and_keys(c, n, c->two_word ? c->key_lo[0] : nullptr); if (r_) return r_; }
  stage_end(c);
  stage_begin(c, ST_SORT);
  {
    if (c->two_word) {     // stable LSD order: low word first
      size_t bytes = c->cub_bytes;
      cub::DoubleBuffer<uint64_t> dl(c->key_lo[0], c->key_lo[1]); cub::DoubleBuffer<int> dv(c->perm[0], c->perm[1]);
      CK(cub::DeviceRadixSort::SortPairs(c->cub_tmp, bytes, dl, dv, n, 0, 63, c->stream));
      if (dv.Current() != c->perm[0]) std::swap(c->perm[0], c->perm[1]);
      LAUNCH(k_gather_u64, cdiv(n, T), T, 0, n, c->perm[0], c->key[0], c->key[1]);
      std::swap(c->key[0], c->key[1]);
    }
    { int r_ = sort_keys(c, n); if (r_) return r_; }
    PermuteArgs pa;
    for (int f = 0; f < 10; ++f) { pa.src[f] = c->st[c->cur][f]; pa.dst[f] = c->st[c->cur ^ 1][f]; }
    pa.id_src = c->id[c->cur]; pa.id_dst = c->id[c->cur ^ 1];
    if (c->late_pending) {      // sph_step_host: columns still arriving are re-ordered when their first reader is due (flush_late)
      for (int f = 0; f < 10; ++f) if ((c->late_pending >> f) & 1u) { c->late_src[f] = pa.src[f]; c->late_dst[f] = pa.dst[f]; pa.src[f] = nullptr; }
      c->late_perm = c->perm[0]; c->late_permuted = true;
    }
    LAUNCH(k_permute, cdiv(n, 4 * T), T, 0, n, c->perm[0], pa);
    c->cur ^= 1;
    if (c->two_word) {     // regenerate both key words in the final order from the re-ordered positions
      StateArrays s = state_of(c, c->cur);
      LAUNCH(k_keys, cdiv(n, T), T, 0, n, s.x, s.y, s.z, c->root, c->dp.lmax, c->key[0], c->key_lo[0], c->perm[1]);
    }
  }
  stage_end(c);
  stage_begin(c, ST_TREE);
  {
    const uint64_t* klo = c->two_word ? c->key_lo[0] : nullptr;
    int nn = 0, key_err = 0;
    { int r_ = octree_leaves(c, n, klo, 0, 0, 0, 0, &nn, &key_err); if (r_) return r_; }
    if (key_err && !c->two_word) {            // a 63-bit key collision: redo this build with two-word keys
      CK(cudaMemsetAsync(&c->sc->err, 0, sizeof(int), c->stream));
      stage_end(c);
      *retry_two_word = true;
      return SPH_OK;
    }
    { int r_ = octree_nodes(c, n, nn, klo); if (r_) return r_; }
    LAUNCH(k_oct_finalize, cdiv(nn, T), T, 0, nn, c->nodes, c->wcount, c->wstart, c->widx, c->wnodes);
    readback(c, c->h_rb, c->d_nsel, sizeof(int));
    CK(cudaStreamSynchronize(c->stream));
    const int ng = c->h_rb[0];
    c->n_groups = ng;
    if (ng + bvh_upper_boxes(ng) > c->bvh_cap) { c->bvh_cap = (ng + bvh_upper_boxes(ng)) * 5 / 4; DA(c->bvh, c->bvh_cap); }
    LAUNCH(k_group_pack, cdiv(ng, T), T, 0, ng, c->gfirst, c->gsize, c->groups);
    StateArrays s = state_of(c, c->cur);
    LAUNCH(k_bvh_leaf, cdiv((int64_t)ng * 32, T), T, 0, ng, c->groups, s.x, s.y, s.z, c->lcx, c->lcy, c->lcz, c->reach, c->bvh);
    bvh_levels(c, c->bvh, ng, c->bvh, ng, c->bi);
    { int r_ = compute_slices(c); if (r_) return r_; }
    // sized here so that the peer mapping (first exchange = density) sees it
    { int r_ = sink_seg_reserve(c, cdiv(ng, GRAV_SEG)); if (r_) return r_; }
  }
  stage_end(c);
  c->tree_valid = true; c->pos_moved = false;
  return SPH_OK;
}


size_t density_smem(const sph_ctx* c, int nwarp) { return (size_t)2 * (c->p.nq + 1) * 8 + (size_t)nwarp * DENS_WARP_DOUBLES * 8 + (size_t)nwarp * WALK_WS * 4; }
size_t force_smem(const sph_ctx* c, int nwarp, bool listed) {
  size_t t = (size_t)((c->p.nq + 1) + ((c->p.nq + 1) & 1)) * 8;
  return t + (size_t)nwarp * FORCE_WARP_DOUBLES * 8 + (size_t)nwarp * WALK_TILE * 4 + (listed ? 0 : (size_t)nwarp * WALK_WS * 4);
}
// warps per block of the pair kernels: as many (<= 16) as the shared memory left beside the kernel table allows
int force_warps(const sph_ctx* c, bool listed) {
  int w = 16;
  while (w > 1 && force_smem(c, w, listed) > (size_t)c->max_smem) --w;
  return w;
}
int walk_grid(const sph_ctx* c, int nwarp) {
  const int nchunk = c->g1 - c->g0;
  return std::max(1, std::min(cdiv(nchunk, nwarp), c->n_sm));
}

DensityArrays dens_arrays(sph_ctx* c) {
  StateArrays s = state_of(c, c->cur);
  return DensityArrays{s.x, s.y, s.z, s.m, c->lcx, c->lcy, c->lcz, c->reach};
}

int run_density(sph_ctx* c) {
  const int W = DENS_WARPS;
  { int r_ = flush_late(c, LF_U | LF_M | LF_H); if (r_) return r_; }
  stage_begin(c, ST_DENSITY);
  StateArrays s = state_of(c, c->cur);
  // pool of 32-int blocks for the saved candidate lists: about one block (30 sources) per local particle, grown
  // when an evaluation overflowed it (that evaluation's pair loop walks by itself instead)
  {
    const size_t want = (size_t)(c->p1 - c->p0) + 4 * (size_t)(c->g1 - c->g0) + 1024 + (size_t)NL_BATCH * 16 * c->n_sm;
    if (c->nl_pool_blocks == 0 && getenv("SPH_B200_LIST_POOL_BLOCKS")) {      // test hook: start with a pool that is too small
      c->nl_pool_blocks = (size_t)std::max(64, atoi(getenv("SPH_B200_LIST_POOL_BLOCKS"))); DA(c->nl_pool, c->nl_pool_blocks * 32);
    } else if (want > c->nl_pool_blocks && !getenv("SPH_B200_LIST_POOL_BLOCKS")) { c->nl_pool_blocks = want + want / 4; DA(c->nl_pool, c->nl_pool_blocks * 32); }
    if ((size_t)c->n_groups + 1 > c->nl_head_cap) { c->nl_head_cap = (size_t)c->n_groups * 5 / 4 + 64; DA(c->nl_head, c->nl_head_cap); }
    CK(cudaMemsetAsync(c->nl_ctl, 0, 2 * sizeof(int), c->stream));      // ctl[2] (overflow) is sticky until the host has seen it
  }
  const NeighbourListSink nl{c->nl_pool, c->nl_head, c->nl_ctl, (int)std::min<size_t>(c->nl_pool_blocks, 0x7fffffff)};
  LAUNCH(k_set_int, 1, 1, 0, c->work, c->g0);
  LAUNCH(k_density<false>, walk_grid(c, W), W * 32, density_smem(c, W), c->g1, c->groups, c->dp, dens_arrays(c), c->bvh, c->bi, c->d_wt, c->d_dwt,
         s.u, s.h, c->rho, c->omega, c->prs, c->cs, c->por2, c->ctr, c->work, c->exact_counters, nl);
  c->nl_valid = true; c->nl_exact = c->exact_counters;
  // a non-finite particle anywhere voids every rank's lists.  Domains: the flag rides the one all-reduce of the evaluation (after the gravity walk)
  if (c->n_ranks > 1 && !c->dd) { int r_ = allreduce(c, c->nl_ctl + 1, 1, 2 /*ncclInt32*/, 2 /*ncclMax*/); if (r_) return r_; }
  stage_end(c);
  c->dd_fields_pending = c->dd;        // the halo's rho, c, P/(Omega rho^2) are pulled after that all-reduce (it is also the "every density pass has finished" barrier)
  if (c->dd) {}
  else if (c->n_ranks > 1) { stage_begin(c, ST_COMM); double* bufs[3] = {c->rho, c->cs, c->por2}; int r_ = allgatherv_begin(c, bufs, 3);   /* what the pair loop reads of its sources (Omega and P stay rank-local until a diagnostic download asks); completes under the gravity walk */ if (r_) return r_; stage_end(c); }
  return SPH_OK;
}
int run_hiter(sph_ctx* c) {
  const int W = DENS_WARPS;
  c->nl_valid = false;                       // h changes: the saved lists' distance culls no longer hold
  stage_begin(c, ST_HITER);
  StateArrays s = state_of(c, c->cur);
  LAUNCH(k_set_int, 1, 1, 0, c->work, c->g0);
  LAUNCH(k_density<true>, walk_grid(c, W), W * 32, density_smem(c, W), c->g1, c->groups, c->dp, dens_arrays(c), c->bvh, c->bi, c->d_wt, c->d_dwt,
         s.u, s.h, c->rho, c->omega, c->prs, c->cs, c->por2, c->ctr, c->work, c->exact_counters, NeighbourListSink{nullptr, nullptr, c->nl_ctl, 0});
  stage_end(c);
  if (c->n_ranks > 1 && !c->dd) { stage_begin(c, ST_COMM); double* bufs[1] = {s.h}; int r_ = allgatherv(c, bufs, 1); if (r_) return r_; stage_end(c); }
  return SPH_OK;
}
int run_force(sph_ctx* c) {
  { int r_ = flush_late(c, LF_ALL); if (r_) return r_; }
  if (c->x_pending) { stage_begin(c, ST_COMM); int r_ = allgatherv_end(c); if (r_) return r_; stage_end(c); }
  stage_begin(c, ST_SPH);
  StateArrays s = state_of(c, c->cur);
  ForceArrays A{s.x, s.y, s.z, s.vx, s.vy, s.vz, s.m, s.h, c->rho, c->cs, s.alpha, c->por2, c->lcx, c->lcy, c->lcz, c->reach, s.id};
  const NeighbourListSink nl{c->nl_pool, c->nl_head, c->nl_ctl, (int)std::min<size_t>(c->nl_pool_blocks, 0x7fffffff)};
  const bool listed = c->nl_valid && c->nl_exact == c->exact_counters && c->use_lists;
  const int WL = force_warps(c, true), WW = force_warps(c, false);
  // peers' copies of the five output arrays: the kernel pushes its results itself (exchanged_arrays slots 3..7)
  PeerOut po; po.n = 0;
  if (c->n_ranks > 1 && !c->dd) {
    if (c->p2p_stale) { int r_ = p2p_setup(c); if (r_) return r_; }
    if (c->p2p_ok && c->n_ranks - 1 <= SPH_MAX_PEERS && c->fused_push) {
      for (int k = 1; k < c->n_ranks; ++k) {
        const int r = (c->rank + k) % c->n_ranks;
        for (int f = 0; f < 5; ++f) po.p[po.n][f] = c->peer[3 + f][r];
        ++po.n;
      }
    }
  }
  if (listed) {
    LAUNCH(k_set_int, 1, 1, 0, c->work, c->g0);
    LAUNCH(k_force<true>, walk_grid(c, WL), WL * 32, force_smem(c, WL, true), c->g1, c->groups, c->dp, A, c->bvh, c->bi, c->d_dwt, c->ax, c->ay, c->az, c->udot, c->adot, c->ctr, c->work, c->exact_counters, nl, 0, po);
  }
  LAUNCH(k_set_int, 1, 1, 0, c->work, c->g0);
  LAUNCH(k_force<false>, walk_grid(c, WW), WW * 32, force_smem(c, WW, false), c->g1, c->groups, c->dp, A, c->bvh, c->bi, c->d_dwt, c->ax, c->ay, c->az, c->udot, c->adot, c->ctr, c->work, c->exact_counters, nl, listed ? 1 : 0, po);
  stage_end(c);
#ifdef WALK_DEBUG
  { unsigned long long d[16]; cudaStreamSynchronize(c->stream); cudaMemcpyFromSymbol(d, wk_dbg, sizeof(d)); unsigned long long z[16] = {}; cudaMemcpyToSymbol(wk_dbg, z, sizeof(z));
    fprintf(stderr, "WKDBG groups %d force: tiles %llu staged %llu trips %llu hits %llu boxpairs %llu | density: tiles %llu staged %llu trips %llu hits %llu\n", c->n_groups, d[0], d[1], d[2], d[3], d[4], d[8], d[9], d[10], d[11]); }
#endif
  if (c->n_ranks > 1 && !c->dd) {
    stage_begin(c, ST_COMM);
    if (po.n > 0) {     // the kernels pushed their slices themselves: only the "every rank's kernel has finished" barrier is left
      { int r_ = coll_allreduce(c, c->stream, c->d_flag + 2, 1, NC_INT32, NC_SUM); if (r_) return r_; }
    } else { double* bufs[5] = {c->ax, c->ay, c->az, c->udot, c->adot}; int r_ = allgatherv(c, bufs, 5); if (r_) return r_; }
    stage_end(c);
  }
  return SPH_OK;
}
int grav_warps(const sph_ctx* c);
size_t gravity_smem(const sph_ctx* c, int nwarp) { return (size_t)((c->p.nq + 1) + ((c->p.nq + 1) & 1)) * 8 + (size_t)nwarp * sizeof(GravWarpSmem); }
int grav_warps(const sph_ctx* c) {     // as many warps (<= GW_WARPS) as the shared memory beside the kernel table holds
  int w = GW_WARPS;
  while (w > 1 && gravity_smem(c, w) > (size_t)c->max_smem) --w;
  return w;
}
__global__ void k_ctr_save(const WalkCounters* ctr, unsigned long long* saved) { saved[0] = ctr->grav_opened; saved[1] = ctr->grav_accepted; }
__global__ void k_ctr_restore(WalkCounters* ctr, const unsigned long long* saved) { ctr->grav_opened += saved[0]; ctr->grav_accepted += saved[1]; }

int run_gravity(sph_ctx* c, int do_grav, int do_sinks) {
  const int GWW = grav_warps(c);
  // far-field reuse (sph_gravity.cuh): the full walk stores the far sums of its tree terms; while they stand (far_valid: same
  // tree, no h beyond its cutoff - decided at the end of step()), the next evaluation adds only the near field and the sinks
  // Stored only where the next evaluation can use it: by evaluation B of a step whose state stayed on the device since the
  // step before (a host that uploads before every step never reuses, and should not pay for the records)
  const bool far_ok = c->far_reuse && do_grav && !c->dp.soft_hi && !c->exact_counters;
  const bool near_only = far_ok && c->far_valid;
  const bool far_on = far_ok && !near_only && c->far_want_store;
  if (near_only) ++c->far_count;
  if (!near_only) c->far_valid = false;      // a full walk re-takes the near / far split (and may not store at all)
  stage_begin(c, near_only ? ST_GRAV_NEAR : ST_GRAVITY);
  StateArrays s = state_of(c, c->cur);
  // upper bound of the number of runs in this rank's slice; unused tail entries stay empty (first = 0, count = 0)
  const int seg0 = c->g0 / GRAV_SEG, nseg = cdiv(c->g1 - c->g0, GRAV_SEG);
  const int ng = cdiv(c->p1 - c->p0, std::min(GRAV_CHUNK_WIDTH, GRAV_MINFILL)) + 2 * nseg;
  const int ns = do_sinks ? c->n_sink : 0;
  if ((size_t)(ng + 8) * std::max(ns, 1) * 3 > c->sink_partial_cap) {
    c->sink_partial_cap = (size_t)(ng + 8) * std::max(ns, 1) * 3 * 2;
    DA(c->sink_partial, c->sink_partial_cap);
  }
  if (ng > 0 && c->g1 > c->g0) {
    const int grid = std::max(1, std::min(cdiv(ng, GWW), c->n_sm));
    if (!c->grav_spill) DA(c->grav_spill, (size_t)c->n_sm * GW_WARPS * GW_SPILL);
    if (!c->grav_groups_valid) {
      if ((size_t)ng > c->ggroups_cap) { c->ggroups_cap = (size_t)ng * 5 / 4 + 64; DA(c->ggroups, c->ggroups_cap); DA(c->gbvh, c->ggroups_cap); }
      if ((size_t)nseg + 1 > c->seg_cap) { c->seg_cap = (size_t)nseg * 5 / 4 + 64; DA(c->seg_cnt, c->seg_cap); DA(c->seg_off, c->seg_cap); }
      CK(cudaMemsetAsync(c->ggroups, 0, sizeof(int2) * (size_t)ng, c->stream));
      LAUNCH(k_seg_count, cdiv(nseg + 1, 64), 64, 0, seg0, nseg, c->g1, GRAV_CHUNK_WIDTH, c->groups, c->seg_cnt);
      size_t bytes = c->cub_bytes;
      CK(cub::DeviceScan::ExclusiveSum(c->cub_tmp, bytes, c->seg_cnt, c->seg_off, nseg + 1, c->stream));
      LAUNCH(k_seg_chunks, cdiv(nseg, 64), 64, 0, seg0, nseg, c->g1, GRAV_CHUNK_WIDTH, c->groups, c->seg_off, c->ggroups);
      LAUNCH(k_grav_boxes, cdiv((int64_t)ng * 32, 256), 256, 0, ng, c->ggroups, s.x, s.y, s.z, c->gbvh);
      c->grav_groups_valid = true;
    }
    if (c->let_pending) { CK(cudaStreamWaitEvent(c->stream, c->let_done, 0)); c->let_pending = false; }      // domains: the locally essential tree was pulled under the density pass
    // recorded near pairs: slots x 32 ints per run (16 KB at 128 slots); without the memory the near field is walked
    if (far_on && c->far_lists && (size_t)ng > c->far_list_runs) {
      if (c->far_list) { cudaFree(c->far_list); cudaFree(c->far_cnt); cudaFree(c->far_ovf); c->far_list = nullptr; c->far_cnt = nullptr; c->far_ovf = nullptr; }
      const size_t runs = (size_t)ng + ng / 50 + 64;
      if (cudaMalloc((void**)&c->far_list, runs * c->far_slots * 32 * sizeof(int)) != cudaSuccess || cudaMalloc((void**)&c->far_cnt, runs * 32 * sizeof(int)) != cudaSuccess ||
          cudaMalloc((void**)&c->far_ovf, runs) != cudaSuccess) {
        cudaGetLastError();
        if (c->far_list) cudaFree(c->far_list); if (c->far_cnt) cudaFree(c->far_cnt); if (c->far_ovf) cudaFree(c->far_ovf);
        c->far_list = nullptr; c->far_cnt = nullptr; c->far_ovf = nullptr; c->far_list_runs = 0; c->far_lists = false;
      } else c->far_list_runs = runs;
    }
    const bool lists = (far_on || near_only) && c->far_lists && c->far_list != nullptr;
    const FarField ff{c->far_fx, c->far_fy, c->far_fz, c->far_hc2, far_on ? 1 : 0, lists ? c->far_list : nullptr, c->far_cnt, c->far_ovf, c->far_slots, &c->sc->far_ovf};
    if (near_only) {
      if (lists) LAUNCH(k_gravity_near, std::max(1, std::min(cdiv(ng, GN_WARPS), 16 * c->n_sm)), GN_WARPS * 32, gravity_smem(c, 0), ng, c->ggroups, c->dp, c->wnodes, s.x, s.y, s.z, s.h, s.m, c->d_gt, c->ax, c->ay, c->az, ns, c->S, c->sink_partial, ff);
      if (!lists || c->far_n_ovf > 0) {       // runs whose lists overflowed (or all of them without lists): the near-only walk
        LAUNCH(k_set_int, 1, 1, 0, c->work, 0);
        LAUNCH(k_gravity<1>, grid, GWW * 32, gravity_smem(c, GWW), 0, ng, c->ggroups, c->gbvh, c->dp, c->wnodes, s.x, s.y, s.z, s.h, s.m, c->d_gt,
               c->ax, c->ay, c->az, do_grav, ns, c->S, c->sink_partial, c->ctr, c->work, c->grav_spill, &c->sc->err, ff);
      }
    } else {
      LAUNCH(k_set_int, 1, 1, 0, c->work, 0);
      CK(cudaMemsetAsync(&c->sc->far_ovf, 0, sizeof(int), c->stream));
      if (far_on) {
        LAUNCH(k_far_hcut, cdiv(c->n, 256), 256, 0, (int)c->n, c->dp, s.h, c->far_hcut, c->far_hc2);
        LAUNCH(k_gravity<0>, grid, GWW * 32, gravity_smem(c, GWW), 0, ng, c->ggroups, c->gbvh, c->dp, c->wnodes, s.x, s.y, s.z, s.h, s.m, c->d_gt,
               c->ax, c->ay, c->az, do_grav, ns, c->S, c->sink_partial, c->ctr, c->work, c->grav_spill, &c->sc->err, ff);
      } else      // nothing to store (first step on a new state, exact counters, reuse switched off): the plain walk, one sum per particle
        LAUNCH(k_gravity<2>, grid, GWW * 32, gravity_smem(c, GWW), 0, ng, c->ggroups, c->gbvh, c->dp, c->wnodes, s.x, s.y, s.z, s.h, s.m, c->d_gt,
               c->ax, c->ay, c->az, do_grav, ns, c->S, c->sink_partial, c->ctr, c->work, c->grav_spill, &c->sc->err, ff);
    }
  }
#ifdef GW_STATS
  { unsigned long long d[16]; cudaStreamSynchronize(c->stream); cudaMemcpyFromSymbol(d, gw_stats, sizeof(d)); unsigned long long z[16] = {}; cudaMemcpyToSymbol(gw_stats, z, sizeof(z));
    fprintf(stderr, "GWSTATS mode %d runs %llu trips %llu pops %llu pruned %llu accept %llu open %llu mixed %llu | far entries %llu (lanes %llu) near entries %llu (lanes %llu) evals %llu\n",
            near_only ? 1 : 0, d[0], d[10], d[1], d[2], d[3], d[4], d[5], d[6], d[8], d[7], d[9], d[12]); }
#endif
  // sink side of the gas terms: per-segment folds -> exchange of the rows -> one fixed fold over all segments (rank-count independent)
  {
    const int nst = cdiv(c->dd ? c->g1 : c->n_groups, GRAV_SEG);
    { int r_ = sink_seg_reserve(c, nst); if (r_) return r_; }
    if (do_sinks && nseg > 0 && c->g1 > c->g0)
      LAUNCH(k_sink_seg_fold, cdiv((int64_t)nseg * c->n_sink * 3, 128), 128, 0, nseg, seg0, c->n_sink, c->seg_off, c->sink_partial, c->sink_seg);
    stage_end(c);
    if (c->n_ranks > 1 && do_sinks && !c->dd) {
      stage_begin(c, ST_COMM);
      std::vector<size_t> roff(c->n_ranks + 1);
      for (int r = 0; r <= c->n_ranks; ++r) roff[r] = (size_t)(r == c->n_ranks ? nst : c->rank_g[r] / GRAV_SEG) * c->n_sink * 3;
      double* bufs[1] = {c->sink_seg};
      int r_ = allgatherv(c, bufs, 1, roff.data()); if (r_) return r_;
      stage_end(c);
    }
    stage_begin(c, near_only ? ST_GRAV_NEAR : ST_GRAVITY);
    LAUNCH(k_sink_reduce, 1, 256, 0, nst, c->n_sink, c->sink_seg, c->S, do_sinks);
    stage_end(c);
    // domains: the segments are per rank (walk groups differ at domain boundaries), so the ranks' totals are added
    if (c->dd) {
      stage_begin(c, ST_COMM);
      if (c->let_pending) { CK(cudaStreamWaitEvent(c->stream, c->let_done, 0)); c->let_pending = false; }
      // ONE all-reduce per evaluation: the ranks' sink sums, their LET overflow flags and their "lists void" flags; it is
      // also the barrier behind which the peers' density fields are final (one sync point per evaluation instead of three)
      LAUNCH(k_dd_flags_pack, 1, 1, 0, c->nl_ctl, c->let_flag);
      int r_ = allreduce(c, c->S.ax, (size_t)3 * SPH_MAX_SINKS + 2, NC_FLOAT64, NC_SUM); if (r_) return r_;
      LAUNCH(k_dd_flags_apply, 1, 1, 0, c->let_flag, &c->sc->err, c->nl_ctl);
      if (c->dd_fields_pending) { r_ = dd_pull_density_fields(c); if (r_) return r_; c->dd_fields_pending = false; }
      stage_end(c);
    }
  }
  stage_begin(c, near_only ? ST_GRAV_NEAR : ST_GRAVITY);
  LAUNCH(k_sink_pairs, 1, 32, 0, c->n_sink, c->S, c->dp.G, do_sinks);
  if (near_only) LAUNCH(k_ctr_restore, 1, 1, 0, c->ctr, c->far_ctr);      // the walk's counters of the evaluation the far sums were taken in (same accepted sets)
  else if (far_on) { LAUNCH(k_ctr_save, 1, 1, 0, c->ctr, c->far_ctr); c->far_valid = true; }
  stage_end(c);
  return SPH_OK;
}

int evaluate(sph_ctx* c, int mask) {
  if (c->n < 2) { c->err = "need at least 2 gas particles"; return SPH_ERR_STATE; }
  int r;
  if (mask & SPH_EVAL_TREE) { if ((r = build_tree(c))) return r; }
  else if (!c->tree_valid) { c->err = "no tree: evaluate with SPH_EVAL_TREE first"; return SPH_ERR_STATE; }
  const size_t nb = (size_t)c->n * 8;        // after the build: under the domain decomposition the build changes which particles live here
  CK(cudaMemsetAsync(c->ax, 0, nb, c->stream)); CK(cudaMemsetAsync(c->ay, 0, nb, c->stream)); CK(cudaMemsetAsync(c->az, 0, nb, c->stream));
  CK(cudaMemsetAsync(c->udot, 0, nb, c->stream)); CK(cudaMemsetAsync(c->adot, 0, nb, c->stream));     // F:824
  CK(cudaMemsetAsync(c->ctr, 0, sizeof(WalkCounters), c->stream));
  if (mask & SPH_EVAL_DENSITY) { if ((r = run_density(c))) return r; }
  if ((r = flush_late(c, LF_M | LF_H))) return r;
  if ((r = run_gravity(c, (mask & SPH_EVAL_GRAVITY) ? 1 : 0, (mask & SPH_EVAL_SINKS) ? 1 : 0))) return r;
  if (mask & SPH_EVAL_SPH) { if ((r = run_force(c))) return r; }
  else if (!c->dd) { double* bufs[3] = {c->ax, c->ay, c->az}; if ((r = allgatherv(c, bufs, 3))) return r; }
  return flush_late(c, LF_ALL);
}

int fetch_counters(sph_ctx* c) {
  { int r_ = allreduce(c, c->ctr, sizeof(WalkCounters) / 8, NC_UINT64, NC_SUM); if (r_) return r_; }
  readback(c, c->h_ctr, c->ctr, sizeof(WalkCounters));
  CK(cudaStreamSynchronize(c->stream));
  c->counts.n_gas = c->dd ? c->n_global : c->n;
  c->counts.density_candidates = (int64_t)c->h_ctr->dens_cand;
  c->counts.density_contributing = (int64_t)c->h_ctr->dens_contrib;
  c->counts.sph_pairs = (int64_t)(c->h_ctr->sph_pairs / 2);
  c->counts.grav_opened = (int64_t)c->h_ctr->grav_opened;
  c->counts.grav_accepted = (int64_t)c->h_ctr->grav_accepted;
  return SPH_OK;
}

int check_device_error(sph_ctx* c) {
  if (c->h_sc->err == 2) { c->err = "gravity walk: node stack overflow (GW_SPILL)"; return SPH_ERR_STATE; }
  if (c->h_sc->err == 5) { c->err = "domain decomposition: the locally essential tree of some rank exceeds its capacity (raise SPH_B200_DOMAIN_SLACK)"; return SPH_ERR_OOM; }
  if (c->h_sc->err == 3) { c->err = "sink table full (SPH_MAX_SINKS): check_sink_creation (V:549-597) could not append a sink"; return SPH_ERR_STATE; }
  if (c->h_sc->err) {
    c->err = "particles share a full 126-bit descent key (closer than root_size/2^42) while max_depth > 42";
    return SPH_ERR_DEPTH;
  }
  return SPH_OK;
}

// compaction after accretion / bounds: order preserving (pack, F:481,554)
int compact(sph_ctx* c) {
  const int n = (int)c->n, T = 256;
  LAUNCH(k_iota, cdiv(n, T), T, 0, n, c->perm[0]);
  size_t bytes = c->cub_bytes;
  CK(cub::DeviceSelect::Flagged(c->cub_tmp, bytes, c->perm[0], c->keep, c->perm[1], c->d_nsel, n, c->stream));
  int nsel = 0;
  CK(cudaMemcpyAsync(&nsel, c->d_nsel, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  PermuteArgs pa;
  for (int f = 0; f < 10; ++f) { pa.src[f] = c->st[c->cur][f]; pa.dst[f] = c->st[c->cur ^ 1][f]; }
  pa.id_src = c->id[c->cur]; pa.id_dst = c->id[c->cur ^ 1];
  if (nsel > 0) LAUNCH(k_permute, cdiv(nsel, 4 * T), T, 0, nsel, c->perm[1], pa);
  c->cur ^= 1;
  c->n = nsel;
  c->tree_valid = false; c->pos_moved = true;
  return SPH_OK;
}

// sph_step_host: columns that are final leave while the step goes on.  Scatter into ascending-number order on the compute
// stream (nothing was removed since the upload of this call: number == id), copies on io_stream.
int io_fetch(sph_ctx* c, const int* fields, int nf) {
  if (!c->io_active || c->n != c->n_upload) return SPH_OK;
  const int n = (int)c->n, T = 256;
  if (c->io_busy) CK(cudaStreamWaitEvent(c->stream, c->io_ev_done, 0));      // the staging buffers of the batch before
  int used = 0; int fl[5];
  for (int k = 0; k < nf && used < 5; ++k) {
    const int f = fields[k];
    if (!c->io_out[f]) continue;
    LAUNCH(k_scatter<double>, cdiv(n, T), T, 0, n, c->id[c->cur], c->st[c->cur][f], c->io_stage[used]);
    fl[used++] = f;
  }
  if (!used) return SPH_OK;
  CK(cudaEventRecord(c->io_ev_out, c->stream));
  CK(cudaStreamWaitEvent(c->io_stream, c->io_ev_out, 0));
  for (int k = 0; k < used; ++k) {
    CK(cudaMemcpyAsync(c->io_out[fl[k]], c->io_stage[k], (size_t)n * 8, cudaMemcpyDeviceToHost, c->io_stream));
    c->io_fetched |= 1u << fl[k];
  }
  CK(cudaEventRecord(c->io_ev_done, c->io_stream));
  c->io_busy = true;
  return SPH_OK;
}

int step(sph_ctx* c) {
  const int T = 256;
  int r;
  int n = (int)c->n;
  c->far_want_store = false;                                                   // the positions move right after this evaluation
  if ((r = evaluate(c, SPH_EVAL_ALL))) return r;                              // F:894-898
  n = (int)c->n;                                                               // domains: the build may have moved particles between ranks
  stage_begin(c, ST_INTEGRATE);
  LAUNCH(k_kick<true>, cdiv(n, T), T, 0, n, state_of(c, c->cur), rates_of(c), c->sc);       // F:900,903
  c->pos_moved = true;
  LAUNCH(k_kick_sinks<true>, 1, SPH_MAX_SINKS, 0, c->S, c->sc);
  stage_end(c);
  if (c->io_active) { const int fl[4] = {0, 1, 2, 7}; if ((r = io_fetch(c, fl, 4))) return r; }      // x y z are final after the drift (F:903), m never changes
  c->far_want_store = c->steps_since_upload >= 1;
  if ((r = evaluate(c, SPH_EVAL_ALL))) return r;                              // F:905-910
  n = (int)c->n;
  stage_begin(c, ST_INTEGRATE);
  LAUNCH(k_kick<false>, cdiv(n, T), T, 0, n, state_of(c, c->cur), rates_of(c), c->sc);      // F:912
  LAUNCH(k_kick_sinks<false>, 1, SPH_MAX_SINKS, 0, c->S, c->sc);
  if (c->io_active) { const int fl[5] = {3, 4, 5, 6, 8}; if ((r = io_fetch(c, fl, 5))) return r; }  // v u alpha are final after the second kick (F:912)
  {
    int nb = std::max(1, std::min(cdiv(c->p1 - c->p0, T), c->n_partial));
    LAUNCH(k_dt_partial, nb, T, 0, c->p0, c->p1, c->dp, state_of(c, c->cur), rates_of(c), c->cs, c->partial);   // F:916
    LAUNCH(k_dt_fold, 1, 32, 0, nb, c->partial, c->sc);
    { int r_ = allreduce(c, &c->sc->dt_min, 1, NC_FLOAT64, NC_MIN); if (r_) return r_; }
    LAUNCH(k_dt_ladder, 1, 1, 0, c->dp, c->sc, 1);                                                   // F:914,855-859
  }
  stage_end(c);
  if (c->dp.variable_h) {
    if ((r = run_hiter(c))) return r;                                         // V:1152
    stage_begin(c, ST_CULL);
    LAUNCH(k_create_scan, cdiv(n, T), T, 0, n, c->dp, state_of(c, c->cur), c->sc);          // V:1155
    if (c->dd) {      // the lowest-numbered over-dense particle of ALL domains; its owner publishes x v h
      CK(cudaMemcpyAsync(c->dd_cand, &c->sc->create_cand, 8, cudaMemcpyDeviceToDevice, c->stream));
      CK(cudaMemcpyAsync(c->dd_cand + 1, &c->sc->create_cand, 8, cudaMemcpyDeviceToDevice, c->stream));
      LAUNCH(k_dd_cand_id, 1, 1, 0, c->dd_cand + 1);
      { int r_ = allreduce(c, c->dd_cand + 1, 1, NC_UINT64, NC_MIN); if (r_) return r_; }
      LAUNCH(k_dd_create_publish, 1, 32, 0, c->dd_cand, c->dd_cand + 1, state_of(c, c->cur), c->dd_create8);
      { int r_ = allreduce(c, c->dd_create8, 8, NC_FLOAT64, NC_SUM); if (r_) return r_; }
      LAUNCH(k_dd_create_apply, 1, 32, 0, c->dd_create8, c->S, c->sc, c->sink_spin);
    } else
    LAUNCH(k_create_apply, 1, 32, 0, state_of(c, c->cur), c->S, c->sc, c->sink_spin);
    stage_end(c);
  }
  stage_begin(c, ST_CULL);
  LAUNCH(k_any_sink_mass, 1, 32, 0, c->S, c->sc);                             // F:919
  auto flags = [&]() -> int {
    LAUNCH(k_flags, cdiv(n, T), T, 0, n, c->dp, state_of(c, c->cur), c->key[0], c->two_word ? c->key_lo[0] : nullptr, c->level, c->lcx, c->lcy, c->lcz, c->reach, c->root,
           c->S, c->sc, c->keep, c->acc_key[0], c->acc_val[0], (int)c->acc_cap);
    readback(c, c->h_sc, c->sc, sizeof(SimScalars));
    CK(cudaStreamSynchronize(c->stream));
    return check_device_error(c);
  };
  if ((r = flags())) return r;
  // k_flags counts every (sink, particle) entry but stores only the first acc_cap: a particle inside several sinks' radii is
  // accreted by each of them, so the list can outgrow the particle count.  Then grow it and flag again - k_flags reads
  // only the state, the tree and the sinks and rewrites keep[] for every row, so the second pass is the first one whole
  if (c->h_sc->n_accreted > c->acc_cap) {
    const int64_t want = (int64_t)c->h_sc->n_accreted;
    if ((r = ensure_acc_capacity(c, want + want / 8 + 1024))) return r;
    CK(cudaMemsetAsync(&c->sc->n_removed, 0, sizeof(int) * 2, c->stream));      // n_removed, n_accreted
    if ((r = flags())) return r;
  }
  int n_acc = c->h_sc->n_accreted;
  int n_removed_global = c->h_sc->n_removed;
  if (c->dd) { int r_ = dd_accrete(c, n_acc, &n_removed_global); if (r_) return r_; }
  else {
    if (n_acc > 1) {
      cub::DoubleBuffer<unsigned long long> dk(c->acc_key[0], c->acc_key[1]); cub::DoubleBuffer<int> dv(c->acc_val[0], c->acc_val[1]);
      size_t bytes = c->cub_bytes;
      CK(cub::DeviceRadixSort::SortPairs(c->cub_tmp, bytes, dk, dv, n_acc, 0, 64, c->stream));
      if (dk.Current() != c->acc_key[0]) std::swap(c->acc_key[0], c->acc_key[1]);
      if (dv.Current() != c->acc_val[0]) std::swap(c->acc_val[0], c->acc_val[1]);
    }
    LAUNCH(k_accrete_apply, 1, SPH_MAX_SINKS, 0, n_acc, c->acc_key[0], c->acc_val[0], state_of(c, c->cur), c->S, c->sc, c->sink_spin);
  }
  if (c->dp.variable_h) LAUNCH(k_cull_sinks, 1, 32, 0, c->dp, c->S, c->sc, c->sink_spin);   // V:613
  if (c->sink_extras) LAUNCH(k_sink_merge, 1, 32, 0, c->S, c->sc, c->sink_spin);            // V:1159 (commented out in the reference)
  const int n_removed = c->h_sc->n_removed;
  // reset per-step device counters
  CK(cudaMemsetAsync(&c->sc->n_removed, 0, sizeof(int) * 2, c->stream));
  if (n_removed > 0) { if ((r = compact(c))) return r; }
  if (c->dd && n_removed_global > 0) { c->tree_valid = false; c->pos_moved = true; c->n_global -= n_removed_global; }      // every domain rebuilds when any lost a particle
  // may evaluation A of the next step keep evaluation B's far-field gravity?  Same particles (no removal anywhere) and no h
  // beyond the cutoff its near / far split was taken with; domains agree through one all-reduce
  const bool far_try = c->far_valid && n_removed == 0 && n_removed_global == 0;
  CK(cudaMemsetAsync(&c->sc->far_bad, 0, sizeof(int), c->stream));
  if (far_try) {
    LAUNCH(k_far_check, cdiv(c->n, T), T, 0, (int)c->n, c->dp, state_of(c, c->cur).h, c->far_hc2, &c->sc->far_bad);
    if (c->dd) { int r_ = allreduce(c, &c->sc->far_bad, 1, NC_INT32, NC_MAX); if (r_) return r_; }
  }
  readback(c, c->h_sc, c->sc, sizeof(SimScalars));
  int* const nl_host = c->h_rb + 4;
  readback(c, nl_host, c->nl_ctl, 4 * sizeof(int));
  CK(cudaStreamSynchronize(c->stream));
  if (nl_host[2]) {                          // the candidate-list pool overflowed in this step: double it for the next one
    const size_t want = c->nl_pool_blocks * 2;
    DA(c->nl_pool, want * 32); c->nl_pool_blocks = want;
    CK(cudaMemsetAsync(c->nl_ctl, 0, 4 * sizeof(int), c->stream));
  }
  c->nl_valid = false;
  c->far_valid = far_try && c->h_sc->far_bad == 0;
  c->far_n_ovf = c->h_sc->far_ovf;
  ++c->steps_since_upload;
  c->n_sink = c->h_sc->n_sink;
  stage_end(c);
  return SPH_OK;
}

// ---- host-facing downloads: the rows in ascending-number order (sph_download, _diag, _tree, _neighbours, sph_step_host)
// Rows covered: under domains every rank's own rows, otherwise this rank's (all of them in the replicated form).
int64_t download_count(const sph_ctx* c) { return c->dd ? c->n_global : c->n; }
// The ascending-number position of every covered row: dd_gpos under domains (collective), else pos.
int download_rows(sph_ctx* c) {
  if (c->dd) return dd_prepare_download(c);
  if (c->n == c->n_upload) {         // nothing was ever removed: number == upload index
    CK(cudaMemcpyAsync(c->pos, c->id[c->cur], (size_t)c->n * 4, cudaMemcpyDeviceToDevice, c->stream));
    return SPH_OK;
  }
  return id_ranks(c, (int)c->n, c->id[c->cur], c->cnt, c->off, c->pos);      // n_upload <= cap: cnt / off (cap + 1 ints) are only read while the octree is being built
}
// One column of the covered rows to the host in ascending-number order (elem = 4 or 8 bytes; nothing if dst_host is null).
// Domains: the ranks' own values are gathered in rank order into the first half of dd_gstage, then scattered into the
// second.  Otherwise the scatter reads the column in place and alternates between two staging buffers, so the scatter of
// the next column overlaps nothing it depends on (stream order protects the buffers); the caller synchronises once.
int fetch_column(sph_ctx* c, Column col, size_t elem, void* dst_host) {
  if (!dst_host) return SPH_OK;
  const int n = (int)download_count(c), T = 256;
  const void* src; void* stage; const int* pos;
  if (c->dd) {
    { int r_ = dd_gather(c, col, elem, c->dd_gstage); if (r_) return r_; }
    src = c->dd_gstage; stage = c->dd_gstage + c->dd_g_cap; pos = c->dd_gpos;
  } else {
    src = dd_exported(c)[column_slot(col, c->cur, c->key[0] == c->key_alloc[0] ? 0 : 1)];
    stage = c->stage_flip ? c->stage_d2 : c->stage_d; c->stage_flip ^= 1; pos = c->pos;
  }
  if (elem == 4) LAUNCH(k_scatter<int>, cdiv(n, T), T, 0, n, pos, (const int*)src, (int*)stage);
  else LAUNCH(k_scatter<unsigned long long>, cdiv(n, T), T, 0, n, pos, (const unsigned long long*)src, (unsigned long long*)stage);
  CK(cudaMemcpyAsync(dst_host, stage, (size_t)n * elem, cudaMemcpyDeviceToHost, c->stream));
  return SPH_OK;
}
int fetch_sink(sph_ctx* c, const double* src, double* dst_host) {
  if (!dst_host || c->n_sink == 0) return SPH_OK;
  CK(cudaMemcpyAsync(dst_host, src, (size_t)c->n_sink * 8, cudaMemcpyDeviceToHost, c->stream));
  return SPH_OK;
}

bool load_nccl(sph_ctx* c) {
  if (c->nccl.lib) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so", nullptr};
  void* h = nullptr;
  for (int i = 0; names[i] && !h; ++i) h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
  if (!h) { c->err = std::string("dlopen libnccl: ") + dlerror(); return false; }
  c->nccl.lib = h;
  *(void**)&c->nccl.GetUniqueId = dlsym(h, "ncclGetUniqueId");
  *(void**)&c->nccl.CommInitRank = dlsym(h, "ncclCommInitRank");
  *(void**)&c->nccl.CommDestroy = dlsym(h, "ncclCommDestroy");
  *(void**)&c->nccl.AllReduce = dlsym(h, "ncclAllReduce");
  *(void**)&c->nccl.AllGather = dlsym(h, "ncclAllGather");
  *(void**)&c->nccl.Broadcast = dlsym(h, "ncclBroadcast");
  *(void**)&c->nccl.GetErrorString = dlsym(h, "ncclGetErrorString");
  *(void**)&c->nccl.GroupStart = dlsym(h, "ncclGroupStart");
  *(void**)&c->nccl.GroupEnd = dlsym(h, "ncclGroupEnd");
  if (!c->nccl.CommInitRank || !c->nccl.Broadcast || !c->nccl.AllReduce || !c->nccl.GroupStart || !c->nccl.GroupEnd) { c->err = "libnccl: missing symbols"; return false; }
  return true;
}

// ---- sph_interpolate (sph_interp.cuh) ------------------------------------------------------------------------------
size_t interp_smem(const sph_ctx* c) {
  return (size_t)((c->p.nq + 1) + ((c->p.nq + 1) & 1)) * 8 + (size_t)INTERP_WARPS * (INTERP_WARP_DOUBLES * 8 + WALK_WS * 4);
}

// The per-chunk scratch for `cap` points: coordinates, the 7 raw columns, sort keys (double-buffered), bounding-box partials.
int interp_scratch(sph_ctx* c, size_t cap) {
  if (cap <= c->ip_cap) return SPH_OK;
  c->ip_cap = 0;
  DA(c->ip_pts, 3 * cap); DA(c->ip_raw, (size_t)SPH_INTERP_COUNT * cap);
  for (int b = 0; b < 2; ++b) { DA(c->ip_key[b], cap); DA(c->ip_tie[b], cap); DA(c->ip_idx[b], cap); }
  if (!c->ip_bpart) { DA(c->ip_bpart, (size_t)c->n_partial * 6); DA(c->ip_rb, 1); }
  size_t bytes = 0;
  cub::DoubleBuffer<uint64_t> dk(c->ip_key[0], c->ip_key[1]); cub::DoubleBuffer<int> dv(c->ip_idx[0], c->ip_idx[1]);
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, dk, dv, (int)cap, 0, 64, c->stream);
  DA(c->ip_cub, bytes + 256); c->ip_cub_bytes = bytes + 256;
  c->ip_cap = cap;
  return SPH_OK;
}

// Private BVH over the source walk groups (domains: the own groups only) with reach boxes that bound |x - x_j| <= 2 h_j.
int interp_bvh(sph_ctx* c, int ng, int n_src) {
  const int T = 256;
  if ((size_t)n_src > c->ip_reach_cap) { c->ip_reach_cap = 0; DA(c->ip_reach, (size_t)c->cap); c->ip_reach_cap = (size_t)c->cap; }
  if (ng + bvh_upper_boxes(ng) > c->ip_bvh_cap) { c->ip_bvh_cap = 0; const size_t cap = (ng + bvh_upper_boxes(ng)) * 5 / 4; DA(c->ip_bvh, cap); c->ip_bvh_cap = cap; }
  if (ng > 0) {
    StateArrays s = state_of(c, c->cur);
    LAUNCH(k_interp_reach, cdiv(n_src, T), T, 0, n_src, s.h, c->dp.variable_h, c->dp.h_fixed, c->ip_reach);
    LAUNCH(k_bvh_leaf, cdiv((int64_t)ng * 32, T), T, 0, ng, c->groups, s.x, s.y, s.z, s.x, s.y, s.z, c->ip_reach, c->ip_bvh);
  }
  bvh_levels(c, c->ip_bvh, ng, c->ip_bvh, ng, c->ip_bi);
  return SPH_OK;
}

// Points [off, off + nc) to the device (pts + k * ip_cap) and their order: sorted by k_interp_keys' Morton key, ties by the
// coordinate-bit hash, so the sorted sequence does not depend on the caller's order.  *perm[i] = the chunk index of the i-th.
int interp_sort(sph_ctx* c, int64_t off, int nc, const double* px, const double* py, const double* pz, double* pts, int** perm_out) {
  const int T = 256;
  const size_t cap = c->ip_cap;
  const double* src[3] = {px, py, pz};
  for (int k = 0; k < 3; ++k) CK(cudaMemcpyAsync(pts + (size_t)k * cap, src[k] + off, (size_t)nc * 8, cudaMemcpyHostToDevice, c->stream));
  const int nb = std::min(cdiv(nc, T), c->n_partial);
  LAUNCH(k_bbox_partial, nb, T, 0, nc, pts, pts + cap, pts + 2 * cap, c->ip_bpart);
  LAUNCH(k_bbox_final, 1, 32, 0, nb, c->ip_bpart, c->ip_rb);
  LAUNCH(k_interp_keys, cdiv(nc, T), T, 0, nc, pts, pts + cap, pts + 2 * cap, c->ip_rb, c->ip_key[0], c->ip_tie[0], c->ip_idx[0]);
  int* perm;
  {   // stable LSD order: by the tie hash, then by the Morton key
    size_t bytes = c->ip_cub_bytes;
    cub::DoubleBuffer<uint64_t> dt(c->ip_tie[0], c->ip_tie[1]); cub::DoubleBuffer<int> dv(c->ip_idx[0], c->ip_idx[1]);
    CK(cub::DeviceRadixSort::SortPairs(c->ip_cub, bytes, dt, dv, nc, 0, 64, c->stream));
    LAUNCH(k_gather_u64, cdiv(nc, T), T, 0, nc, dv.Current(), c->ip_key[0], c->ip_key[1]);
    int* alt = dv.Current() == c->ip_idx[0] ? c->ip_idx[1] : c->ip_idx[0];
    cub::DoubleBuffer<uint64_t> dk(c->ip_key[1], c->ip_key[0]); cub::DoubleBuffer<int> dp(dv.Current(), alt);
    bytes = c->ip_cub_bytes;
    CK(cub::DeviceRadixSort::SortPairs(c->ip_cub, bytes, dk, dp, nc, 0, 63, c->stream));
    perm = dp.Current();
  }
  *perm_out = perm;
  return SPH_OK;
}

// One chunk of points [off, off + nc): sort, walk, (domains) sum the ranks' raw columns, finish, copy out.
int interp_chunk(sph_ctx* c, int64_t off, int nc, const double* px, const double* py, const double* pz, int64_t n_points,
                 double* out, int n_out, bool reduce) {
  const int T = 256;
  const size_t cap = c->ip_cap;
  double* pts = c->ip_pts;
  int* perm;
  { int r = interp_sort(c, off, nc, px, py, pz, pts, &perm); if (r) return r; }
  const int ng = c->ip_bi.cnt[0];
  StateArrays s = state_of(c, c->cur);
  InterpArrays A{s.x, s.y, s.z, s.vx, s.vy, s.vz, s.u, s.m, s.alpha, s.h, c->ip_reach};
  double* raw = c->ip_raw;
  if (ng > 0) {
    const int runs = cdiv(nc, 32);
    LAUNCH(k_interpolate, cdiv(runs, INTERP_WARPS), INTERP_WARPS * 32, interp_smem(c), nc, pts, pts + cap, pts + 2 * cap, perm,
           c->groups, A, c->ip_bvh, c->ip_bi, c->d_wt, c->dp, raw);
  } else CK(cudaMemsetAsync(raw, 0, (size_t)SPH_INTERP_COUNT * nc * 8, c->stream));      // a domain without particles adds zeros
  if (reduce) {      // NCCL: one all-reduce; the host communicator's all-gather carries at most SPH_HC_SLOT bytes per rank
    const size_t tot = (size_t)SPH_INTERP_COUNT * nc, chunk = c->hc ? SPH_HC_SLOT / 8 : tot;
    for (size_t o = 0; o < tot; o += chunk) { int r = coll_allreduce(c, c->stream, raw + o, std::min(chunk, tot - o), NC_FLOAT64, NC_SUM); if (r) return r; }
  }
  LAUNCH(k_interp_finish, cdiv(nc, T), T, 0, nc, raw);
  for (int k = 0; k < n_out; ++k)
    CK(cudaMemcpyAsync(out + (size_t)k * n_points + off, raw + (size_t)k * nc, (size_t)nc * 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return SPH_OK;
}

// ---- sph_gravity_at (sph_gravat.cuh) ------------------------------------------------------------------------------
// One chunk of points [off, off + nc): sort, walk (one thread per point), (domains) sum the ranks' gas columns, sinks, copy out.
int gravat_chunk(sph_ctx* c, int64_t off, int nc, const double* px, const double* py, const double* pz, const double* h,
                 int64_t n_points, double* out, int n_out, bool reduce) {
  const int T = 256;
  const size_t cap = c->ip_cap;
  double* q = c->ga_q;
  int* perm;
  { int r = interp_sort(c, off, nc, px, py, pz, q, &perm); if (r) return r; }
  if (h) CK(cudaMemcpyAsync(q + 3 * cap, h + off, (size_t)nc * 8, cudaMemcpyHostToDevice, c->stream));
  double* raw = c->ga_raw;
  const int rank = c->dd ? c->rank : 0;
  LAUNCH(k_gravity_at, cdiv(nc, GRAVAT_THREADS), GRAVAT_THREADS, 0, nc, q, cap, h ? 1 : 0, perm, c->dp, c->wnodes, c->d_gt,
         c->dd ? DD_TOP_CAP : 0, c->ga_owner, rank, raw);
  if (reduce) {      // NCCL: one all-reduce; the host communicator's all-gather carries at most SPH_HC_SLOT bytes per rank
    const size_t tot = (size_t)GRAVAT_RAW * nc, chunk = c->hc ? SPH_HC_SLOT / 8 : tot;
    for (size_t o = 0; o < tot; o += chunk) { int r = coll_allreduce(c, c->stream, raw + o, std::min(chunk, tot - o), NC_FLOAT64, NC_SUM); if (r) return r; }
  }
  LAUNCH(k_gravity_at_sinks, cdiv(nc, T), T, 0, nc, q, cap, c->dp, c->n_sink, c->S, raw);
  for (int k = 0; k < n_out; ++k)
    CK(cudaMemcpyAsync(out + (size_t)k * n_points + off, raw + (size_t)k * nc, (size_t)nc * 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return SPH_OK;
}

}  // namespace

// =====================================================================================================
extern "C" {

int sph_default_params(int32_t mode, sph_params* p) {
  if (!p) return SPH_ERR_ARG;
  std::memset(p, 0, sizeof(*p));
  p->mode = mode; p->n_ranks = 1; p->h_fixed = 2.5; p->theta = 0.5; p->theta_override = 0;
  p->max_depth = 1000; p->bounding_size = 1500.0; p->gamma = 1.4; p->eta = 1.2;
  p->convergence_criteria = 1e-3; p->max_length = 50.0; p->timestep_scale = 0.25;
  if (mode & SPH_MODE_VARIABLE_H) { p->nq = 2500; p->end_time = 0.1; p->sink_radius = 5.0; }
  else { p->nq = 5000; p->end_time = 1000.0; p->sink_radius = 3.5; }
  return SPH_OK;
}

const char* sph_last_error(const sph_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int sph_create(const sph_params* p, int32_t device, sph_ctx** out) {
  if (!p || !out) { g_create_error = "null argument"; return SPH_ERR_ARG; }
  if (p->nq < 2 || p->nq > 12000 || p->max_depth < 1) { g_create_error = "bad nq / max_depth"; return SPH_ERR_ARG; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); g_create_error = "no CUDA device (there is no CPU fallback)"; return SPH_ERR_NO_DEVICE; }
  if (device < 0 || device >= ndev) { g_create_error = "bad device index"; return SPH_ERR_ARG; }
  sph_ctx* c = new sph_ctx();
  c->p = *p; c->device = device;
  std::memset(&c->counts, 0, sizeof(c->counts));
  auto fail = [&](int code) { g_create_error = c->err; sph_destroy(c); return code; };
  if (cudaSetDevice(device) != cudaSuccess) { c->err = "cudaSetDevice failed"; return fail(SPH_ERR_CUDA); }
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { c->err = "stream create failed"; return fail(SPH_ERR_CUDA); }
  make_dev_params(c);
  c->tree_reuse = getenv("SPH_B200_NO_TREE_REUSE") ? 0 : 1;
  c->fused_push = getenv("SPH_B200_NO_FUSED_PUSH") ? 0 : 1;     // developer switch: copy-engine exchange after the pair kernel
  c->far_reuse = getenv("SPH_B200_NO_FAR_REUSE") ? 0 : 1;        // developer switch: every gravity evaluation walks the whole tree
  c->far_lists = getenv("SPH_B200_NO_FAR_LISTS") ? false : true; // developer switch: the near field is always walked, never read from recorded pairs
  if (getenv("SPH_B200_FAR_HCUT")) c->far_hcut = std::max(1.0, atof(getenv("SPH_B200_FAR_HCUT")));      // test hook: near / far split at this multiple of h (default GW_HCUT)
  if (getenv("SPH_B200_FAR_SLOTS")) c->far_slots = std::max(1, atoi(getenv("SPH_B200_FAR_SLOTS")));      // test hook: recorded near pairs per particle (overflowing runs walk)
  c->use_lists = getenv("SPH_B200_NO_LISTS") ? 0 : 1;            // developer switch: the pair loop always walks by itself     // developer switch: rebuild the tree in every evaluation
  int r;
  if ((r = upload_tables(c))) return fail(r);
  c->n_partial = 4096;
  if ((r = dalloc(c, &c->partial, (size_t)c->n_partial * 6))) return fail(r);
  if ((r = dalloc(c, &c->root, 1))) return fail(r);
  if ((r = dalloc(c, &c->sc, 1))) return fail(r);
  if ((r = dalloc(c, &c->ctr, 1))) return fail(r);
  if ((r = dalloc(c, &c->work, 4))) return fail(r);
  if ((r = dalloc(c, &c->nl_ctl, 4))) return fail(r);
  cudaMemset(c->nl_ctl, 0, 4 * sizeof(int));
  if ((r = dalloc(c, &c->d_nsel, 1))) return fail(r);
  if ((r = dalloc(c, &c->d_same, 1))) return fail(r);
  if ((r = dalloc(c, &c->sink_land, (size_t)SPH_MAX_SINKS * 8))) return fail(r);
  c->resident_check = getenv("SPH_B200_NO_RESIDENT_CHECK") ? 0 : 1;      // developer switch: every upload is a new state
  if ((r = dalloc(c, &c->far_ctr, 2))) return fail(r);
  if ((r = dalloc(c, &c->sink_buf, (size_t)SPH_MAX_SINKS * 11 + 8))) return fail(r);      // + the LET overflow flag right behind az (it rides the sink all-reduce)
  c->let_flag = c->sink_buf + (size_t)SPH_MAX_SINKS * 11;
  { double* b = c->sink_buf; const int M = SPH_MAX_SINKS;
    c->S = SinkArrays{b, b + M, b + 2 * M, b + 3 * M, b + 4 * M, b + 5 * M, b + 6 * M, b + 7 * M, b + 8 * M, b + 9 * M, b + 10 * M}; }
  cudaMemset(c->sink_buf, 0, ((size_t)SPH_MAX_SINKS * 11 + 8) * 8);
  c->sink_extras = (p->mode & SPH_FLAG_SINK_MERGE_SPIN) ? 1 : 0;
  if (c->sink_extras) { if ((r = dalloc(c, &c->sink_spin, (size_t)SPH_MAX_SINKS * 3))) return fail(r); cudaMemset(c->sink_spin, 0, (size_t)SPH_MAX_SINKS * 3 * 8); }
  if (cudaMallocHost((void**)&c->h_sc, sizeof(SimScalars)) != cudaSuccess || cudaMallocHost((void**)&c->h_ctr, sizeof(WalkCounters)) != cudaSuccess) { c->err = "cudaMallocHost failed"; return fail(SPH_ERR_OOM); }
  if (cudaMallocHost((void**)&c->h_rb, 16 * sizeof(int)) != cudaSuccess) { c->err = "cudaMallocHost failed"; return fail(SPH_ERR_OOM); }
  std::memset(c->h_sc, 0, sizeof(SimScalars)); c->h_sc->create_cand = ~0ull; c->h_sc->dt = 1.0e-2;
  cudaMemcpy(c->sc, c->h_sc, sizeof(SimScalars), cudaMemcpyHostToDevice);
  cudaMemset(c->ctr, 0, sizeof(WalkCounters));
  // opt in to large dynamic shared memory
  int maxsm = 0; cudaDeviceGetAttribute(&maxsm, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  c->max_smem = maxsm;
  cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, device);
  size_t need = std::max(std::max(density_smem(c, DENS_WARPS), std::max(force_smem(c, force_warps(c, true), true), force_smem(c, force_warps(c, false), false))), gravity_smem(c, grav_warps(c)));
  if ((size_t)maxsm < need) { c->err = "device shared memory too small for the walk kernels"; return fail(SPH_ERR_CUDA); }
  cudaFuncSetAttribute(k_density<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)density_smem(c, DENS_WARPS));
  cudaFuncSetAttribute(k_density<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)density_smem(c, DENS_WARPS));
  cudaFuncSetAttribute(k_force<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)force_smem(c, force_warps(c, true), true));
  cudaFuncSetAttribute(k_force<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)force_smem(c, force_warps(c, false), false));
  cudaFuncSetAttribute(k_gravity<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gravity_smem(c, grav_warps(c)));
  cudaFuncSetAttribute(k_gravity<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gravity_smem(c, grav_warps(c)));
  cudaFuncSetAttribute(k_gravity<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gravity_smem(c, grav_warps(c)));
  cudaFuncSetAttribute(k_gravity_near, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gravity_smem(c, 0));
  cudaFuncSetAttribute(k_neighbours, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  cudaFuncSetAttribute(k_interpolate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)interp_smem(c));
  if (cudaGetLastError() != cudaSuccess) { c->err = "cudaFuncSetAttribute failed (was the library built for this GPU's architecture?)"; return fail(SPH_ERR_CUDA); }
  *out = c;
  return SPH_OK;
}

int sph_destroy(sph_ctx* c) {
  if (!c) return SPH_OK;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  p2p_close(c);
  for (auto st : c->pstream) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
  for (auto ev : c->pevent) cudaEventDestroy(ev);
  if (c->xstream) { cudaStreamSynchronize(c->xstream); cudaStreamDestroy(c->xstream); cudaEventDestroy(c->x_ready); cudaEventDestroy(c->x_done); }
  if (c->let_done) cudaEventDestroy(c->let_done);
  if (c->io_stream) { cudaStreamSynchronize(c->io_stream); cudaStreamDestroy(c->io_stream); cudaEventDestroy(c->io_ev_xyz); cudaEventDestroy(c->io_ev_out); cudaEventDestroy(c->io_ev_done); for (int f = 0; f < 10; ++f) cudaEventDestroy(c->io_ev_field[f]); }
  for (int k = 0; k < 5; ++k) if (c->io_stage[k]) cudaFree(c->io_stage[k]);
  if (c->d_flag) cudaFree(c->d_flag);
  if (c->d_blob) cudaFree(c->d_blob);
  if (c->comm && c->nccl.CommDestroy) c->nccl.CommDestroy(c->comm);
  if (c->hc) { c->hc->close(); delete c->hc; c->hc = nullptr; }
  auto F = [](void* p) { if (p) cudaFree(p); };
  for (int b = 0; b < 2; ++b) { for (int f = 0; f < 10; ++f) F(c->st[b][f]); F(c->id[b]); F(c->key[b]); F(c->key_lo[b]); F(c->perm[b]); F(c->acc_key[b]); F(c->acc_val[b]); }
  F(c->rho); F(c->omega); F(c->prs); F(c->cs); F(c->por2); F(c->ax); F(c->ay); F(c->az); F(c->udot); F(c->adot);
  F(c->node_count); F(c->gsize); F(c->gfirst); F(c->groups); F(c->level); F(c->lcx); F(c->lcy); F(c->lcz); F(c->reach); F(c->bvh); F(c->nodes); F(c->node_part); F(c->parent); F(c->nchild);
  F(c->nl_pool); F(c->nl_head); F(c->nl_ctl); F(c->ggroups); F(c->gbvh); F(c->seg_cnt); F(c->seg_off); F(c->wnodes); F(c->wcount); F(c->wstart); F(c->widx); F(c->grav_spill);
  F(c->dd_samples); F(c->dd_split); F(c->dd_counts); F(c->dd_sendoff); F(c->dd_segkeys); F(c->dd_cells); F(c->dd_contrib); F(c->dd_obvh); F(c->dd_let_ctl); F(c->dd_create8); F(c->dd_cand);
  F(c->dd_let_f[0]); F(c->dd_let_f[1]); F(c->dd_halo_flag); F(c->dd_halo_list); F(c->dd_halo_size); F(c->dd_halo_poff); F(c->dd_acc_key); F(c->dd_acc_rec);
  F(c->dd_accg_key[0]); F(c->dd_accg_key[1]); F(c->dd_accg_idx[0]); F(c->dd_accg_idx[1]); F(c->dd_accg_rec); F(c->dd_gid); F(c->dd_gpos); F(c->dd_gcnt); F(c->dd_goff); F(c->dd_gstage);
  F(c->cons_partial); F(c->cons_out); F(c->cons_wpart); F(c->img_table); F(c->sink_spin);
  F(c->ip_reach); F(c->ip_bvh); F(c->ip_pts); F(c->ip_raw); F(c->ip_bpart); F(c->ip_rb); F(c->ip_cub);
  F(c->ga_q); F(c->ga_raw); F(c->ga_owner);
  for (int b = 0; b < 2; ++b) { F(c->ip_key[b]); F(c->ip_tie[b]); F(c->ip_idx[b]); }
  F(c->far_fx); F(c->far_fy); F(c->far_fz); F(c->far_hc2); F(c->far_ctr); F(c->far_list); F(c->far_cnt); F(c->far_ovf); F(c->d_same); F(c->sink_land);
  F(c->arrive); F(c->cnt); F(c->off); F(c->root); F(c->partial); F(c->cub_tmp); F(c->d_wt); F(c->d_dwt); F(c->d_gt);
  F(c->sink_buf); F(c->sink_partial); F(c->sink_seg); F(c->sc); F(c->ctr); F(c->work); F(c->keep); F(c->d_nsel); F(c->pos); F(c->stage_d); F(c->stage_d2);
  if (c->h_sc) cudaFreeHost(c->h_sc);
  if (c->h_rb) cudaFreeHost(c->h_rb);
  if (c->h_ctr) cudaFreeHost(c->h_ctr);
  for (auto& e : c->ev_used) { cudaEventDestroy(e.second.first); cudaEventDestroy(e.second.second); }
  for (auto e : c->ev_pool) cudaEventDestroy(e);
  if (c->tm0) { cudaEventDestroy(c->tm0); cudaEventDestroy(c->tm1); }
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return SPH_OK;
}

int sph_comm_unique_id(void* uid) {
  sph_ctx tmp; sph_ctx* c = &tmp;
  if (!uid) return SPH_ERR_ARG;
  if (!load_nccl(c)) { g_create_error = c->err; return SPH_ERR_COMM; }
  int r = c->nccl.GetUniqueId(uid);
  return r == 0 ? SPH_OK : SPH_ERR_COMM;
}

int sph_comm_init(sph_ctx* c, int32_t rank, int32_t n_ranks, const void* uid) {
  if (!c || !uid || n_ranks < 1 || rank < 0 || rank >= n_ranks) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  if (!load_nccl(c)) return SPH_ERR_COMM;
  NcclUid id; std::memcpy(&id, uid, 128);
  int r = c->nccl.CommInitRank(&c->comm, n_ranks, id, rank);
  if (r != 0) { c->err = std::string("ncclCommInitRank: ") + (c->nccl.GetErrorString ? c->nccl.GetErrorString(r) : "?"); return SPH_ERR_COMM; }
  c->rank = rank; c->n_ranks = n_ranks; c->tree_valid = false; c->pos_moved = true; c->p2p_stale = true;
  return SPH_OK;
}

int sph_slice_bounds(int32_t n_groups, int32_t n_ranks, int32_t* first_group) {
  if (n_groups < 0 || n_ranks < 1 || !first_group) return SPH_ERR_ARG;
  slice_first_groups(n_groups, n_ranks, first_group);
  return SPH_OK;
}

int sph_comm_init_host(sph_ctx* c, int32_t rank, int32_t n_ranks, const char* name) {
  if (!c || !name || n_ranks < 1 || rank < 0 || rank >= n_ranks) return SPH_ERR_ARG;
  if (c->comm || c->hc) { c->err = "communicator already initialised"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  if (n_ranks > 1) {
    HostComm* hc = new HostComm();
    const std::string e = hc->open(name, rank, n_ranks);
    if (!e.empty()) { c->err = "sph_comm_init_host: " + e; hc->close(); delete hc; return SPH_ERR_COMM; }
    c->hc = hc;
  }
  c->rank = rank; c->n_ranks = n_ranks; c->tree_valid = false; c->pos_moved = true; c->p2p_stale = true;
  return SPH_OK;
}

// n_local rows starting at global number id_first out of n_global (single rank / replicated: all of them)
// Is the state the host hands over the one this context holds?  A host that keeps bodies(:) / sinks(:) on its side and
// passes them through every step (upload, loop body, download) sends back exactly what it was given.  The geometry columns
// (x y z m h) land in the idle half of the double buffer and are compared bitwise, row `number` against the resident row
// carrying that number, the sinks likewise; when they are the same, the tree, the walk groups, the stored far-field
// sums and their recorded pairs still stand (they are functions of exactly these values), and only the other columns
// (v u alpha) are gathered into the resident order.  Anything else is a new state.
struct SameCols { const double* a[5]; const double* b[5]; int nf; };
// number == nullptr: the host's row j is the particle numbered j (single rank, nothing ever removed).  Otherwise the host's
// rows come with their numbers in the order sph_download_local gave them (domains): row i against resident row i.
__global__ void k_same_state(int n, const int* __restrict__ id, const int* __restrict__ number, SameCols C, int* __restrict__ differ) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool d = false;
  if (i < n) {
    const int j = number ? i : id[i];
    if (number) d = number[i] != id[i];
    for (int f = 0; f < C.nf; ++f) d |= __double_as_longlong(C.a[f][i]) != __double_as_longlong(C.b[f][j]);
  }
  if (__any_sync(FULL_MASK, d) && (threadIdx.x & 31) == 0) atomicOr(differ, 1);
}
__global__ void k_same_sinks(int ns, const double* __restrict__ resident, const double* __restrict__ landed, int* __restrict__ differ) {
  const int t = threadIdx.x;      // 8 arrays (x y z vx vy vz m radius) of SPH_MAX_SINKS
  bool d = false;
  for (int k = 0; k < 8; ++k) if (t < ns) d |= __double_as_longlong(resident[k * SPH_MAX_SINKS + t]) != __double_as_longlong(landed[k * SPH_MAX_SINKS + t]);
  if (d) atomicOr(differ, 1);
}

static int upload_impl(sph_ctx* c, int64_t n_global, int64_t id_first, int64_t n, const double* const* src,
                       int32_t ns, const double* const* ssrc, const double* srad, bool gas_on_device = false, unsigned late_mask = 0, const int32_t* number = nullptr) {
  cudaSetDevice(c->device);
  const bool was_dd = c->dd;
  c->dd = c->n_ranks > 1 && c->p.decomposition == 1;
  int64_t want = n;
  if (c->dd) {      // own share + halo + migration slack; every exported array is sized once here (the peers map them once)
    double slack = 0.6; if (const char* e = getenv("SPH_B200_DOMAIN_SLACK")) slack = atof(e);
    want = std::max<int64_t>(n, (int64_t)((double)(n_global / c->n_ranks) * (1.0 + slack)) + 65536);
  }
  if (c->dd && !c->dd_acc_key) c->cap = 0;        // the exported arrays of the decomposition are sized in ensure_capacity
  // the resident state is a candidate when it came out of a step of this context with every row of its upload still there
  // Domains: every rank hands back its own rows with their numbers, in the order sph_download_local gave them; the ranks
  // agree through one all-reduce (a rank that cannot even try votes "different"), so they all keep or all replace.
  const bool cols_ok = src[0] && src[1] && src[2] && src[3] && src[4] && src[5] && src[6] && src[7] && (src[9] || !c->dp.variable_h);
  const bool try_any = c->resident_check && !gas_on_device && !c->sink_extras && c->tree_valid && !c->pos_moved && c->steps_since_upload >= 1 &&
                       (c->n_ranks == 1 || (c->dd && was_dd));      // the same on every rank of a communicator
  const bool local_ok = try_any && n > 0 && c->n == n && n <= c->cap && want <= c->cap && (ns > 0 ? ns : 1) == c->n_sink && cols_ok &&
                        (c->dd ? (number != nullptr && n_global == c->n_global) : (c->n_upload == n && n_global == n && id_first == 0));
  const bool try_same = try_any && (local_ok || c->dd);
  int r = SPH_OK;
  if (!try_same) { r = ensure_capacity(c, want); if (r) return r; }
  const int L = try_same ? (c->cur ^ 1) : 0;      // where the columns land
  // sinks as the context would hold them (dummy zero sink if none: F:698-707)
  std::vector<double> hb((size_t)SPH_MAX_SINKS * 11, 0.0);
  const int M = SPH_MAX_SINKS;
  for (int k = 0; k < 7; ++k) for (int q = 0; q < ns; ++q) hb[(size_t)k * M + q] = ssrc[k] ? ssrc[k][q] : 0.0;
  for (int q = 0; q < ns; ++q) hb[(size_t)7 * M + q] = (srad && srad[q] == srad[q]) ? srad[q] : c->p.sink_radius;
  c->late_pending = 0; c->late_permuted = false; c->late_n = 0;
  const unsigned geometry = try_same ? ((1u << 0) | (1u << 1) | (1u << 2) | (1u << 7) | (1u << 9)) : 0x7u;      // columns the compute stream waits for
  if (late_mask) late_mask &= ~geometry;
  const bool land = !try_same || local_ok;         // domains: a rank that cannot try only votes (its columns go the plain way afterwards)
  for (int f = 0; f < 10 && !gas_on_device && land; ++f) {
    if (src[f] && ((late_mask >> f) & 1u)) continue;       // follows on io_stream behind the first columns (below)
    if (src[f]) { if (n > 0) CK(cudaMemcpyAsync(c->st[L][f], src[f], (size_t)n * 8, cudaMemcpyHostToDevice, c->stream)); }
    else if (f == 8) CK(cudaMemsetAsync(c->st[L][f], 0, (size_t)std::max<int64_t>(n, 1) * 8, c->stream));            // alpha := 0, F:681
    else if (!try_same) { std::vector<double> hv((size_t)std::max<int64_t>(n, 1), c->p.h_fixed); CK(cudaMemcpyAsync(c->st[L][f], hv.data(), hv.size() * 8, cudaMemcpyHostToDevice, c->stream)); CK(cudaStreamSynchronize(c->stream)); }
  }
  if (late_mask && n > 0 && land) {      // sph_step_host: the other columns in the order their readers come (h: leaf cells, m: node sums, u: EOS, then v, alpha)
    CK(cudaEventRecord(c->io_ev_xyz, c->stream));
    CK(cudaStreamWaitEvent(c->io_stream, c->io_ev_xyz, 0));
    const int order[7] = {9, 7, 6, 3, 4, 5, 8};
    for (int k = 0; k < 7; ++k) {
      const int f = order[k];
      if (!src[f] || !((late_mask >> f) & 1u)) continue;
      CK(cudaMemcpyAsync(c->st[L][f], src[f], (size_t)n * 8, cudaMemcpyHostToDevice, c->io_stream));
      CK(cudaEventRecord(c->io_ev_field[f], c->io_stream));
      c->late_order[c->late_n++] = f; c->late_pending |= 1u << f;
    }
  }
  if (try_same) {
    const int cur = c->cur;
    SameCols C; C.nf = 0;
    const int cols[5] = {0, 1, 2, 7, 9};
    for (int k = 0; k < 5; ++k) { const int f = cols[k]; if (f == 9 && !c->dp.variable_h) continue; C.a[C.nf] = c->st[cur][f]; C.b[C.nf] = c->st[L][f]; ++C.nf; }
    double* landed = c->sink_land;
    CK(cudaMemcpyAsync(landed, hb.data(), (size_t)8 * M * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(c->d_same, 0, sizeof(int), c->stream));
    if (local_ok) {
      const int* d_number = nullptr;
      if (c->dd) { CK(cudaMemcpyAsync(c->pos, number, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream)); d_number = c->pos; }
      LAUNCH(k_same_state, cdiv(n, 256), 256, 0, (int)n, c->id[cur], d_number, C, c->d_same);
      LAUNCH(k_same_sinks, 1, SPH_MAX_SINKS, 0, c->n_sink, c->sink_buf, landed, c->d_same);
    } else LAUNCH(k_set_int, 1, 1, 0, c->d_same, 1);
    if (c->dd) { r = allreduce(c, c->d_same, 1, NC_INT32, NC_MAX); if (r) return r; }
    readback(c, c->h_rb + 8, c->d_same, sizeof(int));
    CK(cudaStreamSynchronize(c->stream));
    if (c->h_rb[8] != 0 && !local_ok) {      // domains, and this rank could not even try (row count, capacity): the plain path from the start
      r = ensure_capacity(c, want); if (r) return r;
      c->tree_valid = false;                 // no second attempt
      return upload_impl(c, n_global, id_first, n, src, ns, ssrc, srad, gas_on_device, late_mask, number);
    }
    if (c->h_rb[8] == 0) {      // the resident state, handed back: keep it and everything derived from its geometry; v u alpha into the resident order
      ++c->resident_hits;
      c->nl_valid = false;
      PermuteArgs pa; std::memset(&pa, 0, sizeof(pa));
      const int rest[5] = {6, 3, 4, 5, 8};
      bool now = false;
      for (int k = 0; k < 5; ++k) {
        const int f = rest[k];
        if (c->dd) CK(cudaMemcpyAsync(c->st[cur][f], c->st[L][f], (size_t)n * 8, cudaMemcpyDeviceToDevice, c->stream));      // rows came in resident order
        else if ((c->late_pending >> f) & 1u) { c->late_src[f] = c->st[L][f]; c->late_dst[f] = c->st[cur][f]; }      // flush_late gathers it when its first reader is due
        else { pa.src[f] = c->st[L][f]; pa.dst[f] = c->st[cur][f]; now = true; }
      }
      c->late_perm = c->id[cur]; c->late_permuted = true;
      if (now) LAUNCH(k_permute, cdiv(n, 4 * 256), 256, 0, (int)n, c->id[cur], pa);
      c->h_sc->n_sink = c->n_sink; c->h_sc->n_removed = 0; c->h_sc->n_accreted = 0; c->h_sc->err = 0; c->h_sc->create_cand = ~0ull;
      CK(cudaMemcpyAsync(c->sc, c->h_sc, sizeof(SimScalars), cudaMemcpyHostToDevice, c->stream));
      CK(cudaStreamSynchronize(c->stream));
      return SPH_OK;
    }
    if (!c->dp.variable_h) { std::vector<double> hv((size_t)n, c->p.h_fixed); CK(cudaMemcpyAsync(c->st[L][9], hv.data(), hv.size() * 8, cudaMemcpyHostToDevice, c->stream)); CK(cudaStreamSynchronize(c->stream)); }
  }
  // a new state
  c->n_halo = 0; c->ng_halo = 0; c->dd_info.clear();
  c->n = n; c->n_upload = n_global; c->n_global = n_global; c->cur = L; c->tree_valid = false; c->pos_moved = true;
  c->far_valid = false; c->steps_since_upload = 0;
  if (n > 0) LAUNCH(k_iota_from, cdiv(n, 256), 256, 0, (int)n, (int)id_first, c->id[L]);
  if (number && n > 0) CK(cudaMemcpyAsync(c->id[L], number, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
  c->n_sink = ns > 0 ? ns : 1;
  CK(cudaMemcpyAsync(c->sink_buf, hb.data(), hb.size() * 8, cudaMemcpyHostToDevice, c->stream));
  if (c->sink_spin) CK(cudaMemsetAsync(c->sink_spin, 0, (size_t)SPH_MAX_SINKS * 3 * 8, c->stream));   // F:695 spin = 0
  CK(cudaStreamSynchronize(c->stream));
  c->h_sc->n_sink = c->n_sink; c->h_sc->n_removed = 0; c->h_sc->n_accreted = 0; c->h_sc->err = 0; c->h_sc->create_cand = ~0ull;
  CK(cudaMemcpyAsync(c->sc, c->h_sc, sizeof(SimScalars), cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return SPH_OK;
}

int sph_upload(sph_ctx* c, int64_t n, const double* x, const double* y, const double* z,
               const double* vx, const double* vy, const double* vz, const double* u, const double* m,
               const double* alpha, const double* h, int32_t ns,
               const double* sx, const double* sy, const double* sz, const double* svx, const double* svy, const double* svz,
               const double* sm, const double* srad) {
  if (!c) return SPH_ERR_ARG;
  if (n < 2 || n > 0x0fffffff * (int64_t)SPH_CHUNK || !x || !y || !z || !vx || !vy || !vz || !u || !m) { c->err = "bad particle arrays"; return SPH_ERR_ARG; }
  if (ns < 0 || ns > SPH_MAX_SINKS - 8) { c->err = "too many sinks"; return SPH_ERR_ARG; }
  if (c->dp.variable_h && !h) { c->err = "variable-h mode needs the smoothing-length column"; return SPH_ERR_ARG; }
  const double* src[10] = {x, y, z, vx, vy, vz, u, m, alpha, c->dp.variable_h ? h : nullptr};   // F ignores column 10
  const double* ssrc[7] = {sx, sy, sz, svx, svy, svz, sm};
  int64_t first = 0, cnt = n;
  if (c->n_ranks > 1 && c->p.decomposition == 1) {      // Morton domains: this rank starts from rows [n r / R, n (r + 1) / R); the first tree build sends every particle to its owner
    first = n * c->rank / c->n_ranks; cnt = n * (c->rank + 1) / c->n_ranks - first;
    for (int f = 0; f < 10; ++f) if (src[f]) src[f] += first;
  }
  return upload_impl(c, n, first, cnt, src, ns, ssrc, srad);
}

int sph_ics_disc(sph_ctx* c, int64_t n, uint64_t seed, double r_in, double r_out, double aspect, double m_star, double m_disc,
                 double u, double alpha, double eta) {
  if (!c) return SPH_ERR_ARG;
  if (n < 2 || n > 0x7fffffff || !(r_out > r_in) || !(r_in > 0.0) || !(m_star > 0.0)) { c->err = "bad disc parameters"; return SPH_ERR_ARG; }
  int64_t first = 0, cnt = n;
  if (c->n_ranks > 1 && c->p.decomposition == 1) { first = n * c->rank / c->n_ranks; cnt = n * (c->rank + 1) / c->n_ranks - first; }
  const double* none[10] = {};
  const double zero = 0.0;
  const double* ssrc[7] = {&zero, &zero, &zero, &zero, &zero, &zero, &m_star};
  int r = upload_impl(c, n, first, cnt, none, 1, ssrc, nullptr, true); if (r) return r;
  IcsDisc P{r_in, r_out, aspect, m_star, m_disc, u, alpha, eta, c->dp.G};
  double** st = c->st[0];
  if (cnt > 0) LAUNCH(k_ics_disc, cdiv(cnt, 256), 256, 0, (long long)n, (long long)first, (int)cnt, seed, P, st[0], st[1], st[2], st[3], st[4], st[5], st[6], st[7], st[8], st[9]);
  if (!c->dp.variable_h && cnt > 0) { std::vector<double> hv((size_t)cnt, c->p.h_fixed); CK(cudaMemcpyAsync(st[9], hv.data(), hv.size() * 8, cudaMemcpyHostToDevice, c->stream)); }
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaGetLastError());
  return SPH_OK;
}

int sph_upload_local(sph_ctx* c, int64_t n_global, int64_t id_first, const int32_t* number, int64_t n_local, const double* x, const double* y, const double* z,
                     const double* vx, const double* vy, const double* vz, const double* u, const double* m,
                     const double* alpha, const double* h, int32_t ns,
                     const double* sx, const double* sy, const double* sz, const double* svx, const double* svy, const double* svz,
                     const double* sm, const double* srad) {
  if (!c) return SPH_ERR_ARG;
  if (!(c->n_ranks > 1 && c->p.decomposition == 1)) { c->err = "sph_upload_local needs the domain decomposition (params.decomposition = 1 and a communicator)"; return SPH_ERR_STATE; }
  if (n_global < 2 || n_local < 0 || id_first < 0 || (!number && id_first + n_local > n_global) || n_local > n_global || n_global > 0x7fffffff) { c->err = "bad row range"; return SPH_ERR_ARG; }
  if (n_local > 0 && (!x || !y || !z || !vx || !vy || !vz || !u || !m)) { c->err = "bad particle arrays"; return SPH_ERR_ARG; }
  if (ns < 0 || ns > SPH_MAX_SINKS - 8) { c->err = "too many sinks"; return SPH_ERR_ARG; }
  if (c->dp.variable_h && !h && n_local > 0) { c->err = "variable-h mode needs the smoothing-length column"; return SPH_ERR_ARG; }
  const double* src[10] = {x, y, z, vx, vy, vz, u, m, alpha, c->dp.variable_h ? h : nullptr};
  const double* ssrc[7] = {sx, sy, sz, svx, svy, svz, sm};
  return upload_impl(c, n_global, id_first, n_local, src, ns, ssrc, srad, false, 0, number);
}

#ifdef SCREEN_AUDIT
static void screen_audit_report(sph_ctx* c, const char* what) {
  unsigned long long d[3]; cudaStreamSynchronize(c->stream); cudaMemcpyFromSymbol(d, screen_audit, sizeof(d)); unsigned long long z[3] = {}; cudaMemcpyToSymbol(screen_audit, z, sizeof(z));
  fprintf(stderr, "SCREEN_AUDIT %s density %llu pair %llu gravity %llu\n", what, d[0], d[1], d[2]);
}
#endif

int sph_evaluate(sph_ctx* c, int32_t mask) {
  if (!c) return SPH_ERR_ARG;
  if (c->n <= 0) { c->err = "no particles uploaded"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  c->far_want_store = c->steps_since_upload >= 1;
  int r = evaluate(c, mask); if (r) return r;
  CK(cudaMemcpyAsync(c->h_sc, c->sc, sizeof(SimScalars), cudaMemcpyDeviceToHost, c->stream));
  if ((r = fetch_counters(c))) return r;
  c->far_n_ovf = c->h_sc->far_ovf;
#ifdef SCREEN_AUDIT
  screen_audit_report(c, "evaluate");
#endif
  stage_collect(c, true);
  CK(cudaGetLastError());
  return check_device_error(c);
}

int sph_step(sph_ctx* c, double* dt, double* t, int64_t* n_out, int32_t* ns_out) {
  if (!c || !dt || !t) return SPH_ERR_ARG;
  if (c->n <= 0) { c->err = "no particles uploaded"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  c->h_sc->dt = *dt; c->h_sc->t = *t;
  CK(cudaMemcpyAsync(c->sc, c->h_sc, 2 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  int r = step(c); if (r) return r;
  if ((r = fetch_counters(c))) return r;
  c->counts.h_iterations = (int64_t)c->h_ctr->h_iters;
#ifdef SCREEN_AUDIT
  screen_audit_report(c, "step");
#endif
  stage_collect(c, true);
  CK(cudaGetLastError());
  *dt = c->h_sc->dt; *t = c->h_sc->t;
  if (n_out) *n_out = c->dd ? c->n_global : c->n;
  if (ns_out) *ns_out = c->n_sink;
  return SPH_OK;
}

// upload + one loop body + download with the copies under the compute (single rank)
int sph_step_host(sph_ctx* c, int64_t n, const double* const* gas_in, int32_t ns, const double* const* sink_in,
                  double* dt, double* t, double* const* gas_out, double* const* sink_out, int64_t* n_out, int32_t* ns_out) {
  if (!c || !gas_in || !dt || !t) return SPH_ERR_ARG;
  if (c->n_ranks > 1) { c->err = "sph_step_host is single-rank: ranks of a multi-GPU run move their rows with sph_upload_local / sph_step / sph_download_local"; return SPH_ERR_ARG; }
  if (n < 2 || n > 0x0fffffff * (int64_t)SPH_CHUNK) { c->err = "bad particle count"; return SPH_ERR_ARG; }
  for (int f = 0; f < 8; ++f) if (!gas_in[f]) { c->err = "bad particle arrays"; return SPH_ERR_ARG; }
  if (ns < 0 || ns > SPH_MAX_SINKS - 8 || (ns > 0 && !sink_in)) { c->err = "bad sink arrays"; return SPH_ERR_ARG; }
  if (c->dp.variable_h && !gas_in[9]) { c->err = "variable-h mode needs the smoothing-length column"; return SPH_ERR_ARG; }
  cudaSetDevice(c->device);
  if (!c->io_stream) {
    if (cudaStreamCreateWithFlags(&c->io_stream, cudaStreamNonBlocking) != cudaSuccess) { c->err = "stream create failed"; return SPH_ERR_CUDA; }
    cudaEventCreateWithFlags(&c->io_ev_xyz, cudaEventDisableTiming); cudaEventCreateWithFlags(&c->io_ev_out, cudaEventDisableTiming); cudaEventCreateWithFlags(&c->io_ev_done, cudaEventDisableTiming);
    for (int f = 0; f < 10; ++f) cudaEventCreateWithFlags(&c->io_ev_field[f], cudaEventDisableTiming);
  }
  const double* src[10]; for (int f = 0; f < 10; ++f) src[f] = gas_in[f];
  if (!c->dp.variable_h) src[9] = nullptr;                                     // F ignores column 10
  // developer switches: SPH_B200_IO_NO_LATE (all columns before the build), SPH_B200_IO_NO_EARLY (all results after the step), SPH_B200_IO_TRACE (host time line on stderr)
  const bool io_trace = getenv("SPH_B200_IO_TRACE") != nullptr, io_no_late = getenv("SPH_B200_IO_NO_LATE") != nullptr, io_no_early = getenv("SPH_B200_IO_NO_EARLY") != nullptr;
  auto now_ms = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
  const double tr0 = now_ms();
  const double* ssrc[7] = {}; const double* srad = nullptr;
  if (ns > 0) { for (int k = 0; k < 7; ++k) ssrc[k] = sink_in[k]; srad = sink_in[7]; }
  int r = upload_impl(c, n, 0, n, src, ns, ssrc, srad, false, io_no_late ? 0u : 0x3f8u /* everything but x y z arrives while the build runs */);
  if (r) return r;
  const double tr1 = now_ms();
  if ((size_t)c->cap > c->io_stage_cap) { for (int k = 0; k < 5; ++k) DA(c->io_stage[k], c->cap); c->io_stage_cap = (size_t)c->cap; }
  for (int f = 0; f < 10; ++f) c->io_out[f] = gas_out ? gas_out[f] : nullptr;
  c->io_active = gas_out != nullptr && !io_no_early; c->io_fetched = 0; c->io_busy = false;
  c->h_sc->dt = *dt; c->h_sc->t = *t;
  CK(cudaMemcpyAsync(c->sc, c->h_sc, 2 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  r = step(c);
  c->io_active = false;
  if (r) { cudaStreamSynchronize(c->io_stream); c->late_pending = 0; return r; }
  if ((r = fetch_counters(c))) return r;
  c->counts.h_iterations = (int64_t)c->h_ctr->h_iters;
  stage_collect(c, true);
  const double tr2 = now_ms();
  if (gas_out && c->n > 0) {
    unsigned have = c->io_fetched;
    if (c->n != c->n_upload) { CK(cudaStreamSynchronize(c->io_stream)); have = 0; }      // rows were removed after the early columns left: all of them again, compacted
    if ((r = download_rows(c))) return r;
    for (int f = 0; f < 10; ++f) if (!((have >> f) & 1u)) { if ((r = fetch_column(c, {DS_ST + f, CB_STATE}, 8, gas_out[f]))) return r; }
  }
  if (sink_out) {
    const double* ss[8] = {c->S.x, c->S.y, c->S.z, c->S.vx, c->S.vy, c->S.vz, c->S.m, c->S.radius};
    for (int k = 0; k < 8; ++k) if ((r = fetch_sink(c, ss[k], sink_out[k]))) return r;
  }
  CK(cudaStreamSynchronize(c->stream));
  const double tr3 = now_ms();
  CK(cudaStreamSynchronize(c->io_stream));
  CK(cudaGetLastError());
  if (io_trace) fprintf(stderr, "sph_step_host: upload %.2f ms, step %.2f ms, last columns %.2f ms, early columns still in flight %.2f ms\n", tr1 - tr0, tr2 - tr1, tr3 - tr2, now_ms() - tr3);
  *dt = c->h_sc->dt; *t = c->h_sc->t;
  if (n_out) *n_out = c->n;
  if (ns_out) *ns_out = c->n_sink;
  return SPH_OK;
}

int sph_run_until(sph_ctx* c, double t_stop, int64_t max_steps, double* dt, double* t, int64_t* steps_out,
                  int64_t* n_out, int32_t* ns_out) {
  if (!c || !dt || !t) return SPH_ERR_ARG;
  if (c->n <= 0) { c->err = "no particles uploaded"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  c->h_sc->dt = *dt; c->h_sc->t = *t;
  CK(cudaMemcpyAsync(c->sc, c->h_sc, 2 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  int64_t steps = 0; int r = SPH_OK;
  bool first = true;
  while (c->h_sc->t < t_stop && (max_steps <= 0 || steps < max_steps) && c->n >= 2) {      // F:879
    if ((r = step(c))) break;
    stage_collect(c, first); first = false;
    ++steps;
  }
  if (!r) { r = fetch_counters(c); c->counts.h_iterations = (int64_t)c->h_ctr->h_iters; }
  *dt = c->h_sc->dt; *t = c->h_sc->t;
  if (steps_out) *steps_out = steps;
  if (n_out) *n_out = c->dd ? c->n_global : c->n;
  if (ns_out) *ns_out = c->n_sink;
  return r;
}

int sph_sizes(sph_ctx* c, int64_t* n, int32_t* ns) {
  if (!c) return SPH_ERR_ARG;
  if (n) *n = c->dd ? c->n_global : c->n;
  if (ns) *ns = c->n_sink;
  return SPH_OK;
}

int sph_download(sph_ctx* c, double* x, double* y, double* z, double* vx, double* vy, double* vz,
                 double* u, double* m, double* alpha, double* h,
                 double* sx, double* sy, double* sz, double* svx, double* svy, double* svz, double* sm, double* srad) {
  if (!c) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  int r;
  const bool any_gas = x || y || z || vx || vy || vz || u || m || alpha || h;
  if (any_gas && download_count(c) > 0) {      // under domains every rank receives all rows (tests, saves of small runs); production hosts use sph_download_local
    if ((r = download_rows(c))) return r;
    double* dst[10] = {x, y, z, vx, vy, vz, u, m, alpha, h};
    for (int f = 0; f < 10; ++f) if ((r = fetch_column(c, {DS_ST + f, CB_STATE}, 8, dst[f]))) return r;
  }
  double* sd[8] = {sx, sy, sz, svx, svy, svz, sm, srad};
  const double* ss[8] = {c->S.x, c->S.y, c->S.z, c->S.vx, c->S.vy, c->S.vz, c->S.m, c->S.radius};
  for (int k = 0; k < 8; ++k) if ((r = fetch_sink(c, ss[k], sd[k]))) return r;
  CK(cudaStreamSynchronize(c->stream));
  return SPH_OK;
}

int sph_state_hash(sph_ctx* c, uint64_t* hash, double* sums5) {
  if (!c || !hash) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  unsigned long long* d = nullptr; DA(d, 8);
  CK(cudaMemsetAsync(d, 0, 64, c->stream));
  const int n = (int)c->n;
  if (n > 0) LAUNCH(k_state_hash, cdiv(n, 256), 256, 0, n, state_of(c, c->cur), d, (double*)(d + 1));
  if (c->dd) {      // the domains' partial fingerprints add up (the hash is a sum; the sums are compared with a tolerance)
    { int r_ = allreduce(c, d, 1, NC_UINT64, NC_SUM); if (r_) { cudaFree(d); return r_; } }
    { int r_ = allreduce(c, d + 1, 5, NC_FLOAT64, NC_SUM); if (r_) { cudaFree(d); return r_; } }
  }
  unsigned long long h[8];
  CK(cudaMemcpyAsync(h, d, 64, cudaMemcpyDeviceToHost, c->stream));
  std::vector<double> sk((size_t)SPH_MAX_SINKS * 8);
  CK(cudaMemcpyAsync(sk.data(), c->sink_buf, sk.size() * 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  cudaFree(d);
  unsigned long long hv = h[0];
  for (int q = 0; q < c->n_sink; ++q) { unsigned long long t = mix64(0x5151ull + q); for (int k = 0; k < 8; ++k) { unsigned long long b; std::memcpy(&b, &sk[(size_t)k * SPH_MAX_SINKS + q], 8); t = mix64(t ^ b); } hv += t; }
  *hash = hv;
  if (sums5) std::memcpy(sums5, h + 1, 40);
  return SPH_OK;
}

int sph_domain_stats(sph_ctx* c, int64_t* out8) {
  if (!c || !out8) return SPH_ERR_ARG;
  out8[0] = c->dd ? 1 : 0; out8[1] = c->n; out8[2] = c->n_halo; out8[3] = c->dd ? c->ng_own : c->n_groups; out8[4] = c->ng_halo;
  if (c->dd && c->dd_let_ctl) { int cur = 0; cudaStreamSynchronize(c->xstream ? c->xstream : c->stream); cudaMemcpy(&cur, c->dd_let_ctl, sizeof(int), cudaMemcpyDeviceToHost); c->dd_let_used = cur > c->dd_let_begin ? cur - c->dd_let_begin : 0; }
  out8[5] = c->dd_let_used; out8[6] = c->dd_top_n; out8[7] = c->dd ? c->n_global : c->n;
  return SPH_OK;
}

int sph_local_size(sph_ctx* c, int64_t* n_local) {
  if (!c || !n_local) return SPH_ERR_ARG;
  *n_local = c->n;
  return SPH_OK;
}

int sph_download_local(sph_ctx* c, int32_t* number, double* x, double* y, double* z, double* vx, double* vy, double* vz,
                       double* u, double* m, double* alpha, double* h) {
  if (!c) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  const size_t n = (size_t)c->n;
  double* dst[10] = {x, y, z, vx, vy, vz, u, m, alpha, h};
  if (n > 0) {
    if (number) CK(cudaMemcpyAsync(number, c->id[c->cur], n * 4, cudaMemcpyDeviceToHost, c->stream));
    for (int f = 0; f < 10; ++f) if (dst[f]) CK(cudaMemcpyAsync(dst[f], c->st[c->cur][f], n * 8, cudaMemcpyDeviceToHost, c->stream));
  }
  CK(cudaStreamSynchronize(c->stream));
  return SPH_OK;
}

int sph_download_diag(sph_ctx* c, double* rho, double* omega, double* pressure, double* sound,
                      double* ax, double* ay, double* az, double* udot, double* alphadot,
                      double* sax, double* say, double* saz) {
  if (!c) return SPH_ERR_ARG;
  if (download_count(c) <= 0) { c->err = "no particles"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  int r;
  if ((r = download_rows(c))) return r;
  // replicated: Omega and P stay rank-local during a step, and calc_smoothing rewrites rho / Omega of the particles it iterated (V:535): bring every slice up to date
  if (!c->dd) { double* bufs[3] = {c->omega, c->prs, c->rho}; if ((r = allgatherv(c, bufs, 3))) return r; }
  const int slots[9] = {DS_RHO, DS_OMEGA, DS_PRS, DS_CS, DS_AX, DS_AY, DS_AZ, DS_UDOT, DS_ADOT};
  double* dst[9] = {rho, omega, pressure, sound, ax, ay, az, udot, alphadot};
  for (int f = 0; f < 9; ++f) if ((r = fetch_column(c, {slots[f], CB_FIXED}, 8, dst[f]))) return r;
  if ((r = fetch_sink(c, c->S.ax, sax))) return r;
  if ((r = fetch_sink(c, c->S.ay, say))) return r;
  if ((r = fetch_sink(c, c->S.az, saz))) return r;
  CK(cudaStreamSynchronize(c->stream));
  return SPH_OK;
}

int sph_download_tree(sph_ctx* c, int32_t* order, uint64_t* key, int32_t* level,
                      double* cx, double* cy, double* cz, double* size) {
  if (!c) return SPH_ERR_ARG;
  if (!c->tree_valid) { c->err = "no tree"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  int r;
  if ((r = download_rows(c))) return r;
  const int n = (int)download_count(c);
  // the global depth-first order = the positions of the rows (under domains: the domains' orders in rank order)
  if (order) CK(cudaMemcpyAsync(order, c->dd ? c->dd_gpos : c->pos, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  std::vector<int> lev(n);
  if ((r = fetch_column(c, {DS_KEY, CB_KEY}, 8, key))) return r;
  if ((r = fetch_column(c, {DS_LEVEL, CB_FIXED}, 4, level || size ? lev.data() : nullptr))) return r;
  if ((r = fetch_column(c, {DS_LCX, CB_FIXED}, 8, cx))) return r;
  if ((r = fetch_column(c, {DS_LCY, CB_FIXED}, 8, cy))) return r;
  if ((r = fetch_column(c, {DS_LCZ, CB_FIXED}, 8, cz))) return r;
  CK(cudaStreamSynchronize(c->stream));
  if (level) std::memcpy(level, lev.data(), (size_t)n * 4);
  if (size) {
    RootBox rb; CK(cudaMemcpy(&rb, c->root, sizeof(rb), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) { double s = rb.size; for (int q = 0; q < lev[i]; ++q) s *= 0.5; size[i] = s; }
  }
  return SPH_OK;
}

int sph_download_neighbours(sph_ctx* c, int32_t* count, uint64_t* hash, int64_t* offsets, int32_t* list, int64_t list_cap) {
  if (!c) return SPH_ERR_ARG;
  if (!c->tree_valid) { c->err = "no tree"; return SPH_ERR_STATE; }
  if (c->dd && list) { c->err = "sph_download_neighbours: the list form is not available under the domain decomposition"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  int r;
  if ((r = download_rows(c))) return r;
  const int n = (int)download_count(c), W = 8, own_groups = c->n_groups - c->ng_halo;
  const size_t smem = (size_t)W * 4 * WALK_TILE * 8 + (size_t)W * WALK_TILE * 4 + (size_t)W * WALK_WS * 4;
  // counts and hashes of the own rows (the walk groups but the halo's), in sorted order, land in the state buffers that
  // are not current: nothing reads those between calls (the next re-order or upload overwrites them), and the staging
  // buffers stay free for the scatter
  const StateArrays spare = state_of(c, c->cur ^ 1);
  int* const d_count = (int*)spare.x; unsigned long long* const d_hash = (unsigned long long*)spare.y;
  LAUNCH(k_neighbours, walk_grid(c, W), W * 32, smem, own_groups, c->groups, dens_arrays(c), c->pos, c->bvh, c->bi, d_count, d_hash, nullptr, nullptr);
  std::vector<int> cnt(n);
  if ((r = fetch_column(c, {DS_ST + 0, CB_SPARE_STATE}, 4, cnt.data()))) return r;
  if ((r = fetch_column(c, {DS_ST + 1, CB_SPARE_STATE}, 8, hash))) return r;
  CK(cudaStreamSynchronize(c->stream));
  if (count) std::memcpy(count, cnt.data(), (size_t)n * 4);
  std::vector<long long> off(n + 1, 0);
  for (int i = 0; i < n; ++i) off[i + 1] = off[i] + cnt[i];
  if (offsets) std::memcpy(offsets, off.data(), (size_t)(n + 1) * 8);
  if (!list) return SPH_OK;
  const long long tot = off[n];
  if (tot > list_cap) { c->err = "neighbour list capacity too small: need " + std::to_string(tot) + " have " + std::to_string((long long)list_cap); return SPH_ERR_ARG; }
  // the list form (single rank / replicated): every row's list is written at its offset, so the offsets go in sorted order
  std::vector<int> pos(n); std::vector<long long> off_sorted(n);
  CK(cudaMemcpy(pos.data(), c->pos, (size_t)n * 4, cudaMemcpyDeviceToHost));
  for (int i = 0; i < n; ++i) off_sorted[i] = off[pos[i]];
  long long* const d_off = (long long*)spare.z; int* d_list = nullptr;
  DA(d_list, std::max<long long>(tot, 1));
  CK(cudaMemcpyAsync(d_off, off_sorted.data(), (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
  LAUNCH(k_neighbours, walk_grid(c, W), W * 32, smem, own_groups, c->groups, dens_arrays(c), c->pos, c->bvh, c->bi, d_count, d_hash, d_off, d_list);
  CK(cudaMemcpyAsync(list, d_list, (size_t)tot * 4, cudaMemcpyDeviceToHost, c->stream)); CK(cudaStreamSynchronize(c->stream));
  cudaFree(d_list);
  for (int i = 0; i < n; ++i) std::sort(list + off[i], list + off[i + 1]);
  return SPH_OK;
}

int sph_set_exact_counters(sph_ctx* c, int32_t on) {
  if (!c) return SPH_ERR_ARG;
  c->exact_counters = on ? 1 : 0;
  return SPH_OK;
}

int sph_counters(sph_ctx* c, sph_counts* out) {
  if (!c || !out) return SPH_ERR_ARG;
  *out = c->counts;
  return SPH_OK;
}

int sph_stage_times(sph_ctx* c, double* ms, int32_t n) {
  if (!c || !ms) return SPH_ERR_ARG;
  for (int i = 0; i < n && i < 16; ++i) ms[i] = i < ST_COUNT ? c->stage_ms[i] : 0.0;
  return SPH_OK;
}

int64_t sph_launch_count(sph_ctx* c) { return c ? c->launches : 0; }
int64_t sph_group_count(sph_ctx* c) { return c ? c->n_groups : 0; }
int64_t sph_far_reuse_count(sph_ctx* c) { return c ? c->far_count : 0; }
int64_t sph_far_overflow_runs(sph_ctx* c) { return c ? c->far_n_ovf : 0; }
int64_t sph_resident_hits(sph_ctx* c) { return c ? c->resident_hits : 0; }
int sph_set_resident_check(sph_ctx* c, int32_t on) { if (!c) return SPH_ERR_ARG; c->resident_check = on ? 1 : 0; return SPH_OK; }

int sph_timer_start(sph_ctx* c) {
  if (!c) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  if (!c->tm0) { CK(cudaEventCreate(&c->tm0)); CK(cudaEventCreate(&c->tm1)); }
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaEventRecord(c->tm0, c->stream));
  return SPH_OK;
}

int sph_timer_stop(sph_ctx* c, double* ms) {
  if (!c || !ms || !c->tm0) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  CK(cudaEventRecord(c->tm1, c->stream));
  CK(cudaEventSynchronize(c->tm1));
  float f = 0.f; CK(cudaEventElapsedTime(&f, c->tm0, c->tm1));
  *ms = f;
  return SPH_OK;
}

int sph_fp64_peak(sph_ctx* c, double* tflops) {
  if (!c || !tflops) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
  double* out = nullptr; DA(out, 1);
  const int iters = 1 << 14, blocks = sms * 8, threads = 256;
  cudaEvent_t a, b; CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    CK(cudaEventRecord(a, c->stream));
    LAUNCH(k_fp64_peak, blocks, threads, 0, iters, 1.0000001, out);
    CK(cudaEventRecord(b, c->stream));
    CK(cudaEventSynchronize(b));
    float ms = 0.f; CK(cudaEventElapsedTime(&ms, a, b));
    const double fl = 2.0 * 8.0 * (double)iters * (double)blocks * threads;
    best = std::max(best, fl / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(out);
  *tflops = best;
  return SPH_OK;
}

int sph_conserved(sph_ctx* c, double* out, int32_t n_out) {
  if (!c || !out || n_out < 1) return SPH_ERR_ARG;
  if ((c->dd ? c->n_global : c->n) < 2) { c->err = "need at least 2 gas particles"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  double keep_ms[ST_COUNT]; std::memcpy(keep_ms, c->stage_ms, sizeof(keep_ms));
  if (!(c->tree_valid && !c->pos_moved)) {        // the octree of the current positions (kept for the next evaluation); domains: migration, halo, LET
    int r = build_tree(c); if (r) return r;
  }
  if (!c->cons_partial) { DA(c->cons_partial, (size_t)(CONS_MAX_BLOCKS + DD_MAX_RANKS) * CONS_SUMS); DA(c->cons_out, CONS_FIELDS); }
  const size_t nslot = c->dd ? (size_t)c->dd_let_end : (size_t)(2 * c->cap);
  if (nslot > c->cons_wpart_n) { c->cons_wpart_n = 0; DA(c->cons_wpart, nslot); c->cons_wpart_n = nslot; }
  const int nn = (int)c->counts.n_nodes, T = 256;
  if (c->dd) {
    CK(cudaMemsetAsync(c->cons_wpart, 0xff, nslot * sizeof(int), c->stream));
    CK(cudaMemcpyAsync(c->cons_wpart, c->dd_top_part.data(), c->dd_top_part.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  }
  LAUNCH(k_conserved_wpart, cdiv(nn, T), T, 0, nn, c->node_part, c->widx, c->dd ? DD_TOP_CAP : 0, c->cons_wpart);
  if (c->dd) {      // the walk reads the LET: every rank's must be complete, and no rank may stop alone
    if (c->let_pending) { CK(cudaStreamWaitEvent(c->stream, c->let_done, 0)); c->let_pending = false; }
    double let_overflow = 0.0;
    CK(cudaMemcpyAsync(&let_overflow, c->let_flag, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(c->h_sc, c->sc, sizeof(SimScalars), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    int code = check_device_error(c);
    if (!code && let_overflow > 0.0) { c->err = "domain decomposition: the locally essential tree of some rank exceeds its capacity (raise SPH_B200_DOMAIN_SLACK)"; code = SPH_ERR_OOM; }
    { int r = dd_agree(c, code, "sph_conserved"); if (r) return r; }
  }
  const int n = (int)c->n;
  const int nb = std::max(1, std::min(cdiv(n, CONS_THREADS), std::min(CONS_MAX_BLOCKS, c->n_sm * 16)));
  LAUNCH(k_conserved_partial, nb, CONS_THREADS, 0, n, c->dp, state_of(c, c->cur), c->wnodes, c->cons_wpart, c->n_sink, c->S, c->cons_partial);
  if (c->dd) {      // each rank's totals, all-gathered and folded in rank order: every rank returns the same bits; the sinks are added once
    double* rank_sums = c->cons_partial + (size_t)CONS_MAX_BLOCKS * CONS_SUMS;
    LAUNCH(k_conserved_fold, 1, 32, 0, nb, c->cons_partial, rank_sums + (size_t)c->rank * CONS_SUMS);
    { int r = coll_allgather(c, c->stream, rank_sums + (size_t)c->rank * CONS_SUMS, rank_sums, CONS_SUMS * sizeof(double)); if (r) return r; }
    LAUNCH(k_conserved_final, 1, 32, 0, c->n_ranks, rank_sums, c->dp, c->n_sink, c->S, c->sink_spin, c->cons_out);
  } else
    LAUNCH(k_conserved_final, 1, 32, 0, nb, c->cons_partial, c->dp, c->n_sink, c->S, c->sink_spin, c->cons_out);
  double host[CONS_FIELDS];
  CK(cudaMemcpyAsync(host, c->cons_out, sizeof(host), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(c->h_sc, c->sc, sizeof(SimScalars), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  stage_collect(c, false);                        // a tree build here is not part of any step's stage times
  std::memcpy(c->stage_ms, keep_ms, sizeof(keep_ms));
  CK(cudaGetLastError());
  { int r = check_device_error(c); if (r) return r; }                  // key-depth error of a tree built here
  for (int k = 0; k < n_out && k < CONS_FIELDS; ++k) out[k] = host[k];
  return SPH_OK;
}

int sph_column_density(sph_ctx* c, int32_t axis, double u0, double u1, double v0, double v1, int32_t nu, int32_t nv, double* image) {
  if (!c || !image) return SPH_ERR_ARG;
  if (axis < 0 || axis > 2 || nu < 1 || nv < 1 || nu > 16384 || nv > 16384 || !(u1 > u0) || !(v1 > v0)) { c->err = "bad image frame"; return SPH_ERR_ARG; }
  if ((c->dd ? c->n_global : c->n) <= 0) { c->err = "no particles uploaded"; return SPH_ERR_STATE; }
  cudaSetDevice(c->device);
  const bool reduce = c->dd && c->n_ranks > 1;      // domains: every rank scatters its own rows (never the halo copies), the images are summed
  if (!c->img_table) {
    // F(q_b) = 2 int_0^sqrt(4 - q_b^2) w(sqrt(q_b^2 + s^2)) ds, w = the M4 shape of F:66,70; composite Simpson, 4096 intervals
    std::vector<double> F(IMG_TABLE + 2, 0.0);
    auto w = [](double q) { return q <= 1.0 ? 1.0 - 1.5 * q * q + 0.75 * q * q * q : (q <= 2.0 ? 0.25 * (2.0 - q) * (2.0 - q) * (2.0 - q) : 0.0); };
    for (int i = 0; i < IMG_TABLE; ++i) {
      const double qb = 2.0 * i / IMG_TABLE, smax = std::sqrt(4.0 - qb * qb);
      const int m = 4096; const double hs = smax / m;
      double acc = w(qb) + w(std::sqrt(qb * qb + smax * smax));
      for (int k = 1; k < m; ++k) { const double sv = k * hs; acc += ((k & 1) ? 4.0 : 2.0) * w(std::sqrt(qb * qb + sv * sv)); }
      F[i] = 2.0 * acc * hs / 3.0;
    }
    DA(c->img_table, IMG_TABLE + 2);
    CK(cudaMemcpy(c->img_table, F.data(), F.size() * 8, cudaMemcpyHostToDevice));
  }
  double* d_img = nullptr;
  const size_t npx = (size_t)nu * nv;
  const bool got = cudaMalloc((void**)&d_img, npx * 8) == cudaSuccess;
  if (!got) { cudaGetLastError(); d_img = nullptr; c->err = "cudaMalloc(image)"; }
  if (reduce) { int r = dd_agree(c, got ? 0 : SPH_ERR_OOM, "sph_column_density"); if (r) { cudaFree(d_img); return r; } }
  else if (!got) return SPH_ERR_OOM;
  int r = SPH_OK;
  cudaError_t e = cudaMemsetAsync(d_img, 0, npx * 8, c->stream);
  if (e == cudaSuccess) {
    const int n = (int)c->n;
    const int grid = std::max(1, std::min(cdiv((int64_t)n * 32, IMG_THREADS), c->n_sm * 8));
    LAUNCH(k_column_density, grid, IMG_THREADS, 0, n, state_of(c, c->cur), c->dp.variable_h, c->dp.h_fixed, (int)axis, u0, v0,
           (u1 - u0) / nu, (v1 - v0) / nv, (int)nu, (int)nv, c->img_table, d_img);
    if (reduce) {      // NCCL: one all-reduce; the host communicator's all-gather carries at most SPH_HC_SLOT bytes per rank
      const size_t chunk = c->hc ? SPH_HC_SLOT / 8 : npx;
      for (size_t o = 0; o < npx && r == SPH_OK; o += chunk) r = coll_allreduce(c, c->stream, d_img + o, std::min(chunk, npx - o), NC_FLOAT64, NC_SUM);
    }
    if (r == SPH_OK) e = cudaMemcpyAsync(image, d_img, npx * 8, cudaMemcpyDeviceToHost, c->stream);
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess) e = cudaGetLastError();
  cudaFree(d_img);
  if (r != SPH_OK) return r;
  if (e != cudaSuccess) { c->err = std::string("sph_column_density: ") + cudaGetErrorString(e); return SPH_ERR_CUDA; }
  return SPH_OK;
}

int sph_interpolate(sph_ctx* c, int64_t n_points, const double* px, const double* py, const double* pz, double* out, int32_t n_out) {
  if (!c) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  const bool coll = c->dd && c->n_ranks > 1;      // domains: every rank walks its own rows for the same points, the raw sums are added
  std::string why;
  if (!px || !py || !pz || !out) why = "null pointer";
  else if (n_out < 1 || n_out > SPH_INTERP_COUNT) why = "n_out must be 1.." + std::to_string(SPH_INTERP_COUNT);
  else if (n_points < 0) why = "n_points < 0";
  uint64_t hash = 0;
  if (why.empty()) {
    const double* col[3] = {px, py, pz};
    for (int64_t i = 0; i < n_points && why.empty(); ++i)
      for (int k = 0; k < 3; ++k) {
        const double v = col[k][i];
        if (!std::isfinite(v)) { why = "non-finite coordinate"; break; }
        if (coll) { uint64_t b; std::memcpy(&b, &v, 8); hash = mix64(hash ^ b); }
      }
  }
  if (coll) {      // the ranks compare their points (count, coordinate-bit hash, n_out) and argument checks: any mismatch stops every rank
    struct Fp { int64_t n; uint64_t h; int32_t n_out, bad; };
    Fp mine = {n_points, hash, n_out, why.empty() ? 0 : 1}, all[DD_MAX_RANKS];
    { int r = dd_allgather_host(c, &mine, sizeof(Fp), all); if (r) return r; }
    for (int q = 0; q < c->n_ranks && why.empty(); ++q) {
      if (all[q].bad) why = "rank " + std::to_string(q) + " passed invalid arguments";
      else if (all[q].n != mine.n || all[q].h != mine.h || all[q].n_out != mine.n_out) why = "the ranks passed different points (the call is collective: every rank passes the same points)";
    }
  }
  if (!why.empty()) { c->err = "sph_interpolate: " + why; return SPH_ERR_ARG; }
  if ((c->dd ? c->n_global : c->n) <= 0) { c->err = "no particles uploaded"; return SPH_ERR_STATE; }
  if (n_points == 0) return SPH_OK;
  double keep_ms[ST_COUNT]; std::memcpy(keep_ms, c->stage_ms, sizeof(keep_ms));
  if (!(c->tree_valid && !c->pos_moved)) {        // the walk groups of the current positions (kept for the next evaluation); domains: migration, halo, LET
    int r = build_tree(c); if (r) return r;
  }
  int code = interp_bvh(c, c->dd ? c->ng_own : c->n_groups, (int)c->n);      // domains: the own groups, never the halo copies
  if (!code) code = interp_scratch(c, (size_t)std::min<int64_t>(n_points, SPH_INTERP_CHUNK));
  CK(cudaMemcpyAsync(c->h_sc, c->sc, sizeof(SimScalars), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  stage_collect(c, false);                        // a tree build here is not part of any step's stage times
  std::memcpy(c->stage_ms, keep_ms, sizeof(keep_ms));
  if (!code) code = check_device_error(c);        // key-depth error of a tree built here
  if (coll) { int r = dd_agree(c, code, "sph_interpolate"); if (r) return r; }
  else if (code) return code;
  for (int64_t off = 0; off < n_points; off += SPH_INTERP_CHUNK) {      // the chunks depend on n_points only: the same on every rank
    const int nc = (int)std::min<int64_t>(SPH_INTERP_CHUNK, n_points - off);
    int r = interp_chunk(c, off, nc, px, py, pz, n_points, out, n_out, coll);
    if (r) return r;
  }
  CK(cudaGetLastError());
  return SPH_OK;
}

int sph_gravity_at(sph_ctx* c, int64_t n_points, const double* px, const double* py, const double* pz, const double* h,
                   double* out, int32_t n_out) {
  if (!c) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  const bool coll = c->dd && c->n_ranks > 1;      // domains: every rank walks the nodes it owns for the same points, the gas sums are added
  std::string why;
  if (!px || !py || !pz || !out) why = "null pointer";
  else if (n_out < 1 || n_out > SPH_GRAVAT_COUNT) why = "n_out must be 1.." + std::to_string(SPH_GRAVAT_COUNT);
  else if (n_points < 0) why = "n_points < 0";
  uint64_t hash = 0;
  if (why.empty()) {
    const double* col[4] = {px, py, pz, h};
    for (int64_t i = 0; i < n_points && why.empty(); ++i)
      for (int k = 0; k < (h ? 4 : 3); ++k) {
        const double v = col[k][i];
        if (!std::isfinite(v)) { why = k < 3 ? "non-finite coordinate" : "h must be finite and positive"; break; }
        if (k == 3 && !(v > 0.0)) { why = "h must be finite and positive"; break; }
        if (coll) { uint64_t b; std::memcpy(&b, &v, 8); hash = mix64(hash ^ b); }
      }
  }
  if (coll) {      // the ranks compare their points (count, hash of the coordinate and h bits, n_out) and argument checks
    struct Fp { int64_t n; uint64_t h; int32_t n_out, bad; };
    Fp mine = {n_points, hash ^ (h ? 1ull : 0ull), n_out, why.empty() ? 0 : 1}, all[DD_MAX_RANKS];
    { int r = dd_allgather_host(c, &mine, sizeof(Fp), all); if (r) return r; }
    for (int q = 0; q < c->n_ranks && why.empty(); ++q) {
      if (all[q].bad) why = "rank " + std::to_string(q) + " passed invalid arguments";
      else if (all[q].n != mine.n || all[q].h != mine.h || all[q].n_out != mine.n_out) why = "the ranks passed different points (the call is collective: every rank passes the same points)";
    }
  }
  if (!why.empty()) { c->err = "sph_gravity_at: " + why; return SPH_ERR_ARG; }
  if ((c->dd ? c->n_global : c->n) <= 0) { c->err = "no particles uploaded"; return SPH_ERR_STATE; }
  if (n_points == 0) return SPH_OK;
  double keep_ms[ST_COUNT]; std::memcpy(keep_ms, c->stage_ms, sizeof(keep_ms));
  if (!(c->tree_valid && !c->pos_moved)) {        // the octree of the current positions (kept for the next evaluation); domains: migration, halo, LET
    int r = build_tree(c); if (r) return r;
  }
  int code = interp_scratch(c, (size_t)std::min<int64_t>(n_points, SPH_INTERP_CHUNK));
  if (!code && c->ga_cap < c->ip_cap) {
    c->ga_cap = 0;
    code = dalloc(c, &c->ga_q, 4 * c->ip_cap);
    if (!code) code = dalloc(c, &c->ga_raw, (size_t)GRAVAT_COLS * c->ip_cap);
    if (!code) c->ga_cap = c->ip_cap;
  }
  if (!code && c->dd) {
    if (!c->ga_owner) code = dalloc(c, &c->ga_owner, DD_TOP_CAP);
    if (!code) CK(cudaMemcpyAsync(c->ga_owner, c->dd_top_owner.data(), c->dd_top_owner.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    if (c->let_pending) { CK(cudaStreamWaitEvent(c->stream, c->let_done, 0)); c->let_pending = false; }      // no LET slot is read, but its pull writes the layout
  }
  CK(cudaMemcpyAsync(c->h_sc, c->sc, sizeof(SimScalars), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  stage_collect(c, false);                        // a tree build here is not part of any step's stage times
  std::memcpy(c->stage_ms, keep_ms, sizeof(keep_ms));
  if (!code) code = check_device_error(c);        // key-depth error of a tree built here
  if (coll) { int r = dd_agree(c, code, "sph_gravity_at"); if (r) return r; }
  else if (code) return code;
  for (int64_t off = 0; off < n_points; off += SPH_INTERP_CHUNK) {      // the chunks depend on n_points only: the same on every rank
    const int nc = (int)std::min<int64_t>(SPH_INTERP_CHUNK, n_points - off);
    int r = gravat_chunk(c, off, nc, px, py, pz, h, n_points, out, n_out, coll);
    if (r) return r;
  }
  CK(cudaGetLastError());
  return SPH_OK;
}

int sph_download_sink_spin(sph_ctx* c, double* sx, double* sy, double* sz) {
  if (!c) return SPH_ERR_ARG;
  cudaSetDevice(c->device);
  double* dst[3] = {sx, sy, sz};
  for (int k = 0; k < 3; ++k) {
    if (!dst[k] || c->n_sink == 0) continue;
    if (c->sink_spin) CK(cudaMemcpyAsync(dst[k], c->sink_spin + (size_t)k * SPH_MAX_SINKS, (size_t)c->n_sink * 8, cudaMemcpyDeviceToHost, c->stream));
    else std::memset(dst[k], 0, (size_t)c->n_sink * 8);        // the reference's sinks keep spin = 0 (F:695)
  }
  CK(cudaStreamSynchronize(c->stream));
  return SPH_OK;
}

}  // extern "C"
