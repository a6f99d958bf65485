/*
 * sph_b200.h — C-ABI of the B200-native SPH step engine.
 *
 * This is the drop-in boundary for the per-step hot path of the Fortran code
 * graves-andrew-02/SUMMERSPH.  The reference has no FFI of its own (no bind(C),
 * SURVEY.md §8(b)); the seam is cut at the body of `simulate`'s time loop:
 *     fixed h    : SUMMER_SPH.f90:886-928            (mode SPH_MODE_FIXED_H)
 *     variable h : "SUMMER_SPH - Variable.f90":1120-1162 (mode SPH_MODE_VARIABLE_H)
 * The host (Fortran via ISO_C_BINDING, the C++ twin in host/, or Python ctypes)
 * keeps `program run_sph`, file I/O, the `do while (t < end_time)` shell, the
 * per-step print and the save cadence; everything inside the loop is one call.
 *
 * Conventions
 *   - every entry point returns 0 on success, <0 on error (SPH_ERR_*); the text
 *     of the last error is available from sph_last_error();
 *   - plain pointers and sizes only; the caller owns its host arrays for the
 *     duration of a call; the context owns all device memory and the
 *     authoritative particle state between calls;
 *   - particle arrays are SoA, FP64; rows come back in ascending `number`
 *     order (the reference's array order after pack, SUMMER_SPH.f90:481,554);
 *   - one host thread drives a context; calls are synchronous at return;
 *   - there is NO CPU fallback: without a CUDA device sph_create fails with
 *     SPH_ERR_NO_DEVICE.
 */
#ifndef SPH_B200_H
#define SPH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPH_MODE_FIXED_H     0   /* SUMMER_SPH.f90                     */
#define SPH_MODE_VARIABLE_H  1   /* "SUMMER_SPH - Variable.f90"        */
#define SPH_FLAG_SOFT_USES_HI 2  /* "(test new)" softening 0.001*h_i (T:298), OR-ed into mode */
#define SPH_FLAG_SINK_MERGE_SPIN 4 /* NOT the reference's behaviour (opt-in, OR-ed into mode): fill the sinks' `spin`
                                      (declared F:33, never updated: "also need something to track the angular momentum",
                                      F:509) at accretion, and run the sink merger the reference leaves as an empty stub
                                      (check_sink_merger, V:1067-1073; call commented out at V:1159) after check_bounds */

#define SPH_OK               0
#define SPH_ERR_ARG         -1
#define SPH_ERR_NO_DEVICE   -2
#define SPH_ERR_CUDA        -3
#define SPH_ERR_OOM         -4
#define SPH_ERR_STATE       -5
#define SPH_ERR_DEPTH       -6   /* particles closer than the key resolution while max_depth exceeds it */
#define SPH_ERR_COMM        -7

/* evaluation phases (sph_evaluate mask); a full reference evaluation is SPH_EVAL_ALL */
#define SPH_EVAL_TREE     1   /* create_tree            F:795-816  V:999-1020 */
#define SPH_EVAL_DENSITY  2   /* get_density + EOS      F:398-468  V:440-512  */
#define SPH_EVAL_GRAVITY  4   /* particle_gravforces    F:249-290  V:270-311  */
#define SPH_EVAL_SINKS    8   /* sink_gravforces        F:559-591  V:691-726  */
#define SPH_EVAL_SPH     16   /* get_SPH                F:295-395  V:324-432  */
#define SPH_EVAL_ALL     31

/* Mirrors V's type(param) (Variable.f90:54-64, file order Variable.f90:899) plus the
 * constants that are compile-time in F (SUMMER_SPH.f90:7-11, 694, 873). */
typedef struct sph_params {
  int32_t mode;                 /* SPH_MODE_* | SPH_FLAG_*                              */
  int32_t max_depth;            /* F:8 (1000) | params%max_depth                        */
  int32_t nq;                   /* kernel-table samples: 5000 (F:8) | 2500 (V:8)        */
  int32_t n_ranks;              /* informational; multi-GPU is set up by sph_comm_init  */
  double  h_fixed;              /* F:11 `smoothing` (2.5). Also the 0.001*smoothing gravity
                                   softening add-on in BOTH modes (F:275, V:296)         */
  double  bounding_size;        /* F:11 (1500) | params%bounding_size                   */
  double  theta;                /* read but unused by the reference (V:1029); the BH
                                   opening angle is the literal 0.5 unless theta_override */
  double  gamma;                /* F:465-466 (1.4) | params%gamma                       */
  double  eta;                  /* V:527                                                */
  double  convergence_criteria; /* V:529                                                */
  double  max_length;           /* V:528                                                */
  double  timestep_scale;       /* F:851 (0.25) | params%timestep_scale                 */
  double  end_time;             /* F:873 (1000) | params%end_time (host loop only)      */
  double  sink_radius;          /* F:694 (3.5) | V:830 (5.0): radius given to IC sinks  */
  int32_t theta_override;       /* 0: use literal 0.5 like the reference; 1: use .theta */
  int32_t decomposition;        /* multi-rank form: 0 = replicated state, Morton-sliced walks (bit-identical to one rank);
                                   1 = Morton-ordered domains with halo exchange and a top-tree all-gather (SURVEY.md 8(e)) */
} sph_params;

/* Interaction counters of the most recent evaluation (for flop rooflines, SURVEY §8(d)). */
typedef struct sph_counts {
  int64_t n_gas;
  int64_t n_nodes;               /* octree nodes incl. leaves                           */
  int64_t density_candidates;    /* leaf box tests passed (F:443 | V:479)               */
  int64_t density_contributing;  /* of those, q <= 2                                    */
  int64_t sph_pairs;             /* unordered pairs reaching F:355 | V:384              */
  int64_t grav_opened;           /* nodes opened (recursed)   F:284                     */
  int64_t grav_accepted;         /* nodes accepted/leaf       F:279                     */
  int64_t h_iterations;          /* calc_smoothing inner re-walks, summed over particles */
} sph_counts;

typedef struct sph_ctx sph_ctx;

/* Fill `p` with the reference's defaults for `mode` (F's compile-time constants, or the
 * values a typical parameters.txt carries for V). */
int sph_default_params(int32_t mode, sph_params* p);

/* Create / destroy a context on CUDA device `device` (use 0; under torchrun LOCAL_RANK). */
int sph_create(const sph_params* p, int32_t device, sph_ctx** out);
int sph_destroy(sph_ctx* ctx);
const char* sph_last_error(const sph_ctx* ctx);   /* ctx may be NULL for create errors */

/* Optional multi-GPU: `unique_id` is the 128-byte ncclUniqueId obtained from
 * sph_comm_unique_id() on rank 0 and broadcast by the host (MPI / torch.distributed). */
int sph_comm_unique_id(void* unique_id_128);
int sph_comm_init(sph_ctx* ctx, int32_t rank, int32_t n_ranks, const void* unique_id_128);

/* The same multi-rank engine with its few small collectives (scalar all-reduces, a few KB of all-gather, barriers)
 * carried through a POSIX shared-memory segment `name` (e.g. "/sph_b200_1234") instead of NCCL.  For ranks that are
 * threads of one process or processes on one node, on any number of devices - several ranks may share one GPU, which
 * NCCL refuses - so the multi-rank logic can be exercised on a single-GPU box.  Bulk data still moves over peer-mapped
 * device memory (CUDA IPC); every collective synchronises the stream: a bring-up / test path, not the fast one.
 * Call on every rank with the same name; rank 0 creates the segment. */
int sph_comm_init_host(sph_ctx* ctx, int32_t rank, int32_t n_ranks, const char* name);

/* Target slices of the replicated-state multi-rank mode (host arithmetic only, no device needed): rank r walks the
 * groups [first_group[r], first_group[r + 1]) of the Morton-ordered group list; first_group has n_ranks + 1 entries. */
int sph_slice_bounds(int32_t n_groups, int32_t n_ranks, int32_t* first_group);

/* Replace the particle state (what read_data_from_file produces, F:594-716 | V:729-852).
 * alpha may be NULL (=0, F:681); h may be NULL in fixed-h mode. n_sink may be 0: the
 * reference's dummy zero-mass sink (F:698-707) is then created internally. */
int sph_upload(sph_ctx* ctx, int64_t n_gas,
               const double* x, const double* y, const double* z,
               const double* vx, const double* vy, const double* vz,
               const double* u, const double* m, const double* alpha, const double* h,
               int32_t n_sink,
               const double* sx, const double* sy, const double* sz,
               const double* svx, const double* svy, const double* svz,
               const double* sm, const double* srad);

/* Domain decomposition only (params.decomposition = 1 after sph_comm_init*): this rank hands over n_local of the gas
 * rows: rows [id_first, id_first + n_local) when `number` is NULL, else the rows with the given 0-based numbers (what
 * sph_download_local returned: a host that owns the state between steps).  n_global = size of the number space (rows
 * of the original file).  Any partition between the ranks: the first tree build sends every particle to the rank that
 * owns its Morton range.  Sinks are replicated: pass the same on every rank. */
int sph_upload_local(sph_ctx* ctx, int64_t n_global, int64_t id_first, const int32_t* number, int64_t n_local,
                     const double* x, const double* y, const double* z,
                     const double* vx, const double* vy, const double* vz,
                     const double* u, const double* m, const double* alpha, const double* h,
                     int32_t n_sink,
                     const double* sx, const double* sy, const double* sz,
                     const double* svx, const double* svy, const double* svz,
                     const double* sm, const double* srad);
/* The rows this rank owns now (domain decomposition; elsewhere: all rows): *n_local of them, `number` = their 0-based
 * row numbers of the upload (persistent across removals), fields as in sph_download; any pointer may be NULL.  Capacity of
 * each array >= the value sph_local_size returns. */
int sph_local_size(sph_ctx* ctx, int64_t* n_local);
int sph_download_local(sph_ctx* ctx, int32_t* number,
                       double* x, double* y, double* z, double* vx, double* vy, double* vz,
                       double* u, double* m, double* alpha, double* h);

/* Seeded synthetic start generated on the device (replaces what Disc_ICs.py:1-41 sketches): n gas particles of a
 * uniform-surface-density Keplerian disc between r_in and r_out (z ~ N(0, (aspect r)^2) clipped at 3 sigma, v_phi =
 * sqrt(G m_star / r), m = m_disc / n, the given u and alpha, h = eta (m / rho)^(1/3)) around one sink of mass m_star at
 * the origin (radius = params.sink_radius).  Row i depends only on (seed, i): under the domain decomposition every rank
 * generates its own rows.  Equivalent to sph_upload of those rows. */
int sph_ics_disc(sph_ctx* ctx, int64_t n_gas, uint64_t seed, double r_in, double r_out, double aspect, double m_star,
                 double m_disc, double u, double alpha, double eta);

/* One evaluation (tree + density + EOS + find_forces) on the current state, no integration:
 * the parity hook. `mask` selects phases (SPH_EVAL_*); rates are zeroed first (F:824). */
int sph_evaluate(sph_ctx* ctx, int32_t mask);

/* One body of the reference loop (F:886-928 | V:1120-1162): two evaluations, two half kicks,
 * drift, t += dt, dt ladder, (V) h Newton-Raphson + sink creation, accretion, bounds cull. */
int sph_step(sph_ctx* ctx, double* dt_inout, double* t_inout,
             int64_t* n_gas_out, int32_t* n_sink_out);

/* sph_upload + sph_step + sph_download in one call for a host that owns the state between steps (the reference's loop,
 * SUMMER_SPH.f90:879-929, keeps bodies(:) / sinks(:) on its side), single rank.  The copies run under the compute when the
 * host arrays are page-locked: x y z go first and the tree build starts on them while the other columns follow in the
 * order their first readers come (h: leaf cells, m: node sums, u: EOS, v / alpha: pair loop); x y z (final after the
 * drift, :903) and m leave while evaluation B runs, v u alpha after the second kick (:912), h after calc_smoothing
 * (Variable.f90:1152).  If the step removed particles every column is sent again, compacted.  Results are bit-identical
 * to the three separate calls.
 *   gas_in[10]  = x y z vx vy vz u m alpha h (alpha may be NULL = 0; h may be NULL in fixed-h mode), n_gas rows each
 *   sink_in[8]  = x y z vx vy vz m radius, n_sink rows each (NULL when n_sink = 0; radius NaN / NULL = params.sink_radius)
 *   gas_out[10] = where the rows go, ascending `number`, capacity >= n_gas each (entries may be NULL; may alias gas_in)
 *   sink_out[8] = capacity >= n_sink + 8 each (entries may be NULL) */
int sph_step_host(sph_ctx* ctx, int64_t n_gas, const double* const* gas_in, int32_t n_sink, const double* const* sink_in,
                  double* dt_inout, double* t_inout, double* const* gas_out, double* const* sink_out,
                  int64_t* n_gas_out, int32_t* n_sink_out);

/* Device-resident loop: step until t >= t_stop or max_steps (<=0: unlimited) steps. */
int sph_run_until(sph_ctx* ctx, double t_stop, int64_t max_steps,
                  double* dt_inout, double* t_inout, int64_t* steps_out,
                  int64_t* n_gas_out, int32_t* n_sink_out);

int sph_sizes(sph_ctx* ctx, int64_t* n_gas, int32_t* n_sink);

/* Download the state in ascending `number` order; any pointer may be NULL. Capacity of each
 * array must be >= the current n_gas (resp. n_sink). */
int sph_download(sph_ctx* ctx,
                 double* x, double* y, double* z, double* vx, double* vy, double* vz,
                 double* u, double* m, double* alpha, double* h,
                 double* sx, double* sy, double* sz, double* svx, double* svy, double* svz,
                 double* sm, double* srad);

/* Per-evaluation quantities the reference never saves (parity hooks), ascending `number`. */
int sph_download_diag(sph_ctx* ctx, double* rho, double* omega, double* pressure, double* sound,
                      double* ax, double* ay, double* az, double* udot, double* alphadot,
                      double* sink_ax, double* sink_ay, double* sink_az);

/* Tree of the most recent evaluation: `order[k]` = number (0-based) of the k-th leaf in the
 * reference's depth-first (Morton) order; per particle (ascending number): 63-bit descent key,
 * leaf level (root=0), leaf cell centre and size. Any pointer may be NULL. */
int sph_download_tree(sph_ctx* ctx, int32_t* order, uint64_t* key, int32_t* level,
                      double* cx, double* cy, double* cz, double* size);

/* Neighbour sets of the most recent evaluation, ascending `number`:
 * count[i]  = #{ j : leaf box test of j passes for x_i }  (self included; F:443 | V:479),
 * hash[i]   = sum over that set of mix64(number_j) (order independent),
 * if list != NULL: CSR with offsets[i] (n_gas+1 entries, caller-provided) and list capacity
 * `list_cap` entries, each row sorted ascending. */
int sph_download_neighbours(sph_ctx* ctx, int32_t* count, uint64_t* hash,
                            int64_t* offsets, int32_t* list, int64_t list_cap);

int sph_counters(sph_ctx* ctx, sph_counts* out);

/* Order-independent 64-bit fingerprint of the resident state (gas: number + the bit patterns of the ten fields; sinks):
 * equal fingerprints <=> bit-identical states, whatever the storage order or the number of ranks.  sums5 (may be NULL):
 * sum m, sum m|x|^2, sum m|v|^2, sum m u, particle count - for comparisons with a tolerance.  Collective under the
 * domain decomposition. */
int sph_state_hash(sph_ctx* ctx, uint64_t* hash, double* sums5);

/* Decomposition figures of the most recent tree build: out8 = { 1 if Morton domains are on, own particles, halo particles,
 * own walk groups, halo walk groups, locally-essential-tree nodes pulled from the peers, top-tree slots, global particles }. */
int sph_domain_stats(sph_ctx* ctx, int64_t* out8);

/* density_candidates / sph_pairs count every pair that passes the reference's leaf-box test (F:443 | V:479),
 * most of which only add exact zeros (q > 2, F:112).  By default the walks drop sources that lie beyond
 * 2 max(h) of a whole walk group before the per-pair tests - every field is bit-identical - and the two
 * counters then cover the pairs that were tested.  on = 1 keeps every box candidate so that the counters
 * equal the reference's (parity tests, flop accounting); it is slower. */
int sph_set_exact_counters(sph_ctx* ctx, int32_t on);

/* Per-stage device time of the most recent sph_step / sph_evaluate in milliseconds:
 * [0]=bbox+keys [1]=sort+reorder [2]=tree build [3]=density+EOS [4]=gravity(+sinks)
 * [5]=SPH pair [6]=integrate+dt [7]=h iteration [8]=accretion+cull [9]=NCCL exchanges (incl. waiting
 * for the slowest rank) ; n <= 16 */
int sph_stage_times(sph_ctx* ctx, double* ms, int32_t n);

/* Number of CUDA kernel launches issued by this context so far. */
int64_t sph_launch_count(sph_ctx* ctx);

/* Number of walk groups (cell-aligned runs of <= 32 particles) in the most recent tree. */
int64_t sph_group_count(sph_ctx* ctx);

/* Number of gravity evaluations so far that kept the far-field sums of the evaluation before them and walked only the
 * near field: evaluation A of a loop body sees the positions, tree and sinks of the previous body's evaluation B
 * (SUMMER_SPH.f90:894 after :905-912), so the accepted (node, particle) pairs of particle_gravforce_one (:264-290) and
 * their distances are the same; only the terms within 2 h change with calc_smoothing (Variable.f90:1152).  Same terms as
 * a full walk, summed in another order.  SPH_B200_NO_FAR_REUSE=1 (environment, read in sph_create) turns it off. */
int64_t sph_far_reuse_count(sph_ctx* ctx);

/* Walk runs (32 Morton-consecutive particles) that the last full gravity walk storing far sums flagged because some
 * particle of the run had more near terms than the records hold per particle (128; SPH_B200_FAR_SLOTS=n, read in
 * sph_create, sets another count): the next near-only evaluation serves those runs by the near-only walk instead of the
 * records.  0 before the first such walk; a full walk that stores nothing (exact counters, first step on a new state)
 * sets it back to 0. */
int64_t sph_far_overflow_runs(sph_ctx* ctx);

/* A host that owns the state between steps (upload, loop body, download - the reference's own loop keeps bodies(:) /
 * sinks(:) on the host side, SUMMER_SPH.f90:879-929) hands back exactly what it was given.  sph_upload / sph_step_host
 * therefore compare the incoming x y z m h and sinks bitwise, on the device, with the state the context holds (rows by
 * `number`); when they are the same - and the resident state came out of a step that removed nothing - the tree, the walk
 * groups and the stored far-field sums still stand and only v u alpha are taken over.  Any difference (one bit, one row,
 * the row count, a sink) makes the upload a new state.  sph_resident_hits counts the uploads that were recognised;
 * sph_set_resident_check(ctx, 0) turns the comparison off (SPH_B200_NO_RESIDENT_CHECK=1 does the same at sph_create). */
int64_t sph_resident_hits(sph_ctx* ctx);
int sph_set_resident_check(sph_ctx* ctx, int32_t on);

/* CUDA-event timer on the context's own stream (bench.py: torch events cannot see this stream). */
int sph_timer_start(sph_ctx* ctx);
int sph_timer_stop(sph_ctx* ctx, double* elapsed_ms);

/* FP64 FMA throughput of the device in TFLOP/s, measured with a register-resident FMA kernel. */
int sph_fp64_peak(sph_ctx* ctx, double* tflops);

/* Conserved-quantity sums of the resident state, for the drift report of a run (north_star: "energy/momentum
 * drift reported over the full run").  The reference keeps no such bookkeeping (nothing in SUMMER_SPH.f90
 * 863-930 sums energies or momenta); the definitions are this build's own, chosen to match the forces the
 * reference applies (SURVEY.md 8(c)):
 *   out[0]  E_kin  = sum 1/2 m v.v over gas and sinks
 *   out[1]  E_int  = sum m u over gas
 *   out[2]  E_pot  = out[10] + out[11]
 *   out[3..5]  linear momentum, out[6..8] angular momentum about the origin (gas + sinks, + sink spin when kept)
 *   out[9]  total mass
 *   out[10] gas-gas potential: 1/2 sum_i m_i G sum_{nodes accepted by the reference's Barnes-Hut walk for i,
 *           F:273-279 | V:294-300} M_node phi(dist/h)/h, phi = the cubic-spline softened potential whose
 *           derivative is the reference's g(q)/q^2 (F:91,94); i's own single-particle leaf is left out
 *   out[11] sink terms: -G m_s m_j / r over sink-gas and sink-sink pairs (unsoftened like F:559-591)
 * n_out <= SPH_CONSERVED_COUNT slots are written.  Builds the octree of the current positions if the context
 * holds none (it is then reused by the next evaluation); in a multi-GPU run every rank returns the same sums.
 * Under decomposition = 1 the call is collective (every rank calls it; the build then includes migration, halo and
 * locally essential tree); every rank returns the same values, equal to the single-rank sums up to rounding (the sum
 * over particles is grouped by rank), not bit for bit. */
#define SPH_CONSERVED_COUNT 12
int sph_conserved(sph_ctx* ctx, double* out, int32_t n_out);

/* Spin of every sink (3 x n_sink doubles; any pointer may be NULL).  All zero unless the context was created with
 * SPH_FLAG_SINK_MERGE_SPIN: the reference declares `sink%spin`, sets it to zero (F:695, V:580) and never updates it.
 * With the flag, accretion and sink mergers move into the spin exactly the orbital angular momentum (about the origin)
 * that the mass-weighted merge removes, so sum(m x cross v) + sum(spin) over sinks and gas only changes through forces;
 * out[6..8] of sph_conserved then include the spin. */
int sph_download_sink_spin(sph_ctx* ctx, double* spin_x, double* spin_y, double* spin_z);

/* Column-density image of the resident gas: what the reference's post-processing script Density_Image.py
 * draws from a save file (a 120^3 density grid with fixed h = 1.25 summed along z, Density_Image.py:105-145),
 * computed on the device from the live state with every particle's own h (`smoothing` in fixed-h mode):
 *   image[iv * nu + iu] = sum_j m_j F(|d| / h_j) / (pi h_j^2),  d = pixel centre - particle in the image plane,
 * F = line-of-sight integral of the M4 kernel shape (F:66,70).  axis = 0|1|2 projects along x|y|z with image
 * axes (y,z)|(z,x)|(x,y); pixel (iu, iv) is centred at (u0 + (iu+1/2)(u1-u0)/nu, v0 + (iv+1/2)(v1-v0)/nv).
 * Particles narrower than a pixel are widened to h = pixel/2.  `image` holds nu*nv doubles (host memory).
 * Under decomposition = 1 the call is collective: every rank scatters the particles it owns and the images are
 * summed over the ranks; every rank returns the same image, equal to the single-rank one up to rounding. */
int sph_column_density(sph_ctx* ctx, int32_t axis, double u0, double u1, double v0, double v1,
                       int32_t nu, int32_t nv, double* image);

/* The SPH interpolant of the resident gas at n_points caller-given points (px, py, pz: host arrays), computed on the
 * device: the point-wise counterpart of the density grid Density_Image.py builds with a KD-tree (:105-141), for slices,
 * profiles along a line and grids.  For a point x and the gas particles j (sinks are point masses, not SPH particles,
 * and take no part):
 *   W(r, h) = w_table(r / h) / (pi h^3), the engine's table-interpolated cubic spline with the density pass's
 *             normalisation: fixed h: h = h_fixed for every j, pi = 3.14159265359 (F:125-126); variable h: h = h_j,
 *             pi in single precision (V:139-140)
 *   members of x = { j : |x - x_j| / h_j <= 2 }  (scatter form, each particle's own h; the leaf-box test of F:443 |
 *             V:479 plays no part, so particles of a depth-limited multi-particle leaf are ordinary members; a particle
 *             whose h is not finite and positive contributes nothing)
 *   out[k * n_points + i], k = 0 .. n_out - 1 (n_out <= SPH_INTERP_COUNT):
 *     0  rho(x) = sum m_j W(|x - x_j|, h_j)
 *     1..3  v = sum m_j v_j W / rho(x),  4  u = sum m_j u_j W / rho(x),  5  alpha = sum m_j alpha_j W / rho(x)
 *           (0 where rho(x) = 0)
 *     6  the number of members, as a double
 * Mass weights, not m_j / rho_j: the result is a function of the resident x m h v u alpha alone, whichever evaluation
 * ran last (the stored rho_j is stale after calc_smoothing, V:1152).  In fixed-h mode rho at x = x_i is the density
 * pass's rho_i up to summation order.
 * SPH_ERR_ARG: a NULL pointer, n_out outside 1..SPH_INTERP_COUNT, n_points < 0 or a non-finite coordinate;
 * SPH_ERR_STATE: no gas uploaded; n_points = 0 is a no-op.  Builds the tree of the current positions if the context
 * holds none (kept for the next evaluation, like sph_conserved); the sources are found through a private BVH over the
 * walk groups, so nothing a later step reads changes, and sph_stage_times still reports the last step.  Points are
 * processed in chunks of 2^22 (scratch is bounded and kept by the context).  A call returns the same bits when repeated,
 * and for a permutation of the points (within one chunk) the permuted output.
 * Replicated multi-GPU form: every rank computes everything locally and returns the same bits.  Under
 * decomposition = 1 the call is collective: every rank passes the same points (checked: count and a hash of the
 * coordinate bits; a mismatch is SPH_ERR_ARG on every rank), each rank sums over the particles it owns, the 7 raw sums
 * are added over the ranks (NCCL all-reduce or the host communicator) and divided after that, so every rank returns
 * the same bits, equal to the single-rank result up to rounding. */
#define SPH_INTERP_COUNT 7
int sph_interpolate(sph_ctx* ctx, int64_t n_points, const double* px, const double* py, const double* pz,
                    double* out, int32_t n_out);

/* The gravitational potential and acceleration at n_points caller-given points (px, py, pz: host arrays): rotation
 * curves, mid-plane potential maps, what a test particle would feel.  Point k is treated as a gas particle of smoothing
 * length h_k (h = NULL: h_k = h_fixed for every point) placed at x_k that adds nothing to the tree; the result is what
 * particle_gravforce_one (F:264-290 | V:285-311) and sink_gravforces (F:559-591 | V:691-726) give that particle:
 *   accepted nodes: the reference's opening test, size / dist < theta or the node has no children (theta = 0.5, or
 *             params.theta under theta_override), dist = sqrt(|x - COM|^2 + soft), soft = 0.001 h_fixed
 *             (0.001 h_k with SPH_FLAG_SOFT_USES_HI); kernel length h' = h_fixed (fixed h, F:280) | h_k (variable h, V:301)
 *   out[c * n_points + k], c = 0 .. n_out - 1 (n_out <= SPH_GRAVAT_COUNT):
 *     0  phi_gas = G sum over the accepted nodes of M phi(dist / h') / h', phi = the softened potential of sph_conserved
 *        (-1/q beyond q = 2).  No node is left out: a point on a particle includes that particle's own softened term,
 *        whereas sph_conserved's E_gg leaves a particle's own leaf out.
 *     1..3  g_gas = -G sum M g(dist / h') (x - COM) / dist^3, the reference's term; at a particle's own position with its
 *        own h this is the gravity pass's gas-gas acceleration of that particle (its own leaf has direction 0)
 *     4  phi_sink = -G sum_s m_s / |x - x_s|, unsoftened (F:572), over the sinks with m_s > 0 and |x - x_s| > 0 (the
 *        zero-mass dummy sink and a point exactly on a sink add nothing)
 *     5..7  g_sink = -G sum_s m_s (x - x_s) / |x - x_s|^3 over the same sinks
 *     8  the number of nodes the walk accepted, as a double (the reference's grav_accepted for such a particle)
 * SPH_ERR_ARG: a NULL px / py / pz / out, n_out outside 1..SPH_GRAVAT_COUNT, n_points < 0, a non-finite coordinate or
 * (h given) an h_k that is not finite and positive; SPH_ERR_STATE: no gas uploaded; n_points = 0 is a no-op.
 * Builds the tree of the current positions if the context holds none (kept for the next evaluation, like
 * sph_interpolate) and changes nothing a later step reads: the stored far-field sums and near-pair records,
 * sph_counters, sph_stage_times, sph_far_reuse_count and the state arrays (ax / ay / az included) are left as they
 * were, and the sinks feel no back-reaction.  A repeated call returns the same bits, and a permutation of the points
 * the permuted output.  Replicated multi-GPU form: every rank computes locally and returns the same bits.  Under
 * decomposition = 1 the call is collective: every rank passes the same points and h (checked: count and a hash of the
 * bits; a mismatch is SPH_ERR_ARG on every rank); each rank adds the tree nodes it owns (a node straddling ranks is
 * added on rank 0), the gas columns are summed over the ranks and the sink columns are computed after that, so every
 * rank returns the same bits: `accepted` equal to the single-rank count, the values equal up to summation order. */
#define SPH_GRAVAT_COUNT 9
int sph_gravity_at(sph_ctx* ctx, int64_t n_points, const double* px, const double* py, const double* pz,
                   const double* h, double* out, int32_t n_out);

#ifdef __cplusplus
}
#endif
#endif /* SPH_B200_H */
