/* b200nest.h -- C ABI of libb200nest.so: the B200 (sm_100a) implementation of
 * dynesty's bounding-and-proposal hot path.
 *
 * The reference (joshspeagle/dynesty @ 99451618, pure Python) has no FFI; its
 * extension seams are three Python duck-types (SURVEY.md section 8b):
 *   bound=<Bound>            py/dynesty/bounding.py:76-122
 *   sample=<InternalSampler> py/dynesty/internal_samplers.py:36-203
 *   pool=<obj with .map>     py/dynesty/utils.py:2358-2381
 * Each entry point below replaces the numeric body of the reference function
 * cited next to it; the Python classes in dynesty_b200/ (ctypes) mirror the
 * three duck-types and call these.  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - all matrices row-major float64; u = unit-cube coordinates (N, n).
 *   - every function returns a b2n_status (0 = ok); the library never returns
 *     owned memory: the caller allocates all outputs.
 *   - pointer mode (b2n_set_pointer_mode): B2N_PTR_HOST (default) = array
 *     arguments are host pointers, the call copies in/out and synchronises
 *     before returning; B2N_PTR_DEVICE = array arguments are device pointers on
 *     the ctx device, work is enqueued on the ctx stream and NOT synchronised
 *     (functions that must return a host scalar synchronise and say so).
 *     Arguments documented "host" are host pointers in both modes.
 *     In B2N_PTR_HOST mode the chain entry points (b2n_{rwalk,rslice,slice,unif}_batch) use PINNED caller
 *     buffers in place: the kernel reads the start points and writes the finished chains through the
 *     buffers' device alias (no staging copy); pageable buffers are staged.  Same results either way.
 *   - one caller thread per ctx (the reference's master is single-threaded,
 *     calls are strictly serialised from Sampler, sampler.py:676-778).
 */
#ifndef B200NEST_H_
#define B200NEST_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2n_ctx b2n_ctx;

/* ---- status codes; the Python layer maps them 1:1 onto the reference's
 *      exceptions (file:line of the raise in the reference) ---------------- */
typedef enum {
    B2N_OK = 0,
    B2N_ERR_CUDA = 1,            /* CUDA runtime failure (b2n_last_error)           */
    B2N_ERR_ARG = 2,             /* bad argument                                    */
    B2N_ERR_SINGLE_POINT = 3,    /* ValueError   bounding.py:1405-1407, RuntimeError :666-668 */
    B2N_ERR_SINGULAR = 4,        /* ValueError   bounding.py:218-222                */
    B2N_ERR_ELL_INIT = 5,        /* RuntimeError bounding.py:1451-1453              */
    B2N_ERR_INVALID_REGION = 6,  /* RuntimeError bounding.py:683-685                */
    B2N_ERR_Q0 = 7,              /* RuntimeError bounding.py:570-574                */
    B2N_ERR_SLICE_FAIL = 8,      /* RuntimeError internal_samplers.py:1191-1203     */
    B2N_ERR_NOMEM = 9,
    B2N_ERR_UNSUPPORTED = 10,
    B2N_ERR_TOO_MANY_ELLS = 11,  /* max_ells too small for the decomposition        */
    B2N_ERR_PEER = 12,           /* peer exchange not configured / a peer never arrived */
    B2N_ERR_PLATEAU = 13         /* RuntimeError sampler.py:473-475: no live point above loglstar   */
} b2n_status;

/* warning bits (the reference issues warnings.warn at the cited lines) */
#define B2N_WARN_IDENTITY_FALLBACK 1u /* bounding.py:1373-1378                       */
#define B2N_WARN_DOUBLING          2u /* internal_samplers.py:694, 839, 1144         */
#define B2N_WARN_Q0_SLACK          4u /* bounding.py:576-579                         */
#define B2N_WARN_UNIF_INEFFICIENT  8u /* internal_samplers.py:316-320                */

#define B2N_PTR_HOST   0
#define B2N_PTR_DEVICE 1

/* per-dimension boundary flags (utils.py:950-976 get_nonbounded) */
#define B2N_DIM_PERIODIC   1u
#define B2N_DIM_REFLECTIVE 2u

int  b2n_init(int device, b2n_ctx** ctx);
void b2n_free(b2n_ctx* ctx);
int  b2n_set_stream(b2n_ctx* ctx, void* cuda_stream);   /* cudaStream_t; NULL = own stream */
int  b2n_set_pointer_mode(b2n_ctx* ctx, int mode);
int  b2n_synchronize(b2n_ctx* ctx);
/* Chains per CTA of the chain kernels: by default a launch spreads its chains over as many CTAs as the GPU holds
 * (small launches: ONE chain per CTA, the shortest latency for a lone run).  When many contexts share the GPU
 * (replicas), packing k chains into a CTA (lock-step, k <= 8 / 16 depending on the kernel) leaves the SMs to the
 * other contexts at a small cost in per-launch latency.  Results do not depend on it. */
int  b2n_set_chain_pack(b2n_ctx* ctx, int32_t chains_per_cta);
/* Start points by INDEX for the next b2n_rwalk_batch call (one call, then reset): `u0` of that call is then the
 * whole live set, `nrows` x ndim, and chain q starts from row idx[q] -- what Sampler.propose_live / _fill_queue do
 * with `self.live_u[i, :]` (sampler.py:469-491, 708-717) moved into the kernel: the caller no longer gathers the Q
 * start rows into a contiguous block (40 us of a 0.32 ms end-to-end step at C2).  idx: nchain int32 in [0, nrows),
 * host or device memory like the other arrays of the call; NULL cancels.  Any other chain entry point called with
 * the setting pending clears it and returns B2N_ERR_UNSUPPORTED. */
int  b2n_set_start_rows(b2n_ctx* ctx, const int32_t* idx, int64_t nrows);
/* diagnostic: host microseconds per launch when `nlaunch` empty kernels are enqueued back to back on the ctx stream
 * (call it from several threads / contexts at once to see what the driver's launch path sustains) */
int  b2n_debug_launch_rate(b2n_ctx* ctx, int32_t nlaunch, double* us_per_launch);
const char* b2n_strerror(int status);
const char* b2n_last_error(b2n_ctx* ctx);
const char* b2n_version(void);
/* number of kernel launches issued through this ctx since b2n_init (bench.py gpu_launches) */
int64_t b2n_launch_count(b2n_ctx* ctx);
/* kernel timing for the roofline: when enabled, the chain entry points bracket their main
 * kernel with CUDA events on the ctx stream; b2n_last_kernel_ms waits for it and returns the
 * duration of the most recent one (ms, <0 if none). */
int  b2n_set_timing(b2n_ctx* ctx, int enabled);
double b2n_last_kernel_ms(b2n_ctx* ctx);

/* ---- device models: the "device-side likelihood callback" -----------------
 * The reference evaluates user Python callables prior_transform(u) and
 * loglikelihood(v) once per proposal (internal_samplers.py:957-958, 1116-1117,
 * 328-329).  Inside a kernel that callback is a closed registry:            */
#define B2N_PRIOR_IDENTITY   0  /* v = u                                          */
#define B2N_PRIOR_UNIFORM    1  /* v = p0[i] + p1[i]*u   (lo, width)               */
#define B2N_PRIOR_NORMAL_PPF 2  /* v = p0[i] + p1[i]*ndtri(u)  (mu, sigma)         */
#define B2N_LIKE_GAUSS_PREC  0  /* -0.5 (v-vec0)^T mat (v-vec0) + s0              */
#define B2N_LIKE_GAUSS_DIAG  1  /* -0.5 sum vec1[i] (v-vec0)[i]^2 + s0            */
#define B2N_LIKE_EGGBOX      2  /* (2 + prod cos((2 s0 v - s0)/2))^s1  (tmax, power) */
#define B2N_LIKE_SHELLS      3  /* logaddexp of two shells: centres vec0, vec1, radius s0, width s1 */
#define B2N_LIKE_REGION2D    4  /* the hard-edged 2-D regions of the reference's sampler-uniformity harness
                                   (tests/test_sampling.py:8-23) on (v[0], v[1]), other dims free:
                                   s0 = 0: diamond_logl, s0 = 1: checker_logl; -inf outside           */

typedef struct {
    int32_t ndim;
    int32_t prior_kind;
    int32_t like_kind;
    int32_t reserved;
    const double* prior_p0;  /* host, ndim (or NULL) */
    const double* prior_p1;  /* host, ndim (or NULL) */
    const double* like_vec0; /* host, ndim (or NULL) */
    const double* like_vec1; /* host, ndim (or NULL) */
    const double* like_mat;  /* host, ndim*ndim symmetric (or NULL) */
    double like_s0, like_s1, like_s2;
} b2n_model_desc;

/* copies the parameters to the device; *model_id is a small integer handle. host args. */
int b2n_model_create(b2n_ctx* ctx, const b2n_model_desc* desc, int32_t* model_id);

/* v = prior_transform(u), logl = loglikelihood(v) for M points (u: M x ndim).
 * Replaces the pool.map of the two callables in sampler.py:148-158. v may be NULL. */
int b2n_model_eval(b2n_ctx* ctx, int32_t model_id, const double* u, int64_t M,
                   double* v, double* logl);

/* ---- ellipsoid membership: MultiEllipsoid.within/overlap/contains
 *      (bounding.py:502-523), Ellipsoid.distance_many/contains (:286-305) ----
 * d2[m,k] = (x_m - c_k)^T A_k (x_m - c_k); mask[m,k] = d2 < 1 (strict != 0) or
 * d2 <= 1 (strict == 0); q[m] = number of ellipsoids containing x_m.
 * mask / q / d2 may each be NULL. */
int b2n_membership(b2n_ctx* ctx, const double* x, int64_t M, int32_t n,
                   const double* ctrs, const double* ams, int32_t K, int32_t strict,
                   uint8_t* mask, int32_t* q, double* d2);

/* ---- bounding construction ------------------------------------------------
 * bounding_ellipsoid (bounding.py:1387-1461) incl. improve_covar_mat
 * (:1311-1384) and the Ellipsoid constructor (:201-240).  Outputs: ctr (n),
 * cov/am/axes (n x n; axes[:,i] = i-th principal axis scaled by its length,
 * columns ordered by ascending eigenvalue), axlens (n), logvol (1).
 * *warn receives B2N_WARN_* bits (host int, may be NULL).  Synchronises. */
int b2n_bounding_ellipsoid(b2n_ctx* ctx, const double* points, int64_t N, int32_t n,
                           double* ctr, double* cov, double* am, double* axes,
                           double* axlens, double* logvol, uint32_t* warn);

/* MultiEllipsoid.update without bootstrap: bounding_ellipsoid + the recursive
 * 2-means split _bounding_ellipsoids (bounding.py:665-686, 1464-1563) + the
 * all-points-contained check (:683-685).  labels[N] = index of the leaf
 * ellipsoid each point was assigned to.  nells: host int out.  Arrays sized
 * for max_ells.  Synchronises.  Internally the update uses two more streams of the
 * context besides its own (the root's eigen fit runs speculatively beside the expansion of
 * the candidate tree, the two halves of a candidate fit run side by side; DESIGN.md 9.7);
 * they are drained before the call returns, the caller sees one synchronous call. */
int b2n_multi_decompose(b2n_ctx* ctx, const double* points, int64_t N, int32_t n,
                        int32_t max_ells, int32_t* nells, int32_t* labels,
                        double* ctrs, double* covs, double* ams, double* axes,
                        double* axlens, double* logvols, uint32_t* warn);

/* Block moments for a row-SHARDED live set (SURVEY.md 8e): mean (n) and sample covariance (n x n, ddof = 1; zeros
 * for a single row) of `points` (N x n) -- np.mean / np.cov of bounding.py:1410-1412 for one shard.  Shards combine
 * exactly: S = sum_r [(N_r - 1) cov_r + N_r (mean_r - mean)(mean_r - mean)^T], cov = S / (N - 1); the ellipsoid then
 * follows from b2n_improve_covar on the combined covariance and an all-reduce(max) of the shard-local
 * max_i delta_i^T am delta_i (b2n_membership's d2).  Synchronises. */
int b2n_moments(b2n_ctx* ctx, const double* points, int64_t N, int32_t n, double* mean, double* cov);

/* improve_covar_mat (bounding.py:1311-1384) on its own: the <= 100-trial repair ladder (eigenvalue clamp at
 * 10 max/1e12, then the identity blend, then the identity fallback) applied to `covar` (n x n).  Outputs:
 * the repaired covariance, its inverse `am`, `axes` = V sqrt(lambda) (columns, ascending eigenvalue);
 * *good = 1 iff the input passed untouched (host int), *warn = B2N_WARN_IDENTITY_FALLBACK bit.  Synchronises. */
int b2n_improve_covar(b2n_ctx* ctx, const double* covar, int32_t n, double* cov_out, double* am,
                      double* axes, int32_t* good, uint32_t* warn);

/* Measured FP64 issue ceilings of this GPU for bench.py's roofline: kind 0 = FP64 FMA (vector pipe),
 * kind 1 = FP64 m8n8k4 MMA (tensor pipe); `iters` rounds of 16 independent chains per thread, all SMs.
 * *tflops, *ms (best of 4 timed launches, CUDA events): host outputs.  Synchronises. */
int b2n_fp64_peak(b2n_ctx* ctx, int32_t kind, int32_t iters, double* tflops, double* ms);

/* Ellipsoid.scale_to_logvol for K ellipsoids (bounding.py:242-276, 478-495).
 * target_logvols: host, K.  covs/ams/axes/axlens/logvols updated in place. */
int b2n_scale_to_logvol(b2n_ctx* ctx, int32_t K, int32_t n, double* covs, double* ams,
                        double* axes, double* axlens, double* logvols,
                        const double* target_logvols);

/* _ellipsoid_bootstrap_expand for nboot replicas (bounding.py:1593-1648):
 * replica r resamples with the B2N stream (seed, chain0 + r) (one integers
 * event, oracle/philox.py), fits in-bag, expand[r] = max(1, max out-of-bag
 * min-over-ellipsoids distance).  expands: host, nboot.  Synchronises. */
int b2n_bootstrap_expand(b2n_ctx* ctx, const double* points, int64_t N, int32_t n,
                         int32_t multi, int32_t nboot, uint64_t seed, uint64_t chain0,
                         double* expands);

/* ---- resident bound for the proposal kernels --------------------------------
 * Uploads K ellipsoids of dimension ncdim (what Sampler ships to every task as
 * `axes` / kwargs['bound'], sampler.py:708-717, internal_samplers.py:229-233).
 * host pointers in both modes.  ctrs/ams/logvols may be NULL if only
 * rwalk/slice are used. */
int b2n_bound_set(b2n_ctx* ctx, int32_t K, int32_t ncdim, const double* ctrs,
                  const double* ams, const double* axes, const double* logvols);

/* b2n_unif_batch only: draw from the bound without the unit-cube test and without
 * evaluating a model (Bound.samples, bounding.py:321-334, 592-606); needs ndim == ncdim,
 * model_id ignored. */
#define B2N_OPT_DRAW_ONLY 1
/* with DRAW_ONLY: MultiEllipsoid.sample(return_q=True) semantics (bounding.py:580-584): the
 * draw is returned WITHOUT the 1/q acceptance test and ncall[q] receives q (the number of
 * ellipsoids containing it) -- the input of monte_carlo_logvol (:608-630). */
#define B2N_OPT_DRAW_MIXTURE 2

/* ---- proposal chains ----------------------------------------------------------
 * One chain per queue slot (sampler.py:690-717).  Chain q consumes the B2N
 * Philox stream (seed, chain0 + q) -- see oracle/philox.py for the layout. */
typedef struct {
    int64_t nchain;          /* Q                                                   */
    int32_t ndim;            /* n                                                   */
    int32_t ncdim;           /* clustered dims (axes are ncdim x ncdim)              */
    int32_t model_id;
    int32_t reserved;        /* option bits: B2N_OPT_*                               */
    const double* u0;        /* Q x ndim start points (live points with logl > loglstar) */
    const int32_t* ell;      /* HOST, Q: index into the resident bound of the axes of
                                each chain (get_random_axes, bounding.py:726-731); NULL = 0 */
    const uint8_t* dimflags; /* HOST, ndim B2N_DIM_* flags or NULL                      */
    double loglstar;
    double scale;
    uint64_t seed;
    uint64_t chain0;
} b2n_chain_args;

/* RWalkSampler.sample -> generic_random_walk (internal_samplers.py:505-561,
 * 866-986, propose_ball_point :989-1035): exactly `walks` proposals per chain.
 * Outputs per chain: u, v (Q x ndim), logl, n_accept, n_reject, ncall (Q). */
int b2n_rwalk_batch(b2n_ctx* ctx, const b2n_chain_args* a, int32_t walks,
                    double* u, double* v, double* logl,
                    int32_t* n_accept, int32_t* n_reject, int32_t* ncall);

/* RSliceSampler.sample (internal_samplers.py:745-855) / SliceSampler.sample
 * (:593-709) -> generic_slice_step (:1075-1206).  flags[q]: B2N_WARN_DOUBLING if
 * the chain switched to doubling; status B2N_ERR_SLICE_FAIL if any chain's
 * interval collapsed. */
int b2n_rslice_batch(b2n_ctx* ctx, const b2n_chain_args* a, int32_t slices,
                     int32_t doubling, double* u, double* v, double* logl,
                     int32_t* n_expand, int32_t* n_contract, int32_t* ncall,
                     uint32_t* flags);
int b2n_slice_batch(b2n_ctx* ctx, const b2n_chain_args* a, int32_t slices,
                    int32_t doubling, double* u, double* v, double* logl,
                    int32_t* n_expand, int32_t* n_contract, int32_t* ncall,
                    uint32_t* flags);

/* UnitCubeSampler.sample (internal_samplers.py:343-441) for a queue: every chain draws u ~ U(0,1)^ndim (one
 * uniform vector event per draw of its B2N stream) until loglikelihood(prior_transform(u)) > loglstar; ncall[q] =
 * number of draws.  u0 / ell / scale / ncdim unused, no resident bound needed.  flags may be NULL. */
int b2n_unitcube_batch(b2n_ctx* ctx, const b2n_chain_args* a, double* u, double* v, double* logl,
                       int32_t* ncall, uint32_t* flags);

/* UniformBoundSampler.sample (internal_samplers.py:243-340) with
 * MultiEllipsoid.sample (bounding.py:525-590) as the bound draw; u0/ell/scale
 * unused.  nprop[q] = draws from the bound incl. out-of-cube ones. */
int b2n_unif_batch(b2n_ctx* ctx, const b2n_chain_args* a, double* u, double* v,
                   double* logl, int32_t* ncall, int32_t* nprop, uint32_t* flags);

/* ---- RadFriends / SupFriends: one ball / cube per live point (bounding.py:734-996, 999-1263) ------------------
 * kind: 0 = balls (RadFriends, Euclidean norm), 1 = cubes (SupFriends, Chebyshev norm).
 * b2n_friends_update  = RadFriends.update / SupFriends.update (:874-958 / 1142-1226): covariance from the clusters
 *     of the single-linkage tree cut at Mahalanobis distance 1 under the CURRENT metric am_prev (use_clustering;
 *     :966-993), am = pinvh(cov), axes = sqrtm(cov), axes_inv = pinvh(axes), radius = leave-one-out nearest-neighbour
 *     distance (nboot = 0; :1683-1705) or the bootstrap radius over nboot realisations (:1651-1680; realisation b
 *     resamples with the B2N stream (seed, chain0 + b), one integers event), everything rescaled by the radius,
 *     logvol = prefactor - slogdet(am) / 2.  Outputs (n x n each, logvol / radius / nclusters host scalars); the
 *     caller keeps `ctrs = points` (:950, sampler.py:481).  Synchronises.
 * b2n_friends_set     makes (ctrs, axes, axes_inv) the resident friends bound of the ctx.
 * b2n_friends_overlap = overlap(x) (:785-790 / 1052-1057) for M query points: q[m] = number of balls / cubes
 *     containing x_m (contains = q > 0, within = the indices).
 * b2n_friends_unif_batch = UniformBoundSampler.sample (internal_samplers.py:243-340) with the bound's own
 *     sample() (:797-831 / 1065-1100: random centre + random offset, accepted with probability 1/q) as the draw;
 *     a->reserved = B2N_OPT_DRAW_ONLY: Bound.samples (no cube test / likelihood), | B2N_OPT_DRAW_MIXTURE:
 *     sample(return_q=True), ncall[q] = q. */
int b2n_friends_update(b2n_ctx* ctx, const double* points, int64_t N, int32_t n, int32_t kind, int32_t use_clustering,
                       const double* am_prev, int32_t nboot, uint64_t seed, uint64_t chain0, double* cov, double* am,
                       double* axes, double* axes_inv, double* logvol, double* radius, int32_t* nclusters);
int b2n_friends_set(b2n_ctx* ctx, int32_t kind, const double* ctrs, int64_t N, int32_t n, const double* axes,
                    const double* axes_inv);
int b2n_friends_overlap(b2n_ctx* ctx, const double* x, int64_t M, int32_t n, int32_t* q);
int b2n_friends_unif_batch(b2n_ctx* ctx, const b2n_chain_args* a, double* u, double* v, double* logl, int32_t* ncall,
                           int32_t* nprop, uint32_t* flags);

/* ---- multi-GPU exchange over NVLink peer memory (SURVEY.md 8e) ------------------------------
 * The path shards by CHAINS: rank r of W runs rows [row0, row0 + nchain) of a `total_rows`-chain
 * queue fill (the reference's pool.map over queue slots, sampler.py:717, one slot = one chain).
 * Every rank needs every finished chain (replicated live set), which is an all-gather.  Instead
 * of a collective after the kernel, the chain kernels themselves store each finished chain into
 * the exchange WINDOW of every rank (peer stores over NVLink/NVSwitch), and the last CTA of the
 * grid runs a cross-GPU arrive/wait on counters in the windows: when a b2n_*_batch launch has
 * completed on a rank, all `total_rows` rows are present in that rank's window.
 *
 *   b2n_peer_export   allocate this rank's window, return its 64-byte CUDA IPC handle
 *   (exchange the handles of all ranks with any host transport, e.g. torch.distributed)
 *   b2n_peer_import   map the windows of all ranks (one process per GPU)
 *   b2n_peer_import_raw  same for ranks living in THIS process (device pointers of the windows)
 *   b2n_peer_rows     switch the following b2n_{rwalk,rslice,slice,unif}_batch calls to gather
 *                     mode: a->nchain local chains are rows [row0, row0+nchain) of total_rows;
 *                     output pointers then receive ALL total_rows rows (they may be NULL in
 *                     device-pointer mode: read the window through b2n_peer_result instead).
 *                     total_rows = 0 switches gather mode off.  All ranks must issue the same
 *                     sequence of gather-mode calls.
 *   b2n_peer_result   window pointer + byte offsets {u, v, logl, int0, int1, int2, int3} of the
 *                     last gather-mode call (int0..3 = the call's int32 outputs in argument order)
 *   b2n_peer_read     synchronise and copy `bytes` at byte `offset` of the own window to HOST memory
 *   b2n_peer_check    synchronise and report B2N_ERR_PEER if a peer never arrived (device mode;
 *                     host-pointer mode checks on return of every call).
 * Windows are double-buffered by call parity, so a rank may consume the rows of call k on its
 * stream while faster peers already store the rows of call k+1. */
#define B2N_PEER_HANDLE_BYTES 64
#define B2N_MAX_PEERS 8
int b2n_peer_export(b2n_ctx* ctx, uint64_t bytes, unsigned char* handle);
int b2n_peer_import(b2n_ctx* ctx, int32_t rank, int32_t world, const unsigned char* handles);
int b2n_peer_import_raw(b2n_ctx* ctx, int32_t rank, int32_t world, void* const* windows);
int b2n_peer_rows(b2n_ctx* ctx, int64_t row0, int64_t total_rows);
int b2n_peer_result(b2n_ctx* ctx, void** window, uint64_t* offsets7);
int b2n_peer_read(b2n_ctx* ctx, uint64_t offset, void* host_dst, uint64_t bytes);
int b2n_peer_check(b2n_ctx* ctx);
/* bytes a window needs for gather-mode calls of total_rows x ndim */
uint64_t b2n_peer_window_bytes(int64_t total_rows, int32_t ndim);

/* ---- device-resident nested-sampling rounds (SURVEY.md 8f-1: "replace K worst points per launch") ----
 * Replaces the reference's per-iteration master loop for the bounded phase of a run: the
 * worst-point search and evidence update of Sampler.sample (sampler.py:1040-1212,
 * utils.py:1470-1492 progress_integration), propose_live (:469-491), _fill_queue / _new_point
 * (:676-778) and the samplers' tune() (internal_samplers.py:460-493, 1209-1239).
 *
 * One ROUND removes the `batch` lowest live points at once (threshold L* = the batch-th lowest
 * logl), evolves `batch` chains from uniformly chosen survivors at L* against the resident bound
 * and writes every chain end point into a freed slot.  Unlike the reference's queue (an entry
 * evolved at an older threshold is kept only if it beats the current one -- a filter that
 * selects the offspring of the best live points when chains stay correlated with their starts,
 * DESIGN.md 9.4) no chain is ever discarded, so there is no selection effect; the live-point
 * count N, N-1, .., N-batch+1 seen by the removed points enters the quadrature the way the
 * reference treats a shrinking live set (ln X -= ln((m+1)/m) at a point with m live points).
 * Tuning (internal_samplers.py:460-493, 1209-1239) happens once per round; for rwalk the update is the product of the
 * `batch` per-iteration updates the reference would have made at that scale, exp(min(batch, ncdim) (abar - facc) /
 * (ncdim facc)) -- batch = 1 is the reference's rule.
 * Launches of R rounds: propose | chains | commit+propose | chains | ... | commit (R chain launches and R + 1
 * single-CTA step launches), no host synchronisation in between;
 * b2n_ns_run enqueues rounds until a stop flag is raised on the device:
 *   done        dlogz / maxiter / maxcall / plateau reached (sampler.py:1095-1120)
 *   need_bound  1 = update interval reached (sampler.py:648-651), 2 = a start point is outside
 *               the bound (forced update, :485-489), 3 = dead-point buffer full, 4 = the FIRST bound is
 *               due (unit-cube phase: enough calls and low efficiency, sampler.py:640-647)
 * The caller then updates the bound from b2n_ns_get_live (b2n_multi_decompose / b2n_bound_set as
 * usual), calls b2n_ns_bound_updated and runs on.  Random streams: chain c of round r is the
 * B2N chain (seed, chain0 + r*batch + c); the round driver (start rows, ellipsoid picks) is the
 * chain (seed, 2^62 + r), tick 0 / 1 = one uniform vector event each (oracle/nsloop.py).      */
typedef struct {
    int32_t nlive, ndim, ncdim, batch;
    int32_t sampler;          /* 0 rwalk, 1 rslice, 2 slice, 3 unif (steps ignored)             */
    int32_t steps;            /* walks / slices                                                  */
    int32_t model_id;
    int32_t strict_contains;  /* 1: MultiEllipsoid.contains (d2 < 1), 0: Ellipsoid.contains (<= 1) */
    double  facc;             /* rwalk target acceptance (internal_samplers.py:449-451)          */
    double  dlogz;
    int64_t maxiter, maxcall; /* in device-buffer iterations / total calls                       */
    int64_t update_interval;  /* bound update every this many calls (dynesty.py:213-240)         */
    uint64_t seed, chain0;
    const uint8_t* dimflags;  /* HOST, ndim B2N_DIM_* flags or NULL (copied)                      */
    /* -- the phase before the first bound (sampler.py:407-409, 625-674; _initialize_live_points + UnitCubeSampler,
     *    sampler.py:56-262, internal_samplers.py:343-441): with unit_cube_phase = 1 the run STARTS with rounds whose
     *    chains draw from the prior (b2n_unitcube_batch) and raises need_bound = 4 once ncall >= first_min_ncall and
     *    the efficiency 100 (it0 + it) / ncall has fallen below first_min_eff; b2n_ns_bound_updated ends the phase. */
    int32_t unit_cube_phase;
    int32_t use_logl_max;     /* 1: stop (done) once the lowest live logl exceeds logl_max (the end of a
                                 dynamic-sampler batch, dynamicsampler.py:1338-1345)                */
    int64_t first_min_ncall;
    double  first_min_eff;
    double  logl_max;
    int64_t it0;              /* iterations of the run before this device phase (enters the efficiency) */
} b2n_ns_config;

typedef struct {
    int64_t it, ncall, rounds;       /* dead points in the device buffer, total calls, rounds done */
    double logz, logvol, loglstar, lmax, delta_logz, scale;
    int32_t done, need_bound, doubling, error;
    int64_t ncall_last_update;       /* calls at the last bound update (restorable state)            */
} b2n_ns_status;

int b2n_ns_create(b2n_ctx* ctx, const b2n_ns_config* cfg, int64_t dead_capacity);
int b2n_ns_destroy(b2n_ctx* ctx);
/* host arrays: the live set (nlive x ndim, nlive) and the scalars of the run so far */
int b2n_ns_set_state(b2n_ctx* ctx, const double* live_u, const double* live_v, const double* live_logl,
                     double logvol, double logz, double loglstar, int64_t it, int64_t ncall, double scale);
/* enqueue up to max_rounds rounds, reading the stop flags every check_every rounds (<= 0: once at
 * the end); synchronises; returns the status (and the sampler error status, e.g.
 * B2N_ERR_SLICE_FAIL, if a chain failed). */
int b2n_ns_run(b2n_ctx* ctx, int32_t max_rounds, int32_t check_every, b2n_ns_status* status);
int b2n_ns_status_get(b2n_ctx* ctx, b2n_ns_status* status);
/* restore the counters a snapshot of a run carries besides b2n_ns_set_state's arguments (utils.py:2321-2355
 * save / restore of the reference pickles the whole sampler; here: live set + scalars + these): the round
 * index (chain ids and the round driver's stream depend on it), the calls at the last bound update, the
 * slice-doubling switch.  A run restored this way continues bit-identically. */
int b2n_ns_set_counters(b2n_ctx* ctx, int64_t rounds, int64_t ncall_last_update, int32_t doubling);
/* after the caller replaced the resident bound: clears need_bound, restarts the update interval, ends the
 * unit-cube phase */
int b2n_ns_bound_updated(b2n_ctx* ctx);
/* Sampler.update_bound (sampler.py:493-510) WITHOUT leaving the device: fits the bound to the run's live points
 * where they lie in HBM (multi = 1: MultiEllipsoid.update, bounding.py:632-686 -- b2n_multi_decompose; 0:
 * Ellipsoid.update, :345-414 -- b2n_bounding_ellipsoid; first ncdim coordinates), enlarges it
 * (scale_to_logvol(logvol + ln enlarge), sampler.py:506-508) and makes it the resident bound of the ctx -- no
 * live-set download, no bound upload.  Bootstrap expansion is not part of this entry (callers that need it take
 * the host route: b2n_ns_get_live + b2n_bootstrap_expand + b2n_bound_set).  nells / logvol (ln of the summed
 * volumes) / warn: host outputs, may be NULL.  Follow with b2n_ns_bound_updated.  Synchronises. */
int b2n_ns_update_bound(b2n_ctx* ctx, int32_t multi, double enlarge, int32_t* nells, double* logvol, uint32_t* warn);
/* the bound b2n_ns_update_bound built last (host outputs sized for max_ells >= nells; each may be NULL) */
int b2n_ns_get_bound(b2n_ctx* ctx, int32_t max_ells, double* ctrs, double* covs, double* ams, double* axes,
                     double* axlens, double* logvols);
/* ---- friends mode: RadFriends / SupFriends bounds (kind 0 balls, 1 cubes; ncdim == ndim) in the rounds.
 * b2n_ns_create starts every run in ellipsoid mode; the first of the two entry points below that installs a bound
 * switches the run to friends mode for the rest of its life (b2n_ns_update_bound is then refused).  In this mode the
 * bound is one ball / cube of common shape (cov, am, axes, axes_inv) around EVERY live point as the live set stands
 * (the reference re-points bound.ctrs = live_u before every proposal, sampler.py:479-482).  A round's chains all use
 * the common axes (get_random_axes); there is no contains test of the start points: a start is a live point, hence a
 * centre (distance 0), so the forced update of sampler.py:485-489 cannot fire.  With sampler 3 every chain draws with
 * RadFriends.sample / SupFriends.sample (bounding.py:797-831 / 1065-1100) around the run's live set, accepted with
 * probability 1/q; the round's commit keeps the transformed centres of the replaced rows current.
 *
 * b2n_ns_update_friends = Sampler.update_bound (sampler.py:493-510) without leaving the device: b2n_friends_update on
 * the run's live set in HBM with am_prev = the run's current am (the identity before the first bound), then
 * scale_to_logvol(logvol + ln enlarge) (the host class's arithmetic: both routes give the same bits).  Bootstrap
 * realisation b (nboot <= 255, else B2N_ERR_ARG) of an update made at round r draws its resample from the B2N chain
 * (seed, 0x6000000000000000 + (r << 8) + b).  logvol / radius / nclusters: host outputs, may be NULL.  Follow with
 * b2n_ns_bound_updated.  Synchronises.
 * b2n_ns_set_friends adopts a bound built elsewhere (host arrays, n x n each) as the run's bound, its centres being the
 * run's live set: a restored run, a dynamic-sampler batch, a host-route update.
 * b2n_ns_get_friends returns the bound the run holds (host outputs, each may be NULL; an adopted bound reports radius
 * NaN and nclusters 0). */
int b2n_ns_update_friends(b2n_ctx* ctx, int32_t kind, double enlarge, int32_t nboot, int32_t use_clustering,
                          double* logvol, double* radius, int32_t* nclusters);
int b2n_ns_set_friends(b2n_ctx* ctx, int32_t kind, const double* cov, const double* am, const double* axes,
                       const double* axes_inv, double logvol);
int b2n_ns_get_friends(b2n_ctx* ctx, double* cov, double* am, double* axes, double* axes_inv, double* logvol,
                       double* radius, int32_t* nclusters);
/* grow the dead-point buffer to `capacity` rows (keeps the rows written so far); clears need_bound == 3 */
int b2n_ns_reserve_dead(b2n_ctx* ctx, int64_t capacity);
/* host outputs (each may be NULL) */
int b2n_ns_get_live(b2n_ctx* ctx, double* live_u, double* live_v, double* live_logl);
int b2n_ns_get_dead(b2n_ctx* ctx, int64_t first, int64_t count, double* u, double* v, double* logl,
                    double* logvol, int32_t* ncall);

#ifdef __cplusplus
}
#endif
#endif /* B200NEST_H_ */
