/* libcmf_sm100 -- C ABI of the B200 (sm_100a) convolutive-NMF fit path.
 *
 * Drop-in boundary for the update-rule plugin interface of degleris1/CMF.jl
 * (`abstract type AbstractCFUpdate`, src/algs/alternating.jl:8): a rule is constructed from
 * (data, W, H) (src/model.jl:79), `update_motifs!` mutates W (alternating.jl:52) and
 * `update_feature_maps!` mutates H and returns the relative loss (alternating.jl:54).
 * Julia binds these entry points with `ccall` (see INTEGRATION.md and julia/CMFsm100.jl);
 * the Python mirror in cmf.jl_b200/ binds the same symbols with ctypes.
 *
 * Conventions
 *  - All HOST arrays are Julia column-major:  data N x T  (X[n + N*t]),
 *    W  K x N x L (W[k + K*(n + N*l)], current-src layout, src/common.jl:18,25),
 *    H  K x T     (H[k + K*t]).  Element type is double (dtype 0) or float (dtype 1).
 *  - The caller owns every host array; the library copies during the call and never keeps
 *    a host pointer.  The library owns all device memory behind the handle.
 *  - Every function returns 0 on success, non-zero on error; the message is available from
 *    cmf_last_error() (thread-local).  No C++ exception crosses this boundary.  There is no
 *    CPU fallback: without a CUDA device every compute entry point fails with CMF_ERR_CUDA.
 *  - One host thread per handle; the call blocks the caller (a Julia task inside `ccall`).  Every call
 *    runs on the handle's device(s) and restores the caller's current CUDA device before returning.
 *
 * Multi-GPU (time axis sharding, SURVEY.md section 8e; the reference is single-process): rank r owns the
 * columns [t_r, t_{r+1}) of X and H, W is replicated.  The collectives (all-reduce of the W-side partials,
 * L-1 column halo exchange of H, all-reduce of the loss scalars, gather/scatter around the HALS H sweep)
 * run INSIDE the library over NCCL (bound at run time with dlopen), so the same reference-facing calls --
 * cmf_set_data, cmf_set_factors, cmf_update_motifs, cmf_update_feature_maps, cmf_loss, cmf_fit,
 * cmf_get_factors -- drive one GPU or many:
 *   - cmf_create_multi: ONE process, one calling thread, `ngpu` devices (ncclCommInitAll + one worker thread
 *     and one stream per device inside the library; Julia never needs `Distributed`).  Host arrays are the
 *     full N x T / K x T arrays, exactly as for cmf_create.
 *   - cmf_create_rank: one process per GPU (torchrun / MPI style); rank 0 obtains cmf_comm_unique_id, the
 *     host passes the 128 bytes to the other ranks by its own means, every rank calls the same sequence of
 *     library calls (they meet inside the collectives).  Host arrays cover the rank's own columns.
 * The older split-phase calls (cmf_w_partials ... cmf_loss_partial on handles from cmf_create_shard, with the
 * HOST doing the collectives on the pointers from cmf_exchange_buffer / cmf_halo_buffers) are kept for hosts
 * that bring their own collective library, and for the CPU (gloo) tests of the step logic.
 */
#ifndef CMF_SM100_H
#define CMF_SM100_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cmf_ctx *cmf_handle;

enum { CMF_F64 = 0, CMF_F32 = 1 };   /* dtype: arithmetic type of the kernels            */
enum { CMF_MULT = 0, CMF_HALS = 1, CMF_PGD = 2 }; /* alg: MultUpdate (src/algs/mult.jl) / HALSUpdate (hals.jl) /
                                                      PGDUpdate (pgd.jl: SquareLoss, Nonneg projection,
                                                      l2 = SquarePenalty weight, l1 = AbsolutePenalty weight) */
enum {
    CMF_OK = 0,
    CMF_ERR_ARG = 1,   /* bad dimensions / null pointer / wrong state                  */
    CMF_ERR_CUDA = 2,  /* CUDA runtime error (including "no device")                   */
    CMF_ERR_UNSUPPORTED = 3,
    CMF_ERR_NCCL = 4   /* NCCL missing or a collective failed                           */
};

/* ---- lifecycle ---------------------------------------------------------------------- */

/* Replaces the rule constructors MultUpdate(data,W,H) / HALSUpdate(data,W,H)
 * (src/algs/mult.jl:11-20, src/algs/hals.jl:18-28) together with cmf_set_data and
 * cmf_set_factors.  Requires 1 <= L <= T (src/common.jl:28-31 would index out of range
 * otherwise).  `device` is the CUDA ordinal. */
int cmf_create(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg,
               int device);

/* Same, for one time-shard [t_begin, t_end) of a T_global-column problem (no reference
 * counterpart: the reference is single-process).  Needs t_end - t_begin >= L-1.
 * PGD is single-shard only in this version (CMF_ERR_UNSUPPORTED otherwise). */
int cmf_create_shard(cmf_handle *out, int64_t N, int64_t T_global, int64_t t_begin, int64_t t_end,
                     int64_t K, int64_t L, int dtype, int alg, int device);

/* The rule constructor (src/model.jl:79) for `ngpu` GPUs driven from ONE host thread: the time axis is
 * split into balanced contiguous shards, one per device (`devices` = CUDA ordinals, NULL = 0..ngpu-1).
 * The returned group handle takes the same calls as a cmf_create handle with the full host arrays;
 * ngpu == 1 is cmf_create.  MultUpdate and HALSUpdate. */
int cmf_create_multi(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg,
                     int ngpu, const int *devices);

/* One process per GPU: the balanced shard of `rank` among `world` ranks on `device`, with its own NCCL
 * communicator built from the 128-byte id that rank 0 got from cmf_comm_unique_id (collective: every
 * rank must call it).  Host arrays passed to this handle start at global column `first_col` as for
 * cmf_create_shard; cmf_get_factors returns the rank's own columns of H.  The communicator is kept by the process and
 * reused by later handles of the same (device, rank, world) created with unique_id == NULL (every rank must then do so). */
int cmf_comm_unique_id(void *id_out_128_bytes);
int cmf_create_rank(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg,
                    int device, const void *unique_id_128_bytes, int rank, int world);
/* The partition rule of both constructors: columns [*t_begin, *t_end) of rank `rank`. */
int cmf_shard_range(int64_t T, int world, int rank, int64_t *t_begin, int64_t *t_end);
/* rank / world / column range of a handle (group handles report rank 0, world = ngpu, the full range). */
int cmf_comm_info(cmf_handle h, int *rank_out, int *world_out, int64_t *t_begin, int64_t *t_end);
/* Re-sends the L-1 column halos of H between neighbouring ranks (after cmf_set_factors from host arrays
 * that hold only the rank's own columns); a no-op without a communicator. */
int cmf_exchange_halos(cmf_handle h);

int cmf_destroy(cmf_handle h);

/* Thread-local message of the last failing call on this thread. */
const char *cmf_last_error(void);

/* ---- data and factors ----------------------------------------------------------------- */

/* `X` is a column-major N x (something) host array whose first column is global column
 * `first_col`; the library reads columns [t_begin, min(t_end + L-1, T)) (owned + right halo)
 * and computes ||X_owned||^2.  Replaces the `data` argument of the rule constructor
 * (src/model.jl:79) and `data_norm = norm(data)` (mult.jl:13, hals.jl:23). */
int cmf_set_data(cmf_handle h, const void *X, int64_t first_col);

/* Synthetic data generated in HBM (benchmarks; SURVEY.md section 8d): the reference's
 * data model (datasets/synthetic.jl:29-61) with a counter-based generator keyed on the global
 * (seed, n, t), so the data are identical for any sharding.  K_true/L_true are the ground-truth
 * rank and lag count, p_h the activation probability, noise the Gaussian noise std. */
int cmf_synth_data(cmf_handle h, uint64_t seed, int64_t K_true, int64_t L_true, double p_h,
                   double noise);

/* Copies the owned columns of X (N x (t_end-t_begin)), plus the right halo clipped to T when
 * with_halo != 0, back to a host array (used by benchmarks to obtain a host copy of the
 * device-generated synthetic data). */
int cmf_get_data(cmf_handle h, void *X_out, int with_halo);

/* sum of squares of the owned columns of X (double), and the global norm used as the loss
 * denominator (defaults to the local one; a sharded host all-reduces and sets it). */
int cmf_data_sumsq(cmf_handle h, double *out);
int cmf_set_data_norm(cmf_handle h, double norm);

/* W: K x N x L host array.  H: column-major K x (something) whose first column is global
 * column `first_col`; the library reads [t_begin-(L-1), t_end+(L-1)) clipped to [0,T)
 * (owned + both halos).  Replaces the W,H arguments of the rule constructor / the deepcopy at
 * src/algs/alternating.jl:33-34.  For HALS this also (re)computes the persistent residual
 * (hals.jl:22). */
int cmf_set_factors(cmf_handle h, const void *W, const void *H, int64_t first_col);

/* Uniform [0,1) initialisation in HBM keyed on the global (seed,k,n,l) / (seed,k,t)
 * (src/model.jl:116-117 restated with a counter-based generator), WITHOUT the alpha rescale:
 * cmf_init_scale_partials returns the local <X, est> and ||est||^2 (model.jl:119-120); the host
 * sums them over shards and calls cmf_scale_factors(sqrt(|alpha|)) (model.jl:121-122). */
int cmf_init_rand(cmf_handle h, uint64_t seed);
int cmf_init_scale_partials(cmf_handle h, double out_dot_norm2[2]);
int cmf_scale_factors(cmf_handle h, double s);

/* Copies W (K x N x L) and the owned columns of H (K x (t_end-t_begin)) to host arrays. */
int cmf_get_factors(cmf_handle h, void *W_out, void *H_out);

/* ---- the update rule (single shard) --------------------------------------------------- */

/* update_motifs!(rule, data, W, H; l1W, l2W)      src/algs/mult.jl:23-39, hals.jl:31-34, pgd.jl:158-178 */
int cmf_update_motifs(cmf_handle h, double l1W, double l2W);
/* loss = update_feature_maps!(rule, data, W, H; l1H, l2H)   mult.jl:42-58, hals.jl:37-42, pgd.jl:181-203 */
int cmf_update_feature_maps(cmf_handle h, double l1H, double l2H, double *loss_out);
/* compute_loss(data, W, H)                         src/common.jl:54-55 */
int cmf_loss(cmf_handle h, double *loss_out);

/* The whole alternating loop on the device (src/algs/alternating.jl:16-71):
 * max_itr < 0 means Inf; loss_hist/time_hist are caller-allocated with capacity `cap`
 * (>= max_itr+1 when max_itr >= 0); *n_hist receives the number of entries written
 * (iterations + 1); *converged_early is set when the early stop of alternating.jl:63-66 fired
 * (the caller prints "Converged early." as the reference does). */
int cmf_fit(cmf_handle h, int64_t max_itr, double max_time, int eval_mode, int check_convergence,
            int patience, double tol, double l1W, double l2W, double l1H, double l2H,
            double *loss_hist, double *time_hist, int64_t cap, int64_t *n_hist,
            int *converged_early);

/* ---- batched restarts: R MultUpdate fits of ONE data set in one handle ------------------------
 *
 * Random restarts, regulariser sweeps and rank sweeps fit the same data many times.  A batch handle holds R factor sets of
 * one L -- of one K (cmf_create_batch) or of a rank K[r] each (cmf_create_batch_ranks) -- over one copy of X and steps all
 * of them with one launch per kernel: numW (mult.jl:32) and numH (mult.jl:47) of all restarts are one correlation / one
 * transposed convolution with sum K[r] components (X is read once per step), and the per-restart pieces (Gram, G*W, W*W',
 * lag tables, denomH, ratio updates, loss) are launches with a restart index.  The launches of an iteration depend
 * neither on R nor on the ranks.  MultUpdate, fp64 and fp32, SIMT engine (0), one GPU, a single shard.
 *
 * Host arrays hold the R restarts one after another, each in the layout of the single-set calls: W is R blocks of
 * K x N x L, H is R blocks of K x T; per-restart vectors have R entries.
 *
 * These calls work on a batch handle as on any other: cmf_set_data / cmf_synth_data (X is stored once), cmf_get_data,
 * cmf_data_sumsq, cmf_destroy, cmf_sync, cmf_launch_count, cmf_stream, cmf_set_stream, cmf_profile, cmf_set_engine(h, 0),
 * cmf_get_engine, cmf_last_error.  Calls that take or return ONE factor set (cmf_set_factors, cmf_init_rand,
 * cmf_init_scale_partials, cmf_scale_factors, cmf_get_factors, cmf_update_motifs, cmf_update_feature_maps, cmf_loss,
 * cmf_fit) return CMF_ERR_ARG with a message naming the batch call to use.  The split-phase calls, engines 1 and 2 and
 * loss mode 1 return CMF_ERR_UNSUPPORTED. */

/* Like cmf_create with R >= 1 restarts.  alg must be CMF_MULT (HALS / PGD: CMF_ERR_UNSUPPORTED).  The device footprint
 * (about (4 R K L N + 3 R K T + (T + L) N) elements plus small per-restart tables) is computed before anything is
 * allocated; when it exceeds the free device memory the call fails with CMF_ERR_ARG and a message stating the bytes needed.
 * Argument checks come before any device query, as for cmf_create. */
int cmf_create_batch(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg, int64_t R,
                     int device);
/* Like cmf_create_batch, restart r with its own rank K[r] >= 1 (same N, T, L, dtype, alg for all): a sweep over K in one
 * handle.  MultUpdate, SIMT engine, one GPU.  Host arrays hold the restarts one after another: W is the R blocks
 * K[r] x N x L, H the R blocks K[r] x T (restart r at W + N*L*sum_{q<r} K[q], H + T*sum_{q<r} K[q]).
 * cmf_create_batch(..., K, ..., R, ...) is this call with K[r] = K for every r.  The footprint grows with sum K[r] and
 * sum K[r]^2 L^2 and is checked, as for cmf_create_batch, before anything is allocated.  Checks as cmf_create_batch, plus
 * a null K (CMF_ERR_ARG) and any K[r] < 1 (CMF_ERR_ARG). */
int cmf_create_batch_ranks(cmf_handle *out, int64_t N, int64_t T, const int64_t *K /* R */, int64_t L, int dtype,
                           int alg, int64_t R, int device);
/* W: R blocks of K x N x L, H: R blocks of K x T (restart r at W + r*K*N*L, H + r*K*T); for cmf_create_batch_ranks the
 * ragged blocks above. */
int cmf_set_factors_batch(cmf_handle h, const void *W, const void *H);
int cmf_get_factors_batch(cmf_handle h, void *W_out, void *H_out);
/* out[2r] = <X, est_r>, out[2r+1] = ||est_r||^2 (model.jl:119-120); the host applies cmf_scale_factors_batch with
 * s[r] = sqrt(|out[2r] / out[2r+1]|) (model.jl:121-122).  Each sum runs in the order of cmf_init_scale_partials. */
int cmf_init_scale_partials_batch(cmf_handle h, double *out /* 2R */);
int cmf_scale_factors_batch(cmf_handle h, const double *s /* R */);
/* compute_loss(data, W_r, H_r) of every restart (src/common.jl:54-55). */
int cmf_loss_batch(cmf_handle h, double *loss_out /* R */);
/* cmf_fit for every restart, restart r with its own l1W[r], l2W[r], l1H[r], l2H[r] and its own early stop.  Restart r
 * writes loss_hist[r*cap .. r*cap + n_hist[r]) and converged_early[r].  A restart that meets the early stop of
 * alternating.jl:63-66 is frozen: nothing updates its factors again while the others go on.  The loop ends when every
 * restart has stopped or max_itr / max_time is reached.  max_time and time_hist use the batch's own wall clock, so every
 * restart shares time_hist (its first n_hist[r] entries are restart r's) -- the one difference from R separate cmf_fit
 * calls, whose clocks would each measure one fit. */
int cmf_fit_batch(cmf_handle h, int64_t max_itr, double max_time, int eval_mode, int check_convergence, int patience,
                  double tol, const double *l1W, const double *l2W, const double *l1H, const double *l2H,
                  double *loss_hist /* R x cap, restart-major */, double *time_hist /* cap */, int64_t cap,
                  int64_t *n_hist /* R */, int *converged_early /* R */);

/* ---- sparse data: X given as compressed sparse columns, the dense N x T X never allocated ---------------------------
 *
 * Spike rasters and event trains are mostly zeros.  A sparse handle holds X as CSC (and a CSR copy built from it, for numW),
 * with int32 row / time indices on the device, and computes the two contractions that read X -- numW (mult.jl:32) and numH
 * (mult.jl:47) -- with nnz K L multiply-adds each instead of N T K L.  Everything else touches W and H only and is unchanged.
 *
 * Rules of a sparse handle:
 *  - The SIMT engine (0) only: cmf_set_engine(h, 1 | 2) returns CMF_ERR_UNSUPPORTED, cmf_get_engine reports 0.
 *  - The loss is always the expansion ||X||^2 - 2 <numH, H> + <W W', Htilde Htilde'>, each term summed in double (||X||^2 from
 *    nzval, once per data set): the direct pass would need the dense residual.  cmf_get_loss_mode reports 1,
 *    cmf_set_loss_mode(h, 0) and cmf_set_loss_guard return CMF_ERR_UNSUPPORTED (there is no calibration), and
 *    cmf_get_loss_stats counts expansions.  cmf_init_scale_partials[_batch] use the same identities:
 *    <X, est> = <numH, H>, ||est||^2 = <W W', Htilde Htilde'>.
 *  - cmf_set_data, cmf_synth_data and cmf_get_data need the dense X and return CMF_ERR_ARG naming cmf_set_data_csc.
 *  - Every other call works as on a dense handle of the same kind (single or batch), including the split-phase diagnostics
 *    cmf_w_partials / cmf_h_update + cmf_exchange_buffer on a single handle.
 *  - MultUpdate and HALSUpdate (batches: MultUpdate), one GPU, one shard.  PGD: CMF_ERR_UNSUPPORTED.
 *  - The footprint of the factors and work buffers (as for a dense handle, without X, plus a transposed copy of W) is checked
 *    at creation, that of the CSC and CSR arrays (2 nnz (4 + sizeof(dtype)) + 8 (N + T + 2) bytes) by cmf_set_data_csc; either
 *    fails with CMF_ERR_ARG and a message stating the bytes needed. */

/* A handle whose data are given as a sparse matrix (cmf_set_data_csc): the dense N x T X is never allocated.
 * alg: CMF_MULT or CMF_HALS (CMF_PGD: CMF_ERR_UNSUPPORTED).  One GPU, one shard.  N <= INT32_MAX, T <= INT32_MAX.  The checks
 * of cmf_create, all before any device query. */
int cmf_create_sparse(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg, int device);

/* Batch form (R MultUpdate restarts of one sparse data set, restart r with rank K[r]); the checks of cmf_create_batch_ranks
 * and of cmf_create_sparse.  numW and numH of all restarts are one sparse launch each (X is read once per step). */
int cmf_create_batch_sparse(cmf_handle *out, int64_t N, int64_t T, const int64_t *K /* R */, int64_t L, int dtype, int alg,
                            int64_t R, int device);

/* X as compressed sparse columns, column t = time bin t, exactly Julia's SparseMatrixCSC{T,Int64} layout:
 * the entries of column t are colptr[t] .. colptr[t+1]-1 (minus index_base), with row indices rowval[] and values nzval[]
 * of the handle dtype.  index_base = 1 lets Julia pass its arrays unchanged; 0 for scipy.  Row indices strictly increasing
 * within a column (no duplicates).  Replaces the data (any nnz).  Sparse handles only (a dense handle: CMF_ERR_ARG naming
 * cmf_create_sparse).  Checked on the host before anything reaches the device, CMF_ERR_ARG with a message naming the first
 * offending column or entry: index_base is 0 or 1; colptr starts at the base, never decreases and ends at nnz + base; every
 * row index is in range; row indices strictly increase within each column; nnz >= 1 (the relative loss of an all-zero X is
 * undefined). */
int cmf_set_data_csc(cmf_handle h, int64_t nnz, const int64_t *colptr /* T+1 */, const int64_t *rowval /* nnz */,
                     const void *nzval /* nnz */, int index_base);

/* ---- split-phase steps for time-sharded fits (MultUpdate only) -------------------------- */

/* 1. local W-side partials: numW (src/algs/mult.jl:32), the H cross-correlation that yields
 *    denomW (mult.jl:28,33 via G = Htilde Htilde'), and the last L-1 columns of H on the last
 *    shard, all into exchange buffers 0 and 1. */
int cmf_w_partials(cmf_handle h);
/* 2. host all-reduces (sum) exchange buffers 0 and 1, then: W update (mult.jl:37-38). */
int cmf_w_apply(cmf_handle h, double l1W, double l2W);
/* 3. H update on the owned columns (mult.jl:44-52); afterwards the host exchanges halos. */
int cmf_h_update(cmf_handle h, double l1H, double l2H);
/* 4. after the halo exchange: local sum of squared residuals (mult.jl:55-57 numerator^2). */
int cmf_loss_partial(cmf_handle h, double *sumsq_out);

/* Exchange buffer `which`: 0 = numW partial (count = K*N*L elements of the handle dtype),
 * 1 = Gram/tail partial (double); diagnostics only: 2 = numH, 3 = denomH of the last cmf_h_update
 * ([t][K], handle dtype).  Returns the device pointer, element count and dtype. */
int cmf_exchange_buffer(cmf_handle h, int which, void **dev_ptr, int64_t *count, int *dtype);
/* H halo regions, each (L-1)*K contiguous elements of the handle dtype:
 * send_left  = first L-1 owned columns (goes to the left neighbour's recv_right),
 * send_right = last  L-1 owned columns (goes to the right neighbour's recv_left). */
int cmf_halo_buffers(cmf_handle h, void **send_left, void **send_right, void **recv_left,
                     void **recv_right, int64_t *count);

/* Blocks until all work queued by this handle has finished (for host-side timing). */
int cmf_sync(cmf_handle h);
/* Number of kernels this handle has launched so far (bench.py's `gpu_launches`). */
int cmf_launch_count(cmf_handle h, int64_t *out);
/* The CUDA stream (cudaStream_t) the handle launches on, for event timing by the host. */
int cmf_stream(cmf_handle h, void **stream_out);
/* Makes the handle launch on a caller-owned stream (e.g. the host framework's current stream,
 * so that host-side collectives on the exchange buffers are stream-ordered with the kernels
 * and no host synchronisation is needed between steps).  NULL selects the legacy default stream. */
int cmf_set_stream(cmf_handle h, void *stream);
/* Per-kernel-class CUDA-event timing on the handle's stream (bench.py's roofline numbers):
 * cmf_profile(h, 1) starts recording an event pair around every launch of the three contraction
 * kernels; cmf_profile_read returns the summed device time and launch count of class
 * `which` (0 = conv/residual/loss, 1 = transposed conv for numH, 2 = correlation for numW, 3 = HALS H sweep). */
int cmf_profile(cmf_handle h, int enable);
int cmf_profile_read(cmf_handle h, int which, double *ms_total, int64_t *count);
/* Selects the contraction engine: 0 = SIMT kernels (fp64 and fp32); 1 = tcgen05 tensor-core kernels in the
 * time domain (fp32 data, split-bf16 operands, K <= 128, N % 8 == 0); 2 = frequency-domain engine: numW
 * (mult.jl:32) and numH (mult.jl:47) through the overlap-save spectrum of X (computed once per data set, the
 * circular-convolution idea of src/common.jl:36-50 made exact) with the per-frequency complex products on
 * tcgen05 -- HBM-bound instead of tensor-bound (fp32, K <= 128, L <= 256, room for ~1.1-1.25x the size of X in
 * bf16 hi/lo planes; the time-domain planes of engine 1 are released).  Returns CMF_ERR_UNSUPPORTED when the
 * handle cannot use the engine.  Default: best available (2 for large problems with L >= 8, else 1, else 0). */
int cmf_set_engine(cmf_handle h, int engine);
/* How the tcgen05 engine evaluates the loss inside the iteration (mult.jl:55-57): 0 = direct fused
 * conv + residual pass (default; always used by the SIMT/fp64 engines), 1 = the exact identity
 * ||conv(W,H)-X||^2 = ||X||^2 - 2<transconv(W,X),H> + <W W', Htilde Htilde'> on the numH and W W' that the
 * H update leaves resident plus the Gram of the new H, which the next cmf_w_partials reuses (a third of the
 * contraction work is saved; the halos must not change between cmf_loss_partial and cmf_w_partials).  The
 * identity cancels like 1/loss^2 (measured error ~2e-6/loss^2 relative: a slowly varying bias from the truncating
 * fp32 adder of the tensor core).  cmf_loss / cmf_update_feature_maps / cmf_fit therefore use it as it is only while
 * the relative loss is above the guard (25 %); at or below the guard they CALIBRATE it: the direct pass runs every
 * `interval` evaluations, the difference to the expansion is kept and subtracted in between, and every direct pass
 * checks the value the previous difference would have predicted -- the interval doubles (up to max_interval) while
 * that prediction is within 5e-6 of the direct loss, halves above 2e-5, and the handle returns to mode 0 for good
 * after three misses above 1e-4.  Split-phase callers (cmf_loss_partial) get the raw expansion and apply their own rule. */
int cmf_set_loss_mode(cmf_handle h, int mode);
/* The loss mode currently in force (handles that select the frequency-domain engine by themselves start with 1). */
int cmf_get_loss_mode(cmf_handle h, int *mode_out);
/* Guard and longest calibration interval of loss mode 1 (defaults 0.25 and 16); a guard above any loss (e.g. 1e30) puts
 * the handle into the calibrated regime from the first evaluation (bench.py measures that regime this way). */
int cmf_set_loss_guard(cmf_handle h, double guard, int max_interval);
/* Loss evaluations so far by the direct pass and by the expansion, the calibration interval in force (0 = not in the
 * calibrated regime) and the relative error of the last checked prediction.  Any output pointer may be NULL. */
int cmf_get_loss_stats(cmf_handle h, int64_t *n_direct, int64_t *n_expansion, int *interval, double *last_err);
/* Overlap-save layout of the frequency-domain engine on this handle (first rank of a group): block length B (the smallest
 * power of two >= 8L, at most 1024; halved when the half is still >= 4L and >= 64 and the shard is so short that the longer
 * block does not cut the per-frequency product work by at least 3 %; the next power of two when memory is short; CMF_FD_B
 * overrides with a power of two in [max(4L, 64), 1024], other values are ignored), hop V = B - L + 1 and the number of
 * blocks (padded to a multiple of 16) whose spectrum the two data-sized products stream.  Zeros when engine 2 is not in force. */
int cmf_get_fd_layout(cmf_handle h, int *block_len, int *hop, int64_t *nblocks);
/* The engine currently selected (0 / 1 / 2). */
int cmf_get_engine(cmf_handle h, int *engine_out);

/* PGDUpdate's pluggable loss (src/algs/pgd.jl:28-70; keyword `loss_func` of update_motifs! / update_feature_maps!, pgd.jl:160,183):
 * loss_func 0 = SquareLoss (default), 1 = AbsoluteLoss; `mask` = NULL or a column-major N x T host array of the handle dtype that
 * wraps the loss in a MaskedLoss (gradient multiplied by the mask, loss evaluated on mask.*data and mask.*est).  With either, the
 * update follows pgd.jl:224-255 literally (conv + loss-gradient epilogue, then the correlation / transposed conv of that gradient);
 * the loss returned by cmf_update_feature_maps is sqrt(eval(loss_func) / ||data||^2) as pgd.jl:202.  PGD handles only. */
int cmf_set_pgd_loss(cmf_handle h, int loss_func, const void *mask);
/* PGDUpdate's projections (keywords `constrW` / `constrH` of update_motifs! / update_feature_maps!, pgd.jl:161,183):
 * 0 = NonnegConstraint (x = max(eps(), x), pgd.jl:91-95; default), 1 = UnitNormConstraint (every component slice whose
 * 2-norm exceeds 1 is divided by it, pgd.jl:98-110; no non-negativity).  PGD handles only. */
int cmf_set_pgd_constraints(cmf_handle h, int constrW, int constrH);

/* ---- primitives (tests; one-shot, host in / host out) ----------------------------------- */

/* tensor_conv(W, H)       src/common.jl:17-34     out: N x T */
int cmf_tensor_conv(int64_t N, int64_t T, int64_t K, int64_t L, int dtype, const void *W,
                    const void *H, void *out);
/* tensor_transconv(W, X)  src/common.jl:62-81     out: K x T */
int cmf_tensor_transconv(int64_t N, int64_t T, int64_t K, int64_t L, int dtype, const void *W,
                         const void *X, void *out);
/* numW of src/algs/mult.jl:31-34                  out: K x N x L */
int cmf_corr_w(int64_t N, int64_t T, int64_t K, int64_t L, int dtype, const void *H,
               const void *X, void *out);
/* compute_resids(data, W, H) = tensor_conv(W,H) - data   src/common.jl:58-59     out: N x T */
int cmf_compute_resids(int64_t N, int64_t T, int64_t K, int64_t L, int dtype, const void *X,
                       const void *W, const void *H, void *out);
/* shift_and_stack(H, L)   src/common.jl:133-142   out: (K*L) x T, row l*K + k holds H[k, :] shifted right by l
 * (the fit never materialises it -- it addresses the same rows through overlapping windows of H; this entry
 * point exists for callers and tests that want the matrix itself) */
int cmf_shift_and_stack(int64_t K, int64_t T, int64_t L, int dtype, const void *H, void *out);

#ifdef __cplusplus
}
#endif
#endif /* CMF_SM100_H */
