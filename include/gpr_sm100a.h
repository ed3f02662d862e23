/*
 * libgpr_sm100a.so -- C ABI of the B200-native exact-GP hot path.
 *
 * Drop-in boundary for srinix007/GaussianProcessRegression.jl (reference paths
 * are relative to /root/reference).  The reference has no FFI; its extension
 * seam is the cache-based non-allocating API (SURVEY.md 8b):
 *     update_cache!(tc, hp, md)            src/cost.jl:74-111
 *     loss(::MarginalLikelihood, md, tc)   src/cost.jl:113-117
 *     grad!(dL, ::MarginalLikelihood, md, tc)  src/cost.jl:119-127
 *     loss_grad! / log_loss_grad!          src/cost.jl:50-70
 *     update_cache!(pc, md)                src/predict.jl:29-34
 *     predict_mean! / predict!             src/predict.jl:36-102
 *     kernel! (SplitKernel), split predict src/split_kernel.jl:137-159, src/split_predict.jl:5-53
 *     kernel / kernel! / grad              src/covariance.jl:29-58, src/compose_covar.jl:35-77, src/deriv_covar.jl:2-32
 * Each entry point below names the reference interface it replaces.  The
 * Julia glue that binds these with ccall is in julia/GPRsm100a.jl and
 * INTEGRATION.md; in this repository the executed binding is the ctypes layer
 * gaussianprocessregression.jl_b200/gpr_sm100a/_ffi.py.
 *
 * Conventions
 *   - All matrices are column major Float64, exactly as Julia passes them:
 *     x is D x N (one point = D contiguous doubles), y is N x ny,
 *     K(x, xp) is N x M, predictive outputs have the test index fastest.
 *   - Hyper-parameters: concatenation in component order; SquaredExp and
 *     Matern52 take [sigma, l_1..l_D] (l multiplies x, no 1/2), WhiteNoise takes [sigma_n]
 *     (src/covariance.jl:27,60,85-95; src/compose_covar.jl:21-28).
 *   - Host pointers unless the function name ends in _device.  The caller owns
 *     every host buffer; the library copies what it needs and retains no
 *     pointer beyond the call.  Handles own all device memory.
 *   - Return value: 0 = ok; GPR_ERR_NOT_POSDEF (1) = the Cholesky hit a
 *     non-positive pivot, *info holds its 1-based index (LAPACK dpotrf info; the
 *     glue throws PosDefException(info) like cholesky!(...; check=true));
 *     negative = argument / CUDA error, text via gpr_last_error().
 *   - Calls on one context are synchronous and must not be issued
 *     concurrently; distinct contexts may be used from distinct threads.
 *   - There is no CPU fallback: every entry point fails with
 *     GPR_ERR_CUDA if no sm_100-class device is usable.
 */
#ifndef GPR_SM100A_H
#define GPR_SM100A_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPR_OK 0
#define GPR_ERR_NOT_POSDEF 1
#define GPR_ERR_ARG (-1)
#define GPR_ERR_CUDA (-2)
#define GPR_ERR_MEMORY (-3)
#define GPR_ERR_STATE (-4)
#define GPR_ERR_UNSUPPORTED (-5)

/* component tags: SquaredExp, WhiteNoise (src/covariance.jl:15-17); Matern52 is an extension */
#define GPR_KERN_SE 1
#define GPR_KERN_NOISE 2
#define GPR_KERN_MATERN52 3

/* gpr_fetch selectors (cache internals pinned by test/test_loss.jl:46-48) */
#define GPR_FETCH_U 0      /* N x N: upper = U, strict lower = K (tc.kchol_base) */
#define GPR_FETCH_ALPHA 1  /* N      (tc.alpha = K^-1 y[:, train_axis]) */
#define GPR_FETCH_KINV 2   /* N x N  (tc.K^-1, full symmetric) */
#define GPR_FETCH_WT 3     /* N x ny (pc.wt = K^-1 y) */

/* gpr_timings slots (milliseconds of the last evaluation, CUDA events on the library stream) */
#define GPR_T_KBUILD 0
#define GPR_T_POTRF 1
#define GPR_T_POTRS 2
#define GPR_T_TRTRI 3
#define GPR_T_LAUUM 4
#define GPR_T_GRAD 5
#define GPR_T_TOTAL 6
#define GPR_T_PRED_KSTAR 7
#define GPR_T_PRED_MEAN 8
#define GPR_T_PRED_TRSM 9
#define GPR_T_PRED_ROWNORM 10
#define GPR_T_EVAL 11        /* one whole gpr_nlml_grad call: hp upload .. F, G on the host side of the stream */
#define GPR_T_SPLIT_BUILD 12 /* gpr_split_predict: A, B^T, Diagonal(wt) C (and C for the variance) builds */
#define GPR_T_SPLIT_GEMM 13  /* gpr_split_predict: sum_k A_k .* (B_k Cw_k), fused epilogue */
#define GPR_T_SPLIT_D2H 14   /* gpr_split_predict: mean tile to the caller's host buffer */
#define GPR_T_COUNT 16

typedef struct gpr_ctx gpr_ctx;
typedef struct gpr_model gpr_model;

int gpr_version(void);
int gpr_device_count(void);                        /* usable sm_100-class devices visible to this process */

/* one context per GPU / per thread */
int gpr_ctx_create(int device, gpr_ctx** ctx);
int gpr_ctx_destroy(gpr_ctx* ctx);
const char* gpr_last_error(gpr_ctx* ctx);          /* ctx may be NULL: last error of a failed gpr_ctx_create */
/* Tuning / A-B options (defaults in brackets); none of them changes what is computed, only how:
 *   "predict_tile" test points per prediction tile; "inplace_lauum" 0/1 [0]; "leaf_lookahead" 0/1 [1]; "alpha_from_inverse" 0/1 [1];
 *   "gemm_cfg" DMMA tile variant [0 = 128x64x16]; "gemm_tma" TMA-fed T,N products 0/1 [1]; "kbuild_gram" TMA-fed Gram covariance build 0/1 [1];
 *   "ozaki" FP64 products on the INT8 tensor cores: -1 automatic from a condition-number bound [default], 0 off, 6 / 7 / 8 digits forced;
 *   "ozaki_lauum" digits of the inverse's W^T W product on that route: 9 [default], 8, 0 = DMMA; "ozaki_split" the same for the
 *   split-predict mean products; "ozaki_min" smallest routed M, N, K [1024];
 *   "ozaki_phases" bit mask potrf 1 | trtri 2 | other solves 8 [11]; "ozaki_panel", "ozaki_kchunk" k-panels [32768];
 *   "ozaki_win_mink" smallest M, N, K for the two-window form of the 8-digit product [8192];
 *   "ozaki_pair" 1 = the INT8 product kernels run as CTA pairs (tcgen05 cta_group::2), 0 = single CTAs [1]; same bits either way. */
int gpr_ctx_set_option(gpr_ctx* ctx, const char* name, int64_t value);
int64_t gpr_ctx_launch_count(gpr_ctx* ctx);        /* kernels launched by this context so far */

/* dim_hp(K, dim): src/covariance.jl:27,60; src/compose_covar.jl:26-28 */
int gpr_dim_hp(const int* comp_types, int ncomp, int D);

/* GPRModel(cov, hp, x, y; train_axis): src/models.jl:17-37.  train_axis is 1-based.
 * Limits of this implementation (the reference has none): at most 8 kernel components (GPR_ERR_ARG beyond, at creation).
 * Any D and any hyper-parameter count are taken (tested up to D = 1024 with 8 components): shapes whose point tiles or
 * per-thread gradient accumulators do not fit in shared memory run a covariance build that stages the coordinates in chunks
 * and a gradient reduction with O(P) state per CTA instead; box integration stages its bounds in chunks of coordinates
 * beyond D = 1816.  Tested up to D = 2048 for box integration. */
int gpr_model_create(gpr_ctx* ctx, const int* comp_types, int ncomp, int D, int64_t N, const double* x,
                     const double* y, int ny, int train_axis, gpr_model** model);
int gpr_model_destroy(gpr_model* model);
int gpr_model_set_y(gpr_model* model, const double* y);   /* md.y .+= dy  (src/update_model.jl:36) */
int gpr_model_set_x(gpr_model* model, const double* x);

/* kernel(K, hp, x[, xp]) / kernel!: src/covariance.jl:29-58, src/compose_covar.jl:35-77.
 * out is N x M.  same_x: the reference's `x === xp` (adds eps per non-noise component on the diagonal);
 * add_noise: self-covariance form (adds sigma_n^2 of the first WhiteNoise on the diagonal). */
int gpr_kernel(gpr_ctx* ctx, const int* comp_types, int ncomp, int D, const double* hp, const double* x, int64_t N,
               const double* xp, int64_t M, int same_x, double eps, int add_noise, double* out);

/* grad(cov, i, hp, x) for one non-noise component: src/deriv_covar.jl:2-29.
 * li: 0 = sigma, d = l_d (1..D).  out is N x N.  (WhiteNoise returns 2*sigma_n*I on the host side.) */
int gpr_kernel_grad(gpr_ctx* ctx, int comp_type, int D, const double* hp_comp, const double* x, int64_t N, int li,
                    double eps, double* out);

/* update_cache!(tc, hp, md) for MllLossCache (want_inverse = 0) / MllGradCache (want_inverse = 1),
 * and update_cache!(pc, md) of the predict caches: src/cost.jl:74-111, src/predict.jl:29-34.
 * Builds K, factors it (upper), solves for all columns of y, optionally forms K^-1. */
int gpr_update_cache(gpr_model* model, const double* hp, int P, double eps, int want_inverse, int64_t* info);
/* loss(::MarginalLikelihood, md, tc): src/cost.jl:113-117, src/loss_grad.jl:39-41 */
int gpr_loss(gpr_model* model, double* F);
/* grad!(dL, ::MarginalLikelihood, md, tc): src/cost.jl:119-127, src/loss_grad.jl:43-52.  log_scale: G .*= hp (src/cost.jl:65) */
int gpr_grad(gpr_model* model, int log_scale, double* G);
/* loss_grad! (log_scale = 0) / log_loss_grad! (log_scale = 1, hp_in holds log hp): src/cost.jl:50-70.
 * F and G may each be NULL (Optim only_fg! contract). */
int gpr_nlml_grad(gpr_model* model, const double* hp_in, int P, int log_scale, double eps, double* F, double* G,
                  int64_t* info);
int gpr_fetch(gpr_model* model, int which, double* out);

/* predict_mean! / predict!: src/predict.jl:36-102.  Requires gpr_update_cache.  xp is D x M.
 * mean: M x ny.  var_diag (nullable): M, the Diagonal path (prior = sum of hp_c[1]^2, no jitter).
 * cov_full (nullable): M x M, the dense path (prior = kernel(cov, hp, xp) incl. jitter and noise). */
int gpr_predict(gpr_model* model, const double* xp, int64_t M, int same_x, double* mean, double* var_diag,
                double* cov_full);
/* same, test points and outputs resident in device memory (mean ld = M) */
int gpr_predict_device(gpr_model* model, const double* d_xp, int64_t M, int same_x, double* d_mean, double* d_var_diag);

/* kernel!(Kxps::SplitKernel, cov, hp, Cmap(+, xe, xq), x): src/split_kernel.jl:137-159.
 * A: ne x nq x k, B: ne x N x k, C: N x nq x k, k = number of non-noise components. */
int gpr_split_kernel(gpr_ctx* ctx, const int* comp_types, int ncomp, int D, const double* hp, const double* xe,
                     int64_t ne, const double* xq, int64_t nq, const double* x, int64_t N, double* A, double* B,
                     double* C);
/* predict!(mu, Sigma::Diagonal, md, Cmap(+, xe, xq), pc): src/predict.jl:51-71, src/split_predict.jl:5-53.
 * mean: ne x nq (e fastest).  var (nullable): ne*nq, laid out q fastest within e; entries of rows
 * e in [e_lo, e_hi] (1-based inclusive, the cache's var_range, default 1:3) get the posterior variance,
 * all others keep the prior. */
int gpr_split_predict(gpr_model* model, const double* xe, int64_t ne, const double* xq, int64_t nq, int64_t e_lo,
                      int64_t e_hi, double* mean, double* var);

int gpr_timings(gpr_model* model, double* ms, int n);
/* which product engine the last factorization of this model took: *digits = 7-bit digits of the INT8-tensor-core route for potrf /
 * trtri / the prediction solves (0 = FP64 DMMA pipe), *digits_inverse = the same for the W^T W product of the inverse. */
int gpr_model_route(gpr_model* model, int* digits, int* digits_inverse);

/* integrate!(Iout, var_Iout, md, hp, a, b, nothing, wc, ac): src/integrate.jl:56-62,103-143 (row f-3 of SURVEY.md 8f,
 * the noise-free path; the per-sample-noise path needs a symmetric eigensolver and is not built).
 * Requires gpr_update_cache (K factored, wt = K^-1 y for all columns).  a, b: D box bounds.
 * Iout[e] = wt[:, e]^T k1 (e < ny), k1 = antideriv!(SquaredExp(), x, hp, a, b) (:15-31, reads hp[1..D+1] of the model);
 * var_out[0] = antideriv2(hp, a, b) - |U^-T k1|^2 (:33-41,131-136). */
int gpr_integrate(gpr_model* model, const double* a, const double* b, double* Iout, double* var_out);
/* integrate!(Iout, var_Iout, md, hp, a, b, nothing, wc, ac) (src/integrate.jl:56-62,103-143) for nbox boxes at once: for each
 * box what gpr_integrate returns for it, with its preconditions and refusals (GPR_ERR_STATE unless the model holds a factor, at
 * that factorization's hp and eps; GPR_ERR_UNSUPPORTED for a WhiteNoise first component).  GPR_ERR_ARG for NULL a, b, Iout or
 * nbox < 1.  a, b: D x nbox (box i is column i).  Iout: nbox x ny, box index fastest (the layout of gpr_mgpu_integrate),
 * Iout[i + e nbox] = wt[:, e]^T k1_i.  var_out: NULL or nbox entries, var_i = antideriv2(hp, a_i, b_i) - |U^-T k1_i|^2, not
 * clamped.  The boxes are the test points of gpr_predict with k1 in place of K(x, xp): tiles of "predict_tile" boxes
 * (GPR_ERR_MEMORY if one does not fit), each one k1 build, one T,N product against wt and one left triangular solve with U^T
 * for all its boxes (on the DMMA pipe or the INT8 route, as the prediction solves), so many boxes per call cost about as much
 * as one.  Timings: PRED_KSTAR = the k1 tile, PRED_MEAN = the wt^T k1 product and its download, PRED_TRSM = the triangular
 * solve, PRED_ROWNORM = the column sums. */
int gpr_integrate_batch(gpr_model* model, int64_t nbox, const double* a, const double* b, double* Iout, double* var_out);

/* sample(gp(x, theta)) / sample(::NormalDistribution): src/distributions.jl:20-45 (row f-5 of SURVEY.md 8f).
 * Sigma = kernel(cov, theta, x) .+ shift  -- the reference adds 1e-7 to EVERY entry, not to the diagonal --
 * factored as Sigma = L L^T; out = L z + mu.  z: N standard-normal draws supplied by the caller (the Xoshiro
 * stream of the reference stays on the host), mu: N means or NULL (zero mean).  x is D x N. */
int gpr_sample_mvn(gpr_ctx* ctx, const int* comp_types, int ncomp, int D, const double* hp, const double* x, int64_t N,
                   double shift, const double* z, const double* mu, double* out, int64_t* info);

/* diagnostics (used by tests / bench only): the DMMA tile GEMM on host matrices, C = alpha op(A) op(B) + beta C.
 * M, N multiples of 128, K multiple of 16; transA/transB in {'N','T'} (TT unsupported).
 * reps > 1 re-runs the kernel and returns the mean kernel time in *ms. */
int gpr_dbg_dgemm(gpr_ctx* ctx, char transA, char transB, int M, int N, int K, double alpha, const double* A,
                  int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int reps,
                  double* ms);
/* diagnostics / prototype: C = alpha A^T B + beta C (T,N form: A is K x M, B is K x N, both k-contiguous) through the INT8
 * tensor cores (tcgen05.mma kind::i8 with TMEM accumulators): Ozaki-type splitting of every row of A^T and column of B
 * into S signed 7-bit digits, S (S + 1) / 2 exact integer products, FP64 recombination (csrc/ozaki_i8.cuh).
 * M % 128 == 0, N % 128 == 0, K % 128 == 0, K <= 32768, S in {2, 6, 7, 8, 9} (9: two diagonal windows, 45 products).
 * flags: 1 = upper only, 2 = K-from-N, 64 = skip tile (0,0) (not with S = 9), 512 = two-window form of the 8-digit product,
 * 2048 = CTA pairs (tcgen05 cta_group::2; S = 6..9, bit-identical to the single-CTA kernels) (csrc/ozaki_i8.cuh); any other flag
 * returns an error. */
int gpr_dbg_ozaki_dgemm(gpr_ctx* ctx, int M, int N, int K, int S, double alpha, const double* A, int64_t lda, const double* B,
                        int64_t ldb, double beta, double* C, int64_t ldc, int flags, int reps, double* ms);
/* factor (and optionally invert) a host SPD matrix in place through the blocked path; A is N x N.
 * mode 0: potrf (upper = U), 1: potrf + trtri (upper = U^-1), 2: potrf + trtri + in-place lauum (upper = A^-1),
 * 3: potrf + trtri + out-of-place W W^T (upper = A^-1; the path gpr_update_cache takes when memory allows). */
int gpr_dbg_factor(gpr_ctx* ctx, double* A, int64_t N, int mode, int64_t* info, double* ms);

/* ---------------------------------------------------------------------------------------------------------
 * Multi-GPU NLML + gradient for training sets whose N x N covariance does not fit (or is too slow on) one
 * device: BASELINE.json config 5 (N = 131072, 137 GB of FP64 K), SURVEY.md 8b ("gpr_ctx_create_multi") / 8e.
 * Single process, one rank per entry of `devices`; K, its factor and K^-1 are 1-D block-cyclic over the ranks
 * (block columns of width nb), panels move between devices as peer-memory reads over NVLink.  Same arithmetic
 * and same results as gpr_nlml_grad (update_cache!(tc::MllGradCache...) + loss + grad!, src/cost.jl:96-127).
 * A device may be listed more than once (several ranks on one GPU; used by the 1-GPU tests of this path).
 * One model per multi-GPU context.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct gpr_mgpu gpr_mgpu;
typedef struct gpr_mgpu_model gpr_mgpu_model;

int gpr_mgpu_create(int nranks, const int* devices, int64_t nb, gpr_mgpu** mg);
int gpr_mgpu_destroy(gpr_mgpu* mg);
/* One rank per PROCESS (torchrun / MPI-style launch) for the same factorization: rank 0 obtains a 128-byte NCCL
 * unique id, ships it to the other processes by whatever means the host has (torch.distributed, MPI, a file), and every
 * process calls gpr_dist_create with it.  The handle is then used with gpr_mgpu_model_create / gpr_mgpu_nlml_grad /
 * gpr_mgpu_fetch(ALPHA) / gpr_mgpu_timings exactly like a single-process one: every process passes the same x, y, hp and
 * receives the same F and G.  Panels travel by ncclBroadcast / ncclAllGather, the P + 3 partial sums by ncclAllReduce.
 * NCCL is loaded with dlopen("libnccl.so.2") on first use; the library itself links the CUDA runtime only. */
int gpr_dist_unique_id(void* id128);
int gpr_dist_create(int device, int rank, int world, const void* id128, int64_t nb, gpr_mgpu** mg);

/* "transport": 0 (default) peer-memory pulls, 1 = the pack / collective / unpack data path of the NCCL transport with
 * in-process copies (test of that path on one GPU); set before creating a model.
 * "prefetch_trtri" / "prefetch_lauum": how the panels of the next step travel while the current step computes:
 * 0 = on the main queue before the step (no overlap), 1 = side queue with SM-driven peer reads, 2 = side queue through
 * the copy engines.  Default 2 for both (measured on 8 x B200, profiles/README.md).
 * "predict_tile" and the "ozaki*" options (incl. "ozaki_split") are forwarded to every rank's context (meaning as in
 * gpr_ctx_set_option). */
int gpr_mgpu_set_option(gpr_mgpu* mg, const char* name, int64_t value);
const char* gpr_mgpu_last_error(gpr_mgpu* mg);     /* mg may be NULL: last error of a failed gpr_mgpu_create */
int64_t gpr_mgpu_launch_count(gpr_mgpu* mg);
/* GPRModel(cov, hp, x, y; train_axis): src/models.jl:17-37; x and y are replicated on every rank */
int gpr_mgpu_model_create(gpr_mgpu* mg, const int* comp_types, int ncomp, int D, int64_t N, const double* x,
                          const double* y, int ny, int train_axis, gpr_mgpu_model** model);
int gpr_mgpu_model_destroy(gpr_mgpu_model* model);
/* loss_grad! / log_loss_grad!: src/cost.jl:50-70 (same contract as gpr_nlml_grad) */
int gpr_mgpu_nlml_grad(gpr_mgpu_model* model, const double* hp_in, int P, int log_scale, double eps, double* F,
                       double* G, int64_t* info);
/* update_cache!(pc, md) of a predict cache on the multi-GPU model (src/predict.jl:29-34): covariance, potrf, trtri, lauum
 * (K^-1 block-cyclic), K^-1 Y for all ny columns; no gradient reduction.  Collective; same contract and info as gpr_update_cache. */
int gpr_mgpu_update_cache(gpr_mgpu_model* model, const double* hp, int P, double eps, int64_t* info);
/* predict_mean! / predict! (src/predict.jl:36-102) from the K^-1 left by the last gpr_mgpu_update_cache, or by a
 * gpr_mgpu_nlml_grad call with G != NULL, at that call's hp and eps.  GPR_ERR_STATE if there is none (no evaluation yet,
 * loss-only evaluation, failed factorization).  Arguments and outputs exactly as gpr_predict (mean M x ny, var_diag and
 * cov_full nullable, same_x = the reference's xp === md.x).  Collective: under gpr_dist_create every process passes the
 * same xp and receives the same outputs.
 * No triangular solve: with Uu the upper triangle of K^-1 (diagonal included) every rank forms T = K(x, xp)^T Uu for its
 * own block columns, the variance is the quadratic form of K^-1 = Uu + Uu^T - diag(K^-1), and one sum of
 * M (ny + 1) doubles (+ M^2 for cov_full) over the ranks finishes a tile.  Test points go in tiles of "predict_tile"
 * (gpr_mgpu_set_option, default 16384), halved while a tile does not fit (GPR_ERR_MEMORY below 128 points); cov_full
 * takes all M points in one tile.  Timings (gpr_mgpu_timings): PRED_KSTAR = K(x, xp) build on every rank, PRED_TRSM =
 * the products, PRED_ROWNORM = the fix-up / row-dot kernel, PRED_MEAN = the sum over the ranks and the download. */
int gpr_mgpu_predict(gpr_mgpu_model* model, const double* xp, int64_t M, int same_x, double* mean, double* var_diag,
                     double* cov_full);
/* integrate!(Iout, var_Iout, md, hp, a, b, nothing, wc, ac) (src/integrate.jl:56-62,103-143) for nbox boxes at once on the
 * multi-GPU model, from the K^-1 of gpr_mgpu_predict (same preconditions: GPR_ERR_STATE unless predict-ready, at that
 * factorization's hp and eps).  a, b: D x nbox (box i is column i).  Iout: nbox x ny, box index fastest (the layout of the
 * gpr_mgpu_predict mean; for nbox = 1 gpr_integrate's Iout[ny]), Iout[i + e nbox] = Y[:, e]^T K^-1 k1_i.  var_out: NULL or
 * nbox entries, var_i = k2_i - k1_i^T K^-1 k1_i, not clamped.  As gpr_integrate, k1 = antideriv!(SquaredExp(), x, hp, a, b)
 * (:15-31) and k2 = antideriv2 (:33-41) read hp[1..D+1] of the first component whatever the others are;
 * GPR_ERR_UNSUPPORTED unless that component is a SquaredExp.  GPR_ERR_ARG for NULL a, b, Iout or nbox < 1.
 * Collective like gpr_mgpu_predict: under gpr_dist_create every process passes the same boxes and receives the same outputs.
 * The boxes are the test points of gpr_mgpu_predict with k1 in place of K(x, xp): tiles of "predict_tile" boxes (halved while
 * they do not fit, GPR_ERR_MEMORY below 128), each one pass over every rank's K^-1 columns, so many boxes per call cost
 * about as much as one.  Timings: PRED_KSTAR = the k1 tile build, PRED_TRSM = the products, PRED_ROWNORM = the fix-up,
 * PRED_MEAN = the sum over the ranks and the download. */
int gpr_mgpu_integrate(gpr_mgpu_model* model, int64_t nbox, const double* a, const double* b, double* Iout, double* var_out);
/* predict_mean! / predict!(mu, Sigma::Diagonal, md, Cmap(+, xe, xq), pc) (src/split_predict.jl:5-53) on the multi-GPU model.
 * Arguments and outputs exactly as gpr_split_predict (mean ne x nq, e fastest; var nullable, ne*nq entries, q fastest within e;
 * rows e in [e_lo, e_hi] get the posterior variance, all others keep the prior; e_lo = e_hi + 1: no variance rows); the
 * preconditions of gpr_mgpu_predict (GPR_ERR_STATE unless predict-ready, at that factorization's hp and eps), GPR_ERR_UNSUPPORTED
 * for ny != 1.  Collective like gpr_mgpu_predict.
 * Mean: nothing in mu = sum_k A_k .* (B_k diag(alpha) C_k) touches K^-1 and every rank holds x and alpha, so the q columns are
 * sharded: a chunk of q columns is cut into one slab of whole 128-column tiles per rank, every rank builds B^T for all e rows
 * and A, diag(alpha) C for its slab and runs the Hadamard-epilogue products of gpr_split_predict, and one sum over the ranks
 * (zeros outside each slab) assembles the chunk.  Slabs hold at most "predict_tile" columns and are halved while they do not
 * fit (GPR_ERR_MEMORY below 128).  With "ozaki" = 0 the mean does not depend on the number of ranks, the transport or the slab
 * width.  Variance rows: ordinary test points through the quadratic form of gpr_mgpu_predict, in tiles of at most
 * "predict_tile" points (whole rows e when one fits, else a slab of a row's q columns), halved while they do not fit.
 * Timings: SPLIT_BUILD / SPLIT_GEMM / SPLIT_D2H (incl. the sum over the ranks) for the mean, PRED_KSTAR / PRED_TRSM /
 * PRED_ROWNORM / PRED_MEAN for the variance rows as in gpr_mgpu_predict. */
int gpr_mgpu_split_predict(gpr_mgpu_model* model, const double* xe, int64_t ne, const double* xq, int64_t nq, int64_t e_lo,
                           int64_t e_hi, double* mean, double* var);
/* GPR_FETCH_ALPHA (N) or GPR_FETCH_KINV (N x N full symmetric; after an evaluation with G != NULL) */
int gpr_mgpu_fetch(gpr_mgpu_model* model, int which, double* out);
int gpr_mgpu_timings(gpr_mgpu_model* model, double* ms, int n);   /* GPR_T_* slots; POTRS = alpha extraction + broadcast */
/* diagnostics: block-cyclic factorization of a host SPD matrix A (N x N, upper triangle referenced; the strict
 * lower triangle comes back zero) with right-hand sides Y (N x ny; NULL with ny = 0).
 * mode 0: potrf (upper(A) <- U, Y <- U^-T Y), 1: + trtri (upper(A) <- U^-1, Y <- -A^-1 Y), 2: + lauum (upper(A) <- A^-1).
 * ms[0..2]: potrf / trtri / lauum milliseconds. */
int gpr_mgpu_dbg_factor(gpr_mgpu* mg, double* A, int64_t N, double* Y, int ny, int mode, int64_t* info, double* ms);

#ifdef __cplusplus
}
#endif
#endif /* GPR_SM100A_H */
