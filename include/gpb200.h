/*
 * gpb200.h -- C ABI of libgpb200.so: the B200-native exact-GP hot path behind the
 * GaussianProcesses.jl `CovarianceStrategy` seam.
 *
 * There is no FFI in the reference (pure Julia); the boundary this library slots into is the
 * reference's own strategy-dispatch API (src/GP.jl:10 `abstract type CovarianceStrategy`).  Each
 * entry point below names the reference method (file:line under /root/reference) it replaces;
 * INTEGRATION.md shows the Julia `ccall` shim (`B200Covariance <: CovarianceStrategy`) and the
 * Python ctypes binding that drive exactly these symbols.
 *
 * Conventions
 *   - all matrices FP64.  `x` is Julia's d x N column-major Matrix{Float64} (== N x d row-major,
 *     one observation per column), passed with its leading dimension `ldx` (>= d).
 *   - caller owns every host buffer for the duration of the call only; the library owns all
 *     device memory behind the opaque handle.  Calls are synchronous.
 *   - return value: 0 OK;  k > 0 = LAPACK-style "leading minor k is not positive definite"
 *     (shim throws LinearAlgebra.PosDefException(k), cf. src/GP.jl:110, src/optimize.jl:46-61);
 *     GPB200_EINVAL (<0) invalid argument (-> ArgumentError);  GPB200_ECUDA / GPB200_ENCCL
 *     runtime failure, message via gpb200_last_error().  A failed factorisation leaves the
 *     handle reusable with new hyper-parameters.
 *   - one handle must not be used from two threads at once; distinct handles may be.
 *   - there is NO CPU fallback: without a CUDA device gpb200_create fails with GPB200_ECUDA.
 */
#ifndef GPB200_H
#define GPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpb200_handle gpb200_handle;

#define GPB200_OK        0
#define GPB200_EINVAL   (-1)
#define GPB200_ECUDA    (-2)
#define GPB200_ENCCL    (-3)
#define GPB200_ESTATE   (-4)   /* call order violated (e.g. solve before factorize) */

/* ---- kernel program: post-order (RPN) list of ops; 6 int32 per op ------------------------
 *   {opcode, theta_off, n_theta, dims_off, n_dims, extra}
 * leaves read theta[theta_off .. theta_off+n_theta) (log-scale, exactly get_params(kernel) order,
 * src/kernels/pair_kernel.jl:15, src/common.jl:98-104) and the active input dimensions
 * dims[dims_off .. dims_off+n_dims) (0-based; `Masked`, src/kernels/masked_kernel.jl:23, is
 * resolved into this list by the shim).  `extra` = polynomial degree for GPB200_OP_POLY.
 * SUM / PROD pop two values (src/kernels/sum_kernel.jl:15-16, prod_kernel.jl:14-15).
 * FixedKernel (src/kernels/fixed_kernel.jl:64-69) is resolved in the shim: pass the full
 * parameter vector of the wrapped kernel, select gradient entries `free` on the host.        */
#define GPB200_OP_SE_ISO     1   /* src/kernels/se_iso.jl:39-50     theta = [ll, lsigma]          */
#define GPB200_OP_SE_ARD     2   /* src/kernels/se_ard.jl:43-50     theta = [ll_1..ll_nd, lsigma] */
#define GPB200_OP_MAT12_ISO  3   /* src/kernels/mat12_iso.jl:41-43                                */
#define GPB200_OP_MAT32_ISO  4   /* src/kernels/mat32_iso.jl:41-45                                */
#define GPB200_OP_MAT52_ISO  5   /* src/kernels/mat52_iso.jl:40-44                                */
#define GPB200_OP_MAT12_ARD  6   /* src/kernels/mat12_ard.jl:43-45, mat.jl:5-18                   */
#define GPB200_OP_MAT32_ARD  7   /* src/kernels/mat32_ard.jl:43-46                                */
#define GPB200_OP_MAT52_ARD  8   /* src/kernels/mat52_ard.jl:43-47                                */
#define GPB200_OP_RQ_ISO     9   /* src/kernels/rq_iso.jl:44-52     theta = [ll, lsigma, lalpha]  */
#define GPB200_OP_RQ_ARD    10   /* src/kernels/rq_ard.jl:47-54     theta = [ll.., lsigma, lalpha]*/
#define GPB200_OP_PERIODIC  11   /* src/kernels/periodic.jl:45-51   theta = [ll, lsigma, lp]      */
#define GPB200_OP_LIN_ISO   12   /* src/kernels/lin_iso.jl:42,71    theta = [ll]                  */
#define GPB200_OP_LIN_ARD   13   /* src/kernels/lin_ard.jl:69-92    theta = [ll_1..ll_nd]         */
#define GPB200_OP_POLY      14   /* src/kernels/poly.jl:44,69-70    theta = [lc, lsigma]          */
#define GPB200_OP_NOISE     15   /* src/kernels/noise.jl:31-52      theta = [lsigma]              */
#define GPB200_OP_CONST     16   /* src/kernels/const.jl:41         theta = [lsigma]              */
#define GPB200_OP_SUM       32
#define GPB200_OP_PROD      33

#define GPB200_MAX_OPS     16
#define GPB200_MAX_THETA   96
#define GPB200_MAX_DIMS   128
#define GPB200_OP_STRIDE    6

/* ---- lifetime ------------------------------------------------------------------------- */
/* replaces alloc_cK(covstrat, nobs) (src/GP.jl:14-20): creates the engine on CUDA device
 * `device`; device buffers are sized at gpb200_set_data.                                   */
int  gpb200_create(gpb200_handle** out, int device);
/* Julia finalizer on B200PDMat */
void gpb200_destroy(gpb200_handle* h);
/* message of the last failure on this handle (h == NULL: last create failure) */
const char* gpb200_last_error(gpb200_handle* h);
int  gpb200_version(void);

/* ---- data + model ---------------------------------------------------------------------- */
/* GPE ctor / fit! (src/GPE.jl:63-69, 128-136): upload the d x N inputs once; hyper-parameter
 * independent.  No N x N distance matrix is precomputed (cf. IsotropicData,
 * src/kernels/stationary.jl:34-40): distances are recomputed from x inside the Gram kernel. */
int  gpb200_set_data(gpb200_handle* h, int64_t N, int32_t d, const double* x, int64_t ldx);
/* flattened kernel tree (see opcodes above) */
int  gpb200_set_kernel(gpb200_handle* h, int32_t n_ops, const int32_t* ops,
                       int32_t n_dims, const int32_t* dims, int32_t n_theta);

/* ---- update_cK! (src/GPE.jl:169-186) + make_posdef! (src/GP.jl:101-112) ------------------
 * Gram build cov!(...) (src/kernels/kernels.jl:39-50) with K_ii += exp(2*log_noise) (n_noise==1)
 * or += exp(2*log_noise[i]) (n_noise==N), plus `extra_nugget`, then the Cholesky factorisation.
 * Returns k>0 if the leading minor k is not positive definite.                              */
int  gpb200_factorize(gpb200_handle* h, const double* theta, const double* log_noise,
                      int64_t n_noise, double extra_nugget);
/* logdet(cK) (src/GPE.jl:210; PDMats: 2*sum(log(diag(U)))) */
int  gpb200_logdet(gpb200_handle* h, double* logdet);
/* cK \ rhs (src/GPE.jl:208; PDMats `\` == dpotrs): out = K_y^-1 rhs, both length N on host */
int  gpb200_solve(gpb200_handle* h, const double* rhs, double* out);
/* update_mll! body (src/GPE.jl:206-210): alpha = K_y^-1 r, mll = -(r'alpha + logdet + N log 2pi)/2;
 * alpha stays resident on the device for grad/predict.                                      */
int  gpb200_mll(gpb200_handle* h, const double* y_minus_mean, double* alpha, double* mll);

/* ---- gradient -------------------------------------------------------------------------- */
/* precompute!(precomp, gp) -> get_ααinvcKI! (src/GPE.jl:151-164, 262-264): builds K_y^-1 from
 * the factor (triangular inverse + W'W, N^3*2/3 flop instead of the reference's 2N^3 potrs on
 * the identity).  The factor is kept: predict after grad needs no refactorisation.           */
int  gpb200_grad_prepare(gpb200_handle* h);
/* dmll_kern! (src/GPE.jl:219-241) + dmll_noise's tr(A) (src/GPE.jl:273-275), fused:
 * dmll_kernel[p] = 1/2 sum_ij A_ij dK_ij/dtheta_p, A = alpha alpha' - K_y^-1;  *trA = tr(A).
 * `alpha` may be NULL to use the alpha left resident by gpb200_mll.                          */
int  gpb200_grad_kernel(gpb200_handle* h, const double* alpha, double* dmll_kernel, double* trA);

/* ---- latent-variable GP (src/GPA.jl; single-GPU handles, after gpb200_factorize) -------------------------------------
 * GPA whitens the latent values, f = L v + mu with K = L L' (the shim factorises with logNoise = -20, GPA.jl:111-114).
 * Multi-rank handles (replicated or row-sharded) return GPB200_EINVAL.                                                 */
/* unwhiten(cK, v) (GPA.jl:106,125,159): f = L v, both length N on host                                                 */
int  gpb200_unwhiten(gpb200_handle* h, const double* v, double* f);
/* update_dll! (GPA.jl:183-228), process and kernel blocks: dll_v[N] = L' dl_df (may be NULL; GPA.jl:200) and
 * dll_kernel[n_theta] = dll_kern! (GPA.jl:164-173: chol_unblocked_rev! on tril(dl_df v'), diagonal doubled, dmll_kern!),
 * computed in closed form: 1/2 sum_ij (P + P')_ij dK_ij/dtheta_p with P = W' Phi(w v') W, W = L^-1, w = L' dl_df,
 * Phi = lower triangle with the diagonal halved.  G no longer holds K^-1 afterwards: gpb200_grad_kernel, the
 * cross-validation calls and gpb200_get_inverse(_diag) return GPB200_ESTATE until gpb200_grad_prepare runs again, and
 * the resident alpha is cleared (pass alpha explicitly to gpb200_predict).  solve, logdet, predict and unwhiten keep
 * working on the unchanged factor.                                                                                     */
int  gpb200_gpa_grad(gpb200_handle* h, const double* v, const double* dl_df, double* dll_v, double* dll_kernel);
/* debug: the N x N symmetric P + P' of the last gpb200_gpa_grad (row-major)                                           */
int  gpb200_get_chol_bar(gpb200_handle* h, double* out);

/* ---- predictMVN / predict_f (src/GP.jl:25-79) ---------------------------------------------
 * xs: d x M column-major test inputs (leading dim ldxs).  mu_minus_mean[M] = K*' alpha;
 * var[M] (may be NULL) = k** - |L^-1 k*|^2, NOT clamped (the shim applies max(.,0) as
 * src/GP.jl:75 does only on the diagonal path); cov[M*M] (may be NULL) = K** - V'V, symmetric.
 * Batched: one cross-Gram + one blocked triangular solve for all M points (the reference loops
 * over test points, src/GP.jl:72-76).                                                       */
int  gpb200_predict(gpb200_handle* h, int64_t M, const double* xs, int64_t ldxs,
                    const double* alpha, double* mu_minus_mean, double* var, double* cov);

/* rand(gp, X, n) (src/GP.jl:120-146): n posterior draws at the M test points, on the device: predictMVN's full covariance,
 * make_posdef!(Sigma; nugget) (Cholesky of the M x M matrix), unwhiten!(Sigma, Z) and + mu.  z and samples are M x nsamp
 * column-major (Julia `randn(M, n)` / the returned matrix); mu_minus_mean[M] as in gpb200_predict (the shim adds mean(x*) to
 * it and to every draw).  Returns k > 0 if Sigma + nugget I is not positive definite (PosDefException).               */
int  gpb200_rand(gpb200_handle* h, int64_t M, const double* xs, int64_t ldxs, const double* alpha, int64_t nsamp,
                 const double* z, double nugget, double* mu_minus_mean, double* samples);

/* append!(gp::ElasticGPE, x, y) (src/GPEelastic.jl:13-22): k more observations (xnew: d x k column-major) with UNCHANGED
 * hyper-parameters; the factor is extended in place (rows from the first touched tile on are rebuilt: O(k N^2)), alpha / mll are
 * then refreshed with gpb200_mll on the longer y.  Needs room reserved by option "capacity" (ElasticGPE's capacity) before
 * gpb200_set_data; GPB200_EINVAL when the capacity is exceeded (the shim refits, like ElasticPDMats.resize!).             */
int  gpb200_append(gpb200_handle* h, int64_t k, const double* xnew, int64_t ldx);

/* ---- cross-validation on the resident inverse (src/crossvalidation.jl; after gpb200_grad_prepare, single GPU) ------------
 * Per hyper-parameter the reference forms Z_j = inv(Sigma) dK_j and Z_j inv(Sigma) as host matrices (crossvalidation.jl:86-108,
 * 270-283).  gpb200_cv_param does the two N^3 products on the device and returns the two vectors the LOO formulas need:
 * Zj_alpha[N] = Z_j alpha and diag_ZjSinv[N] = diag(Z_j inv(Sigma)); `param` indexes the kernel's full parameter vector, -1 is the
 * noise variance (Z = inv(Sigma), crossvalidation.jl:124-126).  M_j = Z_j inv(Sigma) stays resident for gpb200_cv_block.        */
int  gpb200_cv_param(gpb200_handle* h, int32_t param, const double* alpha, double* Zj_alpha, double* diag_ZjSinv);
/* principal sub-matrix on the index set idx[nV] (0-based) of inv(Sigma) (which = 0) or of the last M_j (which = 1), row-major
 * nV x nV: `Matrix(invΣ)[V,V]` / `ZjΣinv[V,V]` of predict_CVfold / gradient_fold (crossvalidation.jl:180-191, 248-262)     */
int  gpb200_cv_block(gpb200_handle* h, int32_t which, int64_t nV, const int64_t* idx, double* out);

/* ---- debug / introspection (Base.Matrix(::P), mat(::P), tests) ----------------------------- */
int  gpb200_get_gram(gpb200_handle* h, double* K);        /* N x N, K_y rebuilt from x, theta   */
int  gpb200_get_factor(gpb200_handle* h, double* U);      /* N x N column-major upper U, K_y=U'U */
int  gpb200_get_inverse(gpb200_handle* h, double* Kinv);  /* N x N, after gpb200_grad_prepare    */
/* diag(K_y^-1)[N] after gpb200_grad_prepare: all predict_LOO / logp_LOO need besides alpha
 * (src/crossvalidation.jl:8-13, 37-49: sigma_i^2 = 1/[K^-1]_ii, mu_i = y_i - alpha_i sigma_i^2)  */
int  gpb200_get_inverse_diag(gpb200_handle* h, double* diag);
/* per-phase device times (ms) of the last calls:
 * [0] gram  [1] cholesky  [2] solve+mll  [3] inverse (trtri+lauum)  [4] trace  [5] predict
 * with option "profile"=1, accumulated since the option was set:
 * [6] number of DMMA GEMM launches  [7] sum of their device durations (ms, CUDA events around
 * every launch)  [8] FP64 flops those launches executed (tile-granular)
 * of the last gpb200_unwhiten / gpb200_gpa_grad: [9] L v  [10] L' g  [11] inverse merges  [12] row scan
 * [13] the two GEMMs of P + P'  (the trace of gpb200_gpa_grad goes to [4]); up to n = 16 values    */
int  gpb200_get_timings(gpb200_handle* h, double* ms, int32_t n);
/* number of kernel launches issued by this handle since creation */
int64_t gpb200_launch_count(gpb200_handle* h);
/* tuning knobs (string key):
 *   "nb"         outer Cholesky block: 0 (default) = fully recursive, else 128*2^k <= 4096 (right-looking panels)
 *   "gemm"       0 = TMA/mbarrier DMMA kernel (default), 1 = simple-loader kernel (bring-up / cross-check)
 *   "lookahead"  1 (default) = next diagonal tile factored on a side stream behind the Schur update
 *   "trsv_fused" single-launch flag-synchronised triangular solves: 2 (default) = critical tiles resident in registers / shared
 *                memory, 1 = round-1 kernels (L2 prefetch only), 0 = one launch per block step
 *   "profile"    1 = CUDA events around every GEMM launch (see gpb200_get_timings)
 *   "dist_nb"    multi-GPU: width of an owned block column, 0 = auto (~N/(8*ranks))
 *   "p2p"        multi-GPU: 1 = fused panel push over peer memory (after gpb200_ipc_import), 0 = NCCL broadcast
 *   "gram_fast"  1 (default) = TMA-staged SEIso Gram / trace kernels (gram_fast.cu) when the kernel is one SEIso leaf over
 *                <= 8 dimensions, 0 = always the generic kernel-program kernels (cross-check)
 *   "leaf"       1 (default) = blocked 128 x 128 diagonal-tile kernel (16-column panels, 74.5 us), 0 = column-per-barrier kernel
 *                (123 us; cross-check); process-wide
 *   "capacity"   rows reserved by the next gpb200_set_data (>= N) so that gpb200_append can extend the factor in place
 *   "shard"      multi-GPU storage of the two N x N buffers: 1 = row-sharded (each rank maps only its own block rows),
 *                0 = replicated, -1 (default) = sharded only when the replicated form would not fit the device
 *   "shard_la"   1 (default) = look-ahead schedules of the row-sharded Cholesky / inverse (panel chain on a side stream),
 *                0 = the plain one-stream schedules (cross-check)
 *   "shard_rb"   row-sharded ownership block in 128-row tiles (panel width 128*rb): 0 auto, 1, 2, 4, 8
 * Returns GPB200_EINVAL for unknown keys or values.                                           */
int  gpb200_set_option(gpb200_handle* h, const char* key, int64_t value);

/* run all work of this handle on the caller's CUDA stream (cudaStream_t; NULL = a private
 * stream again), so that the caller's events bracket it (bench.py: torch.cuda.Event).         */
int  gpb200_set_stream(gpb200_handle* h, void* cuda_stream);
/* FP64 roofline denominators measured on this device: DMMA.8x8x4 (mma.sync f64, the FP64 tensor
 * path on sm_100a) and DFMA issue rates, TFLOP/s.                                             */
int  gpb200_fp64_peak(gpb200_handle* h, double* tflops_dmma, double* tflops_dfma);

/* ---- raw kernels exposed for the parity tests and the roofline bench ----------------------
 * C[M x N] = alpha * A[M x K] * B[N x K]' + beta * C   (all row-major, device pointers,
 * M,N multiples of 128, K multiple of 16, leading dims multiples of 2); runs the same DMMA
 * kernel the factorisation uses.  `impl` 0 = TMA/mbarrier kernel, 1 = simple kernel.
 * Returns the device time of `reps` launches in *ms (reps>=1).                               */
int  gpb200_dgemm_nt_device(gpb200_handle* h, int impl, int64_t M, int64_t N, int64_t K,
                            double alpha, const double* dA, int64_t lda,
                            const double* dB, int64_t ldb, double beta,
                            double* dC, int64_t ldc, int lower_only, int reps, double* ms);

/* ---- multi-GPU (one process per GPU; NCCL over NVLink) -------------------------------------- */
/* rank 0 obtains a 128-byte NCCL unique id, the host side broadcasts it (torch.distributed /
 * Julia Distributed), every rank then joins.                                                */
int  gpb200_nccl_unique_id(char* id128);
int  gpb200_comm_init(gpb200_handle* h, int nranks, int rank, const char* id128);
/* Fused panel broadcast over NVLink peer memory (optional, after comm_init and set_data): every rank
 * exports CUDA-IPC handles of its factor buffers (GPB200_IPC_BYTES bytes), the host layer all-gathers
 * the blobs (rank order) and every rank imports them.  From then on the kernels that PRODUCE a panel
 * (tile leaf, 128-wide TRSM GEMM) store it straight into all peers' buffers and raise a device-side
 * flag; NCCL stays on the small collectives only.  Re-export after a gpb200_set_data that changes N. */
#define GPB200_IPC_BYTES 512
int  gpb200_ipc_export(gpb200_handle* h, char* out);
int  gpb200_ipc_import(gpb200_handle* h, int nranks, const char* all_blobs);

/* In-process group of `n` (<= 8) handles on ONE device acting as n ranks of the ROW-SHARDED schedules (the storage
 * layout of config C4: each rank keeps only its own block rows of the N x N factor / inverse; see csrc/shard_impl.cuh).
 * Collectives become event-ordered device copies, so a single-GPU box exercises exactly the multi-rank code.  Every
 * handle needs the same gpb200_set_data / gpb200_set_kernel; factorize / mll / solve / grad_* / predict are then called
 * on hs[0] only.  (One process per GPU uses gpb200_comm_init instead and option "shard".)                       */
int  gpb200_group_create(gpb200_handle** hs, int n);
/* storage of the two N x N buffers of this handle: out[0] = 1 if row-sharded, out[1] / out[2] = bytes of F / G physically
 * backed on this device, out[3] = ownership block (tiles), out[4] = ranks, out[5] = rank, out[6] = 1 if the GEMMs run on
 * TMA descriptors (0: plain-load fallback)  (cf. test/memory.jl:14-19)                                              */
int  gpb200_storage_info(gpb200_handle* h, int64_t* out, int32_t n);

/* ---- sparse FITC strategy (src/sparse/fully_indep_train_conditional.jl) ------------------------
 * FITC(x, Xu, y, mean, kern, logNoise) (fitc.jl:335-338) == GPE(..., FullyIndepStrat(Xu)).
 * Covers update_cK!(::FullyIndepPDMat) (fitc.jl:134-156), `\` (fitc.jl:33-36), logdet (fitc.jl:77),
 * dmll_noise (fitc.jl:243-257), get_alpha_u (fitc.jl:279-286) and predictMVN (fitc.jl:324-332 ->
 * determ_train_conditional.jl:41-59 -> subsetofregressors.jl:302-321) and the kernel-parameter
 * gradient dmll_kern! (fitc.jl:200-234 on top of subsetofregressors.jl:140-151, 219-253).
 * N is streamed in chunks; only M x M matrices and O(N) vectors persist on the device.          */
typedef struct gpb200_fitc gpb200_fitc;
int  gpb200_fitc_create(gpb200_fitc** out, int device);
void gpb200_fitc_destroy(gpb200_fitc* f);
const char* gpb200_fitc_last_error(gpb200_fitc* f);
/* multi-GPU (one process per GPU): after gpb200_nccl_unique_id / broadcast of the id, every rank joins; each rank then passes
 * ITS OWN slice of the observations to gpb200_fitc_set_data / _mll (alpha is returned for that slice) and the same inducing points
 * and hyper-parameters.  Exchanged over NCCL: one all-reduce of the M x M accumulator Sigma_QR per factorisation (0.54 GB at
 * M = 8192), one of H per kernel gradient, M-vectors and scalars; K_uu / Sigma_QR factorisations and predictions are replicated. */
int  gpb200_fitc_comm_init(gpb200_fitc* f, int nranks, int rank, const char* id128);
/* x: d x N training inputs, xu: d x M inducing inputs (both column-major, one point per column) */
int  gpb200_fitc_set_data(gpb200_fitc* f, int64_t N, int32_t d, const double* x, int64_t ldx,
                          int64_t M, const double* xu, int64_t ldxu);
int  gpb200_fitc_set_kernel(gpb200_fitc* f, int32_t n_ops, const int32_t* ops, int32_t n_dims,
                            const int32_t* dims, int32_t n_theta);
/* update_cK!: K_uu (+1e-10 I), Lambda, Sigma_QR (+1e-10 I) and both Cholesky factors */
int  gpb200_fitc_factorize(gpb200_fitc* f, const double* theta, double log_noise);
/* alpha = Sigma^-1 r, logdet(Sigma), mll = -(r'alpha + logdet + N log 2pi)/2 */
int  gpb200_fitc_mll(gpb200_fitc* f, const double* y_minus_mean, double* alpha, double* mll, double* logdet);
int  gpb200_fitc_grad_noise(gpb200_fitc* f, double* dmll_noise);
/* dmll_kernel[n_theta], full parameter vector of the un-fixed kernel tree (as gpb200_grad_kernel) */
int  gpb200_fitc_grad_kernel(gpb200_fitc* f, double* dmll_kernel);
/* mu_minus_mean[Ms], var[Ms] (may be NULL; not clamped) */
int  gpb200_fitc_predict(gpb200_fitc* f, int64_t Ms, const double* xs, int64_t ldxs, double* mu_minus_mean, double* var);
/* predictMVN with the full covariance cov[Ms x Ms] (fitc.jl:324-332, dtc.jl:41-59, sor.jl:302-321); Ms <= 32768 */
int  gpb200_fitc_predict_cov(gpb200_fitc* f, int64_t Ms, const double* xs, int64_t ldxs, double* mu_minus_mean, double* cov);
/* 0 = FITC (default), 1 = DTC (src/sparse/determ_train_conditional.jl), 2 = SoR
 * (src/sparse/subsetofregressors.jl): the two share Lambda = sigma^2 I (sor.jl:96-106, `\` sor.jl:50,
 * logdet sor.jl:53, dmll_noise sor.jl:159-166, dmll_kern! sor.jl:219-253); SoR's predictive covariance is
 * K_xu S^-1 K_ux (sor.jl:302-321), DTC's adds K_xx - Q_xx (dtc.jl:41-59).                         */
int  gpb200_fitc_set_mode(gpb200_fitc* f, int mode);
int64_t gpb200_fitc_launch_count(gpb200_fitc* f);

#ifdef __cplusplus
}
#endif
#endif /* GPB200_H */
