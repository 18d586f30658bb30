/* gpx.h — C ABI of the B200-native exact-GP engine (libgpx.so).
 *
 * This is the drop-in boundary for ONE hot path of SheffieldML/GPy:
 *     GPRegression -> GP.parameters_changed -> ExactGaussianInference.inference -> Kern.K/Kdiag/update_gradients_full
 * Each entry point names the reference interface it replaces (paths relative to the GPy repository root).
 * Plain C: pointers and sizes only, no torch / numpy types. All inputs, outputs and stored matrices are IEEE fp64; the N^3
 * products run on fp64 tensor instructions (DMMA) or, from N = 8192 on one GPU, as int8 digit-split products on the tcgen05
 * tensor cores whose exact s32 sums are recombined in fp64 (8 digits for the Cholesky part, 7 for the inverse part:
 * |dLML| <= 1e-8 and 1e-6 relative on gradients against the reference, DESIGN.md section 5.1; option "ozaki" selects).
 *
 * Conventions
 *   - Return value: 0 ok; >0 "matrix not positive definite, leading minor <ret>" (the caller raises
 *     numpy.linalg.LinAlgError as GPy/util/linalg.py:64,75 does); <0 CUDA / argument error, text via gpx_last_error().
 *   - Host buffers are caller-owned and only read/written during the call. Device state lives behind gpx_ctx.
 *   - Matrices returned to the host are column-major (Fortran order) N x N unless stated, which is the layout
 *     LAPACK hands GPy (GPy/util/linalg.py:31-38 force_F_ordered); symmetric results are fully populated.
 *   - kind: 0 RBF (GPy/kern/src/rbf.py:51-52,177-178), 1 Exponential (stationary.py:382-386),
 *           2 Matern32 (stationary.py:488-492), 3 Matern52 (stationary.py:585-589).
 *   - ard:  0 -> `lengthscale` points at 1 double; 1 -> at D doubles (stationary.py:64-79).
 *   - Gradient vector order is paramz's: [kern.variance, kern.lengthscale (1 or D), Gaussian_noise.variance]
 *     (link order stationary.py:81, GPy/core/gp.py:106-107).
 */
#ifndef GPX_H_
#define GPX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpx_ctx gpx_ctx;

enum { GPX_RBF = 0, GPX_EXPONENTIAL = 1, GPX_MATERN32 = 2, GPX_MATERN52 = 3,
       GPX_WHITE = 4, GPX_BIAS = 5, /* static parts of a composite kernel only (GPy/kern/src/static.py:63-99,142-185) */
       GPX_COREGIONALIZE = 6        /* coregionalization part, gpx_exact_eval_coreg only (GPy/kern/src/coregionalize.py:82-137) */ };

/* gpx_get selectors */
enum {
  GPX_GET_L = 0,     /* woodbury_chol: lower Cholesky factor of K + (noise+jitter) I, N x N col-major, zeros above diag
                        (GPy/inference/latent_function_inference/exact_gaussian_inference.py:58,74) */
  GPX_GET_ALPHA = 1, /* woodbury_vector alpha = Ky^-1 Y, N x P row-major (exact_gaussian_inference.py:60) */
  GPX_GET_KINV = 2,  /* Wi = Ky^-1, symmetric N x N (GPy/util/linalg.py:210-212) */
  GPX_GET_DLDK = 3,  /* dL_dK = 0.5 (alpha alpha^T - P Ky^-1), symmetric N x N (exact_gaussian_inference.py:70) */
  GPX_GET_K = 4,     /* noise-free K(X,X), symmetric N x N (exact_gaussian_inference.py:53) */
  GPX_GET_LINV = 5   /* L^-1 lower, N x N col-major (GPy/util/linalg.py:209 dtrtri; unused by the exact-GP caller) */
};

/* Library / device ----------------------------------------------------------------------------------------------- */
const char* gpx_last_error(void);      /* thread-local text of the last <0 return */
const char* gpx_version(void);
int gpx_device_count(void);            /* number of visible CUDA devices, <0 on error */

/* One context per model: owns the stream(s), the N x N workspace and (multi-GPU) the NCCL communicator. */
int gpx_create(int device, gpx_ctx** out);
int gpx_destroy(gpx_ctx* ctx);

/* Replaces Kern._slice_X + ObsAr wiring (GPy/kern/src/kern.py:112-117, GPy/core/gp.py:42-62): host X (N x D, row-major,
 * already sliced to active dims) and Y (N x P row-major) are copied to HBM once per (X, Y) identity. */
int gpx_set_data(gpx_ctx* ctx, const double* X, int64_t N, int D, const double* Y, int P);

/* The hot call. Replaces, fused: Stationary.K (stationary.py:105-168) -> diag.add (exact_gaussian_inference.py:55-56)
 * -> pdinv/jitchol/dpotri (GPy/util/linalg.py:56-75,193-214) -> dpotrs (:116-125) -> log marginal + dL_dK
 * (exact_gaussian_inference.py:62-72) -> Stationary.update_gradients_full (stationary.py:193-243, incl.
 * stationary_cython.pyx:53-62) -> Gaussian.exact_inference_gradients (GPy/likelihoods/gaussian.py:78-79).
 *   jitter     : added unconditionally to the diagonal (the reference uses 1e-8, exact_gaussian_inference.py:56)
 *   max_tries  : jitchol ladder length (reference: 5). On a non-PD factorisation the diagonal gets
 *                mean(diag)*1e-6*10^k, k = 0..max_tries-1 (linalg.py:66-74); *jitter_used reports the extra jitter.
 *   lml        : out, log marginal likelihood;  grad: out, (1 + (ard?D:1) + 1) doubles. */
int gpx_exact_eval(gpx_ctx* ctx, int kind, int ard, double variance, const double* lengthscale, double noise,
                   double jitter, int max_tries, double* lml, double* grad, double* jitter_used);

/* The same evaluation with one noise variance PER DATA POINT (HeteroscedasticGaussian, GPy/likelihoods/gaussian.py:347-362;
 * GPy/models/gp_heteroscedastic_regression.py:10-37): Ky = K + diag(noise_variances + jitter)
 * (exact_gaussian_inference.py:55-56 with a vector `variance`), and dL_dthetaL = diag(dL_dK) per point
 * (gaussian.py:358-359 applied to exact_gaussian_inference.py:72) written to dnoise (N doubles) by the fused K^-1
 * epilogue. grad keeps the layout of gpx_exact_eval; its last entry is the sum of dnoise. Single-GPU. */
int gpx_exact_eval_het(gpx_ctx* ctx, int kind, int ard, double variance, const double* lengthscale,
                       const double* noise_variances, double jitter, int max_tries, double* lml, double* grad,
                       double* dnoise, double* jitter_used);

/* Composite kernels on the fused path: K = sum over terms of products of parts (GPy/kern/src/add.py:60-99 Add.K /
 * update_gradients_full; prod.py:59-68,377-396 Prod.K, where every factor's gradient sees dL_dK times the other factors;
 * static.py:63-99 White, :142-185 Bias). Each part is a stationary kernel on its own active dims (column indices into
 * the X of gpx_set_data; kernel_slice_operations.py:59-79), a White or a Bias kernel. Parts with the same `term` are
 * multiplied, terms are summed; parts must be ordered by term. The whole evaluation runs on the device like
 * gpx_exact_eval (K-build, factor-and-invert sweep, K^-1, one gradient-reduction pass per part over the stored K^-1).
 *   grad: out, concatenation over the parts in the given order of [d/d variance, d/d lengthscale (1 or ndims; none for
 *         White / Bias)], then d/d noise — the order paramz gives Add/Prod parameters (kern.py:363-451 link order).
 * gpx_get / gpx_predict afterwards use the composite kernel. Single-GPU. */
typedef struct {
  int kind;                  /* GPX_RBF .. GPX_MATERN52, GPX_WHITE, GPX_BIAS (GPX_COREGIONALIZE: gpx_exact_eval_coreg) */
  int ard;                   /* stationary kinds: 0 -> lengthscale points at 1 double, 1 -> at ndims doubles */
  int term;                  /* additive term this factor belongs to */
  int ndims;                 /* number of active dims (0 for White / Bias, 1 for a coregionalization part) */
  const int* dims;           /* column indices into X, ndims entries */
  double variance;
  const double* lengthscale;
} gpx_kern_part;
int gpx_exact_eval_multi(gpx_ctx* ctx, const gpx_kern_part* parts, int nparts, double noise, double jitter, int max_tries,
                         double* lml, double* grad, double* jitter_used);

/* Multi-output regression (intrinsic / linear coregionalization: GPy/kern/src/coregionalize.py, GPy/util/multioutput.py:48-135,
 * GPy/models/gp_coregionalized_regression.py:31-46) on the fused path: gpx_exact_eval_multi with two additions.
 *  - Parts of kind GPX_COREGIONALIZE. Such a part has one active dim, the output-index column of X (a float column as
 *    build_XY makes it, multioutput.py:48-67); its value at (x_i, x_j) is B[idx_i, idx_j] with idx = the truncated integer
 *    (np.asarray(X, dtype=int), coregionalize.py:88-108). B = W W^T + diag(kappa) is formed by the caller
 *    (coregionalize.py:80) and passed in `coreg`, one entry per GPX_COREGIONALIZE part in part order; the part's `variance`
 *    and `lengthscale` are ignored (its factor in a product is B itself). An index outside [0, output_dim) makes the call
 *    return <0 with a message; nothing is read out of bounds.
 *  - noise_variances: NULL -> the scalar `noise` on the diagonal; else N per-point variances (MixedNoise /
 *    HeteroscedasticGaussian: exact_gaussian_inference.py:55-56 with a vector), and dnoise (N doubles) receives diag(dL_dK),
 *    which the likelihood's exact_inference_gradients sums per output (mixed_noise.py:38-41, gaussian.py:358-359).
 *  grad: concatenation over the parts in the given order of [d/d variance, d/d lengthscale (1 or ndims; none for White /
 *        Bias)] or, for a GPX_COREGIONALIZE part, S = dL_dK_small (output_dim x output_dim, row-major): S[a][b] = sum over
 *        idx_i = a, idx_j = b of (dL_dK o other factors of the term)_ij (coregionalize.py:130-137, prod.py:377-385). The
 *        caller forms dkappa = diag(S), dW = (S + S^T) W (coregionalize.py:123-128). Last entry: d/d noise (the sum of
 *        dnoise when noise_variances was given). Every reduction runs in a fixed order: results are bit-identical run to run.
 *  Caps: output_dim <= 16, nparts <= 8. gpx_get / gpx_predict afterwards use this kernel (gpx_predict checks the indices of
 *  Xnew as well). Single-GPU. */
typedef struct {
  int output_dim;            /* O: B is O x O */
  const double* B;           /* O x O row-major, finite and exactly symmetric (else the call returns <0) */
} gpx_coreg;
int gpx_exact_eval_coreg(gpx_ctx* ctx, const gpx_kern_part* parts, int nparts, const gpx_coreg* coreg, double noise,
                         const double* noise_variances, double jitter, int max_tries, double* lml, double* grad,
                         double* dnoise, double* jitter_used);

/* Lazy device->host fetch of N^2 / N*P results of the last gpx_exact_eval (Posterior / grad_dict consumers:
 * GPy/inference/latent_function_inference/posterior.py:21-77; exact_gaussian_inference.py:74). */
int gpx_get(gpx_ctx* ctx, int which, double* out_host);

/* PosteriorExact._raw_predict (posterior.py:273-302) on device with the factor of the last eval:
 * mu (M x P row-major) = K(X,Xnew)^T alpha; var (M) = Kdiag(Xnew) - colsum((L^-1 K(X,Xnew))^2)   [full_cov = 0]
 * or var (M x M col-major) = K(Xnew) - tmp^T tmp                                                 [full_cov = 1]. */
int gpx_predict(gpx_ctx* ctx, const double* Xnew, int64_t M, int full_cov, double* mu, double* var);

/* Standalone kernel plugin calls (no context needed beyond a device; ctx may be NULL -> device 0 scratch context).
 * Replaces Stationary.K (stationary.py:105-168): out is N x M ROW-major (what Kern.K returns to NumPy callers).
 * out == NULL: build on the device only and report the kernel time via gpx_get_stats (kbuild_ms, kbuild_bytes). */
int gpx_kern_K(gpx_ctx* ctx, int kind, int ard, double variance, const double* lengthscale, const double* X, int64_t N,
               const double* X2 /* NULL -> K(X,X) with exact zero-distance diagonal */, int64_t M, int D, double* out);
/* Replaces Stationary.Kdiag (stationary.py:170-173). */
int gpx_kern_Kdiag(int kind, double variance, int64_t N, double* out);
/* Replaces Stationary.update_gradients_full (stationary.py:193-243) for a caller-supplied dL_dK (N x M row-major). */
int gpx_kern_grad_full(gpx_ctx* ctx, int kind, int ard, double variance, const double* lengthscale, const double* X,
                       int64_t N, const double* X2, int64_t M, int D, const double* dL_dK, double* dvariance,
                       double* dlengthscale);

/* Replaces Stationary.gradients_X (stationary.py:245-252,348-366 and the OpenMP helper GPy/kern/src/stationary_utils.c:1-14
 * _grad_X): grad (N x D row-major) = d/dX of sum(dL_dK * K(X, X2)); X2 == NULL is the symmetric case (tmp + tmp^T). */
int gpx_kern_grad_X(gpx_ctx* ctx, int kind, int ard, double variance, const double* lengthscale, const double* X,
                    int64_t N, const double* X2, int64_t M, int D, const double* dL_dK, double* grad);

/* Replaces pdinv / jitchol for a caller-supplied symmetric positive (semi-)definite matrix A (N x N, dense, symmetric so
 * row- and column-major coincide): GPy/util/linalg.py:193-214 (pdinv -> Ai, L, Li, logdet) and :56-75 (jitchol: first a
 * plain factorisation; on failure LinAlgError if any diagonal entry is <= 0, else jitter mean(diag)*1e-6*10^k, k <
 * max_tries). Ai / L / Li may be NULL (not wanted); L, Li are lower, column-major; returns >0 when not PD. */
int gpx_pdinv(gpx_ctx* ctx, const double* A, int64_t N, int max_tries, double* Ai, double* L, double* Li, double* logdet,
              double* jitter_used);

/* Sparse GP regression (VarDTC): the N-dependent work of GPy/inference/latent_function_inference/var_dtc.py:66-215 and of
 * the gradient wiring GPy/core/sparse_gp.py:108-119 (Gaussian likelihood, homoscedastic, certain inputs). psi1 = K(X, Z)
 * (8 N M bytes) is built and kept in HBM; only M x M / M x P / M x D results cross PCIe.
 *   gpx_sparse_set_data : X (N x D row-major), Y (N x P row-major) -> HBM (no N x N workspace is allocated).
 */
int gpx_sparse_set_data(gpx_ctx* ctx, const double* X, int64_t N, int D, const double* Y, int P);
/* One whole VarDTC evaluation on the device: VarDTC.inference (var_dtc.py:66-215, Gaussian homoscedastic noise, certain
 * inputs, no mean function) + SparseGP._update_gradients (core/sparse_gp.py:108-119) + Gaussian.update_gradients
 * (likelihoods/gaussian.py:78-79). Kmm + 1e-8 I and B = I + A are factored-and-inverted by the same sweep as the exact
 * path (jitchol ladder, util/linalg.py:56-75); every M x M product of :130-156,:201-233 is a DMMA GEMM; only the
 * scalars, dZ (M x D row-major) and the (1 + nl + 1) gradient entries [variance, lengthscale.., noise variance] return.
 * A = beta (Lm^-1 psi1^T)(Lm^-1 psi1^T)^T is formed from tmp = Lm^-1 psi1^T like the reference does (:130-132), not by
 * sandwiching psi1^T psi1, which loses ~cond(Kmm) digits. With a communicator attached (gpx_comm_init) X, Y are THIS
 * rank's rows and A, tmp Y and the Knm gradient pieces are all-reduced (var_dtc_parallel.py:113-131).
 *   gpx_sparse_get: posterior pieces of the last evaluation (var_dtc.py:201-214): 0 woodbury_vector (M x P row-major),
 *                   1 woodbury_inv (M x M), 2 Kmm (+ const_jitter on the diagonal), 3 Lm (lower, column-major). */
int gpx_sparse_eval(gpx_ctx* ctx, int kind, int ard, double variance, const double* lengthscale, const double* Z,
                    int64_t M, double noise_variance, double* lml, double* grad, double* dZ);
int gpx_sparse_get(gpx_ctx* ctx, int which, double* out);
/* The same evaluation with ONE NOISE VARIANCE PER DATA POINT (HeteroscedasticGaussian, likelihoods/gaussian.py:347-362):
 * the `het_noise` branches of VarDTC.inference — tmp = Lm^-1 (psi1 sqrt(beta))^T (var_dtc.py:127-131), dL_dpsi1 += 2
 * (dL_dpsi2_beta (psi1 beta)^T)^T (:221-227), the bound with sum(log beta_n) and sum(beta_n |Y_n|^2) (:267-269) and the
 * per-point noise gradients dL_dR (:241-257). noise_variances: N values (this rank's rows); grad: (1 + nl) entries
 * [variance, lengthscale..]; dL_dR: N x P row-major, what HeteroscedasticGaussian.exact_inference_gradients indexes by
 * output_index (gaussian.py:358-359). dL_dR needs three column reductions over M x N matrices (|Lm^-1 psi1^T[:, n]|^2,
 * |LB^-1 Lm^-1 psi1^T[:, n]|^2, v^T LB^-1 Lm^-1 psi1^T[:, n]); nothing of size N x M crosses PCIe. gpx_sparse_get serves
 * the posterior of this evaluation as well. */
int gpx_sparse_eval_het(gpx_ctx* ctx, int kind, int ard, double variance, const double* lengthscale, const double* Z,
                        int64_t M, const double* noise_variances, double* lml, double* grad, double* dZ, double* dL_dR);

/* Measurement hooks (bench.py): device time of the last eval between CUDA events on the launching stream, the number
 * of kernels this library launched since creation, and per-phase accounting of the last eval. */
typedef struct {
  float total_ms;       /* whole eval, H2D of theta .. D2H of (lml, grad) */
  float kbuild_ms;      /* covariance build kernel */
  float sweep_ms;       /* blocked factor-and-invert sweep (all launches) */
  float update_ms;      /* sum over the outer trailing-update GEMM launches (dominant kernel); on the tcgen05 path these launches
                           also accumulate K^-1 = U U^T */
  float lauum_ms;       /* DMMA path: K^-1 = U U^T + fused gradient epilogue; tcgen05 path: gradient reductions from the stored K^-1 */
  float solve_ms;       /* alpha / quadratic form */
  double update_flops;  /* algorithmic flops executed by the outer trailing-update launches */
  double lauum_flops;
  double kbuild_bytes;  /* algorithmic bytes of the covariance build (8 N^2 + 8 N D) */
  int64_t launches;     /* kernels launched by the last eval */
  int32_t update_launches;
  int32_t tries;        /* factorisation attempts (1 = no jitter ladder) */
  double update_int8_ops; /* tcgen05 path: int8 multiply-add operations (2 per MAC) issued by the update / K^-1 launches, summed
                             over the digit pairs actually computed; 0 on the DMMA path */
} gpx_stats;
int gpx_get_stats(gpx_ctx* ctx, gpx_stats* out);
int64_t gpx_total_launches(gpx_ctx* ctx);
/* Roofline denominator measured on this device: fp64 tensor (DMMA.8x8x4) issue rate in TFLOP/s, CUDA-event timed. */
int gpx_measure_fp64_peak(gpx_ctx* ctx, double* tflops);

/* Tunables (block sizes etc.), mainly for tests: name in {"nb", "lookahead", "profile", "ozaki" (0 = fp64 DMMA only,
 * 1 = trailing update and K^-1 on the tcgen05 int8 path where applicable, -1 = default), "oz_dig_up" (digits per operand
 * for the inverse-part tiles, 4..8), "oz_ctas" (CTAs of the persistent tcgen05 GEMM, 0 = one per SM), "fine" (1 = 64 x 64-tile DMMA kernels inside
 * the diagonal-block chain, 0 = 128 x 128 tiles), "chain" (1 = tcgen05 path: diagonal-block chain alone on the side stream, the
 * rest of the panel / digit split / forward substitution on a third stream; 0 = round-2 schedule), "base" (generation of the
 * 128 x 128 base-block kernel, process-wide: 0 = default, 1..3)}. */
int gpx_set_option(gpx_ctx* ctx, const char* name, int64_t value);

/* Multi-GPU (one process per GPU). The caller obtains a 128-byte NCCL unique id on rank 0 (gpx_comm_unique_id),
 * ships it to the other ranks with its own plumbing (torch.distributed broadcast), and every rank calls
 * gpx_comm_init. Afterwards gpx_set_data / gpx_exact_eval are collective: block rows are dealt block-cyclically
 * to the ranks, the inverted diagonal block is broadcast and the panel all-gathered (NCCL over NVLink), scalars all-reduced. */
int gpx_comm_unique_id(char id_out[128]);
int gpx_comm_init(gpx_ctx* ctx, const char id[128], int rank, int nranks);

#ifdef __cplusplus
}
#endif
#endif /* GPX_H_ */
