/*
 * gpk.h -- C ABI of libgpk.so: the B200 (sm_100a) dense Gaussian-process hot path of scikit-gpuppy.
 *
 * The reference has no FFI layer on this path: its boundary is the Python class protocol
 * (GaussianCovariance / GaussianProcess / UncertaintyPropagationApprox) plus one Cython module.
 * Each entry point below names the reference call site it replaces (paths relative to the
 * reference tree, skgpuppy/...). The drop-in Python classes under scikit-gpuppy_b200/skgpuppy/
 * bind these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; `double*` arguments named *_dev are DEVICE pointers (FP64, row-major),
 *     `*_host` are host pointers. theta = [log v, log vt, log w_1..log w_d] is always a host pointer.
 *   - every function returns int: 0 ok; k > 0: leading minor k of K is not positive definite
 *     (the Python layer raises numpy.linalg.LinAlgError so the reference's retry-at-0.999*theta and
 *     1e20 sentinel logic keep working, Covariance.py:209-214, 306-311); < 0: CUDA / argument error,
 *     text in gpk_last_error().
 *   - a handle is bound to the CUDA device current at gpk_create; one host thread drives a handle at a time. Different
 *     handles may be driven from different threads: gpk_last_error() and the measurement counters are per thread.
 *   - all work is enqueued on the handle's stream (gpk_set_stream); functions that return host scalars
 *     synchronise that stream, the others are asynchronous.
 *   - matrices owned by the handle are padded to npad = gpk_npad(n) (multiple of 128) with an identity
 *     diagonal in the padding block.
 */
#ifndef GPK_H
#define GPK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpk_handle_s* gpk_handle;

#define GPK_MAX_D 64

/* version / diagnostics */
int gpk_version(void);
const char* gpk_last_error(void);   /* text of the last failure on the calling thread */

/* padded order used for all n x n buffers of a handle */
int64_t gpk_npad(int64_t n);

/*
 * Create a handle for n training points in d dimensions.
 * Xbuf_dev / Wbuf_dev: two caller-owned device buffers of gpk_npad(n)^2 doubles each (e.g. torch tensors;
 * they are what gets broadcast over NCCL for query-sharded prediction), or NULL to let the library allocate.
 * After gpk_factorize: Xbuf = X = L^-1 (lower, L L^T = K); Wbuf = K^-1 (lower tiles) when the inverse was requested.
 * Replaces the object state of GaussianProcess.__init__ (GaussianProcess.py:19-41: x, t, Kinv).
 */
int gpk_create(int64_t n, int64_t d, double* Xbuf_dev, double* Wbuf_dev, gpk_handle* out);
int gpk_destroy(gpk_handle h);
int gpk_set_stream(gpk_handle h, void* cuda_stream);

/* Copy training inputs x (n x d) and centred targets t (n) from device memory into the handle. */
int gpk_set_data(gpk_handle h, const double* x_dev, const double* t_dev);

/*
 * out[i*ld + j] = v exp(-1/2 sum_k w_k (x1_ik - x2_jk)^2) (+ vt where i == j if add_noise).
 * Replaces GaussianCovariance.cov_matrix_ij / cov_matrix (Covariance.py:466-483, 461-464).
 */
int gpk_kernel_matrix(const double* x1_dev, int64_t n1, const double* x2_dev, int64_t n2, int64_t d,
                      const double* theta_host, int add_noise, double* out_dev, int64_t ld, void* cuda_stream);

/*
 * Build K(theta) on the device, factor it and form X = L^-1, y = X t, alpha = K^-1 t, log det K;
 * with want_inverse also K^-1 = X^T X. Results are cached by theta.
 * Replaces inv_cov_matrix / _log_det_cov_matrix (Covariance.py:167-195: scipy inv + numpy slogdet).
 */
int gpk_factorize(gpk_handle h, const double* theta_host, int want_inverse);

/*
 * The same factorisation stack on a caller-supplied symmetric positive definite matrix K (n x n, device, leading
 * dimension ldk; only the lower triangle is read): X = L^-1, alpha = K^-1 t, log det K, optionally K^-1.
 * Replaces the cov_matrix= branch of Covariance.inv_cov_matrix (Covariance.py:186-187) and serves covariance classes
 * whose K is built on the host (user subclasses of Covariance, Covariance.py:137-152; SPGP's low-rank systems).
 * gpk_logdet / gpk_solve / gpk_inverse / gpk_get_alpha / gpk_nll_matrix apply afterwards; the theta-keyed entry points
 * (gpk_nll_grad, gpk_predict, gpk_propagate_*) need gpk_factorize.
 */
int gpk_factorize_matrix(gpk_handle h, const double* K_dev, int64_t ldk, int want_inverse);
/* n/2 log(2 pi) + 1/2 log det K + 1/2 t^T K^-1 t of the cached factorisation (Covariance.py:211). */
int gpk_nll_matrix(gpk_handle h, double* nll_host);

/* log det K of the cached factorisation (Covariance.py:189-195). */
int gpk_logdet(gpk_handle h, double* out_host);

/*
 * nll = n/2 log(2 pi) + 1/2 log det K + 1/2 t^T K^-1 t            (Covariance.py:197-216)
 * grad[j] = 1/2 tr(K^-1 dK_j) - 1/2 t^T K^-1 dK_j K^-1 t, j < d+2  (Covariance.py:266-282, 505-512, 605-657)
 * One factorisation is shared between a nll call and a grad call at the same theta.
 * want_grad: 0 = nll only; 1 = nll and grad; 2 = nll now, and K^-1 with the trace sums of the gradient are queued behind
 * it without waiting (Gaussian family; grad_host is not written): the want_grad = 1 call at the same theta then only
 * collects them. For callers that know the gradient call follows, as in an L-BFGS iteration (Covariance.py:314-337).
 */
int gpk_nll_grad(gpk_handle h, const double* theta_host, double* nll_host, double* grad_host, int want_grad);

/*
 * Raw trace sums over tile rows [tile_row_begin, tile_row_end) of the cached K^-1 (128-row tiles):
 * out_host[0] = sum_ab M_ab Knl_ab, out_host[1+k] = sum_ab M_ab Knl_ab (x_ak - x_bk)^2, M = K^-1 - alpha alpha^T,
 * out_host[d+1] = sum_a (K^-1)_aa, out_host[d+2] = sum_a alpha_a^2 over the rows of those tiles (d+3 doubles).
 * This is the shard a rank owns before the all-reduce; the d+2 gradient scalars follow from the reduced sums.
 */
int gpk_grad_trace_partial(gpk_handle h, int64_t tile_row_begin, int64_t tile_row_end, double* out_host);

/* out = K^-1 b for nrhs right-hand sides stored as columns of length n, contiguous one after another. */
int gpk_solve(gpk_handle h, const double* b_dev, int64_t nrhs, double* out_dev);

/* Dense symmetric n x n K^-1 (GaussianProcess.Kinv, GaussianProcess.py:41); computes it if not cached. */
int gpk_inverse(gpk_handle h, double* Kinv_out_dev, int64_t ldo);

/*
 * Backward-error check of the cached factorisation: out_host[0] = max_i |(K alpha)_i - t_i| with K regenerated from the
 * training inputs (K itself was consumed by the factorisation), [1] = max_i |alpha_i|, [2] = max_i |t_i|. One extra
 * K build (O(n^2 d)); the Python layer runs it once per GaussianProcess, not per likelihood evaluation. The reference
 * has no counterpart; it guards the choice of tensor pipe / operand width of gpk_set_route.
 */
int gpk_solve_residual(gpk_handle h, double* out_host);

/* alpha = K^-1 t (GaussianProcess._get_beta, GaussianProcess.py:114-119), n doubles. */
int gpk_get_alpha(gpk_handle h, double* alpha_out_dev);

/*
 * Mark a handle as factored from state produced on another rank: Xbuf (and Wbuf if have_inverse) were
 * filled by the caller (NCCL broadcast), alpha_dev holds alpha. Used for query-sharded predict/propagate.
 */
int gpk_import_state(gpk_handle h, const double* theta_host, const double* alpha_dev, int have_inverse);

/*
 * mean[q] = k*_q . alpha + meant ; var[q] = v + vt - |X k*_q|^2      (GaussianProcess.estimate_many,
 * GaussianProcess.py:68-80; the m x m temporaries of the reference are never formed).
 */
int gpk_predict(gpk_handle h, const double* xs_dev, int64_t m, double meant, double* mean_dev, double* var_dev,
                int want_var);

/*
 * The same prediction from a caller-built cross covariance (covariance classes without device kernels, whose scalar
 * function runs on the host; works after gpk_factorize or gpk_factorize_matrix): Ks_dev is m x n (leading dimension
 * ldk) with Ks[q][i] = k(x*_q, x_i), prior_dev[q] = k(x*_q, x*_q) incl. noise;
 * mean[q] = Ks_q . alpha + meant, var[q] = prior[q] - |X Ks_q|^2 (GaussianProcess.py:75-80). var_dev may be NULL.
 */
int gpk_predict_cross(gpk_handle h, const double* Ks_dev, int64_t ldk, int64_t m, const double* prior_dev, double meant,
                      double* mean_dev, double* var_dev);

/*
 * Joint predictive covariance (the matrix the reference forms inside estimate_many, GaussianProcess.py:75-80):
 * cov[a*ldc + b] = k(xa_a, xb_b) + noise - k(xa_a, x) K^-1 k(x, xb_b), with k(., x) = K* rows as in gpk_predict.
 * xb_dev == NULL: B = A (mb is ignored). The output is ma x ma and exactly symmetric, and the noise term follows
 * cov_matrix(A) of the family. xb_dev != NULL: the noise term follows cov_matrix_ij(A, B).
 * Needs gpk_factorize (theta state), like gpk_predict. ma == 0 or mb == 0 does nothing.
 * Workspace: the rows of V = X k(x, .) of both sets stay resident for the call (8 * m_pad * npad bytes per set, plus
 * moduli * m_pad * npad bytes of their residues on the INT8 route) with a padded ma x mb output block and one query
 * batch; if that does not fit the call returns -4 before any work is queued (byte counts in gpk_last_error()).
 */
int gpk_predict_cov(gpk_handle h, const double* xa_dev, int64_t ma, const double* xb_dev, int64_t mb,
                    double* cov_dev, int64_t ldc);

/*
 * Same from caller-built cross covariances (covariance classes without device kernels; works after
 * gpk_factorize or gpk_factorize_matrix): Ka is ma x n (lda), Kb is mb x n (ldb) or NULL for B = A,
 * prior is the caller's ma x mb block k(A, B) including its noise (ldp). cov_dev may equal prior_dev.
 */
int gpk_predict_cov_cross(gpk_handle h, const double* Ka_dev, int64_t lda, int64_t ma,
                          const double* Kb_dev, int64_t ldb, int64_t mb,
                          const double* prior_dev, int64_t ldp, double* cov_dev, int64_t ldc);

/*
 * Gradients of the predictive mean and variance with respect to the query point (both device families):
 *   mean[q] and var[q] as gpk_predict (noise included), dmean[q*d + k] = d mean[q] / d x*_qk = D_k . alpha,
 *   dvar[q*d + k] = d var[q] / d x*_qk = -2 (X k*_q) . (X D_k),   D_k,i = d k(x*_q, x_i) / d x*_qk,
 * with k*_q the row gpk_predict builds (prior k(x*, x*) is constant for both families).
 * D is the true derivative: the reference's get_Jacobian (Covariance.py:676-689) has the opposite sign. Noise is a jump,
 * not a slope: the vt added where a query coincides with a training point (periodic family, and the scalar rule of the
 * Gaussian covariance) is left out of D. var_dev and dvar_dev: both NULL skips the O(n^2)
 * product (rows and dots with alpha only); one of them NULL returns -2. Needs gpk_factorize (theta state), like
 * gpk_predict. m == 0 does nothing.
 * Workspace: one batch of d + 1 rows per query and, with the variances, its V^T (plus its residues on the INT8 route);
 * if that does not fit the call returns -4 before any work is queued (byte counts in gpk_last_error()).
 */
int gpk_predict_grad(gpk_handle h, const double* xs_dev, int64_t m, double meant, double* mean_dev, double* var_dev,
                     double* dmean_dev, double* dvar_dev);

/*
 * Girard Gaussian approximation, batched over Q queries (UncertaintyPropagationApprox.propagate_GA,
 * UncertaintyPropagation2.pyx:266-299 with :208-257). U: Q x d means. S: Q x d (diagonal of Sigma_x) or,
 * with sigma_full, Q x d x d. Includes the equality-noise quirk of the scalar covariance (Covariance.py:451).
 */
int gpk_propagate_ga(gpk_handle h, const double* U_dev, const double* S_dev, int64_t Q, int sigma_full,
                     double meant, double* mean_dev, double* var_dev);

/*
 * The two addends of the propagated variance, per query: sigma2 = cov(u,u) - C^T K^-1 C (pyx:221-232) and
 * variance_rest = variance2 + variance3 (pyx:234-257). They are what UncertaintyPropagationApprox._getFactor
 * (pyx:302-336: (v - sigma2)/variance_rest) and ._get_variance_dv_h (pyx:340-380: variance_rest for
 * Sigma = e_h e_h^T) need; inverse uncertainty propagation is built on them.
 */
int gpk_propagate_ga_parts(gpk_handle h, const double* U_dev, const double* S_dev, int64_t Q, int sigma_full,
                           double* sigma2_dev, double* rest_dev);

/*
 * Girard's exact mean / variance for the SE kernel, batched over Q queries (UncertaintyPropagationExact.propagate_GA,
 * UncertaintyPropagation2.pyx:57-184). The d x d constants of each query are built by the caller (they are O(d^3)
 * host work in the reference too, pyx:67-78, 116-128): Lam = 2 W^-1 - (W/2 + Sigma)^-1 (Q x d x d, symmetric),
 * Dinv = diag of Delta^-1 (Q x d), norms = (|I + W^-1 o Sigma|^-1/2, |2 W^-1 o Sigma + I|^-1/2) (Q x 2). d <= 32.
 */
int gpk_propagate_exact(gpk_handle h, const double* U_dev, const double* Lam_dev, const double* Dinv_dev,
                        const double* norms_dev, int64_t Q, double meant, double* mean_dev, double* var_dev);

/*
 * Covariance family of a handle: 0 = GaussianCovariance (default), 1 = PeriodicCovariance
 * (k = v exp(-1/2 sum_k [w2_k sin^2(pi diff_k / p_k) + w_k diff_k^2]) + vt where the points are equal; theta =
 * [log v, log vt, log w (d), log p (d), log w2 (d)]; reference Covariance.py:361-433; d <= 16). With kind 1,
 * gpk_factorize / gpk_nll_grad / gpk_solve / gpk_inverse / gpk_predict work as above with theta and grad of length
 * 2 + 3d; the propagation entry points need kind 0 (the reference has no propagation for this kernel either).
 */
int gpk_set_kernel(gpk_handle h, int kind);

/* Periodic-kernel counterpart of gpk_kernel_matrix. noise_mode: 0 none, 1 + vt on the diagonal, 2 + vt wherever the two
 * points are equal element-wise (the rule of the reference's scalar __call__, used by its generic cov_matrix_ij). */
int gpk_kernel_matrix_periodic(const double* x1_dev, int64_t n1, const double* x2_dev, int64_t n2, int64_t d,
                               const double* theta_host, int noise_mode, double* out_dev, int64_t ld, void* cuda_stream);

/*
 * Tensor pipe of the O(n^3) contractions of a handle (factorisation, inverse, predictive variances, Girard quadratic
 * forms). int8 != 0: blocks of order >= min_dim run as EXACT INT8 products on the tcgen05 tensor cores (csrc/oz_gemm.cuh:
 * Chinese-remainder form, one int8 GEMM per modulus, int32 accumulation in TMEM, exact reconstruction to FP64), smaller
 * blocks on the FP64 DMMA kernel; int8 == 0: FP64 DMMA everywhere. min_dim: 0 = default (2048), else a multiple of 128
 * >= 256. moduli: 0 = the fewest that carry 54-bit operands (one bit more than an FP64 significand) at K = npad
 * (16 up to n = 65536), else 8..18. plane_cap_bytes: cap of the residue-plane buffer of the products, 0 = default
 * (16 GiB, 8 GiB at npad >= 49152); larger products run as row panels.
 * Default of a new handle: int8 on when gpk_npad(n) >= 2048. The INT8 workspace (moduli * npad^2 bytes of operand
 * residues + the plane buffer) is allocated by the first call that needs it; if it does not fit that call fails with
 * -4 -- there is NO silent fallback to the slower pipe, the caller selects it with gpk_set_route(h, 0, 0, 0, 0).
 * Calling gpk_set_route drops the cached factorisation.
 * gpk_get_route: out_host[0] = INT8 route requested, [1] = moduli, [2] = min_dim, [3] = operand bits at K = npad (53 for DMMA).
 */
int gpk_set_route(gpk_handle h, int int8, int64_t min_dim, int moduli, int64_t plane_cap_bytes);
int gpk_get_route(gpk_handle h, int* out_host);

/* Upper bound on the rows of the per-batch workspace (queries per GEMM); 0 restores the default. */
int gpk_set_batch_rows(gpk_handle h, int64_t rows);

#ifdef __cplusplus
}
#endif
#endif /* GPK_H */
