/*
 * gpk_test.h -- measurement and test hooks of libgpk.so. NOT part of the drop-in boundary (include/gpk.h): nothing in
 * the product's Python layer calls these; they exist so that tests/ and bench.py can exercise single kernels (a GEMM
 * with a given k-range, the residue conversion, one tensor-pipe probe) and read per-launch CUDA-event timings.
 */
#ifndef GPK_TEST_H
#define GPK_TEST_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* In: A (lower tiles of an SPD matrix, order npad, ld). Out: X = L^-1, dL = diag(L), *info_host (0 = ok). FP64 DMMA. */
int gpk_test_potrf_inv(double* A_dev, double* X_dev, int64_t ld, int64_t npad, double* dL_dev, int* info_host,
                       void* cuda_stream);

/*
 * FP64 GEMM through the INT8 tcgen05 tensor cores (csrc/oz_gemm.cuh).
 * gpk_test_oz_residues: reduce an operand (trans == 0: rows x K, leading dimension ld; trans == 1: K x rows; lower != 0:
 * source 128-tiles above the diagonal read as zero) into `moduli` tiled planes of rows x K int8 residues and the
 * per-row scales 2^(e - bits).
 * gpk_test_oz_gemm: C = beta*C + alpha * A(M,K) B(N,K)^T over the per-tile k range with `moduli` moduli; transA/transB
 * as above; panel_rows > 0 limits the residue-plane buffer to that many rows, so the product runs panel by panel;
 * ms_out_host[0] = residue conversion time of both operands, [1] = average GEMM + reconstruction time over `reps`.
 */
int gpk_test_oz_residues(const double* src_dev, int64_t ld, int64_t rows, int64_t K, int trans, int lower, int moduli,
                         void* planes_out_dev, double* scales_out_dev, void* cuda_stream);
int gpk_test_oz_gemm(const double* A_dev, int64_t lda, int transA, int lowerA, const double* B_dev, int64_t ldb,
                     int transB, int lowerB, double* C_dev, int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha,
                     double beta, int krange, int lower_only, int moduli, int64_t panel_rows, int reps,
                     float* ms_out_host, void* cuda_stream);

/* Planes kernel (calling thread only): 0 = a CTA pair that starts a tile adopts the modulus of the most advanced pair and
 * starts at its first k-block; 1 = it adopts the (modulus, k-block) position, splitting its first modulus; 2 = in
 * addition every tile of a raster band takes the band's k range when K >= 16384 (default). Same bits in all three
 * (exact integer sums). Other values leave the setting unchanged. Returns the setting. */
int gpk_test_position_lock(int on);

/* Unwritten-memory check (calling thread only): while byte != 0, every device buffer the library allocates (handle
 * buffers, query and gradient scratch, INT8 residue workspaces) is filled with `byte` right after allocation; switching
 * it on also refills the device's position-lock scratch. 0xFF makes every double a NaN, 0x7F every double 1.4e306.
 * Outputs must not depend on it. Returns the KiB of allocations filled since the previous call (so that a test can
 * check the fill took place; the refill of the position-lock scratch is not counted), or -1 on a CUDA error. */
int gpk_test_poison(int byte);

/* INT8 route (calling thread only): 1 = T = L21 X11 of each node overlaps the right sub-tree on its own stream when
 * the handle has the memory (default), 0 = every product on one stream; any other value leaves it unchanged. Takes
 * effect at the next factorisation (the workspaces follow at the next gpk_set_route). Returns the setting. */
int gpk_test_overlap(int on);

/*
 * gpk_profile(1): record a CUDA-event pair around every tensor-pipe GEMM launch (on the launching stream) of the
 * calling thread. gpk_profile_read: sum of those durations in ms (over all streams, so overlapping launches add up),
 * number of GEMM launches, number of ALL kernel launches issued by the library on this thread since the last read, and
 * the duration of the single longest GEMM launch (in a fit iteration: K^-1 = X^T X, n^3/3 flops); resets the counters.
 */
int gpk_profile(int on);
int gpk_profile_read(double* gemm_ms_host, int64_t* gemm_launches_host, int64_t* all_launches_host,
                     double* max_gemm_ms_host);

/*
 * INT8 tensor-pipe peak of this GPU: every SM pair issues tcgen05.mma.cta_group::2.kind::i8 (M = 256, N = 256, K = 32)
 * back to back from operand tiles that stay in shared memory (no TMA, no epilogue), accumulators in TMEM.
 * out_host[0] = burst TOP/s (best single launch of `iters` x 4 instructions per pair), out_host[1] = sustained TOP/s
 * over `seconds` of back-to-back launches (the power-capped rate a long step sees). ops = 2 x int8 multiply-adds.
 */
int gpk_microbench_i8(int64_t iters, double seconds, double* out_host);

#ifdef __cplusplus
}
#endif
#endif /* GPK_TEST_H */
