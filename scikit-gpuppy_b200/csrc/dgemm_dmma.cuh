// FP64 tile GEMM on the Blackwell DMMA pipe (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4).
//
//   C[m,n] = beta*C[m,n] + alpha * sum_{k in krange(bi,bj)} A(m,k) * B(n,k)
//
// This is the one dense contraction behind the whole factorisation stack: the
// recursive Cholesky+inverse (TRSM-as-GEMM, SYRK trailing update, TRMM), the
// explicit inverse K^-1 = X^T X, and the predictive-variance / Girard quadratic
// forms ||X k*||^2 (EPI_COLSQ epilogue, V never stored).
//
// All extents are multiples of the 128x128 CTA tile (matrices are padded by the
// handle), so the kernel has no bounds checks. Triangular structure is expressed
// as a per-tile k-range, never as masked arithmetic.
//
// There is no f64 kind for tcgen05/wgmma; DMMA is the FP64 tensor path on sm_100a.
#pragma once
#include <cstdlib>

#include "gpk_common.cuh"

namespace gpk {

// CTA tile TM x TN x 16, warps arranged (TM/32) x 2, warp tile 32 x TN/2 (= 4 x TN/16 DMMA.8x8x4 fragments),
// STAGES-deep cp.async pipeline, MINCTAS co-resident CTAs per SM. Several small CTAs per SM hide each other's
// barrier / LDS bubbles (ncu: one 128x128 CTA/SM kept the DMMA pipe 89% busy, three 64x64 CTAs 93+%).
// k-ranges stay expressed in 128-blocks whatever the tile.
constexpr int GEMM_BM = 128, GEMM_BN = 128, GEMM_BK = 16;   // extent granularity of every operand
constexpr int GEMM_LDK = GEMM_BK + 4;                       // 20: smem leading dim when k is contiguous
template <int TM_, int TN_, int STAGES_, int MINCTAS_>
struct GemmTile {
  static constexpr int TM = TM_, TN = TN_, STAGES = STAGES_, MINCTAS = MINCTAS_;
  static constexpr int WARPS_M = TM / 32;
  static constexpr int THREADS = WARPS_M * 2 * 32;
  static constexpr int NJ = TN / 16;                 // column fragments per warp
  static constexpr int LDMA = TM + 4, LDMB = TN + 4; // leading dims when m/n is contiguous (== 4 mod 16)
  static constexpr int A_ELEMS = TM * GEMM_LDK;      // >= 16 * LDMA
  static constexpr int B_ELEMS = TN * GEMM_LDK;      // >= 16 * LDMB
  static constexpr int PA = TM * 8 / THREADS;        // 16-byte cp.async per thread per chunk (A): 4
  static constexpr int PB = TN * 8 / THREADS;        // (B): 4*TN/TM
  static constexpr int SMEM_BYTES = STAGES * (A_ELEMS + B_ELEMS) * (int)sizeof(double);
};
using Tile128 = GemmTile<128, 128, 3, 1>;   // 8 warps, 1 CTA/SM (needed by the EPI_COLSQ consumers' 128-row partials)
using Tile64 = GemmTile<64, 64, 3, 3>;      // 4 warps, 3 CTAs/SM
using Tile64x128 = GemmTile<64, 128, 3, 2>; // 4 warps (warp tile 32x64), 2 CTAs/SM: best measured on large grids
constexpr int GEMM_SMEM_BYTES = Tile128::SMEM_BYTES;

// operand layouts
constexpr int LAY_KC = 0;  // element (m,k) at ptr[m*ld + k]   (k contiguous)
constexpr int LAY_MC = 1;  // element (m,k) at ptr[k*ld + m]   (m contiguous)

// per-tile k ranges (bi = tile row, bj = tile col, in units of 128)
enum KRange : int {
  K_FULL = 0,     // [0, K)
  K_UPTO_BJ = 1,  // [0, (bj+1)*128)
  K_FROM_BJ = 2,  // [bj*128, K)
  K_UPTO_BI = 3,  // [0, (bi+1)*128)
  K_FROM_BI = 4   // [bi*128, K)
};

constexpr int EPI_STORE = 0;  // C = beta*C + alpha*acc
constexpr int EPI_COLSQ = 1;  // colsq[bi][n] = sum_m acc[m,n]^2 ; pairdot[bi][p] = sum_m acc[m,2p]*acc[m,2p+1]

struct GemmArgs {
  const double* A; long lda;
  const double* B; long ldb;
  double* C; long ldc;
  int M, N, K;
  double alpha, beta;
  int krange;
  int lower_only;   // skip tiles entirely above the diagonal
  int reverse_bi;   // schedule large bi first (heavy-first for K_UPTO_BI)
  double* colsq; double* pairdot; long ldo;  // EPI_COLSQ outputs: colsq[bi*ldo + n], pairdot[bi*(ldo/2) + n/2]
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// Part r of an (EXT x 16) operand chunk global -> shared: one 16-byte cp.async per thread. The main loop
// spreads the parts over the k-steps so the LDGSTS never queue in front of the fragment LDS in the LSU FIFO
// (a burst right after the barrier cost ~10% of the DMMA pipe).
template <int LAY, int EXT, int THREADS>
__device__ __forceinline__ void load_chunk_part(double* s, const double* g, long ld, int mn0, int k0, int tid,
                                                int r) {
  const int idx = tid + r * THREADS;
  if (LAY == LAY_KC) {
    // EXT rows (m) x 8 chunks of 2 doubles
    const int row = idx >> 3, ch = idx & 7;
    cp_async16(s + row * GEMM_LDK + ch * 2, g + (long)(mn0 + row) * ld + k0 + ch * 2);
  } else {
    // 16 rows (k) x EXT/2 chunks of 2 doubles
    const int row = idx / (EXT / 2), ch = idx % (EXT / 2);
    cp_async16(s + row * (EXT + 4) + ch * 2, g + (long)(k0 + row) * ld + mn0 + ch * 2);
  }
}

template <int ALAY, int BLAY, int EPI, class T>
__global__ void __launch_bounds__(T::THREADS, T::MINCTAS) dgemm_dmma_kernel(GemmArgs p) {
  constexpr int TM = T::TM, TN = T::TN, NJ = T::NJ, STAGES = T::STAGES;
  extern __shared__ __align__(16) double smem[];
  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x;
  // Raster: the CTAs resident at one time (148 x MINCTAS) should share as few A/B panels as possible, so the
  // linear CTA id walks column-major through bands of GROUP_M tile rows (a near-square working set) instead of
  // along whole tile rows. ncu on 8192^3: DRAM reads 64 GB row-major vs the 1.6 GB the operands occupy.
  constexpr int GROUP_M = (TM >= 128) ? 8 : 16;   // band height in tile rows
  const int pid = blockIdx.y * gridDim.x + blockIdx.x;
  const int per_band = GROUP_M * gridDim.x;
  const int band = pid / per_band;
  const int first = band * GROUP_M;
  const int rows = min((int)gridDim.y - first, GROUP_M);
  const int rem = pid - band * per_band;
  const int by = first + rem % rows;
  const int bj = rem / rows;
  const int bi = p.reverse_bi ? (gridDim.y - 1 - by) : by;
  if (p.lower_only && bj * TN > bi * TM + (TM - 1)) return;

  // k-ranges are defined on 128-blocks whatever the CTA tile
  const int bi128 = (bi * TM) / TILE, bj128 = (bj * TN) / TILE;
  int kb = 0, ke = p.K;
  switch (p.krange) {
    case K_UPTO_BJ: ke = min(p.K, (bj128 + 1) * TILE); break;
    case K_FROM_BJ: kb = min(p.K, bj128 * TILE); break;
    case K_UPTO_BI: ke = min(p.K, (bi128 + 1) * TILE); break;
    case K_FROM_BI: kb = min(p.K, bi128 * TILE); break;
    default: break;
  }
  const int nk = (ke - kb) / GEMM_BK;

  double* As = smem;
  double* Bs = smem + STAGES * T::A_ELEMS;

  const int warp = tid >> 5, lane = tid & 31;
  const int wm = warp % T::WARPS_M, wn = warp / T::WARPS_M;
  const int g = lane >> 2, tg = lane & 3;

  double acc[4][NJ][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < NJ; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  // Software pipeline (needs STAGES >= 3):
  //  * chunks kc+1 .. kc+STAGES-2 are in flight while chunk kc is consumed; the cp.async of chunk kc+STAGES-1
  //    are spread over the 4 k-steps of iteration kc;
  //  * fragments are double-buffered in registers across k-steps AND across the chunk boundary: the barrier
  //    that publishes chunk kc+1 sits BEFORE the last k-step's DMMAs, so barrier skew and LDS latency are
  //    covered by DMMAs already issued (ncu: barrier + short-scoreboard stalls were ~10% of samples).
  static_assert(STAGES >= 3, "the cross-chunk fragment pipeline needs at least 3 stages");
#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) {
    if (s < nk) {
#pragma unroll
      for (int r = 0; r < T::PA; ++r)
        load_chunk_part<ALAY, TM, T::THREADS>(As + s * T::A_ELEMS, p.A, p.lda, bi * TM, kb + s * GEMM_BK, tid, r);
#pragma unroll
      for (int r = 0; r < T::PB; ++r)
        load_chunk_part<BLAY, TN, T::THREADS>(Bs + s * T::B_ELEMS, p.B, p.ldb, bj * TN, kb + s * GEMM_BK, tid, r);
    }
    cp_async_commit();
  }
  cp_async_wait<STAGES - 2>();
  __syncthreads();

  double fa[2][4], fb[2][NJ];
  auto load_frags = [&](const double* as, const double* bs, int ks, double (&a)[4], double (&b)[NJ]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      a[i] = (ALAY == LAY_KC) ? as[(wm * 32 + i * 8 + g) * GEMM_LDK + ks * 4 + tg]
                              : as[(ks * 4 + tg) * T::LDMA + wm * 32 + i * 8 + g];
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      b[j] = (BLAY == LAY_KC) ? bs[(wn * (TN / 2) + j * 8 + g) * GEMM_LDK + ks * 4 + tg]
                              : bs[(ks * 4 + tg) * T::LDMB + wn * (TN / 2) + j * 8 + g];
    }
  };
  if (nk > 0) load_frags(As, Bs, 0, fa[0], fb[0]);

  for (int kc = 0; kc < nk; ++kc) {
    const int nxt = kc + STAGES - 1;
    const bool do_load = nxt < nk;
    double* as_n = As + (nxt % STAGES) * T::A_ELEMS;
    double* bs_n = Bs + (nxt % STAGES) * T::B_ELEMS;
    const int k_n = kb + nxt * GEMM_BK;
    const double* as = As + (kc % STAGES) * T::A_ELEMS;
    const double* bs = Bs + (kc % STAGES) * T::B_ELEMS;
    const double* as1 = As + ((kc + 1) % STAGES) * T::A_ELEMS;
    const double* bs1 = Bs + ((kc + 1) % STAGES) * T::B_ELEMS;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const int cur = ks & 1, nx = cur ^ 1;
      if (ks == 3) {
        // chunk kc+1 must be visible before its first fragments are read below; after this barrier nobody
        // reads stage kc-1 any more, which is where iteration kc+1 will put chunk kc+STAGES
        cp_async_wait<STAGES - 3>();
        __syncthreads();
        if (kc + 1 < nk) load_frags(as1, bs1, 0, fa[nx], fb[nx]);
      } else {
        load_frags(as, bs, ks + 1, fa[nx], fb[nx]);
      }
      if (do_load) {
#pragma unroll
        for (int r = (ks * T::PA) / 4; r < ((ks + 1) * T::PA) / 4; ++r)
          load_chunk_part<ALAY, TM, T::THREADS>(as_n, p.A, p.lda, bi * TM, k_n, tid, r);
#pragma unroll
        for (int r = (ks * T::PB) / 4; r < ((ks + 1) * T::PB) / 4; ++r)
          load_chunk_part<BLAY, TN, T::THREADS>(bs_n, p.B, p.ldb, bj * TN, k_n, tid, r);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < NJ; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[cur][i], fb[cur][j]);
    }
    cp_async_commit();
  }
  cp_async_wait<0>();

  if (EPI == EPI_STORE) {
    const double alpha = p.alpha, beta = p.beta;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long row = (long)bi * TM + wm * 32 + i * 8 + g;
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        const long col = (long)bj * TN + wn * (TN / 2) + j * 8 + 2 * tg;
        double2* ptr = reinterpret_cast<double2*>(p.C + row * p.ldc + col);
        double2 v;
        v.x = alpha * acc[i][j][0];
        v.y = alpha * acc[i][j][1];
        if (beta != 0.0) {
          double2 o = *ptr;
          v.x += beta * o.x;
          v.y += beta * o.y;
        }
        *ptr = v;
      }
    }
  } else {
    // column sums of squares and adjacent-pair dots over the tile's TM rows -> partial row bi of colsq/pairdot
    __syncthreads();  // pipeline smem is dead now; reuse it
    double* red_sq = smem;                         // [WARPS_M][TN]
    double* red_pd = smem + T::WARPS_M * TN;       // [WARPS_M][TN/2]
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      double s0 = 0.0, s1 = 0.0, pd = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const double c0 = acc[i][j][0], c1 = acc[i][j][1];
        s0 = fma(c0, c0, s0);
        s1 = fma(c1, c1, s1);
        pd = fma(c0, c1, pd);
      }
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        pd += __shfl_xor_sync(0xffffffffu, pd, o);
      }
      if (g == 0) {
        const int c = wn * (TN / 2) + j * 8 + 2 * tg;
        red_sq[wm * TN + c] = s0;
        red_sq[wm * TN + c + 1] = s1;
        red_pd[wm * (TN / 2) + (c >> 1)] = pd;
      }
    }
    __syncthreads();
    for (int c = tid; c < TN + TN / 2; c += T::THREADS) {
      if (c < TN) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < T::WARPS_M; ++w) s += red_sq[w * TN + c];
        p.colsq[(long)bi * p.ldo + (long)bj * TN + c] = s;
      } else {
        const int cc = c - TN;
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < T::WARPS_M; ++w) s += red_pd[w * (TN / 2) + cc];
        p.pairdot[(long)bi * (p.ldo / 2) + (long)bj * (TN / 2) + cc] = s;
      }
    }
  }
}

template <int ALAY, int BLAY, int EPI, class T = Tile128>
inline int gemm_launch(const GemmArgs& a, cudaStream_t st) {
  static bool configured_on[GPK_MAX_DEVICES] = {};
  bool& configured = configured_on[current_device_slot()];
  if (!configured) {
    GPK_CUDA_OK(cudaFuncSetAttribute(dgemm_dmma_kernel<ALAY, BLAY, EPI, T>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, T::SMEM_BYTES));
    configured = true;
  }
  if (a.M <= 0 || a.N <= 0) return 0;
  if (a.M % GEMM_BM || a.N % GEMM_BN || a.K % GEMM_BK) {
    snprintf(g_err, sizeof(g_err), "gemm_launch: extents %d,%d,%d not tile multiples", a.M, a.N, a.K);
    return -2;
  }
  dim3 grid(a.N / T::TN, a.M / T::TM);
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (g_prof_on) {
    GPK_CUDA_OK(cudaEventCreate(&e0));
    GPK_CUDA_OK(cudaEventCreate(&e1));
    GPK_CUDA_OK(cudaEventRecord(e0, st));
  }
  GPK_CUDA_OK(launch_pdl(dgemm_dmma_kernel<ALAY, BLAY, EPI, T>, grid, dim3(T::THREADS), (size_t)T::SMEM_BYTES, st, a));
  GPK_LAUNCH_OK();
  if (g_prof_on) {
    GPK_CUDA_OK(cudaEventRecord(e1, st));
    prof_push(e0, e1);
  }
  return 0;
}

// Tile choice of the store-epilogue GEMMs: 64x128 (2 CTAs/SM) when the grid has at least two full waves of
// them, else 64x64 (3 CTAs/SM) so that the small nodes of the recursion still spread over the SMs.
template <int ALAY, int BLAY>
inline int gemm_store_auto(const GemmArgs& a, cudaStream_t st) {
  long tiles = (long)(a.M / 64) * (a.N / 128);
  if (a.lower_only) tiles /= 2;
  if (tiles >= 2 * 2 * 148) return gemm_launch<ALAY, BLAY, EPI_STORE, Tile64x128>(a, st);
  // sub-2048 nodes of the recursion: 64x64 tiles leave 1.7 CTAs per SM at order 1024 and 4-64 CTAs in all below;
  // 64x32 tiles (4 CTAs/SM) double the CTA count for the same work: 16.9 -> 12.2 ms of small GEMMs per fit iteration at
  // n = 32768, 2.0 -> 1.45 ms at n = 4096 (32x32 tiles measured the same as 64x32)
  const long t64 = (long)(a.M / 64) * (a.N / 64);
  if (t64 <= 512) return gemm_launch<ALAY, BLAY, EPI_STORE, GemmTile<64, 32, 4, 4>>(a, st);
  return gemm_launch<ALAY, BLAY, EPI_STORE, Tile64>(a, st);
}

inline GemmArgs gemm_args(const double* A, long lda, const double* B, long ldb, double* C, long ldc,
                          int M, int N, int K, double alpha, double beta, int krange, int lower_only) {
  GemmArgs a;
  memset(&a, 0, sizeof(a));
  a.A = A; a.lda = lda; a.B = B; a.ldb = ldb; a.C = C; a.ldc = ldc;
  a.M = M; a.N = N; a.K = K; a.alpha = alpha; a.beta = beta;
  a.krange = krange; a.lower_only = lower_only;
  a.reverse_bi = (krange == K_UPTO_BI) ? 1 : 0;
  return a;
}

}  // namespace gpk
