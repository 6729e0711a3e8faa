// FP64 GEMM through the INT8 tcgen05 tensor cores (Ozaki scheme II: Chinese-remainder form, exact int32 accumulation in
// TMEM, exact reconstruction to FP64).
//
//   C[m,n] = beta*C[m,n] + alpha * sum_{k in krange(bi,bj)} A(m,k) * B(n,k)        (same contract as dgemm_dmma.cuh)
//
// Why: every O(n^3) flop of the GP hot path (recursive Cholesky + triangular inverse, K^-1 = X^T X, the predictive
// variance / Girard quadratic forms) is this contraction. The FP64 DMMA pipe of B200 peaks at 37 TFLOP/s and
// dgemm_dmma.cuh already keeps it 97% busy; the INT8 tensor pipe (tcgen05.mma.kind::i8, 8192 MAC/clk/SM) is ~120x
// wider, and an FP64 product can be computed EXACTLY from int8 products:
//
//   A' = rn(A * 2^(bits - eA[m]))  (integers, |A'| <= 2^bits, eA[m] = exponent of the row maximum), B' likewise;
//   C' = A' B'^T is an exact integer matrix with |C'| <= K 2^(2 bits) < P/2,  P = m_0 m_1 ... m_{N-1}
//   (pairwise coprime moduli <= 256, tools/gen_crt_tables.py).  R_i = (A' mod m_i)(B' mod m_i)^T is an exact int32 GEMM
//   of balanced int8 residues (|R_i| <= K 2^14), and
//   C'/P = sum_i s_i/m_i (mod 1),  s_i = (R_i u_i) mod m_i,  u_i = (P/m_i)^-1 mod m_i      (Chinese remainder theorem).
//   16 moduli give P = 2^125.4: bits = 54 at K = 32768, one bit more than an FP64 significand, no dropped products.
//
// One route, three kernels (this file + oz_crt_planes.cuh):
//   oz_absmax_* + oz_residue_*_kernel   operand -> per-row power-of-two scale + one int8 residue plane per modulus
//   oz_crt_planes_kernel                one tcgen05 GEMM per modulus (CTA pair, 256x256 tile, TMA ring, TMEM double
//                                       buffer), epilogue writes s_i as one byte per element and modulus
//   oz_crt_reconstruct_kernel           96-bit fixed-point sum of s_i round(2^96/m_i) -> FP64, scales, alpha/beta or the
//                                       row reductions of the query path
// Earlier variants (digit products: 36 int8 GEMMs; CRT with the 96-bit sum kept in TMEM: tensor pipe 47 % active;
// 4-CTA multicast clusters; split-K) were measured in round 1 (profiles/r1_*) and removed: this is the only route.
#pragma once
#include <cuda.h>

#include "dgemm_dmma.cuh"
#include "oz_crt_tables.h"

namespace gpk {
namespace oz {

constexpr int BM = 128, BN = 128, BK = 128;        // operand tile; BK int8 elements = one 128-byte swizzle row
constexpr int TILE_BYTES = BM * BK;                // 16 KB per (modulus, k-block) operand tile
constexpr int EPI_WARPS = 8;
constexpr int THREADS = 64 + EPI_WARPS * 32;       // 320: TMA warp, MMA warp, 8 epilogue warps
constexpr int TMEM_COLS = 512;

constexpr int OZ_EPI_STORE = 0;   // C = beta*C + alpha*acc
// per-row sums over a 128-column block of acc^2 and of acc[m]*acc[m^1] (adjacent rows): the quadratic forms
// |X k*|^2 and (X C).(X tr) of prediction / propagation with queries as ROWS
constexpr int OZ_EPI_ROWSQ = 1;

// ---- PTX wrappers ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// A protocol error must end the kernel with a trap (reported as a launch failure), never hang the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- CTA-pair (cta_group::2) pieces --------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}\n"
      ::"r"(smem_u32(bar)), "r"(rank)
      : "memory");
}
// Residue planes are stored tiled: [plane][row tile][k block][128 rows][128 bytes], so one operand tile is 16 KB of
// contiguous memory; the tensor map is 5-D {128 B, 128 rows, k blocks, row tiles, planes}.
// TMA load issued by either CTA of the pair; the transaction bytes are counted on the LEADER CTA's barrier
// (bit 24 of a shared::cluster address selects the CTA of the pair: cute's Sm100MmaPeerBitMask)
__device__ __forceinline__ void tma_load_tile_pair(void* dst, const CUtensorMap* tm, uint64_t* bar, int row_in_tile,
                                                   int kb, int row_tile, int plane) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
      "%7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(0), "r"(row_in_tile), "r"(kb), "r"(row_tile),
        "r"(plane)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrives on the barrier at this offset in BOTH CTAs of the pair when the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t mask = 3) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void umma_i8_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// exact int32 -> double without the conversion pipe: 2^52 + (v + 2^31) is built in the mantissa, one DADD removes the bias
__device__ __forceinline__ double i32_to_f64(uint32_t v) {
  return __hiloint2double(0x43300000, (int)(v ^ 0x80000000u)) - 4503601774854144.0;
}

// UMMA shared-memory descriptor of a K-major operand tile written by TMA with SWIZZLE_128B: rows of 128 bytes,
// 8-row groups 1024 bytes apart (stride byte offset), 1024-byte aligned tile (base offset 0), descriptor version 1.
// Bit layout: cute::UMMA::SmemDescriptor (start [0,14), LBO [16,30), SBO [32,46), version [46,48), layout [61,64)).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;             // leading byte offset: unused for swizzled K-major layouts
  d |= (uint64_t)(1024 >> 4) << 32;   // stride byte offset
  d |= (uint64_t)1 << 46;             // version (Blackwell)
  d |= (uint64_t)2 << 61;             // SWIZZLE_128B
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D = S32, A = B = signed int8, both K-major, M x N.
__host__ __device__ constexpr uint32_t umma_idesc_i8(int M, int N) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- slicing ---------------------------------------------------------------------------------------------------
// Operand element (r, k): TRANS == 0 -> src[r*ld + k]; TRANS == 1 -> src[k*ld + r].
// lower != 0: only source elements with (source col tile) <= (source row tile) are valid, the rest read as zero
// (the upper 128-tiles of X = L^-1 are never written).
template <int TRANS>
__device__ __forceinline__ bool oz_valid(int r, int k, int lower) {
  if (!lower) return true;
  return TRANS ? ((r >> 7) <= (k >> 7)) : ((k >> 7) <= (r >> 7));
}
// Masked-out tiles are written as zeros only next to the diagonal: the GEMM k-ranges never read a masked tile further
// away, so those stay unwritten. `extra` = how many tiles beyond the diagonal: 1 for the CTA-pair union of the 128-tile
// ranges, 1 + WIDEN_TILES when the product is long enough (K >= WIDEN_MIN_K) for the planes kernel to give every tile
// of a raster band the same k range (see oz_crt_planes_kernel: tiles in step share their operand panels in L2).
constexpr int WIDEN_MIN_K = 16384;   // at K = 8192 the added k-blocks and zero tiles cost more than the sharing saves (propagate_GA -3 %)
// CTA raster of the planes kernel: consecutive CTA pairs sweep bands of PLANES_BAND pair rows (or pair columns). Bands
// of 2 / 6 / 8 / 16 ran 6-22 % slower on the K^-1 launch at n = 32768 (profiles/r2_tune_planes.txt).
constexpr int PLANES_BAND = 4;
constexpr int WIDEN_TILES = 2 * (PLANES_BAND - 1);   // k-blocks between the first and the last pair row of a band
inline int zero_fill_extra(int K) { return K >= WIDEN_MIN_K ? 1 + WIDEN_TILES : 1; }
template <int TRANS>
__device__ __forceinline__ bool oz_needed(int r, int k, int lower, int extra) {
  if (!lower) return true;
  return TRANS ? ((r >> 7) <= (k >> 7) + extra) : ((k >> 7) <= (r >> 7) + extra);
}

// byte offset of element (plane p, operand row r, k) in the tiled slice layout
__device__ __forceinline__ size_t slice_offset(int rows, int K, int p, int r, int k) {
  const size_t tiles_per_plane = (size_t)(rows >> 7) * (size_t)(K >> 7);
  return (((size_t)p * tiles_per_plane + (size_t)(r >> 7) * (size_t)(K >> 7) + (size_t)(k >> 7)) << 14) +
         ((size_t)(r & 127) << 7) + (size_t)(k & 127);
}

// mx[r] = bits of max_k |operand(r,k)| over the valid tiles, or of +Inf if one of them is not finite. The maximum is
// taken on the bit patterns: non-negative doubles order like them, and |NaN| orders above +Inf (fmax would drop it).
constexpr unsigned long long OZ_INF_BITS = 0x7ff0000000000000ull;
__device__ __forceinline__ unsigned long long oz_abs_bits(double x) {
  return (unsigned long long)__double_as_longlong(x) & 0x7fffffffffffffffull;
}
__global__ void __launch_bounds__(256) oz_absmax_rows_kernel(const double* __restrict__ src, long ld, int K, int lower,
                                                             unsigned long long* __restrict__ mx) {
  __shared__ unsigned long long red[8];
  const int r = blockIdx.x;
  const int kend = lower ? min(K, ((r >> 7) + 1) << 7) : K;
  const double* row = src + (long)r * ld;
  unsigned long long m = 0ull;
  for (int k = threadIdx.x; k < kend; k += 256) m = max(m, oz_abs_bits(row[k]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) m = max(m, red[i]);
    mx[r] = min(m, OZ_INF_BITS);
  }
}
// transposed operand: rows of the operand are columns of the source. grid (rows/32, ceil(K/1024)), 256 threads.
__global__ void __launch_bounds__(256) oz_absmax_cols_kernel(const double* __restrict__ src, long ld, int K, int lower,
                                                             unsigned long long* __restrict__ mx) {
  __shared__ unsigned long long red[8][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int r = blockIdx.x * 32 + lane;
  const int k0 = blockIdx.y * 1024, k1 = min(K, k0 + 1024);
  const int kfirst = lower ? ((r >> 7) << 7) : 0;
  unsigned long long m = 0ull;
  for (int k = k0 + w; k < k1; k += 8)
    if (k >= kfirst) m = max(m, oz_abs_bits(src[(long)k * ld + r]));
  red[w][lane] = m;
  __syncthreads();
  if (w == 0) {
#pragma unroll
    for (int i = 1; i < 8; ++i) m = max(m, red[i][lane]);
    atomicMax(mx + r, min(m, OZ_INF_BITS));
  }
}

// exponent e with |x| < 2^e for every element of the row; rows that are zero (or not finite) get e = 0.
// Rows whose maximum is below 2^-900 are flushed to zero: their elements scale below 2^(bits - 900 - 1) and round to 0.
__device__ __forceinline__ int oz_row_exponent(unsigned long long bits) {
  const double m = __longlong_as_double((long long)bits);
  if (!(m > 0.0) || bits >= OZ_INF_BITS) return 0;
  int e = ilogb(m) + 1;
  if (e < -900) e = -900;
  return e;
}

// ---- residues ---------------------------------------------------------------------------------------------------
__constant__ CrtModulus c_crt[CRT_MAX_MODULI];   // m, magic, W, c1..c3 do not depend on the number of moduli in use

inline int crt_upload_constants() {
  static bool done_on[GPK_MAX_DEVICES] = {};
  bool& done = done_on[current_device_slot()];
  if (done) return 0;
  const CrtSet& last = CRT_SETS[CRT_MAX_MODULI - CRT_MIN_MODULI];
  GPK_CUDA_OK(cudaMemcpyToSymbol(c_crt, last.mod, sizeof(CrtModulus) * CRT_MAX_MODULI));
  done = true;
  return 0;
}
inline const CrtSet& crt_set(int nmod) { return CRT_SETS[nmod - CRT_MIN_MODULI]; }
// largest operand width with K 2^(2 bits + 1) < P
inline int crt_bits(int K, int nmod) {
  int b = (int)floor((crt_set(nmod).log2P - 1.0 - log2((double)K) - 1e-6) / 2.0);
  return b > 60 ? 60 : b;
}

// fewest moduli that carry `want_bits`-bit operands over an inner dimension K (the largest set if none does)
inline int crt_moduli_for(int K, int want_bits) {
  for (int nmod = CRT_MIN_MODULI; nmod < CRT_MAX_MODULI; ++nmod)
    if (crt_bits(K, nmod) >= want_bits) return nmod;
  return CRT_MAX_MODULI;
}

// Residues of 16 elements for one modulus at a time, balanced into int8. X + 2^62 >= 0 is split into its 8 bytes; two
// dp4a against the balanced residues of 2^(8j) give t == X + half (mod m), 0 <= t < 2^22 (the offsets sit in the dp4a
// accumulator constant); the quotient umulhi(t, ceil(2^32/m)) is exact for such t, so r = t mod m is canonical and r - half is the
// balanced residue. The modulus loop is the OUTER loop: its 5 constants are loaded once per 16 elements and the 16 bytes
// of a plane are stored as soon as they are complete (no per-plane register arrays).
// The kernel is bound by instruction ISSUE (6 per residue: 2 IDP.4A, IMAD.HI, IMAD, IADD, PRMT), not by the multiply pipe
// alone: a variant with 4 multiply-pipe and 4-5 ALU operations per residue (32-bit multiply + shift for the quotient,
// compare / subtract for the balancing; exhaustively checked, parity-clean) ran 33 % SLOWER (6.43 vs 4.85 ms for two
// 16384^2 operands, round 2). Fewer instructions per residue need the byte dot products on mma.sync fragments.
__device__ __forceinline__ int dp4a_us(uint32_t a, uint32_t b, int c) {
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ void oz_split(double x, double scale, uint32_t& lo, uint32_t& hi) {
  const unsigned long long X = (unsigned long long)(__double2ll_rn(x * scale) + (1ll << 62));
  lo = (uint32_t)X;
  hi = (uint32_t)(X >> 32);
}
__device__ __forceinline__ uint4 oz_residues16(const uint32_t (&lo)[16], const uint32_t (&hi)[16], int i) {
  const uint32_t dlo = c_crt[i].dlo, dhi = c_crt[i].dhi, m32c = c_crt[i].m32c;
  const int dinit = c_crt[i].dinit, m = c_crt[i].m, half = c_crt[i].half;
  uint32_t w[4];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint32_t word = 0u;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int e = g * 4 + b;
      const int t = dp4a_us(lo[e], dlo, dp4a_us(hi[e], dhi, dinit));
      const uint32_t q = __umulhi((uint32_t)t, m32c);
      const int r = t - (int)q * m - half;
      word = __byte_perm(word, (uint32_t)r, 0x3210u ^ ((0x4u ^ (uint32_t)b) << (4 * b)));
    }
    w[g] = word;
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

__global__ void __launch_bounds__(256) oz_residue_rows_kernel(const double* __restrict__ src, long ld, int rows, int K,
                                                              int lower, int nmod, int bits, int extra,
                                                              const unsigned long long* __restrict__ mx,
                                                              int8_t* __restrict__ sl, double* __restrict__ sc) {
  const long idx = (long)blockIdx.x * 256 + threadIdx.x;
  const int cpr = K >> 4;
  if (idx >= (long)rows * cpr) return;
  const int r = (int)(idx / cpr), ch = (int)(idx % cpr);
  // a row with a non-finite element: scale NaN, residues zero, so the reconstruction makes the whole output row NaN
  const bool finite = mx[r] < OZ_INF_BITS;
  const int e = oz_row_exponent(mx[r]);
  if (ch == 0) sc[r] = finite ? ldexp(1.0, e - bits) : __longlong_as_double(0x7ff8000000000000ll);
  const double scale = ldexp(1.0, bits - e);
  const int k0 = ch << 4;
  if (!oz_needed<0>(r, k0, lower, extra)) return;
  uint32_t lo[16], hi[16];
  if (finite && oz_valid<0>(r, k0, lower)) {
    const double2* s2 = reinterpret_cast<const double2*>(src + (long)r * ld + k0);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const double2 v = s2[i];
      oz_split(v.x, scale, lo[2 * i], hi[2 * i]);
      oz_split(v.y, scale, lo[2 * i + 1], hi[2 * i + 1]);
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) oz_split(0.0, scale, lo[i], hi[i]);
  }
  for (int p = 0; p < nmod; ++p)
    *reinterpret_cast<uint4*>(sl + slice_offset(rows, K, p, r, k0)) = oz_residues16(lo, hi, p);
}

// transposed operand: lane = operand row (source column), thread = 16 consecutive k. grid (rows/32, ceil(K/128)).
__global__ void __launch_bounds__(256) oz_residue_cols_kernel(const double* __restrict__ src, long ld, int rows, int K,
                                                              int lower, int nmod, int bits, int extra,
                                                              const unsigned long long* __restrict__ mx,
                                                              int8_t* __restrict__ sl, double* __restrict__ sc) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int r = blockIdx.x * 32 + lane;
  const int k0 = (blockIdx.y * 8 + w) * 16;
  if (k0 >= K) return;
  const bool finite = mx[r] < OZ_INF_BITS;   // as in oz_residue_rows_kernel
  const int e = oz_row_exponent(mx[r]);
  if (k0 == 0) sc[r] = finite ? ldexp(1.0, e - bits) : __longlong_as_double(0x7ff8000000000000ll);
  const double scale = ldexp(1.0, bits - e);
  if (!oz_needed<1>(r, k0, lower, extra)) return;
  uint32_t lo[16], hi[16];
  const bool valid = finite && oz_valid<1>(r, k0, lower);
#pragma unroll
  for (int i = 0; i < 16; ++i) oz_split(valid ? src[(long)(k0 + i) * ld + r] : 0.0, scale, lo[i], hi[i]);
  for (int p = 0; p < nmod; ++p)
    *reinterpret_cast<uint4*>(sl + slice_offset(rows, K, p, r, k0)) = oz_residues16(lo, hi, p);
}

#include "oz_crt_planes.cuh"

// ---- host side -----------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      f = nullptr;
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}

// 5-D view {128 B, 128 rows, k blocks, row tiles, planes} of a tiled slice buffer; box = one tile (or its row half)
inline int make_tmap(CUtensorMap* tm, const int8_t* base, int rows, int K, int S, int box_rows = BM) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled entry point not available");
    return -1;
  }
  const cuuint64_t kbs = (cuuint64_t)(K / BK), rts = (cuuint64_t)(rows / BM);
  cuuint64_t dims[5] = {(cuuint64_t)BK, (cuuint64_t)BM, kbs, rts, (cuuint64_t)S};
  cuuint64_t strides[4] = {(cuuint64_t)BK, (cuuint64_t)TILE_BYTES, (cuuint64_t)TILE_BYTES * kbs,
                           (cuuint64_t)TILE_BYTES * kbs * rts};
  cuuint32_t box[5] = {(cuuint32_t)BK, (cuuint32_t)box_rows, 1, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 5, const_cast<int8_t*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled failed (%d) rows=%d K=%d S=%d", (int)r, rows, K, S);
    return -1;
  }
  return 0;
}
// One operand in residue form: S planes of rows x K int8 (K-major, tiled) and the per-row scales 2^(e - bits).
struct Operand {
  int8_t* sl = nullptr;
  double* sc = nullptr;
  int rows = 0, K = 0, S = 0;
  int bits = 0;                  // operand width (|A'| <= 2^bits)
  uint8_t* out = nullptr;        // residue planes of the product (owned by the operand's workspace)
  size_t out_cap = 0;
  static size_t slice_bytes(int rows, int K, int S) { return (size_t)S * rows * K; }
};

// Reduce `src` (trans == 0: rows x K with leading dimension ld; trans == 1: K x rows) into op.sl / op.sc.
// mx: scratch of `rows` 64-bit words.
inline int slice_operand(const double* src, long ld, int trans, int lower, Operand& op, unsigned long long* mx,
                         cudaStream_t st) {
  if (op.rows % BM || op.K % BK || op.S < CRT_MIN_MODULI || op.S > CRT_MAX_MODULI) {
    snprintf(g_err, sizeof(g_err), "slice_operand: bad shape rows=%d K=%d moduli=%d", op.rows, op.K, op.S);
    return -2;
  }
  GPK_TRY(crt_upload_constants());
  op.bits = crt_bits(op.K, op.S);
  if (!trans) {
    oz_absmax_rows_kernel<<<op.rows, 256, 0, st>>>(src, ld, op.K, lower, mx);
    GPK_LAUNCH_OK();
    const long chunks = (long)op.rows * (op.K >> 4);
    oz_residue_rows_kernel<<<(unsigned)((chunks + 255) / 256), 256, 0, st>>>(src, ld, op.rows, op.K, lower, op.S,
                                                                            op.bits, zero_fill_extra(op.K), mx, op.sl, op.sc);
    GPK_LAUNCH_OK();
  } else {
    GPK_CUDA_OK(cudaMemsetAsync(mx, 0, (size_t)op.rows * sizeof(unsigned long long), st));
    dim3 g1(op.rows / 32, (op.K + 1023) / 1024);
    oz_absmax_cols_kernel<<<g1, 256, 0, st>>>(src, ld, op.K, lower, mx);
    GPK_LAUNCH_OK();
    dim3 g2(op.rows / 32, (op.K + 127) / 128);
    oz_residue_cols_kernel<<<g2, 256, 0, st>>>(src, ld, op.rows, op.K, lower, op.S, op.bits, zero_fill_extra(op.K), mx, op.sl, op.sc);
    GPK_LAUNCH_OK();
  }
  return 0;
}

// scratch of the position lock (oz_crt_planes_kernel): one slot per SM, shared by every launch on the device (a slot
// belongs to the one CTA that is resident on that SM)
inline int* g_spill_dev[GPK_MAX_DEVICES] = {};
constexpr size_t SPILL_BYTES = (size_t)SPILL_SLOTS * BM * Q_BN * sizeof(int);

thread_local int g_position_lock = 2;   // gpk_test_position_lock: 0 = lock on the modulus only, 1 = + split first modulus, 2 = + band-uniform k ranges

// C = beta*C + alpha * A * B^T over the per-tile k range, from operands in residue form (A.K == B.K, A.S == B.S):
// per row panel that fits A.out, one GEMM launch (all moduli) and one reconstruction launch.
inline int gemm_sliced(const Operand& A, const Operand& B, double* C, long ldc, double alpha, double beta, int krange,
                       int lower_only, cudaStream_t st, int epi = OZ_EPI_STORE, double* colsq = nullptr,
                       double* pairdot = nullptr, long ldo = 0) {
  if (A.K != B.K || A.S != B.S) {
    snprintf(g_err, sizeof(g_err), "gemm_sliced: operand mismatch K %d/%d moduli %d/%d", A.K, B.K, A.S, B.S);
    return -2;
  }
  if (A.bits != B.bits || A.bits != crt_bits(A.K, A.S)) {
    snprintf(g_err, sizeof(g_err), "gemm_sliced: operand widths %d/%d do not match K=%d", A.bits, B.bits, A.K);
    return -2;
  }
  const long Nc = ((long)B.rows + Q_BN - 1) / Q_BN * Q_BN;
  const size_t per_row = (size_t)A.S * (size_t)Nc;
  const long panel = (long)(A.out_cap / per_row) / 256 * 256;
  if (!A.out || panel < 256) {
    snprintf(g_err, sizeof(g_err), "gemm_sliced: the residue-plane buffer (%zu bytes) cannot hold a 256-row panel of %ld columns",
             A.out_cap, Nc);
    return -4;
  }
  static bool configured_on[GPK_MAX_DEVICES] = {};
  bool& configured = configured_on[current_device_slot()];
  if (!configured) {
    GPK_CUDA_OK(cudaFuncSetAttribute(oz_crt_planes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Q_SMEM_BYTES));
    configured = true;
  }
  CUtensorMap tmA, tmB;
  GPK_TRY(make_tmap(&tmA, A.sl, A.rows, A.K, A.S, BM));
  GPK_TRY(make_tmap(&tmB, B.sl, B.rows, B.K, B.S, BM));
  const CrtSet& cs = crt_set(A.S);
  PlaneArgs g;
  memset(&g, 0, sizeof(g));
  g.res = A.out; g.res_ld = Nc;
  g.M = A.rows; g.N = B.rows; g.K = A.K; g.krange = krange; g.lower_only = lower_only; g.nmod = A.S;
  // band-uniform k ranges (and column bands for the column-dependent ranges) when the operands are far larger than L2
  g.widen = (g_position_lock >= 2 && A.K >= WIDEN_MIN_K &&
             (krange == K_FROM_BI || krange == K_UPTO_BI || krange == K_FROM_BJ || krange == K_UPTO_BJ)) ? 1 : 0;
  g.band_cols = (g.widen && (krange == K_FROM_BJ || krange == K_UPTO_BJ)) ? 1 : 0;
  ReconArgs r;
  memset(&r, 0, sizeof(r));
  r.res = A.out; r.res_ld = Nc;
  r.C = C; r.ldc = ldc; r.scA = A.sc; r.scB = B.sc; r.alpha = alpha; r.beta = beta;
  r.M = A.rows; r.N = B.rows; r.K = A.K; r.krange = krange; r.lower_only = lower_only; r.nmod = A.S;
  r.p_scaled = cs.p_scaled;
  r.colsq = colsq; r.pairdot = pairdot; r.ldo = ldo;
  for (int i = 0; i < A.S; ++i) {
    g.m[i] = cs.mod[i].m; g.magic[i] = cs.mod[i].magic; g.u[i] = (uint32_t)cs.mod[i].u;
    const uint32_t w[3] = {cs.mod[i].w0, cs.mod[i].w1, cs.mod[i].w2};
    for (int j = 0; j < 6; ++j) {
      const uint32_t limb = (w[j >> 1] >> (16 * (j & 1))) & 0xffffu;
      r.wp[i >> 1][j] |= limb << (16 * (i & 1));
    }
  }
  // position counters (see oz_crt_planes_kernel): a fresh one per launch, launches on different streams may overlap
  static unsigned int* phase_dev_on[GPK_MAX_DEVICES] = {};
  unsigned int*& phase_dev = phase_dev_on[current_device_slot()];
  if (!phase_dev) {
    GPK_CUDA_OK(cudaMalloc((void**)&phase_dev, 64 * sizeof(unsigned int)));
    GPK_CUDA_OK(poison_fill(phase_dev, 64 * sizeof(unsigned int)));
  }
  static thread_local int phase_next = 0;
  int*& spill_dev = g_spill_dev[current_device_slot()];
  if (!spill_dev) {
    GPK_CUDA_OK(cudaMalloc((void**)&spill_dev, SPILL_BYTES));
    GPK_CUDA_OK(poison_fill(spill_dev, SPILL_BYTES));
  }
  g.spill = g_position_lock ? spill_dev : nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (g_prof_on) {
    GPK_CUDA_OK(cudaEventCreate(&e0));
    GPK_CUDA_OK(cudaEventCreate(&e1));
    GPK_CUDA_OK(cudaEventRecord(e0, st));
  }
  for (long row0 = 0; row0 < A.rows; row0 += panel) {
    const long rows = (A.rows - row0 < panel) ? A.rows - row0 : panel;
    const long rows_pad = (rows + 255) / 256 * 256;
    g.row_tile0 = (int)(row0 / 256);
    g.res_plane = rows_pad * Nc;
    r.row0 = (int)row0;
    r.res_plane = g.res_plane;
    // lower-only products: the tiles right of the panel's last row are never computed
    long ncol_tiles = Nc / Q_BN;
    if (lower_only && (row0 + rows_pad) / Q_BN < ncol_tiles) ncol_tiles = (row0 + rows_pad) / Q_BN;
    g.phase = phase_dev + (phase_next++ & 63);
    GPK_CUDA_OK(cudaMemsetAsync(g.phase, 0, sizeof(unsigned int), st));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3((unsigned)(2 * ncol_tiles), (unsigned)(rows_pad / 256));
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = Q_SMEM_BYTES;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    GPK_CUDA_OK(cudaLaunchKernelEx(&cfg, oz_crt_planes_kernel, tmA, tmB, g));
    GPK_LAUNCH_OK();
    long ncol_blocks = B.rows / 128;
    if (lower_only && (row0 + rows) / 128 < ncol_blocks) ncol_blocks = (row0 + rows) / 128;
    dim3 rg((unsigned)ncol_blocks, (unsigned)(rows / 8));   // rows are multiples of 8
    const int ng = (A.S + 3) / 4;      // 2..RECON_GROUPS
    const bool store = epi == OZ_EPI_STORE;
    auto kernel = (ng <= 2) ? (store ? oz_crt_reconstruct_kernel<OZ_EPI_STORE, 2> : oz_crt_reconstruct_kernel<OZ_EPI_ROWSQ, 2>)
                : (ng == 3) ? (store ? oz_crt_reconstruct_kernel<OZ_EPI_STORE, 3> : oz_crt_reconstruct_kernel<OZ_EPI_ROWSQ, 3>)
                : (ng == 4) ? (store ? oz_crt_reconstruct_kernel<OZ_EPI_STORE, 4> : oz_crt_reconstruct_kernel<OZ_EPI_ROWSQ, 4>)
                            : (store ? oz_crt_reconstruct_kernel<OZ_EPI_STORE, 5> : oz_crt_reconstruct_kernel<OZ_EPI_ROWSQ, 5>);
    kernel<<<rg, 256, 0, st>>>(r);
    GPK_LAUNCH_OK();
  }
  if (g_prof_on) {
    GPK_CUDA_OK(cudaEventRecord(e1, st));
    prof_push(e0, e1);
  }
  return 0;
}

// Residue workspace of a handle: one int8 region (bump-allocated, reset between GEMM groups; everything that uses it
// is ordered on one stream), the per-row scales, the row-max scratch and the residue planes of the products.
struct Workspace {
  int8_t* buf = nullptr; size_t cap = 0, top = 0;
  double* sc = nullptr; size_t sc_cap = 0, sc_top = 0;
  unsigned long long* mx = nullptr; size_t mx_cap = 0;
  uint8_t* out = nullptr; size_t out_cap = 0;   // residue planes of the products
  int S = CRT_MIN_MODULI;   // moduli per operand
  int min_dim = 2048;       // GEMMs with a smaller inner block stay on the DMMA kernel
  void reset() { top = 0; sc_top = 0; }
  Operand alloc(int rows, int K) {
    Operand op;
    const size_t bytes = Operand::slice_bytes(rows, K, S);
    if (top + bytes > cap || sc_top + (size_t)rows > sc_cap || (size_t)rows > mx_cap) return op;
    op.sl = buf + top; op.sc = sc + sc_top; op.rows = rows; op.K = K; op.S = S;
    op.out = out; op.out_cap = out_cap;
    top += bytes; sc_top += (size_t)rows;
    return op;
  }
  int ensure_out(size_t bytes) {
    if (bytes <= out_cap) return 0;
    if (out) cudaFree(out);
    out = nullptr; out_cap = 0;
    if (cudaMalloc((void**)&out, bytes) != cudaSuccess) { cudaGetLastError(); out = nullptr; return -1; }
    out_cap = bytes;
    if (poison_fill(out, bytes) != cudaSuccess) return -1;
    return 0;
  }
  int ensure(size_t bytes, size_t rows_total, size_t rows_max) {
    if (bytes > cap) {
      if (buf) cudaFree(buf);
      buf = nullptr; cap = 0;
      if (cudaMalloc((void**)&buf, bytes) != cudaSuccess) { cudaGetLastError(); buf = nullptr; return -1; }
      cap = bytes;
      if (poison_fill(buf, bytes) != cudaSuccess) return -1;
    }
    if (rows_total > sc_cap) {
      if (sc) cudaFree(sc);
      sc = nullptr; sc_cap = 0;
      if (cudaMalloc((void**)&sc, rows_total * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return -1; }
      sc_cap = rows_total;
      if (poison_fill(sc, rows_total * sizeof(double)) != cudaSuccess) return -1;
    }
    if (rows_max > mx_cap) {
      if (mx) cudaFree(mx);
      mx = nullptr; mx_cap = 0;
      if (cudaMalloc((void**)&mx, rows_max * sizeof(unsigned long long)) != cudaSuccess) { cudaGetLastError(); return -1; }
      mx_cap = rows_max;
      if (poison_fill(mx, rows_max * sizeof(unsigned long long)) != cudaSuccess) return -1;
    }
    return 0;
  }
  void release() {
    if (buf) cudaFree(buf);
    if (sc) cudaFree(sc);
    if (mx) cudaFree(mx);
    if (out) cudaFree(out);
    buf = nullptr; sc = nullptr; mx = nullptr; out = nullptr; cap = sc_cap = mx_cap = out_cap = 0;
  }
};

// C = beta*C + alpha * A * B^T with both operands reduced on the fly into the workspace (reset first).
// 0 on success, < 0 on error (-4: the workspace is too small; there is no fallback to another pipe).
inline int gemm_f64(Workspace& ws, const double* A, long lda, int transA, int lowerA, int M, const double* B, long ldb,
                    int transB, int lowerB, int N, int K, double* C, long ldc, double alpha, double beta, int krange,
                    int lower_only, cudaStream_t st) {
  ws.reset();
  Operand a = ws.alloc(M, K);
  const bool same = (A == B && lda == ldb && transA == transB && lowerA == lowerB && M == N);
  Operand b = same ? a : ws.alloc(N, K);
  if (!a.sl || !b.sl) {
    snprintf(g_err, sizeof(g_err), "gemm_f64: residue workspace too small for %d x %d and %d x %d operands", M, K, N, K);
    return -4;
  }
  GPK_TRY(slice_operand(A, lda, transA, lowerA, a, ws.mx, st));
  if (same) b = a;
  else GPK_TRY(slice_operand(B, ldb, transB, lowerB, b, ws.mx, st));
  return gemm_sliced(a, b, C, ldc, alpha, beta, krange, lower_only, st);
}

}  // namespace oz
}  // namespace gpk
