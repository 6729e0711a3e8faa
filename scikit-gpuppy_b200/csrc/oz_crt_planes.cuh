// CRT route: the tcgen05 GEMM kernel (residue planes out) and the reconstruction pass.   (included by oz_gemm.cuh, inside
// namespace gpk::oz)
//
// The int32 product of ONE modulus is all that lives in TMEM: 256 x 256 per CTA pair (each CTA 128 lanes x 256
// columns), double buffered (2 x 256 columns), so the MMAs of modulus i+1 run while the epilogue drains modulus i.
// The epilogue only maps R -> s = (R u_i) mod m_i in [0, m_i) and stores it as one byte per element into a residue
// plane; oz_crt_reconstruct_kernel then reads the nmod bytes of an element, forms the 96-bit sum
// sum_i s_i round(2^96/m_i) in registers and applies scales, alpha/beta or the row reductions. The price is 2 x nmod
// bytes of HBM traffic per output element (16 + 16 B next to the 8 B of the FP64 result); what it buys is N = 256
// tcgen05.mma instructions and 32 KB of operands per 4 M multiply-adds: ncu shows the tensor pipe 95 % active
// (profiles/r2c_ncu_oz_planes_lauum_n32768.txt) against 47 % for the round-1 kernel that kept the 96-bit sums in TMEM
// (384 of the 512 columns, tiles pinned to 256 x 128). With the pipe that busy the kernel's speed is its clock under the
// 1 kW cap, and the clock is set by what the kernel moves: see the position lock in the kernel body.

struct PlaneArgs {
  uint8_t* res; long res_ld; long res_plane;   // residue planes [nmod][panel rows][res_ld] (one byte per element)
  int M, N, K;
  int row_tile0;                               // first 256-row tile of this row panel
  int krange, lower_only;
  int widen, band_cols;                        // band-uniform k ranges; raster bands over columns instead of rows
  int nmod;
  unsigned int* phase;                         // position (modulus step, k-block) of the most advanced CTA pair of the launch
  int* spill;                                  // per-SM scratch for a split first modulus: [SPILL_SLOTS][128][256] int32
  int m[CRT_MAX_MODULI]; uint32_t magic[CRT_MAX_MODULI]; uint32_t u[CRT_MAX_MODULI];
};

constexpr int RECON_GROUPS = (CRT_MAX_MODULI + 3) / 4;   // groups of 4 moduli in the reconstruction kernel

struct ReconArgs {
  const uint8_t* res; long res_ld; long res_plane;
  double* C; long ldc;
  const double* scA; const double* scB;
  double alpha, beta;
  int M, N, K;
  int row0;                                    // first row of this panel (multiple of 256)
  int krange, lower_only;
  int nmod;
  double p_scaled;                             // P * 2^-96
  double* colsq; double* pairdot; long ldo;    // OZ_EPI_ROWSQ outputs
  uint32_t wp[2 * RECON_GROUPS][6];            // 16-bit limbs of W = round(2^96/m) of moduli 2k (low half) and 2k+1 (high)
};

constexpr int SPILL_SLOTS = 256;                                     // >= %nsmid
constexpr int Q_BN = 256;                                            // columns of a pair tile
constexpr int Q_STAGES = 7;
constexpr int Q_STAGE_BYTES = 2 * TILE_BYTES;                        // 32 KB: this CTA's A tile + its half (128 rows) of B
constexpr int Q_SMEM_BYTES = Q_STAGES * Q_STAGE_BYTES + 1024 + 256;

// k-block range [kb0, kb1) of the 256 x 256 tile (pair row bi2, pair column bx2): the union over its 128-tiles; the
// extra k-blocks meet operand tiles the slicer wrote as zeros (triangular masks), so the results agree
__host__ __device__ __forceinline__ void planes_krange(int krange, int K, int bi2, int bx2, int& kb0, int& kb1) {
  kb0 = 0;
  kb1 = K / BK;
  switch (krange) {
    case K_UPTO_BJ: kb1 = (kb1 < 2 * bx2 + 2) ? kb1 : 2 * bx2 + 2; break;
    case K_FROM_BJ: kb0 = (kb1 < 2 * bx2) ? kb1 : 2 * bx2; break;
    case K_UPTO_BI: kb1 = (kb1 < 2 * bi2 + 2) ? kb1 : 2 * bi2 + 2; break;
    case K_FROM_BI: kb0 = (kb1 < 2 * bi2) ? kb1 : 2 * bi2; break;
    default: break;
  }
}

__global__ void __launch_bounds__(THREADS, 1)
oz_crt_planes_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const __grid_constant__ PlaneArgs p) {
  extern __shared__ uint8_t oz_smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pp = (int)(rank & 1u);            // CTA within its pair: M half of the tile and N half of the B rows it loads

  const int nx = gridDim.x >> 1, ny = (int)gridDim.y;
  const int pid = (int)blockIdx.y * nx + (int)(blockIdx.x >> 1);
  int bx, by;
  int band_lo, band_hi;                       // first / last pair row (or column) of this tile's raster band
  if (!p.band_cols) {                         // bands of PLANES_BAND pair rows, column-major inside a band
    const int per_band = PLANES_BAND * nx;
    const int band = pid / per_band;
    const int first = band * PLANES_BAND;
    const int rows = min(ny - first, PLANES_BAND);
    const int rem = pid - band * per_band;
    by = first + rem % rows;
    bx = rem / rows;
    band_lo = first + p.row_tile0;
    band_hi = first + rows - 1 + p.row_tile0;
  } else {                                    // bands of PLANES_BAND pair columns, row-major inside a band
    const int per_band = PLANES_BAND * ny;
    const int band = pid / per_band;
    const int first = band * PLANES_BAND;
    const int cols = min(nx - first, PLANES_BAND);
    const int rem = pid - band * per_band;
    bx = first + rem % cols;
    by = rem / cols;
    band_lo = first;
    band_hi = first + cols - 1;
  }
  const int bi2 = by + p.row_tile0;           // global pair-row tile
  const int bi = 2 * bi2 + pp;                // 128-row tile of A this CTA loads
  const int bjt = 2 * bx + pp;                // 128-row tile of B this CTA loads
  if (p.lower_only && 2 * bx > 2 * bi2 + 1) return;           // the whole tile lies above the diagonal
  int kb0, kb1;
  planes_krange(p.krange, p.K, bi2, bx, kb0, kb1);
  if (kb1 <= kb0) return;                                     // empty range: the reconstruction reads it as zero
  if (p.widen) {
    // Every tile of the band gets the union of the band's k ranges (at most WIDEN_TILES more k-blocks than its own):
    // tiles with equal ranges that start in step stay in step, so the panels they share are read from DRAM once. The
    // added k-blocks meet residue tiles the slicer wrote as zeros (zero_fill_extra), the sums do not change.
    const int kbt = p.K / BK;
    switch (p.krange) {
      case K_FROM_BI: case K_FROM_BJ: { const int u = min(kb0, 2 * band_lo); kb0 = max(u, kb0 - WIDEN_TILES); if (kb0 < 0) kb0 = 0; } break;
      case K_UPTO_BI: case K_UPTO_BJ: { const int u = max(kb1, min(kbt, 2 * band_hi + 2)); kb1 = min(u, kb1 + WIDEN_TILES); if (kb1 > kbt) kb1 = kbt; } break;
      default: break;
    }
  }
  const int nmod = p.nmod;

  const uint32_t raw = smem_u32(oz_smem_raw);
  uint8_t* smem = oz_smem_raw + ((1024u - (raw & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Q_STAGES * Q_STAGE_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + Q_STAGES;
  uint64_t* tmem_full = bars + 2 * Q_STAGES;        // [2]
  uint64_t* tmem_empty = bars + 2 * Q_STAGES + 2;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * Q_STAGES + 4);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Q_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 2 * EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_pair(tmem_slot, TMEM_COLS);
  // Position lock. All CTA pairs of a launch that share operand panels should walk the same residue plane at the same
  // k-block at the same time: then they find each other's lines in L2 (a pass over one modulus takes 55-110 us, L2 keeps a
  // line for ~25-50 us at this kernel's fill rate). Every plane is written independently and the int32 sums are exact, so
  // both the order of the moduli and the order of the k-blocks are free:
  //   * the in-frame producers publish their position (modulus step << 16 | k-block offset) with atomicMax;
  //   * a pair that starts a tile adopts the position of the most advanced pair: it starts modulus i0 at k-block
  //     k_start, goes on with full passes over the other moduli in step with everybody else, and adds the missing part
  //     [kb0, k_start) of modulus i0 at the very end. The partial int32 sums of that split modulus wait in a per-SM
  //     scratch area (128 KB per CTA, L2-resident) and are added in the epilogue of the closing segment.
  // History: no lock, 364 GB of DRAM reads for 9 GB of residues at n = 16384 (round 1); lock on the modulus only, 116 GB
  // there and 175 GB for the K^-1 launch at n = 32768 (pairs up to a whole pass apart in k); triangular products ran
  // 12-16 % slower than the SYRK of the same size, whose equal tiles stay in step by themselves.
  uint32_t* phase_slot = tmem_slot + 1;
  if (rank == 0 && threadIdx.x == 0) *phase_slot = p.phase ? *reinterpret_cast<volatile unsigned int*>(p.phase) : 0u;
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  uint32_t phase0;
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %1, 0;\n\t"
      "ld.shared::cluster.u32 %0, [ra];\n\t}\n"
      : "=r"(phase0)
      : "r"(smem_u32(phase_slot))
      : "memory");
  uint32_t smid;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
  const int nk = kb1 - kb0;
  uint32_t mstep0 = phase0 >> 16;
  int k_start = kb0 + (int)(phase0 & 0xffffu);
  if (k_start >= kb1) { k_start = kb0; ++mstep0; }          // the leaders' pass is longer than this tile's: next modulus
  // both CTAs of the pair must take the same decision: the scratch test uses a bound, not this CTA's own SM id
  const bool split = k_start > kb0 && p.spill != nullptr;
  if (!split) k_start = kb0;
  const int i0 = (int)(mstep0 % (uint32_t)nmod);
  const int nseg = nmod + (split ? 1 : 0);
  // segment s: modulus (i0 + s) mod nmod over [kb0, kb1); with a split, segment 0 covers [k_start, kb1) and the closing
  // segment nmod covers [kb0, k_start) of modulus i0
#define SEG_MOD(sx) ((sx) < nmod ? ((i0 + (sx)) >= nmod ? i0 + (sx) - nmod : i0 + (sx)) : i0)
#define SEG_BEG(sx) ((split && (sx) == 0) ? k_start : kb0)
#define SEG_END(sx) ((split && (sx) == nmod) ? k_start : kb1)

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int sg = 0; sg < nseg; ++sg) {
        const int i = SEG_MOD(sg);
        const int kbeg = SEG_BEG(sg), kend = SEG_END(sg);
        for (int kb = kbeg; kb < kend; ++kb) {
          if (rank == 0 && p.phase && sg < nmod && ((kb - kbeg) & 3) == 0)
            atomicMax(p.phase, ((mstep0 + (uint32_t)sg) << 16) | (uint32_t)(kb - kb0));
          mbar_wait(&empty[stage], phase ^ 1u);
          uint8_t* st = smem + stage * Q_STAGE_BYTES;
          if (pp == 0) mbar_expect_tx(&full[stage], 2u * (uint32_t)Q_STAGE_BYTES);
          tma_load_tile_pair(st, &tmA, &full[stage], 0, kb, bi, i);
          tma_load_tile_pair(st + TILE_BYTES, &tmB, &full[stage], 0, kb, bjt, i);
          if (++stage == Q_STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && pp == 0) {
      constexpr uint32_t idesc = umma_idesc_i8(2 * BM, Q_BN);
      int stage = 0;
      uint32_t phase = 0;
      for (int sg = 0; sg < nseg; ++sg) {
        const int buf = sg & 1;
        if (sg >= 2) {
          mbar_wait(&tmem_empty[buf], (uint32_t)((sg >> 1) - 1) & 1u);   // the epilogue has drained this buffer
          tc_fence_after();
        }
        const uint32_t acc = tmem_base + (uint32_t)(buf * Q_BN);
        const int kbeg = SEG_BEG(sg), kend = SEG_END(sg);
        for (int kb = kbeg; kb < kend; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + stage * Q_STAGE_BYTES);
          const uint64_t ad = umma_desc_sw128(st);
          const uint64_t bd = umma_desc_sw128(st + TILE_BYTES);
#pragma unroll
          for (int k4 = 0; k4 < BK / 32; ++k4)
            umma_i8_pair(acc, ad + (uint64_t)(k4 * 2), bd + (uint64_t)(k4 * 2), idesc, (kb > kbeg) | (k4 > 0));
          umma_commit_pair(&empty[stage], 3);
          if (++stage == Q_STAGES) { stage = 0; phase ^= 1u; }
        }
        umma_commit_pair(&tmem_full[buf], 3);
      }
    }
  } else {
    const int quad = warp & 3, half = (warp - 2) >> 2;
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
    const long lrow = (long)by * (2 * BM) + pp * BM + row;           // row within the panel
    uint8_t* dst0 = p.res + lrow * p.res_ld + (long)bx * Q_BN + half * 128;
    // this thread's 128 int32 of the split modulus: [slot = SM][row][256 columns]
    int4* sp = split ? reinterpret_cast<int4*>(p.spill + ((size_t)(smid % SPILL_SLOTS) * BM + row) * Q_BN + half * 128) : nullptr;
    for (int sg = 0; sg < nseg; ++sg) {
      const int i = SEG_MOD(sg);
      const bool spill_out = split && sg == 0, add_in = split && sg == nmod;
      const int buf = sg & 1;
      if (lane == 0) mbar_wait(&tmem_full[buf], (uint32_t)(sg >> 1) & 1u);
      __syncwarp();
      tc_fence_after();
      const int m = p.m[i];
      const int magic = (int)p.magic[i];
      const uint32_t u = p.u[i];
      uint8_t* dst = dst0 + (long)i * p.res_plane;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t R[2][16];
        const uint32_t ta = lane_addr + (uint32_t)(buf * Q_BN + half * 128 + c * 32);
        tmem_ld16(ta, R[0]);
        tmem_ld16(ta + 16u, R[1]);
        tmem_ld_wait();
        if (c == 3) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(&tmem_empty[buf], rank & ~1u);   // segment sg+2 may overwrite the buffer
        }
        if (spill_out) {                 // partial sums of the split modulus: keep them for the closing segment
#pragma unroll
          for (int x = 0; x < 8; ++x) {
            const uint32_t* r4 = &R[x >> 2][(x & 3) * 4];
            sp[c * 8 + x] = make_int4((int)r4[0], (int)r4[1], (int)r4[2], (int)r4[3]);
          }
          continue;
        }
        if (add_in) {
#pragma unroll
          for (int x = 0; x < 8; ++x) {
            const int4 v = sp[c * 8 + x];
            uint32_t* r4 = &R[x >> 2][(x & 3) * 4];
            r4[0] += (uint32_t)v.x; r4[1] += (uint32_t)v.y; r4[2] += (uint32_t)v.z; r4[3] += (uint32_t)v.w;
          }
        }
        uint32_t pk[8];
#pragma unroll
        for (int x = 0; x < 32; ++x) {
          const int Rv = (int)R[x >> 4][x & 15];
          const int r = Rv - __mulhi(Rv, magic) * m + m;                        // == R (mod m), in [0, 3m)
          const uint32_t t = (uint32_t)r * u;
          uint32_t s = t - __umulhi(t, (uint32_t)magic) * (uint32_t)m;          // == R u (mod m), in [0, m+2]
          s = (s >= (uint32_t)m) ? s - (uint32_t)m : s;                         // canonical: one byte
          if ((x & 3) == 0) pk[x >> 2] = s;
          else pk[x >> 2] |= s << (8 * (x & 3));
        }
        uint4* o = reinterpret_cast<uint4*>(dst + c * 32);
        o[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        o[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
      }
    }
  }
#undef SEG_MOD
#undef SEG_BEG
#undef SEG_END
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

// Reconstruction: value = scA[row] scB[col] P 2^-96 * signed96( sum_i s_i W_i mod 2^96 ), W_i = round(2^96/m_i).
// One thread: 4 consecutive columns of one row (one 32-bit word per residue plane); a warp covers the 128 columns of a
// row, a block 8 rows x 128 columns (inside one 128-tile, so every range / triangle test is uniform over the block).
// The sum runs on the integer dot-product unit: the bytes of 4 moduli for one column are gathered into one word
// (two PRMT levels per 4 x 4 byte block) and multiplied against the 16-bit limbs of W_i with dp2a
// (sum of 2 products 16 bit x 8 bit): 12 dp2a per column and modulus group instead of ~47 multiply-add / carry /
// extract instructions; the six limb sums (< 2^29 each) are folded into the 96-bit value once per element.
// All loads of a thread are issued before the arithmetic starts; ~64 registers keep 4 blocks per SM resident
// (the first version, 16 columns per thread with 64-bit multiply-adds, ran at 16 warps per SM and 5.8 ms for the
// n = 32768 inverse; 8 columns + dp2a 4.2 ms; this one 3.5 ms; per fit iteration 31 -> 16.7 ms).
__device__ __forceinline__ uint32_t dp2a_lo(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t dp2a_hi(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// NG = groups of 4 moduli (compile time: no per-plane predicates or index multiplies for the groups that are full).
// Blocks of 2 or 4 warps side by side in a row (longer contiguous reads and writes per row) made no measurable
// difference (profiles/r2_tune_planes.txt).
template <int EPI, int NG>
__global__ void __launch_bounds__(256, 4) oz_crt_reconstruct_kernel(const __grid_constant__ ReconArgs p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int bjc = blockIdx.x;                                   // 128-column block
  const long lrow = (long)blockIdx.y * 8 + warp;
  const long grow = (long)p.row0 + lrow;
  const long gcol = (long)bjc * 128 + lane * 4;
  const int bi = (int)(grow >> 7), bi2 = (int)(grow >> 8), bx2 = bjc >> 1;
  if (EPI == OZ_EPI_STORE && p.lower_only && bjc > bi) return;  // never stored
  int kb0, kb1;
  planes_krange(p.krange, p.K, bi2, bx2, kb0, kb1);
  const bool computed = (kb1 > kb0) && !(p.lower_only && 2 * bx2 > 2 * bi2 + 1);

  uint32_t acc[4][6];
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int j = 0; j < 6; ++j) acc[x][j] = 0u;
  if (computed) {
    const uint8_t* src = p.res + lrow * p.res_ld + gcol;
    uint32_t q[NG * 4];
#pragma unroll
    for (int i = 0; i < NG * 4; ++i) {
      q[i] = (i < 4 * (NG - 1) || i < p.nmod) ? __ldcs(reinterpret_cast<const uint32_t*>(src)) : 0u;
      src += p.res_plane;
    }
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      {
        const uint32_t ab_lo = __byte_perm(q[4 * g], q[4 * g + 1], 0x5140), ab_hi = __byte_perm(q[4 * g], q[4 * g + 1], 0x7362);
        const uint32_t cd_lo = __byte_perm(q[4 * g + 2], q[4 * g + 3], 0x5140),
                       cd_hi = __byte_perm(q[4 * g + 2], q[4 * g + 3], 0x7362);
        const uint32_t t[4] = {__byte_perm(ab_lo, cd_lo, 0x5410), __byte_perm(ab_lo, cd_lo, 0x7632),
                               __byte_perm(ab_hi, cd_hi, 0x5410), __byte_perm(ab_hi, cd_hi, 0x7632)};
#pragma unroll
        for (int e = 0; e < 4; ++e)
#pragma unroll
          for (int j = 0; j < 6; ++j) {
            uint32_t v = acc[e][j];
            v = dp2a_lo(p.wp[2 * g][j], t[e], v);
            v = dp2a_hi(p.wp[2 * g + 1][j], t[e], v);
            acc[e][j] = v;
          }
      }
    }
  }
  const bool row_ok = grow < p.M;
  const bool col_ok = gcol < p.N;
  const double sa = row_ok ? p.scA[grow] * p.p_scaled : 0.0;
  double v[4];
#pragma unroll
  for (int x = 0; x < 4; ++x) {
    // fold the limb sums: F = sum_j acc_j 2^(16 j) mod 2^96
    const unsigned long long t0 = ((unsigned long long)acc[x][1] << 16) + acc[x][0];
    const unsigned long long t1 = ((unsigned long long)acc[x][3] << 16) + acc[x][2] + (t0 >> 32);
    const unsigned long long t2 = ((unsigned long long)acc[x][5] << 16) + acc[x][4] + (t1 >> 32);
    const long long hi = (long long)((t2 << 32) | (t1 & 0xffffffffull));
    const double frac = fma((double)hi, 4294967296.0, (double)(uint32_t)t0);   // signed 96-bit integer, 53 leading bits
    // (sa scB) frac rounds once. When sa scB underflows (eA + eB - 2 bits + log2 p_scaled < -1022: subnormal, or 0 below
    // about -1074) it has lost bits while the value itself may be normal: (sa frac) scB rounds once too there (sa frac is
    // normal, scB a power of two), and gives the same bits wherever both orders are exact. sa and scB are never 0 for a
    // valid row and column, so the test is on the range, not on sab itself.
    const double sab = col_ok ? sa * p.scB[gcol + x] : 0.0;
    v[x] = col_ok ? sab * frac : 0.0;
    if (row_ok && col_ok && fabs(sab) < 2.2250738585072014e-308) v[x] = sa * frac * p.scB[gcol + x];
  }
  if (EPI == OZ_EPI_STORE) {
    if (row_ok && col_ok) {
      double* crow = p.C + grow * p.ldc + gcol;
#pragma unroll
      for (int x = 0; x < 4; x += 2) {
        double2 o;
        o.x = p.alpha * v[x];
        o.y = p.alpha * v[x + 1];
        if (p.beta != 0.0) {
          const double2 old = *reinterpret_cast<const double2*>(crow + x);
          o.x = fma(p.beta, old.x, o.x);
          o.y = fma(p.beta, old.y, o.y);
        }
        *reinterpret_cast<double2*>(crow + x) = o;
      }
    }
  } else {
    // per row: sum of squares over this 128-column block, and the dot with the adjacent row (the neighbouring warp)
    __shared__ double vrow[8][128];
#pragma unroll
    for (int x = 0; x < 4; ++x) vrow[warp][lane * 4 + x] = v[x];
    __syncthreads();
    double sq = 0.0, pd = 0.0;
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      sq = fma(v[x], v[x], sq);
      pd = fma(v[x], vrow[warp ^ 1][lane * 4 + x], pd);
    }
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      sq += __shfl_xor_sync(0xffffffffu, sq, off);
      pd += __shfl_xor_sync(0xffffffffu, pd, off);
    }
    if (lane == 0 && row_ok) {
      p.colsq[(long)bjc * p.ldo + grow] = sq;
      if (!(grow & 1)) p.pairdot[(long)bjc * (p.ldo / 2) + (grow >> 1)] = pd;
    }
  }
}
