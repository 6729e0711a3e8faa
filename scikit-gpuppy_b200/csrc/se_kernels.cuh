// ARD squared-exponential covariance kernels (GaussianCovariance of the reference):
//   k(a,b) = v * exp(-1/2 * sum_k w_k (a_k - b_k)^2)        Covariance.py:440-451, 466-483
// fused distance+exp tiles, the NLL-gradient trace with dK/dtheta generated on the fly
// (Covariance.py:266-282, 605-657 never materialised), and the per-query vectors of the
// Girard Gaussian approximation (UncertaintyPropagation2.pyx:266-299, Covariance.py:660-689).
#pragma once
#include "gpk_common.cuh"

namespace gpk {

constexpr int MAX_D = 64;   // input dimension limit of this build
constexpr int SE_DCH = 16;  // dimensions staged per shared-memory pass

constexpr int KIND_SE = 0;        // GaussianCovariance
constexpr int KIND_PERIODIC = 1;  // PeriodicCovariance (periodic_kernels.cuh)

struct SEHyper {
  double v, vt;
  double w[MAX_D];   // inverse squared length scales exp(theta[2:])
  double sw[MAX_D];  // sqrt(w)
  int kind;
  double pf[16];     // KIND_PERIODIC: pi / p_k
  double w2[16];     // KIND_PERIODIC: weights of the sin^2 terms
  double pr[16];     // KIND_PERIODIC: p_k
};

struct SETileArgs {
  const double* x1; int n1;   // rows   (n1 x d, row-major)
  const double* x2; int n2;   // cols   (n2 x d, row-major)
  int d;
  double* out; long ld;
  int rows_out, cols_out;     // extents written (>= n1, n2 when padding)
  int add_noise;              // += vt where row == col (training K)
  int pad_identity;           // 1 on the diagonal of the padding block, else 0
  int lower_only;             // skip tiles strictly above the diagonal
  int vec_ok;                 // 16-byte stores allowed (ld even, out 16B aligned)
};

// 128x128 output tile per CTA, 512 threads, 4x8 outputs per thread, direct differences (no |a|^2+|b|^2-2ab
// cancellation). The kernel is bound by FP64 latency (3 FP64 operations per element and dimension + exp): with 8x8
// outputs per thread (196 registers, 8 warps per SM) ncu showed the FP64 pipe 36 % active; half the register tile and
// twice the warps keep more independent work in flight.
constexpr int SE_THREADS = 512;
__global__ void __launch_bounds__(SE_THREADS, 1) se_tile_kernel(SETileArgs p, SEHyper h) {
  const int bj = blockIdx.x, bi = blockIdx.y;
  if (p.lower_only && bj > bi) return;
  __shared__ __align__(16) double xa[SE_DCH][TILE];
  __shared__ __align__(16) double xb[SE_DCH][TILE];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = (tid >> 4) & 15, tz = tid >> 8;   // rows ty + 16 (a + 4 tz), a < 4
  const int row0 = bi * TILE, col0 = bj * TILE;

  double acc[4][8];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) acc[a][b] = 0.0;

  for (int k0 = 0; k0 < p.d; k0 += SE_DCH) {
    const int kc = min(SE_DCH, p.d - k0);
    __syncthreads();
    for (int idx = tid; idx < TILE * SE_DCH; idx += SE_THREADS) {
      const int r = idx / SE_DCH, k = idx % SE_DCH;
      double va = 0.0, vb = 0.0;
      if (k < kc) {
        const double s = h.sw[k0 + k];
        if (row0 + r < p.n1) va = p.x1[(long)(row0 + r) * p.d + k0 + k] * s;
        if (col0 + r < p.n2) vb = p.x2[(long)(col0 + r) * p.d + k0 + k] * s;
      }
      xa[k][r] = va;
      xb[k][r] = vb;
    }
    __syncthreads();
    for (int k = 0; k < kc; ++k) {
      double av[4];
      double2 bv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) av[a] = xa[k][ty + 16 * (a + 4 * tz)];
#pragma unroll
      for (int b = 0; b < 4; ++b) bv[b] = *reinterpret_cast<const double2*>(&xb[k][32 * b + 2 * tx]);
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const double d0 = av[a] - bv[b].x, d1 = av[a] - bv[b].y;
          acc[a][2 * b] = fma(d0, d0, acc[a][2 * b]);
          acc[a][2 * b + 1] = fma(d1, d1, acc[a][2 * b + 1]);
        }
    }
  }

#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int row = row0 + ty + 16 * (a + 4 * tz);
    if (row >= p.rows_out) continue;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int col = col0 + 32 * b + 2 * tx;
      double o[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = col + e;
        double val;
        if (row < p.n1 && c < p.n2) {
          val = h.v * exp(-0.5 * acc[a][2 * b + e]);
          if (p.add_noise && row == c) val += h.vt;
        } else {
          val = (p.pad_identity && row == c) ? 1.0 : 0.0;
        }
        o[e] = val;
      }
      double* dst = p.out + (long)row * p.ld + col;
      if (p.vec_ok && col + 1 < p.cols_out) {
        *reinterpret_cast<double2*>(dst) = make_double2(o[0], o[1]);
      } else {
        if (col < p.cols_out) dst[0] = o[0];
        if (col + 1 < p.cols_out) dst[1] = o[1];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// NLL gradient trace:  g_j = 1/2 sum_ab (Kinv - alpha alpha^T)_ab dK_j,ab   (Covariance.py:280)
// One CTA per lower tile of Kinv. Per tile partial sums P[tile][0] = sum M*Knl,
// P[tile][1+k] = sum M*Knl*(x_ak-x_bk)^2 ; only elements with col <= row are read (K^-1 is stored as a
// lower triangle) and the strictly-lower ones count twice (symmetry).
// DP = padded dimension (template) so the per-thread accumulators stay in registers.
// ncu (round 2, n = 16384, d = 16): FP64 pipe 36 % active, issue slots 49 % busy, 16 warps/SM at 128 registers; a
// variant with one row per step (80 registers, 24 warps/SM) was measured SLOWER (13.1 vs 11.5 ms at n = 32768): the
// kernel is bound by the dependent FP64 chains of each element (distance sum, exp), not by occupancy.
template <int DP>
__global__ void __launch_bounds__(256, (DP <= 16) ? 2 : 1)
grad_trace_kernel(const double* __restrict__ Kinv, long ld, const double* __restrict__ alpha,
                  const double* __restrict__ x, int n, int d, int d0 /*first dim of this pass*/, SEHyper h,
                  int tile_row_begin, double* __restrict__ partial /*[gridDim.y*gridDim.x][DP+1]*/) {
  // grid: x = tile column, y = tile row offset from tile_row_begin; tiles above the diagonal
  // only clear their partial slot.
  const int bj = blockIdx.x, bi = tile_row_begin + blockIdx.y;
  double* out = partial + ((long)blockIdx.y * gridDim.x + blockIdx.x) * (DP + 1);
  if (bj > bi) {
    if (threadIdx.x <= DP) out[threadIdx.x] = 0.0;
    return;
  }

  // dynamic smem: xa[d][XLD], xb[d][XLD] hold ALL d dimensions of the tile's rows / columns
  extern __shared__ __align__(16) double gsm[];
  constexpr int XLD = TILE + 2;            // even: rows r0..r0+RT-1 of one dimension are a 16-byte aligned run
  constexpr int RT = 2;                    // rows per thread per step (register tile RT x 1); 2 CTAs/SM for DP <= 16
  double* xa = gsm;
  double* xb = gsm + (long)d * XLD;
  __shared__ double al_a[TILE], al_b[TILE];
  __shared__ double red[8];
  const int tid = threadIdx.x;
  const int row0 = bi * TILE, col0 = bj * TILE;

  for (int idx = tid; idx < TILE * d; idx += 256) {
    const int r = idx / d, k = idx % d;
    xa[k * XLD + r] = (row0 + r < n) ? x[(long)(row0 + r) * d + k] : 0.0;
    xb[k * XLD + r] = (col0 + r < n) ? x[(long)(col0 + r) * d + k] : 0.0;
  }
  if (tid < TILE) {
    al_a[tid] = (row0 + tid < n) ? alpha[row0 + tid] : 0.0;
    al_b[tid] = (col0 + tid < n) ? alpha[col0 + tid] : 0.0;
  }
  __syncthreads();

  double g0 = 0.0;
  double gk[DP];
#pragma unroll
  for (int k = 0; k < DP; ++k) gk[k] = 0.0;

  // thread = one column c of the tile and half of its rows, RT rows at a time: the column's coordinates are
  // loaded once per dimension and reused for RT rows (the rows' coordinates are broadcast 128-bit loads)
  const int c = tid & 127;
  const int rhalf = (tid >> 7) * (TILE / 2);
  const bool col_ok = (col0 + c) < n;
  const bool diag_tile = (bi == bj);
  const double alc = al_b[c];
  // K^-1 elements are fetched two steps ahead (one step ahead measured 5 % slower, no prefetch 8 % slower) (ncu round 2: 27 % of the stall samples were long-scoreboard waits on
  // this load, issued right before its first use; the matrix is read once from DRAM, nothing hits in L2). The padded
  // matrix makes every address valid; rows the tile does not use are masked below.
  const double* kcol = Kinv + (long)row0 * ld + col0 + c;
  double kq[2][RT];
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int i = 0; i < RT; ++i) kq[s][i] = kcol[(long)(rhalf + s * RT + i) * ld];
  for (int r0 = rhalf; r0 < rhalf + TILE / 2; r0 += RT) {
    double m[RT], dist[RT], sq[RT][DP];
    double kcur[RT];
#pragma unroll
    for (int i = 0; i < RT; ++i) {
      kcur[i] = kq[0][i];
      kq[0][i] = kq[1][i];
      const int rn = r0 + 2 * RT + i;                          // two steps ahead, clamped inside the tile
      kq[1][i] = kcol[(long)(rn < rhalf + TILE / 2 ? rn : r0 + i) * ld];
    }
#pragma unroll
    for (int i = 0; i < RT; ++i) {
      const int r = r0 + i;
      const bool ok = col_ok && (row0 + r) < n && !(diag_tile && c > r);
      const double sym = (diag_tile && c == r) ? 1.0 : 2.0;   // strictly-lower elements stand for their mirror
      m[i] = ok ? sym * (kcur[i] - al_a[r] * alc) : 0.0;
      dist[i] = 0.0;
    }
    for (int k = 0; k < d0; ++k) {          // dimensions handled by another pass (d > 32 only)
      const double bv = xb[k * XLD + c];
#pragma unroll
      for (int i = 0; i < RT; ++i) {
        const double df = xa[k * XLD + r0 + i] - bv;
        dist[i] = fma(h.w[k] * df, df, dist[i]);
      }
    }
#pragma unroll
    for (int k = 0; k < DP; ++k) {
      if (d0 + k < d) {
        const double bv = xb[(d0 + k) * XLD + c];
        const double wk = h.w[d0 + k];
        const double2* arow = reinterpret_cast<const double2*>(&xa[(d0 + k) * XLD + r0]);
#pragma unroll
        for (int i2 = 0; i2 < RT / 2; ++i2) {
          const double2 av = arow[i2];
          const double d0v = av.x - bv, d1v = av.y - bv;
          sq[2 * i2][k] = d0v * d0v;
          sq[2 * i2 + 1][k] = d1v * d1v;
          dist[2 * i2] = fma(wk, sq[2 * i2][k], dist[2 * i2]);
          dist[2 * i2 + 1] = fma(wk, sq[2 * i2 + 1][k], dist[2 * i2 + 1]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < RT; ++i) sq[i][k] = 0.0;
      }
    }
    for (int k = d0 + DP; k < d; ++k) {
      const double bv = xb[k * XLD + c];
#pragma unroll
      for (int i = 0; i < RT; ++i) {
        const double df = xa[k * XLD + r0 + i] - bv;
        dist[i] = fma(h.w[k] * df, df, dist[i]);
      }
    }
#pragma unroll
    for (int i = 0; i < RT; ++i) {
      const double pk = m[i] * h.v * exp(-0.5 * dist[i]);
      g0 += pk;
#pragma unroll
      for (int k = 0; k < DP; ++k) gk[k] = fma(pk, sq[i][k], gk[k]);
    }
  }

  double s = block_sum_256(g0, red);
  if (tid == 0) out[0] = s;
#pragma unroll
  for (int k = 0; k < DP; ++k) {
    s = block_sum_256(gk[k], red);
    if (tid == 0) out[1 + k] = s;
  }
}

// out[0] = sum_{i in [r0,r1)} W[i][i] (trace of K^-1 rows) ; out[1] = sum_{i in [r0,r1)} alpha_i^2
__global__ void __launch_bounds__(256) diag_sum_kernel(const double* __restrict__ W, long ld,
                                                       const double* __restrict__ alpha, int r0, int r1,
                                                       double* __restrict__ out) {
  __shared__ double red[8];
  double s = 0.0, a2 = 0.0;
  for (int i = r0 + threadIdx.x; i < r1; i += 256) {
    s += W[(long)i * ld + i];
    a2 = fma(alpha[i], alpha[i], a2);
  }
  s = block_sum_256(s, red);
  a2 = block_sum_256(a2, red);
  if (threadIdx.x == 0) {
    out[0] = s;
    out[1] = a2;
  }
}

// ---------------------------------------------------------------------------------------------
// Girard GA per-query vectors. For query q (mean u, input covariance Sigma) and training point i:
//   E_i  = v exp(-1/2 sum_k w_k (x_ik-u_k)^2)
//   C_i  = E_i (+ vt when x_i == u element-wise: the scalar-covariance quirk, Covariance.py:451)
//   tr_i = tracedot(H_i, Sigma),  H_i = ((delta w)(delta w)^T - diag(w)) E_i     Covariance.py:660-674
//   J_ik = -(x_ik-u_k) w_k E_i                                                    Covariance.py:676-689
// Row layout of G: row q*P + 0 = C, +1 = tr, +2+k = J_k ; columns i (contiguous), zero for i >= n.
struct GAArgs {
  const double* xT; long ldxt;  // x transposed: xT[k*ldxt + i]
  int n, npad, d, P;
  const double* U;              // [Q][d]
  const double* S;              // [Q][d] (diag) or [Q][d][d] (full)
  int sigma_full;
  double* G; long ldg;
  int rows_pad;                 // rows of G to clear beyond Q*P
  int Q;
};

__global__ void __launch_bounds__(256) ga_build_kernel(GAArgs p, SEHyper h) {
  const int q = blockIdx.y;
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= p.npad) return;
  if (q >= p.Q) {
    // padding rows (beyond Q*P): zero
    const long row = (long)p.Q * p.P + (q - p.Q);
    if (row < p.rows_pad) p.G[row * p.ldg + i] = 0.0;
    return;
  }
  double* g = p.G + (long)q * p.P * p.ldg + i;
  if (i >= p.n) {
    for (int c = 0; c < p.P; ++c) g[(long)c * p.ldg] = 0.0;
    return;
  }
  const double* u = p.U + (long)q * p.d;
  double dist = 0.0;
  bool same = true;
  for (int k = 0; k < p.d; ++k) {
    const double xv = p.xT[(long)k * p.ldxt + i];
    const double df = xv - u[k];
    same = same && (xv == u[k]);
    dist = fma(h.w[k] * df, df, dist);
  }
  const double E = h.v * exp(-0.5 * dist);
  double tr = 0.0;
  if (!p.sigma_full) {
    const double* s = p.S + (long)q * p.d;
    for (int k = 0; k < p.d; ++k) {
      const double df = p.xT[(long)k * p.ldxt + i] - u[k];
      const double dw = df * h.w[k];
      tr += (dw * dw - h.w[k]) * s[k];
      g[(long)(2 + k) * p.ldg] = -dw * E;
    }
  } else {
    const double* s = p.S + (long)q * p.d * p.d;
    for (int a = 0; a < p.d; ++a) {
      const double dwa = (p.xT[(long)a * p.ldxt + i] - u[a]) * h.w[a];
      g[(long)(2 + a) * p.ldg] = -dwa * E;
      for (int b = 0; b < p.d; ++b) {
        const double dwb = (p.xT[(long)b * p.ldxt + i] - u[b]) * h.w[b];
        // tracedot(H,Sigma) = sum_ab H[b][a]*Sigma[a][b]  (Covariance.py:101-109)
        double hba = dwa * dwb;
        if (a == b) hba -= h.w[a];
        tr = fma(hba, s[(long)a * p.d + b], tr);
      }
    }
  }
  g[0] = same ? (E + h.vt) : E;
  g[p.ldg] = tr * E;
  for (int c = 2 + p.d; c < p.P; ++c) g[(long)c * p.ldg] = 0.0;
}

// dots[row] = sum_i G[row][i] * alpha[i]   (one warp per row)
__global__ void __launch_bounds__(256) rows_dot_kernel(const double* __restrict__ G, long ldg, int rows, int len,
                                                       const double* __restrict__ alpha, double* __restrict__ dots) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const double* Gr = G + (long)row * ldg;
  double s0 = 0.0, s1 = 0.0;
  int i = lane;
  for (; i + 32 < len; i += 64) {
    s0 = fma(Gr[i], alpha[i], s0);
    s1 = fma(Gr[i + 32], alpha[i + 32], s1);
  }
  if (i < len) s0 = fma(Gr[i], alpha[i], s0);
  const double s = warp_sum(s0 + s1);
  if (lane == 0) dots[row] = s;
}

// Combine per-row-block partials into the propagated moments (closed form of pyx:208-257):
//   mean = a.C + 1/2 a.tr + meant
//   var  = (v+vt) - |XC|^2 - sum_k S_kk (|XJ_k|^2 - (a.J_k)^2) - (XC).(Xtr)
__global__ void __launch_bounds__(256) ga_finalize_kernel(const double* __restrict__ colsq,
                                                          const double* __restrict__ pairdot, long ldo, int nbi,
                                                          const double* __restrict__ dots, const double* __restrict__ S,
                                                          int sigma_full, int Q, int d, int P, double v, double vt,
                                                          double meant, double* __restrict__ mean,
                                                          double* __restrict__ var, double* __restrict__ sigma2_out,
                                                          double* __restrict__ rest_out) {
  const int q = blockIdx.x * 256 + threadIdx.x;
  if (q >= Q) return;
  const long base = (long)q * P;
  auto csum = [&](long col) {
    double s = 0.0;
    for (int b = 0; b < nbi; ++b) s += colsq[(long)b * ldo + col];
    return s;
  };
  double pd = 0.0;
  for (int b = 0; b < nbi; ++b) pd += pairdot[(long)b * (ldo / 2) + base / 2];
  const double sC = csum(base);
  double v2 = 0.0;
  for (int k = 0; k < d; ++k) {
    const double skk = sigma_full ? S[(long)q * d * d + (long)k * d + k] : S[(long)q * d + k];
    const double aj = dots[base + 2 + k];
    v2 += skk * (csum(base + 2 + k) - aj * aj);
  }
  // sigma2 = cov(u,u) - C^T Kinv C (pyx:221-232); variance_rest = variance2 + variance3 (pyx:234-257)
  const double sigma2 = (v + vt) - sC;
  const double rest = -v2 - pd;
  if (mean) mean[q] = dots[base] + 0.5 * dots[base + 1] + meant;
  if (var) var[q] = sigma2 + rest;
  if (sigma2_out) sigma2_out[q] = sigma2;
  if (rest_out) rest_out[q] = rest;
}

// var[q] = prior[q] - sum_b colsq[b][q], or v + vt - sum_b colsq[b][q] without a prior vector
__global__ void __launch_bounds__(256) predict_var_kernel(const double* __restrict__ colsq, long ldo, int nbi, int m,
                                                          const double* __restrict__ prior, double vpvt,
                                                          double* __restrict__ var) {
  const int q = blockIdx.x * 256 + threadIdx.x;
  if (q >= m) return;
  double s = 0.0;
  for (int b = 0; b < nbi; ++b) s += colsq[(long)b * ldo + q];
  var[q] = (prior ? prior[q] : vpvt) - s;
}

__global__ void __launch_bounds__(256) add_scalar_kernel(double* __restrict__ y, int len, double a) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < len) y[i] += a;
}

// xT[k*ld + i] = x[i*d + k], zero padded to ld columns
__global__ void __launch_bounds__(256) transpose_x_kernel(const double* __restrict__ x, int n, int d,
                                                          double* __restrict__ xT, long ld) {
  const long i = (long)blockIdx.x * 256 + threadIdx.x;
  if (i >= ld) return;
  for (int k = 0; k < d; ++k) xT[(long)k * ld + i] = (i < n) ? x[i * d + k] : 0.0;
}

}  // namespace gpk
