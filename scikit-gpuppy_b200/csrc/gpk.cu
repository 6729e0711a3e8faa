// libgpk.so -- C ABI (include/gpk.h) over the sm_100a kernels in this directory.
// No CPU fallback exists: every entry point runs CUDA kernels or fails with an error code.
#include "../../include/gpk.h"
#include "../../include/gpk_test.h"

#include <climits>
#include <new>
#include <type_traits>
#include <vector>

#include "dgemm_dmma.cuh"
#include "factor.cuh"
#include "se_kernels.cuh"
#include "exact_kernels.cuh"
#include "periodic_kernels.cuh"

namespace gpk {
// Error text and measurement state belong to the calling host thread (the contract is one host thread per handle,
// include/gpk.h): two handles driven from two threads do not see each other's errors or event pairs.
thread_local char g_err[512] = {0};
thread_local long g_launch_count = 0;
thread_local bool g_prof_on = false;
static thread_local std::vector<ProfPair> g_prof;
void prof_push(cudaEvent_t a, cudaEvent_t b) { g_prof.push_back(ProfPair{a, b}); }

struct Handle {
  int n = 0, d = 0, npad = 0;
  double *X = nullptr, *W = nullptr;
  bool own_X = false, own_W = false;
  double *x = nullptr, *xT = nullptr, *t = nullptr, *y = nullptr, *alpha = nullptr, *dL = nullptr;
  double* scal = nullptr;  // device scalars [3] of nll_scalars_kernel
  int* info = nullptr;
  double* part = nullptr; size_t part_elems = 0;      // partial-sum workspace
  double* G = nullptr; size_t G_elems = 0;            // per-batch query workspace rows x npad
  double* colsq = nullptr; size_t colsq_elems = 0;    // [nbi][rows]
  double* pairdot = nullptr;                          // [nbi][rows/2]
  double* dots = nullptr; size_t dots_elems = 0;      // [rows]
  double* V = nullptr; size_t V_elems = 0;            // gpk_predict_cov: rows of V^T = G X^T of both query sets;
                                                      // gpk_predict_grad: V^T of one batch
  double* C = nullptr; size_t C_elems = 0;            // gpk_predict_cov: padded output block
  long batch_rows = 0;                                // user cap on rows per batch (0 = default)
  SEHyper hyp;
  int kind = KIND_SE;                     // covariance family (gpk_set_kernel)
  double theta[3 * MAX_D + 2];
  bool factored = false, have_inverse = false;
  bool matrix_state = false;              // factored from a caller-supplied matrix (gpk_factorize_matrix), not from theta
  double logdet = 0.0, quad = 0.0, alpha2 = 0.0;
  cudaStream_t st = nullptr;
  cudaStream_t side = nullptr;            // side stream of the factorisation (off-critical-path TRMMs)
  std::vector<cudaEvent_t> events;        // fork/join events, 2 per internal node of the recursion
  int ev_next = 0;
  // INT8 tensor-core route (gpk_set_route): requested at create / set_route, workspace allocated at first use
  bool oz_want = false;                   // route requested for this handle
  bool oz_on = false;                     // workspace allocated, route active
  int oz_moduli_req = 0;                  // 0 = the fewest moduli that carry 54-bit operands at K = npad
  size_t oz_out_cap = 0;                  // byte cap of the residue-plane buffer (0 = default)
  oz::Workspace oz;                       // residues of the factorisation operands + residue planes of the products
  oz::Workspace ozq;                      // residues of the per-batch query operand G
  oz::Operand xs;                         // cached residues of X = L^-1 (rows, lower) for prediction / propagation
  bool x_sliced = false;
  // overlap of T = L21 X11 with the right sub-tree (factor.cuh): critical path on a high-priority stream, one
  // lower-priority stream + workspace per recursion depth; allocated with the route when the memory is there
  cudaStream_t chain_st = nullptr;
  std::vector<cudaStream_t> ovl_st;
  std::vector<oz::Workspace> ovl_ws;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  bool ovl_on = false;
  // gradient prefetch (gpk_nll_grad with want_grad = 2): K^-1 and the trace sums are queued behind the factorisation
  // and land in pinned host memory; the gradient call at the same theta only waits for them
  double* raw_pinned = nullptr;           // [TRACE_SUMS]
  bool grad_pending = false;
};

thread_local int g_overlap_T = 1;   // gpk_test_overlap: 0 keeps every INT8 product on one stream (A/B timings)

static void release_overlap(Handle* h) {
  for (auto& w : h->ovl_ws) w.release();
  h->ovl_ws.clear();
  for (auto& s : h->ovl_st) if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
  h->ovl_st.clear();
  if (h->chain_st) { cudaStreamSynchronize(h->chain_st); cudaStreamDestroy(h->chain_st); h->chain_st = nullptr; }
  if (h->ev_in) { cudaEventDestroy(h->ev_in); h->ev_in = nullptr; }
  if (h->ev_out) { cudaEventDestroy(h->ev_out); h->ev_out = nullptr; }
  h->ovl_on = false;
}

// Streams and workspaces for the overlapped T products: depth k serves the nodes of half-size h = npad >> (k + 1) >=
// min_dim. An optimisation only: when the memory is not there (n = 65536 uses 163 of 180 GB already) the
// factorisation runs on one stream as before and gives the same bits.
static int ensure_overlap(Handle* h) {
  if (h->ovl_on || !h->oz_on || !g_overlap_T) return 0;
  int depths = 0;
  size_t need = 0;
  for (long hh = h->npad / 2 / TILE * TILE; hh >= h->oz.min_dim; hh = hh / 2 / TILE * TILE) {
    need += (size_t)h->oz.S * (hh + TILE) * (3 * (hh + TILE) + round_up_l(hh + TILE, 256)) + 6 * hh * sizeof(double);
    ++depths;
  }
  if (depths == 0) return 0;
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return 0; }
  if (free_b < need + ((size_t)28 << 30)) return 0;      // keep room for the query batches (G, its residues, planes)
  int least = 0, greatest = 0;
  GPK_CUDA_OK(cudaDeviceGetStreamPriorityRange(&least, &greatest));
  GPK_CUDA_OK(cudaStreamCreateWithPriority(&h->chain_st, cudaStreamNonBlocking, greatest));
  GPK_CUDA_OK(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
  GPK_CUDA_OK(cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming));
  h->ovl_st.assign(depths, nullptr);
  h->ovl_ws.assign(depths, oz::Workspace());
  long hs = h->npad / 2 / TILE * TILE;
  for (int k = 0; k < depths; ++k, hs = hs / 2 / TILE * TILE) {
    int prio = greatest + (depths - k);                  // deeper products are joined sooner: higher priority
    if (prio > least) prio = least;
    GPK_CUDA_OK(cudaStreamCreateWithPriority(&h->ovl_st[k], cudaStreamNonBlocking, prio));
    oz::Workspace& w = h->ovl_ws[k];
    w.S = h->oz.S;
    const long hmax = hs + TILE;                         // odd splits: halves differ by one tile
    if (w.ensure((size_t)w.S * 3 * hmax * hmax, (size_t)(3 * hmax), (size_t)hmax) != 0 ||
        w.ensure_out((size_t)w.S * hmax * round_up_l(hmax, 256)) != 0) {
      release_overlap(h);
      return 0;
    }
  }
  h->ovl_on = true;
  return 0;
}

static int theta_len(int kind, int d) { return kind == KIND_PERIODIC ? 2 + 3 * d : 2 + d; }

// noise mode of the covariance tiles (periodic_tile_kernel): the periodic family adds vt wherever two points coincide,
// the Gaussian family on the diagonal of the training K only
static int noise_mode(int kind, bool training) { return kind == KIND_PERIODIC ? 2 : training ? 1 : 0; }

// n/2 log(2 pi) + 1/2 log det K + 1/2 t^T K^-1 t of the cached factorisation (Covariance.py:211)
static double nll_of(const Handle* h) {
  const double two_pi = 6.283185307179586476925286766559;
  return 0.5 * h->n * log(two_pi) + 0.5 * h->logdet + 0.5 * h->quad;
}

static int set_hyper(SEHyper& h, const double* theta, int d, int kind = KIND_SE) {
  if (d < 1 || d > MAX_D || (kind == KIND_PERIODIC && d > PER_MAX_D)) {
    snprintf(g_err, sizeof(g_err), "d=%d outside [1,%d]", d, kind == KIND_PERIODIC ? PER_MAX_D : MAX_D);
    return -2;
  }
  memset(&h, 0, sizeof(h));
  h.kind = kind;
  h.v = exp(theta[0]);
  h.vt = exp(theta[1]);
  for (int k = 0; k < d; ++k) {
    h.w[k] = exp(theta[2 + k]);
    h.sw[k] = sqrt(h.w[k]);
  }
  if (kind == KIND_PERIODIC) {
    const double pi = 3.14159265358979323846;
    for (int k = 0; k < d; ++k) {
      h.pr[k] = exp(theta[2 + d + k]);
      h.pf[k] = pi / h.pr[k];
      h.w2[k] = exp(theta[2 + 2 * d + k]);
    }
  }
  return 0;
}

static int ensure(double** p, size_t* have, size_t need) {
  if (*have >= need) return 0;
  if (*p) GPK_CUDA_OK(cudaFree(*p));
  *p = nullptr;
  *have = 0;
  GPK_CUDA_OK(cudaMalloc((void**)p, need * sizeof(double)));
  *have = need;
  GPK_CUDA_OK(poison_fill(*p, need * sizeof(double)));
  return 0;
}

// deterministic column sums of a [nrows][ncols] row-major array: one CTA per column
__global__ void __launch_bounds__(256) col_sum_kernel(const double* __restrict__ part, long nrows, int ncols,
                                                      double* __restrict__ out) {
  __shared__ double red[8];
  const int c = blockIdx.x;
  double s = 0.0;
  for (long r = threadIdx.x; r < nrows; r += 256) s += part[r * ncols + c];
  s = block_sum_256(s, red);
  if (threadIdx.x == 0) out[c] = s;
}

__global__ void set_int_kernel(int* p, int v) { *p = v; }
__global__ void __launch_bounds__(256) axpy_kernel(double* __restrict__ y, const double* __restrict__ x, int n, double a) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) y[i] = fma(a, x[i], y[i]);
}

static int launch_se_tiles(const double* x1, int n1, const double* x2, int n2, int d, const SEHyper& hyp, double* out,
                           long ld, int rows_out, int cols_out, int add_noise, int pad_identity, int lower_only,
                           cudaStream_t st) {
  SETileArgs a;
  a.x1 = x1; a.n1 = n1; a.x2 = x2; a.n2 = n2; a.d = d;
  a.out = out; a.ld = ld; a.rows_out = rows_out; a.cols_out = cols_out;
  a.add_noise = add_noise; a.pad_identity = pad_identity; a.lower_only = lower_only;
  a.vec_ok = ((ld % 2) == 0 && (reinterpret_cast<uintptr_t>(out) % 16) == 0) ? 1 : 0;
  if (rows_out <= 0 || cols_out <= 0) return 0;
  if (hyp.kind == KIND_PERIODIC) {
    dim3 pgrid((cols_out + PER_T - 1) / PER_T, (rows_out + PER_T - 1) / PER_T);
    periodic_tile_kernel<<<pgrid, 256, 0, st>>>(a, hyp);
    GPK_LAUNCH_OK();
    return 0;
  }
  dim3 grid((cols_out + TILE - 1) / TILE, (rows_out + TILE - 1) / TILE);
  se_tile_kernel<<<grid, SE_THREADS, 0, st>>>(a, hyp);
  GPK_LAUNCH_OK();
  return 0;
}

// y = X b ; out = X^T y   (K^-1 b through the triangular inverse)
static int solve_one(Handle* h, const double* b_pad, double* y, double* out) {
  const int npad = h->npad;
  trmv_lower_kernel<<<(npad + 7) / 8, 256, 0, h->st>>>(h->X, npad, npad, b_pad, y);
  GPK_LAUNCH_OK();
  const int nchunks = (npad + TRMVT_ROWS - 1) / TRMVT_ROWS;
  GPK_TRY(ensure(&h->part, &h->part_elems, (size_t)nchunks * npad));
  dim3 grid(npad / 128, nchunks);
  trmv_lower_T_partial_kernel<<<grid, 128, 0, h->st>>>(h->X, npad, npad, y, h->part);
  GPK_LAUNCH_OK();
  sum_chunks_kernel<<<(npad + 255) / 256, 256, 0, h->st>>>(h->part, nchunks, npad, npad, out, 1.0, 0.0);
  GPK_LAUNCH_OK();
  return 0;
}

// Pass width of the gradient-trace and exact-pair kernels: the dimensions of one pass are padded to DP, so the
// per-thread accumulators are register arrays; the SE trace takes ceil(d / 32) passes beyond d = 32.
static int pass_dim(int d) { return d <= 4 ? 4 : d <= 8 ? 8 : d <= 16 ? 16 : 32; }

// f(std::integral_constant<int, pass_dim(d)>()), with only the widths up to MAX_DP instantiated
template <int MAX_DP, int DP = 4, class F>
static int dispatch_pass_dim(int d, F&& f) {
  if constexpr (DP < MAX_DP) {
    if (pass_dim(d) > DP) return dispatch_pass_dim<MAX_DP, 2 * DP>(d, f);
  }
  return f(std::integral_constant<int, DP>());
}

// doubles of the trace-sum vector (trace_enqueue): SE ceil(d / 32) passes of 33 + 2, periodic 3 * 16 + 2
constexpr int TRACE_SUMS = (MAX_D + 31) / 32 * 33 + 2;
static_assert(3 * PER_MAX_D + 2 <= TRACE_SUMS, "periodic trace sums exceed the trace-sum vector");

template <int DP>
static int launch_trace(Handle* h, int d0, int trb, int tre, double* partial) {
  const int nt = h->npad / TILE;
  const size_t smem = (size_t)2 * h->d * (TILE + 2) * sizeof(double);
  // set per launch: the attribute is per device and per function, the call is cheap, and a cached flag would be wrong
  // for a process that drives several devices or threads
  GPK_CUDA_OK(cudaFuncSetAttribute(grad_trace_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(nt, tre - trb);
  grad_trace_kernel<DP><<<grid, 256, smem, h->st>>>(h->W, h->npad, h->alpha, h->x, h->n, h->d, d0, h->hyp, trb, partial);
  GPK_LAUNCH_OK();
  return 0;
}

// Queue the trace sums of tile rows [trb, tre) of K^-1 and one copy of them to the host buffer dst (TRACE_SUMS doubles),
// without synchronising. An empty range launches nothing and leaves dst alone. The device vector at the tail of h->part
// has the layout dst receives, which only trace_unpack reads:
//   SE, per pass p of DP dimensions: [p (DP + 1)] = sum M Knl, then sum M Knl diff_k^2 for k = p DP + j, j < DP;
//       after the passes the sums of diag(K^-1) and of alpha^2 over the rows of the range
//   periodic: the 3 DP + 2 column sums of periodic_trace_kernel<DP>
static int trace_enqueue(Handle* h, int trb, int tre, double* dst) {
  if (tre <= trb) return 0;
  const int d = h->d, nt = h->npad / TILE;
  const long nslots = (long)nt * (tre - trb);
  double* sums = nullptr;
  int nsums = 0;
  if (h->kind == KIND_PERIODIC) {
    GPK_TRY(dispatch_pass_dim<16>(d, [&](auto dp) {
      constexpr int DP = decltype(dp)::value;
      nsums = 3 * DP + 2;
      GPK_TRY(ensure(&h->part, &h->part_elems, (size_t)nslots * nsums + nsums));
      sums = h->part + (size_t)nslots * nsums;
      periodic_trace_kernel<DP><<<dim3(nt, tre - trb), 256, 0, h->st>>>(h->W, h->npad, h->alpha, h->x, h->n, d, h->hyp,
                                                                        trb, h->part);
      GPK_LAUNCH_OK();
      col_sum_kernel<<<nsums, 256, 0, h->st>>>(h->part, nslots, nsums, sums);
      GPK_LAUNCH_OK();
      return 0;
    }));
  } else {
    GPK_TRY(dispatch_pass_dim<32>(d, [&](auto dp) {
      constexpr int DP = decltype(dp)::value;
      const int npass = (d + DP - 1) / DP;
      nsums = npass * (DP + 1) + 2;
      GPK_TRY(ensure(&h->part, &h->part_elems, (size_t)nslots * (DP + 1) + nsums));
      sums = h->part + (size_t)nslots * (DP + 1);
      const int r0 = trb * TILE, r1 = (tre * TILE < h->n) ? tre * TILE : h->n;
      diag_sum_kernel<<<1, 256, 0, h->st>>>(h->W, h->npad, h->alpha, r0, r1, sums + npass * (DP + 1));
      GPK_LAUNCH_OK();
      for (int p = 0; p < npass; ++p) {
        GPK_TRY(launch_trace<DP>(h, p * DP, trb, tre, h->part));
        col_sum_kernel<<<DP + 1, 256, 0, h->st>>>(h->part, nslots, DP + 1, sums + p * (DP + 1));
        GPK_LAUNCH_OK();
      }
      return 0;
    }));
  }
  GPK_CUDA_OK(cudaMemcpyAsync(dst, sums, nsums * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  return 0;
}

// raw sums from the trace-sum vector of trace_enqueue:
//   SE (d + 3): [0] = sum M Knl, [1 + k] = sum M Knl diff_k^2, [d + 1] = sum of diag(K^-1), [d + 2] = sum of alpha^2
//   periodic (3 d + 3): [0] = sum M K, [1 + k] diff^2 sums, [1 + d + k] diff sin cos sums, [1 + 2d + k] sin^2 sums,
//   [3d + 1] = sum of M over coincident pairs (the noise derivative), [3d + 2] = 0
// Every SE pass sums M Knl again; the first pass's sum is the one used.
static void trace_unpack(const Handle* h, const double* src, double* raw) {
  const int d = h->d, DP = pass_dim(d);
  raw[0] = src[0];
  if (h->kind == KIND_PERIODIC) {
    for (int k = 0; k < d; ++k) {
      raw[1 + k] = src[1 + k];
      raw[1 + d + k] = src[1 + DP + k];
      raw[1 + 2 * d + k] = src[1 + 2 * DP + k];
    }
    raw[3 * d + 1] = src[3 * DP + 1];
    raw[3 * d + 2] = 0.0;
    return;
  }
  for (int k = 0; k < d; ++k) raw[1 + k] = src[k / DP * (DP + 1) + 1 + k % DP];
  const double* diag = src + (d + DP - 1) / DP * (DP + 1);
  raw[d + 1] = diag[0];
  raw[d + 2] = diag[1];
}

// the gradient from the raw trace sums of the whole K^-1 (trace_unpack)
static void grad_from_raw(const Handle* h, const double* raw, double* grad) {
  const int d = h->d;
  grad[0] = 0.5 * raw[0];
  if (h->kind == KIND_PERIODIC) {
    // dK/dlog w_k = -1/2 w_k diff^2 K ; dK/dlog p_k = pi w2_k/p_k diff sin cos K ; dK/dlog w2_k = -1/2 w2_k sin^2 K
    // (reference Covariance.py:420-433); the noise derivative is vt wherever two points coincide (:412-413)
    grad[1] = 0.5 * h->hyp.vt * raw[3 * d + 1];
    for (int k = 0; k < d; ++k) {
      grad[2 + k] = -0.25 * h->hyp.w[k] * raw[1 + k];
      grad[2 + d + k] = 0.5 * h->hyp.pf[k] * h->hyp.w2[k] * raw[1 + d + k];
      grad[2 + 2 * d + k] = -0.25 * h->hyp.w2[k] * raw[1 + 2 * d + k];
    }
    return;
  }
  grad[1] = 0.5 * h->hyp.vt * (raw[d + 1] - raw[d + 2]);
  for (int k = 0; k < d; ++k) grad[2 + k] = -0.25 * h->hyp.w[k] * raw[1 + k];
}

static int ensure_route(Handle* h);

static int do_lauum(Handle* h) {
  if (h->have_inverse) return 0;
  GPK_TRY(ensure_route(h));
  h->x_sliced = false;   // the residue workspace is about to be reused
  GPK_TRY(lauum_launch(h->X, h->W, h->npad, h->npad, h->st, h->oz_on ? &h->oz : nullptr));
  h->have_inverse = true;
  return 0;
}

static bool same_theta(const Handle* h, const double* theta) {
  if (!h->factored || h->matrix_state) return false;
  return memcmp(h->theta, theta, sizeof(double) * theta_len(h->kind, h->d)) == 0;
}

// rows available per batch for the query workspace
static long batch_rows_for(const Handle* h, long want) {
  long cap = (long)(4.0e9 / (8.0 * h->npad));      // ~4 GB of workspace
  cap = cap / TILE * TILE;
  if (cap > 16384) cap = 16384;
  if (cap < TILE) cap = TILE;
  if (h->batch_rows > 0 && h->batch_rows < cap) cap = round_up_l(h->batch_rows, TILE);
  long r = round_up_l(want, TILE);
  return r < cap ? r : cap;
}

static int ensure_query_ws(Handle* h, long rows) {
  const long nbi = h->npad / TILE;
  GPK_TRY(ensure(&h->G, &h->G_elems, (size_t)rows * h->npad));
  size_t need = (size_t)nbi * rows + (size_t)nbi * (rows / 2);
  if (h->colsq_elems < need) {
    GPK_TRY(ensure(&h->colsq, &h->colsq_elems, need));
  }
  h->pairdot = h->colsq + (size_t)nbi * rows;
  GPK_TRY(ensure(&h->dots, &h->dots_elems, (size_t)rows));
  return 0;
}

// plane buffer of the factorisation products: a whole product at n <= 32768 (16 GiB), 8 GiB row panels at the orders
// where the matrices themselves take most of the 180 GB (n = 65536: 2 x 34 GB + 69 GB of operand residues)
static size_t oz_out_cap_bytes(const Handle* h) {
  if (h->oz_out_cap) return h->oz_out_cap;
  return (size_t)(h->npad >= 49152 ? 8192 : 16384) << 20;
}

// Allocate the INT8 workspace of a handle whose route asks for it. No silent fallback: if it does not fit, the call
// that needed it fails with -4 and the caller decides (gpk_set_route(h, 0, ...) selects FP64 DMMA explicitly).
static int ensure_route(Handle* h) {
  if (!h->oz_want || h->oz_on) return 0;
  const size_t np = h->npad;
  oz::Workspace& w = h->oz;
  w.S = h->oz_moduli_req ? h->oz_moduli_req : oz::crt_moduli_for(h->npad, 54);
  if (w.S < oz::CRT_MIN_MODULI) w.S = oz::CRT_MIN_MODULI;
  if (w.S > oz::CRT_MAX_MODULI) w.S = oz::CRT_MAX_MODULI;
  size_t want_out = (size_t)w.S * np * round_up_l((long)np, 256);
  if (want_out > oz_out_cap_bytes(h)) want_out = oz_out_cap_bytes(h);
  if (w.ensure((size_t)w.S * np * np, 4 * np, np) != 0 || w.ensure_out(want_out) != 0) {
    w.release();
    snprintf(g_err, sizeof(g_err),
             "INT8 route: %.1f GB of residue workspace + %.1f GB of residue planes do not fit on the device at n=%d "
             "(gpk_set_route(h, 0, 0, 0, 0) selects the FP64 DMMA kernels explicitly)",
             (double)w.S * np * np / 1e9, (double)want_out / 1e9, h->n);
    return -4;
  }
  h->ozq.S = w.S;
  h->oz_on = true;
  return ensure_overlap(h);
}

// residue planes of a rows x cols query product (INT8 route): 4 GiB at most, row panels beyond
static int ensure_query_planes(Handle* h, long rows, long cols) {
  size_t want_out = (size_t)h->oz.S * round_up_l(rows, 256) * round_up_l(cols, 256);
  const size_t qcap = oz_out_cap_bytes(h) < ((size_t)4 << 30) ? oz_out_cap_bytes(h) : ((size_t)4 << 30);
  if (want_out > qcap) want_out = qcap;
  return h->ozq.ensure_out(want_out);
}

// V = X * G^T for `rows` rows of G (multiple of 128). Vt == nullptr: only its colsq/pairdot partials (predictive
// variances, Girard quadratic forms); else V^T = G X^T itself, stored to Vt (rows x npad, leading dimension npad).
static int quad_forms(Handle* h, long rows, double* Vt = nullptr) {
  GPK_TRY(ensure_route(h));
  const int npad = h->npad;
  if (h->oz_on) {
    // INT8 tensor-core route: V^T = G X^T with the queries as rows, so each reconstruction warp sums its own row.
    // X is reduced once per factorisation (kept in the workspace), G once per batch.
    if (!h->x_sliced) {
      h->oz.reset();
      h->xs = h->oz.alloc(npad, npad);
      if (!h->xs.sl) { snprintf(g_err, sizeof(g_err), "INT8 route: residue workspace too small for X"); return -4; }
      GPK_TRY(oz::slice_operand(h->X, npad, 0, 1, h->xs, h->oz.mx, h->st));
      h->x_sliced = true;
    }
    h->ozq.S = h->oz.S;
    if (h->ozq.ensure((size_t)h->oz.S * rows * npad, (size_t)rows, (size_t)rows) != 0 ||
        ensure_query_planes(h, rows, npad) != 0) {
      snprintf(g_err, sizeof(g_err), "INT8 route: query workspace for %ld rows does not fit on the device", rows);
      return -4;
    }
    h->ozq.reset();
    oz::Operand g = h->ozq.alloc((int)rows, npad);
    GPK_TRY(oz::slice_operand(h->G, npad, 0, 0, g, h->ozq.mx, h->st));
    if (Vt) return oz::gemm_sliced(g, h->xs, Vt, npad, 1.0, 0.0, K_UPTO_BJ, 0, h->st);
    return oz::gemm_sliced(g, h->xs, nullptr, 0, 1.0, 0.0, K_UPTO_BJ, 0, h->st, oz::OZ_EPI_ROWSQ, h->colsq, h->pairdot,
                           rows);
  }
  if (Vt)   // the L21 = A21 X11^T form of the factorisation
    return gemm_store_auto<LAY_KC, LAY_KC>(
        gemm_args(h->G, npad, h->X, npad, Vt, npad, (int)rows, npad, npad, 1.0, 0.0, K_UPTO_BJ, 0), h->st);
  GemmArgs a = gemm_args(h->X, h->npad, h->G, h->npad, nullptr, 0, h->npad, (int)rows, h->npad, 1.0, 0.0, K_UPTO_BI, 0);
  a.colsq = h->colsq;
  a.pairdot = h->pairdot;
  a.ldo = rows;
  return gemm_launch<LAY_KC, LAY_KC, EPI_COLSQ>(a, h->st);
}

// ---- microbenchmarks -----------------------------------------------------------------------
// INT8 tensor-pipe probe: one CTA pair per two SMs, tcgen05.mma.cta_group::2.kind::i8 M=256 N=256 K=32 issued back to
// back from shared-memory tiles filled with pseudo-random bytes (so the datapath toggles like real operands), two
// 256-column TMEM accumulators alternating. No TMA, no epilogue: the ceiling of oz_crt_planes_kernel's MMA stream.
__global__ void __launch_bounds__(128, 1) mb_i8_kernel(long iters) {
  extern __shared__ uint8_t mb_smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = oz::cluster_ctarank();
  const uint32_t raw = oz::smem_u32(mb_smem_raw);
  uint8_t* smem = mb_smem_raw + ((1024u - (raw & 1023u)) & 1023u);
  uint64_t* done = reinterpret_cast<uint64_t*>(smem + 2 * oz::TILE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
  uint32_t* w = reinterpret_cast<uint32_t*>(smem);
  for (int i = threadIdx.x; i < 2 * oz::TILE_BYTES / 4; i += blockDim.x) {
    uint32_t x = (uint32_t)i * 2654435761u + blockIdx.x * 40503u + 12345u;
    x ^= x >> 15; x *= 2246822519u; x ^= x >> 13;
    w[i] = x;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
  if (warp == 1 && lane == 0) {
    oz::mbar_init(done, 1);
    oz::fence_barrier_init();
  }
  if (warp == 2) oz::tmem_alloc_pair(tmem_slot, oz::TMEM_COLS);
  oz::tc_fence_before();
  oz::cluster_sync_all();
  oz::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 1 && lane == 0 && rank == 0) {
    constexpr uint32_t idesc = oz::umma_idesc_i8(256, 256);
    const uint32_t st = oz::smem_u32(smem);
    const uint64_t ad = oz::umma_desc_sw128(st), bd = oz::umma_desc_sw128(st + oz::TILE_BYTES);
    for (long it = 0; it < iters; ++it) {
      const uint32_t acc = tmem_base + (uint32_t)((it & 1) * 256);
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4)
        oz::umma_i8_pair(acc, ad + (uint64_t)(k4 * 2), bd + (uint64_t)(k4 * 2), idesc, k4 > 0);
    }
    oz::umma_commit_pair(done, 3);
  }
  if (lane == 0) oz::mbar_wait(done, 0);
  __syncwarp();
  oz::tc_fence_before();
  oz::cluster_sync_all();
  if (warp == 2) oz::tmem_dealloc_pair(tmem_base, oz::TMEM_COLS);
}

}  // namespace gpk

using namespace gpk;

#define H_OR_FAIL(h)                                                     \
  Handle* hh = reinterpret_cast<Handle*>(h);                             \
  if (!hh) {                                                             \
    snprintf(g_err, sizeof(g_err), "null handle");                       \
    return -2;                                                           \
  }

extern "C" {

int gpk_version(void) { return 100; }
const char* gpk_last_error(void) { return g_err; }
int64_t gpk_npad(int64_t n) { return round_up_l(n < 1 ? 1 : n, TILE); }

// allocations of a new handle; on any failure the caller releases what was allocated so far
static int create_fill(Handle* h, int64_t n, int64_t d, double* Xbuf, double* Wbuf) {
  h->n = (int)n; h->d = (int)d; h->npad = (int)gpk_npad(n);
  const size_t np = h->npad;
  h->X = Xbuf; h->W = Wbuf;
  if (!h->X) { GPK_CUDA_OK(cudaMalloc((void**)&h->X, np * np * sizeof(double))); h->own_X = true; }
  if (!h->W) { GPK_CUDA_OK(cudaMalloc((void**)&h->W, np * np * sizeof(double))); h->own_W = true; }
  GPK_CUDA_OK(cudaMalloc((void**)&h->x, (size_t)n * d * sizeof(double)));
  GPK_CUDA_OK(cudaMalloc((void**)&h->xT, (size_t)d * np * sizeof(double)));
  GPK_CUDA_OK(cudaMalloc((void**)&h->t, np * sizeof(double)));
  GPK_CUDA_OK(cudaMalloc((void**)&h->y, np * sizeof(double)));
  GPK_CUDA_OK(cudaMalloc((void**)&h->alpha, np * sizeof(double)));
  GPK_CUDA_OK(cudaMalloc((void**)&h->dL, np * sizeof(double)));
  GPK_CUDA_OK(cudaMalloc((void**)&h->scal, 3 * sizeof(double)));
  GPK_CUDA_OK(cudaMalloc((void**)&h->info, sizeof(int)));
  if (h->own_X) GPK_CUDA_OK(poison_fill(h->X, np * np * sizeof(double)));
  if (h->own_W) GPK_CUDA_OK(poison_fill(h->W, np * np * sizeof(double)));
  GPK_CUDA_OK(poison_fill(h->x, (size_t)n * d * sizeof(double)));
  GPK_CUDA_OK(poison_fill(h->xT, (size_t)d * np * sizeof(double)));
  GPK_CUDA_OK(poison_fill(h->y, np * sizeof(double)));
  GPK_CUDA_OK(poison_fill(h->dL, np * sizeof(double)));
  GPK_CUDA_OK(poison_fill(h->scal, 3 * sizeof(double)));
  GPK_CUDA_OK(poison_fill(h->info, sizeof(int)));
  GPK_CUDA_OK(cudaMemset(h->t, 0, np * sizeof(double)));
  GPK_CUDA_OK(cudaMemset(h->alpha, 0, np * sizeof(double)));
  {
    // the off-critical-path products of the sub-2048 nodes are joined within microseconds: never behind the overlapped
    // INT8 products of the outer nodes
    int least = 0, greatest = 0;
    GPK_CUDA_OK(cudaDeviceGetStreamPriorityRange(&least, &greatest));
    GPK_CUDA_OK(cudaStreamCreateWithPriority(&h->side, cudaStreamNonBlocking, greatest));
  }
  h->events.resize(2 * (np / TILE) + 2 + 256);   // 2 per DMMA node, 5 per overlapped INT8 node
  for (auto& e : h->events) GPK_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  // INT8 tensor-core route for the large contractions: requested by default when the padded order reaches 2048
  // (gpk_set_route changes it); its workspace is allocated at the first factorisation / query (ensure_route).
  // Exact int32 accumulation bounds the inner dimension: K * 2^14 < 2^31 (residues in [-128,127]).
  h->oz.min_dim = 2048;
  h->oz_want = h->npad >= h->oz.min_dim && h->npad <= 98304;
  return 0;
}

int gpk_create(int64_t n, int64_t d, double* Xbuf, double* Wbuf, gpk_handle* out) {
  if (!out) { snprintf(g_err, sizeof(g_err), "gpk_create: null output pointer"); return -2; }
  *out = nullptr;
  if (n < 1 || d < 1 || d > MAX_D || n > (1 << 20)) {
    snprintf(g_err, sizeof(g_err), "gpk_create: bad shape n=%ld d=%ld", (long)n, (long)d);
    return -2;
  }
  Handle* h = new (std::nothrow) Handle();
  if (!h) return -3;
  const int rc = create_fill(h, n, d, Xbuf, Wbuf);
  if (rc != 0) {
    cudaGetLastError();   // clear the sticky allocation error so the release below is not misreported
    gpk_destroy(reinterpret_cast<gpk_handle>(h));
    return rc;
  }
  *out = reinterpret_cast<gpk_handle>(h);
  return 0;
}

int gpk_destroy(gpk_handle h) {
  H_OR_FAIL(h);
  cudaStreamSynchronize(hh->st);
  if (hh->own_X) cudaFree(hh->X);
  if (hh->own_W) cudaFree(hh->W);
  cudaFree(hh->x); cudaFree(hh->xT); cudaFree(hh->t); cudaFree(hh->y); cudaFree(hh->alpha); cudaFree(hh->dL);
  cudaFree(hh->scal); cudaFree(hh->info);
  for (auto& e : hh->events) if (e) cudaEventDestroy(e);
  if (hh->side) { cudaStreamSynchronize(hh->side); cudaStreamDestroy(hh->side); }
  if (hh->part) cudaFree(hh->part);
  if (hh->G) cudaFree(hh->G);
  if (hh->colsq) cudaFree(hh->colsq);
  if (hh->dots) cudaFree(hh->dots);
  if (hh->V) cudaFree(hh->V);
  if (hh->C) cudaFree(hh->C);
  hh->oz.release();
  hh->ozq.release();
  release_overlap(hh);
  if (hh->raw_pinned) cudaFreeHost(hh->raw_pinned);
  delete hh;
  return 0;
}

int gpk_set_stream(gpk_handle h, void* stream) {
  H_OR_FAIL(h);
  hh->st = reinterpret_cast<cudaStream_t>(stream);
  return 0;
}

int gpk_set_kernel(gpk_handle h, int kind) {
  H_OR_FAIL(h);
  if (kind != KIND_SE && kind != KIND_PERIODIC) { snprintf(g_err, sizeof(g_err), "unknown kernel kind %d", kind); return -2; }
  if (kind == KIND_PERIODIC && hh->d > PER_MAX_D) {
    snprintf(g_err, sizeof(g_err), "the periodic covariance supports d <= %d", PER_MAX_D);
    return -2;
  }
  hh->kind = kind;
  hh->factored = false;
  hh->have_inverse = false;
  hh->x_sliced = false;
  return 0;
}

int gpk_kernel_matrix_periodic(const double* x1, int64_t n1, const double* x2, int64_t n2, int64_t d, const double* theta,
                               int noise_mode, double* out, int64_t ld, void* stream) {
  SEHyper hyp;
  GPK_TRY(set_hyper(hyp, theta, (int)d, KIND_PERIODIC));
  return launch_se_tiles(x1, (int)n1, x2, (int)n2, (int)d, hyp, out, ld, (int)n1, (int)n2, noise_mode, 0, 0,
                         reinterpret_cast<cudaStream_t>(stream));
}

int gpk_set_route(gpk_handle h, int int8, int64_t min_dim, int moduli, int64_t plane_cap_bytes) {
  H_OR_FAIL(h);
  if (int8 && (min_dim != 0 && (min_dim < 2 * TILE || min_dim % TILE))) {
    snprintf(g_err, sizeof(g_err), "gpk_set_route: min_dim must be 0 (default 2048) or a multiple of 128 >= 256");
    return -2;
  }
  if (int8 && moduli != 0 && (moduli < oz::CRT_MIN_MODULI || moduli > oz::CRT_MAX_MODULI)) {
    snprintf(g_err, sizeof(g_err), "gpk_set_route: moduli must be 0 (automatic) or in [%d, %d]", oz::CRT_MIN_MODULI,
             oz::CRT_MAX_MODULI);
    return -2;
  }
  if (int8 && hh->npad > 98304) {
    snprintf(g_err, sizeof(g_err), "gpk_set_route: exact int32 accumulation needs npad <= 98304");
    return -2;
  }
  GPK_CUDA_OK(cudaStreamSynchronize(hh->st));
  hh->oz.release();
  hh->ozq.release();
  release_overlap(hh);
  hh->oz_on = false;
  hh->x_sliced = false;
  hh->factored = false;
  hh->have_inverse = false;
  hh->oz.min_dim = (int8 && min_dim) ? (int)min_dim : 2048;
  hh->oz_moduli_req = int8 ? moduli : 0;
  hh->oz_out_cap = plane_cap_bytes > 0 ? (size_t)plane_cap_bytes : 0;
  hh->oz_want = int8 != 0 && hh->npad >= hh->oz.min_dim;
  return 0;
}

int gpk_get_route(gpk_handle h, int* out) {
  H_OR_FAIL(h);
  const int S = hh->oz_on ? hh->oz.S
                          : (hh->oz_moduli_req ? hh->oz_moduli_req : oz::crt_moduli_for(hh->npad, 54));
  out[0] = hh->oz_want ? 1 : 0;
  out[1] = hh->oz_want ? S : 0;
  out[2] = hh->oz.min_dim;
  out[3] = hh->oz_want ? oz::crt_bits(hh->npad, S) : 53;
  return 0;
}

int gpk_set_batch_rows(gpk_handle h, int64_t rows) {
  H_OR_FAIL(h);
  hh->batch_rows = rows < 0 ? 0 : rows;
  return 0;
}

int gpk_set_data(gpk_handle h, const double* x_dev, const double* t_dev) {
  H_OR_FAIL(h);
  GPK_CUDA_OK(cudaMemcpyAsync(hh->x, x_dev, (size_t)hh->n * hh->d * sizeof(double), cudaMemcpyDeviceToDevice, hh->st));
  GPK_CUDA_OK(cudaMemsetAsync(hh->t, 0, (size_t)hh->npad * sizeof(double), hh->st));
  GPK_CUDA_OK(cudaMemcpyAsync(hh->t, t_dev, (size_t)hh->n * sizeof(double), cudaMemcpyDeviceToDevice, hh->st));
  transpose_x_kernel<<<(hh->npad + 255) / 256, 256, 0, hh->st>>>(hh->x, hh->n, hh->d, hh->xT, hh->npad);
  GPK_LAUNCH_OK();
  hh->factored = false;
  hh->have_inverse = false;
  return 0;
}

int gpk_kernel_matrix(const double* x1, int64_t n1, const double* x2, int64_t n2, int64_t d, const double* theta,
                      int add_noise, double* out, int64_t ld, void* stream) {
  SEHyper hyp;
  GPK_TRY(set_hyper(hyp, theta, (int)d));
  return launch_se_tiles(x1, (int)n1, x2, (int)n2, (int)d, hyp, out, ld, (int)n1, (int)n2, add_noise, 0, 0,
                         reinterpret_cast<cudaStream_t>(stream));
}

// W holds K (lower tiles, identity in the padding block): factor it, form X = L^-1, y = X t, alpha, log det
static int factorize_W(Handle* hh) {
  const int n = hh->n, npad = hh->npad;
  set_int_kernel<<<1, 1, 0, hh->st>>>(hh->info, INT_MAX);
  GPK_LAUNCH_OK();
  FactorCtx c{hh->W, hh->X, (long)npad, hh->dL, hh->info, hh->st};
  hh->ev_next = 0;
  c.side = hh->side; c.ev = hh->events.data(); c.ev_next = &hh->ev_next;
  c.oz = hh->oz_on ? &hh->oz : nullptr;
  const bool ovl = hh->oz_on && hh->ovl_on && g_overlap_T;
  if (ovl) {
    // the critical path moves to the high-priority stream for the duration of the recursion
    GPK_CUDA_OK(cudaEventRecord(hh->ev_in, hh->st));
    GPK_CUDA_OK(cudaStreamWaitEvent(hh->chain_st, hh->ev_in, 0));
    c.st = hh->chain_st;
    c.ovl_ws = hh->ovl_ws.data(); c.ovl_st = hh->ovl_st.data(); c.ovl_depths = (int)hh->ovl_ws.size();
  }
  const int rc_rec = potrf_inv_node(c, 0, npad);
  if (rc_rec < 0) {
    // a failed launch / allocation in the middle of the recursion leaves forked streams behind: drain them before the
    // caller can touch the buffers again
    cudaDeviceSynchronize();
    return rc_rec;
  }
  if (ovl) {
    GPK_CUDA_OK(cudaEventRecord(hh->ev_out, hh->chain_st));
    GPK_CUDA_OK(cudaStreamWaitEvent(hh->st, hh->ev_out, 0));
  }
  GPK_TRY(solve_one(hh, hh->t, hh->y, hh->alpha));
  nll_scalars_kernel<<<1, 256, 0, hh->st>>>(hh->dL, hh->y, hh->alpha, n, hh->scal);
  GPK_LAUNCH_OK();
  int info = 0;
  double sc[3];
  GPK_CUDA_OK(cudaMemcpyAsync(&info, hh->info, sizeof(int), cudaMemcpyDeviceToHost, hh->st));
  GPK_CUDA_OK(cudaMemcpyAsync(sc, hh->scal, 3 * sizeof(double), cudaMemcpyDeviceToHost, hh->st));
  GPK_CUDA_OK(cudaStreamSynchronize(hh->st));
  if (info != INT_MAX) {
    snprintf(g_err, sizeof(g_err), "leading minor %d of K is not positive definite", info);
    return info > 0 ? info : 1;
  }
  hh->logdet = sc[0]; hh->quad = sc[1]; hh->alpha2 = sc[2];
  return 0;
}

int gpk_factorize(gpk_handle h, const double* theta, int want_inverse) {
  H_OR_FAIL(h);
  if (!same_theta(hh, theta)) {
    hh->factored = false;
    hh->have_inverse = false;
    hh->x_sliced = false;
    hh->grad_pending = false;   // sums of another theta (stream order keeps the pinned buffer consistent)
    GPK_TRY(set_hyper(hh->hyp, theta, hh->d, hh->kind));
    GPK_TRY(ensure_route(hh));
    const int n = hh->n, npad = hh->npad;
    // K (lower tiles) -> W
    GPK_TRY(launch_se_tiles(hh->x, n, hh->x, n, hh->d, hh->hyp, hh->W, npad, npad, npad, noise_mode(hh->kind, true), 1,
                            1, hh->st));
    const int rc = factorize_W(hh);
    if (rc != 0) return rc;
    memcpy(hh->theta, theta, sizeof(double) * theta_len(hh->kind, hh->d));
    hh->factored = true;
    hh->matrix_state = false;
  }
  if (want_inverse) GPK_TRY(do_lauum(hh));
  return 0;
}

// W[r][c] = K[r][c] for the lower 128-tiles (c tile <= r tile), identity in the padding block
__global__ void __launch_bounds__(256) load_matrix_kernel(const double* __restrict__ K, long ldk, int n,
                                                          double* __restrict__ W, long ld, int npad) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  const int r = blockIdx.y;
  if (c >= npad || (c >> 7) > (r >> 7)) return;
  W[(long)r * ld + c] = (r < n && c < n) ? K[(long)r * ldk + c] : (r == c ? 1.0 : 0.0);
}

int gpk_factorize_matrix(gpk_handle h, const double* K_dev, int64_t ldk, int want_inverse) {
  H_OR_FAIL(h);
  if (!K_dev || ldk < hh->n) { snprintf(g_err, sizeof(g_err), "gpk_factorize_matrix: bad matrix argument"); return -2; }
  hh->factored = false;
  hh->have_inverse = false;
  hh->x_sliced = false;
  GPK_TRY(ensure_route(hh));
  dim3 grid((hh->npad + 255) / 256, hh->npad);
  load_matrix_kernel<<<grid, 256, 0, hh->st>>>(K_dev, ldk, hh->n, hh->W, hh->npad, hh->npad);
  GPK_LAUNCH_OK();
  const int rc = factorize_W(hh);
  if (rc != 0) return rc;
  hh->factored = true;
  hh->matrix_state = true;   // theta-keyed entry points (nll_grad, predict, propagate) do not apply to this state
  if (want_inverse) GPK_TRY(do_lauum(hh));
  return 0;
}

int gpk_nll_matrix(gpk_handle h, double* nll) {
  H_OR_FAIL(h);
  if (!hh->factored) { snprintf(g_err, sizeof(g_err), "not factored"); return -2; }
  *nll = nll_of(hh);
  return 0;
}

int gpk_logdet(gpk_handle h, double* out) {
  H_OR_FAIL(h);
  if (!hh->factored) { snprintf(g_err, sizeof(g_err), "not factored"); return -2; }
  *out = hh->logdet;
  return 0;
}

int gpk_grad_trace_partial(gpk_handle h, int64_t trb, int64_t tre, double* out) {
  H_OR_FAIL(h);
  if (!hh->factored || !hh->have_inverse || hh->matrix_state) { snprintf(g_err, sizeof(g_err), "inverse not available"); return -2; }
  if (hh->kind != KIND_SE) { snprintf(g_err, sizeof(g_err), "sharded trace: Gaussian covariance only"); return -2; }
  const int nt = hh->npad / TILE;
  if (trb < 0) trb = 0;
  if (tre > nt) tre = nt;
  double sums[TRACE_SUMS] = {};   // stays zero for an empty range
  GPK_TRY(trace_enqueue(hh, (int)trb, (int)tre, sums));
  GPK_CUDA_OK(cudaStreamSynchronize(hh->st));
  trace_unpack(hh, sums, out);
  return 0;
}

int gpk_nll_grad(gpk_handle h, const double* theta, double* nll, double* grad, int want_grad) {
  H_OR_FAIL(h);
  const bool prefetch = want_grad == 2 && hh->kind == KIND_SE;
  const bool cached = same_theta(hh, theta);
  if (!cached && hh->grad_pending) {            // a prefetch for another theta is still in flight: let it finish
    GPK_CUDA_OK(cudaStreamSynchronize(hh->st));
    hh->grad_pending = false;
  }
  int rc = gpk_factorize(h, theta, want_grad == 1);
  if (rc != 0) return rc;
  if (nll) *nll = nll_of(hh);
  if (prefetch && !hh->grad_pending) {
    // the caller announced that the gradient at this theta follows: queue K^-1 = X^T X and the trace sums now, so the
    // device keeps working while the host returns the likelihood
    if (!hh->raw_pinned) GPK_CUDA_OK(cudaMallocHost((void**)&hh->raw_pinned, TRACE_SUMS * sizeof(double)));
    GPK_TRY(do_lauum(hh));
    GPK_TRY(trace_enqueue(hh, 0, hh->npad / TILE, hh->raw_pinned));
    hh->grad_pending = true;
    return 0;
  }
  if (want_grad == 1 && grad) {
    double sums[TRACE_SUMS], raw[3 * MAX_D + 3];
    if (!hh->grad_pending) GPK_TRY(trace_enqueue(hh, 0, hh->npad / TILE, sums));
    GPK_CUDA_OK(cudaStreamSynchronize(hh->st));
    trace_unpack(hh, hh->grad_pending ? hh->raw_pinned : sums, raw);
    hh->grad_pending = false;
    grad_from_raw(hh, raw, grad);
  }
  return 0;
}

int gpk_solve(gpk_handle h, const double* b, int64_t nrhs, double* out) {
  H_OR_FAIL(h);
  if (!hh->factored) { snprintf(g_err, sizeof(g_err), "not factored"); return -2; }
  const int npad = hh->npad, n = hh->n;
  GPK_TRY(ensure_query_ws(hh, TILE));  // borrow G as padded rhs / result scratch (>= 3*npad doubles)
  double* bp = hh->G;
  double* yy = hh->G + npad;
  double* oo = hh->G + 2 * (size_t)npad;
  for (int64_t r = 0; r < nrhs; ++r) {
    GPK_CUDA_OK(cudaMemsetAsync(bp, 0, npad * sizeof(double), hh->st));
    GPK_CUDA_OK(cudaMemcpyAsync(bp, b + r * n, n * sizeof(double), cudaMemcpyDeviceToDevice, hh->st));
    GPK_TRY(solve_one(hh, bp, yy, oo));
    GPK_CUDA_OK(cudaMemcpyAsync(out + r * n, oo, n * sizeof(double), cudaMemcpyDeviceToDevice, hh->st));
  }
  return 0;
}

int gpk_inverse(gpk_handle h, double* Kinv_out, int64_t ldo) {
  H_OR_FAIL(h);
  if (!hh->factored) { snprintf(g_err, sizeof(g_err), "not factored"); return -2; }
  GPK_TRY(do_lauum(hh));
  const int n = hh->n;
  dim3 grid((n + 31) / 32, (n + 31) / 32);
  symmetrize_out_kernel<<<grid, 256, 0, hh->st>>>(hh->W, hh->npad, n, Kinv_out, ldo);
  GPK_LAUNCH_OK();
  return 0;
}

// G[q][i] = Ks[q][i] for q < m, i < n; zero in the padding
__global__ void __launch_bounds__(256) load_rows_kernel(const double* __restrict__ Ks, long ldk, int m, int n,
                                                        double* __restrict__ G, long ldg, int npad) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  const int q = blockIdx.y;
  if (i >= npad) return;
  G[(long)q * ldg + i] = (q < m && i < n) ? Ks[(long)q * ldk + i] : 0.0;
}

// The query batches of gpk_predict, gpk_predict_cross and the K alpha of gpk_solve_residual. Row q of G is the
// covariance k(xq_q, x_i) from the family's tile kernel, or the caller's row Ks[q] when xq is null.
// With mean: mean[q] = G_q . alpha (+ meant). With var: var[q] = prior[q] - |X G_q|^2, and v + vt in place of a null
// prior. With Vt (gpk_predict_cov): row q of Vt = (X G_q)^T, round_up(m, 128) rows of npad, zero beyond row m.
static int query_batches(Handle* h, const double* xq, const double* Ks, long ldk, long m, double meant, double* mean,
                         double* var, const double* prior, double* Vt = nullptr) {
  const int npad = h->npad, n = h->n, d = h->d, nbi = npad / TILE;
  const long rows_max = batch_rows_for(h, m);
  GPK_TRY(ensure_query_ws(h, rows_max));
  for (long q0 = 0; q0 < m; q0 += rows_max) {
    const long mb = (m - q0) < rows_max ? m - q0 : rows_max;
    const long rows = round_up_l(mb, TILE);   // G zero padded to rows x npad
    if (xq) {
      GPK_TRY(launch_se_tiles(xq + q0 * d, (int)mb, h->x, n, d, h->hyp, h->G, npad, (int)rows, npad,
                              noise_mode(h->kind, false), 0, 0, h->st));
    } else {
      load_rows_kernel<<<dim3((npad + 255) / 256, (unsigned)rows), 256, 0, h->st>>>(Ks + q0 * ldk, ldk, (int)mb, n,
                                                                                    h->G, npad, npad);
      GPK_LAUNCH_OK();
    }
    if (mean) {
      rows_dot_kernel<<<(unsigned)((mb + 7) / 8), 256, 0, h->st>>>(h->G, npad, (int)mb, npad, h->alpha, mean + q0);
      GPK_LAUNCH_OK();
      if (meant != 0.0) {
        add_scalar_kernel<<<(unsigned)((mb + 255) / 256), 256, 0, h->st>>>(mean + q0, (int)mb, meant);
        GPK_LAUNCH_OK();
      }
    }
    if (Vt) GPK_TRY(quad_forms(h, rows, Vt + q0 * npad));
    if (var) {
      GPK_TRY(quad_forms(h, rows));
      predict_var_kernel<<<(unsigned)((mb + 255) / 256), 256, 0, h->st>>>(h->colsq, rows, nbi, (int)mb,
                                                                          prior ? prior + q0 : nullptr,
                                                                          h->hyp.v + h->hyp.vt, var + q0);
      GPK_LAUNCH_OK();
    }
  }
  return 0;
}

// Joint predictive covariance Sigma(A, B) = prior(A, B) - V_A^T V_B, V_Q = X k(x, Q), for gpk_predict_cov and
// gpk_predict_cov_cross. Rows of A / B come from the query points xa / xb through the family's tile kernel, or from the
// caller's cross covariances Ka / Kb; prior is the caller's block (ldp), else k(A, B) with the family's noise rule.
// xb and Kb both null: B = A, only the lower tiles are formed and mirrored on the way out, so the result is exactly
// symmetric. V^T of both sets stays resident for the call and the product runs once over K = npad, on the route of
// the factorisation; if its workspace does not fit, the call fails with -4 before any work is queued.
static int predict_cov_impl(Handle* h, const double* xa, const double* Ka, long lda, long ma, const double* xb,
                            const double* Kb, long ldb, long mb, const double* prior, long ldp, double* cov, long ldc) {
  const bool sym = !xb && !Kb;
  const long npad = h->npad;
  const long ma_pad = round_up_l(ma, TILE), mb_pad = sym ? ma_pad : round_up_l(mb, TILE);
  const long vrows = sym ? ma_pad : ma_pad + mb_pad;
  GPK_TRY(ensure_route(h));
  // every allocation of the call, before any of its work is queued: V, the output block, the query batch (G and its
  // partials), and on the INT8 route the residues of V (which also hold those of G) and the planes of both products
  const long mmax = ma_pad > mb_pad ? ma_pad : mb_pad;
  const long rows_max = batch_rows_for(h, mmax);
  const size_t res_bytes = h->oz_on ? (size_t)h->oz.S * vrows * npad : 0;
  if (ensure(&h->V, &h->V_elems, (size_t)vrows * npad) != 0 || ensure(&h->C, &h->C_elems, (size_t)ma_pad * mb_pad) != 0 ||
      ensure_query_ws(h, rows_max) != 0 ||
      (h->oz_on && (h->ozq.ensure(res_bytes, (size_t)vrows, (size_t)mmax) != 0 ||
                    ensure_query_planes(h, rows_max, npad) != 0 || ensure_query_planes(h, ma_pad, mb_pad) != 0))) {
    cudaGetLastError();   // the failed allocation is reported here, not by the next call
    snprintf(g_err, sizeof(g_err),
             "predictive covariance %ld x %ld at n=%d: %.2f GB of V + %.2f GB of output block + %.2f GB of query batch "
             "+ %.2f GB of V residues do not fit on the device",
             ma, mb, h->n, 8.0 * vrows * npad / 1e9, 8.0 * ma_pad * mb_pad / 1e9, 8.0 * rows_max * npad / 1e9,
             (double)res_bytes / 1e9);
    return -4;
  }
  double* Va = h->V;
  double* Vb = sym ? h->V : h->V + ma_pad * npad;
  GPK_TRY(query_batches(h, xa, Ka, lda, ma, 0.0, nullptr, nullptr, nullptr, Va));
  if (!sym) GPK_TRY(query_batches(h, xb, Kb, ldb, mb, 0.0, nullptr, nullptr, nullptr, Vb));
  // the padding of the output block is never copied out: a caller's prior leaves it unset
  if (prior) {
    GPK_CUDA_OK(cudaMemcpy2DAsync(h->C, mb_pad * sizeof(double), prior, ldp * sizeof(double), mb * sizeof(double), ma,
                                  cudaMemcpyDeviceToDevice, h->st));
  } else {
    GPK_TRY(launch_se_tiles(xa, (int)ma, sym ? xa : xb, (int)mb, h->d, h->hyp, h->C, mb_pad, (int)ma_pad, (int)mb_pad,
                            noise_mode(h->kind, sym), 0, sym ? 1 : 0, h->st));
  }
  if (h->oz_on) {
    // the residues of G are consumed by the V products queued above; the residues of V replace them
    h->ozq.reset();
    oz::Operand a = h->ozq.alloc((int)ma_pad, (int)npad);
    oz::Operand b = sym ? a : h->ozq.alloc((int)mb_pad, (int)npad);
    GPK_TRY(oz::slice_operand(Va, npad, 0, 0, a, h->ozq.mx, h->st));
    if (!sym) GPK_TRY(oz::slice_operand(Vb, npad, 0, 0, b, h->ozq.mx, h->st));
    GPK_TRY(oz::gemm_sliced(a, sym ? a : b, h->C, mb_pad, -1.0, 1.0, K_FULL, sym ? 1 : 0, h->st));
  } else {
    GPK_TRY((gemm_store_auto<LAY_KC, LAY_KC>(
        gemm_args(Va, npad, Vb, npad, h->C, mb_pad, (int)ma_pad, (int)mb_pad, (int)npad, -1.0, 1.0, K_FULL, sym ? 1 : 0),
        h->st)));
  }
  if (sym) {
    dim3 grid((unsigned)((ma + 31) / 32), (unsigned)((ma + 31) / 32));
    symmetrize_out_kernel<<<grid, 256, 0, h->st>>>(h->C, mb_pad, (int)ma, cov, ldc);
    GPK_LAUNCH_OK();
  } else {
    GPK_CUDA_OK(cudaMemcpy2DAsync(cov, ldc * sizeof(double), h->C, mb_pad * sizeof(double), mb * sizeof(double), ma,
                                  cudaMemcpyDeviceToDevice, h->st));
  }
  return 0;
}

// out[0] = max_i |(K alpha)_i - t_i|, out[1] = max_i |alpha_i|, out[2] = max_i |t_i| over the n training points
__global__ void __launch_bounds__(256) residual_max_kernel(const double* __restrict__ Ka, const double* __restrict__ t,
                                                           const double* __restrict__ alpha, int n,
                                                           unsigned long long* __restrict__ out) {
  __shared__ double red[3][8];
  double r = 0.0, a = 0.0, tm = 0.0;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
    r = fmax(r, fabs(Ka[i] - t[i]));
    a = fmax(a, fabs(alpha[i]));
    tm = fmax(tm, fabs(t[i]));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    r = fmax(r, __shfl_xor_sync(0xffffffffu, r, o));
    a = fmax(a, __shfl_xor_sync(0xffffffffu, a, o));
    tm = fmax(tm, __shfl_xor_sync(0xffffffffu, tm, o));
  }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = r; red[1][threadIdx.x >> 5] = a; red[2][threadIdx.x >> 5] = tm; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double m = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) m = fmax(m, red[threadIdx.x][i]);
    atomicMax(out + threadIdx.x, (unsigned long long)__double_as_longlong(m));   // non-negative doubles order like their bits
  }
}

int gpk_solve_residual(gpk_handle h, double* out_host) {
  H_OR_FAIL(h);
  if (!hh->factored || hh->matrix_state) { snprintf(g_err, sizeof(g_err), "not factored from theta"); return -2; }
  const int n = hh->n;
  // K alpha with K regenerated tile row by tile row in the query workspace (K itself was consumed by the factorisation)
  GPK_TRY(ensure(&hh->part, &hh->part_elems, (size_t)hh->npad + 8));
  double* Ka = hh->part;
  unsigned long long* mx = reinterpret_cast<unsigned long long*>(hh->part + hh->npad);
  GPK_CUDA_OK(cudaMemsetAsync(mx, 0, 3 * sizeof(unsigned long long), hh->st));
  GPK_TRY(query_batches(hh, hh->x, nullptr, 0, n, 0.0, Ka, nullptr, nullptr));
  if (hh->kind != KIND_PERIODIC) {
    // the Gaussian family adds vt on the diagonal only (Covariance.py:461-464): (K alpha)_i += vt alpha_i
    axpy_kernel<<<(n + 255) / 256, 256, 0, hh->st>>>(Ka, hh->alpha, n, hh->hyp.vt);
    GPK_LAUNCH_OK();
  }
  residual_max_kernel<<<64, 256, 0, hh->st>>>(Ka, hh->t, hh->alpha, n, mx);
  GPK_LAUNCH_OK();
  unsigned long long bits[3];
  GPK_CUDA_OK(cudaMemcpyAsync(bits, mx, sizeof(bits), cudaMemcpyDeviceToHost, hh->st));
  GPK_CUDA_OK(cudaStreamSynchronize(hh->st));
  for (int i = 0; i < 3; ++i) memcpy(out_host + i, bits + i, sizeof(double));
  return 0;
}

int gpk_get_alpha(gpk_handle h, double* out) {
  H_OR_FAIL(h);
  if (!hh->factored) { snprintf(g_err, sizeof(g_err), "not factored"); return -2; }
  GPK_CUDA_OK(cudaMemcpyAsync(out, hh->alpha, (size_t)hh->n * sizeof(double), cudaMemcpyDeviceToDevice, hh->st));
  return 0;
}

int gpk_import_state(gpk_handle h, const double* theta, const double* alpha_dev, int have_inverse) {
  H_OR_FAIL(h);
  GPK_TRY(set_hyper(hh->hyp, theta, hh->d, hh->kind));
  memcpy(hh->theta, theta, sizeof(double) * theta_len(hh->kind, hh->d));
  GPK_CUDA_OK(cudaMemsetAsync(hh->alpha, 0, (size_t)hh->npad * sizeof(double), hh->st));
  GPK_CUDA_OK(cudaMemcpyAsync(hh->alpha, alpha_dev, (size_t)hh->n * sizeof(double), cudaMemcpyDeviceToDevice, hh->st));
  hh->factored = true;
  hh->matrix_state = false;
  hh->x_sliced = false;
  hh->have_inverse = have_inverse != 0;
  hh->logdet = NAN; hh->quad = NAN; hh->alpha2 = NAN;  // scalars stay on the factorising rank
  return 0;
}

int gpk_predict(gpk_handle h, const double* xs, int64_t m, double meant, double* mean, double* var, int want_var) {
  H_OR_FAIL(h);
  if (!hh->factored || hh->matrix_state) { snprintf(g_err, sizeof(g_err), "not factored from theta"); return -2; }
  if (m <= 0) return 0;
  return query_batches(hh, xs, nullptr, 0, m, meant, mean, want_var ? var : nullptr, nullptr);
}

int gpk_predict_cross(gpk_handle h, const double* Ks, int64_t ldk, int64_t m, const double* prior, double meant,
                      double* mean, double* var) {
  H_OR_FAIL(h);
  if (!hh->factored) { snprintf(g_err, sizeof(g_err), "not factored"); return -2; }
  if (m <= 0) return 0;
  if (!Ks || ldk < hh->n || (var && !prior)) {
    snprintf(g_err, sizeof(g_err), "gpk_predict_cross: bad cross-covariance argument");
    return -2;
  }
  return query_batches(hh, nullptr, Ks, ldk, m, meant, mean, var, prior);
}

int gpk_predict_cov(gpk_handle h, const double* xa, int64_t ma, const double* xb, int64_t mb, double* cov, int64_t ldc) {
  H_OR_FAIL(h);
  if (!hh->factored || hh->matrix_state) { snprintf(g_err, sizeof(g_err), "not factored from theta"); return -2; }
  if (!xb) mb = ma;
  if (ma < 0 || mb < 0) { snprintf(g_err, sizeof(g_err), "gpk_predict_cov: negative query count"); return -2; }
  if (ma == 0 || mb == 0) return 0;
  if (!xa || !cov || ldc < mb) { snprintf(g_err, sizeof(g_err), "gpk_predict_cov: bad query or output argument"); return -2; }
  return predict_cov_impl(hh, xa, nullptr, 0, ma, xb, nullptr, 0, mb, nullptr, 0, cov, ldc);
}

int gpk_predict_cov_cross(gpk_handle h, const double* Ka, int64_t lda, int64_t ma, const double* Kb, int64_t ldb,
                          int64_t mb, const double* prior, int64_t ldp, double* cov, int64_t ldc) {
  H_OR_FAIL(h);
  if (!hh->factored) { snprintf(g_err, sizeof(g_err), "not factored"); return -2; }
  if (!Kb) mb = ma;
  if (ma < 0 || mb < 0) { snprintf(g_err, sizeof(g_err), "gpk_predict_cov_cross: negative query count"); return -2; }
  if (ma == 0 || mb == 0) return 0;
  if (!Ka || lda < hh->n || (Kb && ldb < hh->n) || !prior || ldp < mb || !cov || ldc < mb) {
    snprintf(g_err, sizeof(g_err), "gpk_predict_cov_cross: bad cross-covariance, prior or output argument");
    return -2;
  }
  return predict_cov_impl(hh, nullptr, Ka, lda, ma, nullptr, Kb, ldb, mb, prior, ldp, cov, ldc);
}

// Gradients of the predictive mean and variance at the query points xq (gpk_predict_grad). Each query owns P = d + 1
// rows of G: k* from the family's tile kernel (leading dimension P npad, so the means are those of gpk_predict), then
// D_1 .. D_d from grad_build_kernel; a batch holds whole queries. One rows_dot_kernel gives the means and their
// gradients. With var: V^T = G X^T through the store product, group_dots_kernel forms V_0 . V_r per query, and
// grad_finalize_kernel writes var = v + vt - |V_0|^2, dvar_k = -2 V_0 . V_k. Every allocation precedes the work.
static int predict_grad_impl(Handle* h, const double* xq, long m, double meant, double* mean, double* var,
                             double* dmean, double* dvar) {
  const int npad = h->npad, n = h->n, d = h->d, P = d + 1, nbi = npad / TILE;
  long qb_max = batch_rows_for(h, m * (long)P) / P;
  if (qb_max < 1) qb_max = 1;
  const long rows_max = round_up_l(qb_max * P, TILE);
  if (var) GPK_TRY(ensure_route(h));
  const size_t res_bytes = var && h->oz_on ? (size_t)h->oz.S * rows_max * npad : 0;
  if (ensure_query_ws(h, rows_max) != 0 ||
      (var && (ensure(&h->V, &h->V_elems, (size_t)rows_max * npad) != 0 ||
               (h->oz_on && (h->ozq.ensure(res_bytes, (size_t)rows_max, (size_t)rows_max) != 0 ||
                             ensure_query_planes(h, rows_max, npad) != 0))))) {
    cudaGetLastError();   // the failed allocation is reported here, not by the next call
    snprintf(g_err, sizeof(g_err),
             "predictive gradient at n=%d, d=%d: %.2f GB of query batch + %.2f GB of V^T batch + %.2f GB of its residues "
             "do not fit on the device",
             n, d, 8.0 * rows_max * npad / 1e9, var ? 8.0 * rows_max * npad / 1e9 : 0.0, (double)res_bytes / 1e9);
    return -4;
  }
  for (long q0 = 0; q0 < m; q0 += qb_max) {
    const long qb = (m - q0) < qb_max ? m - q0 : qb_max;
    const long rows = round_up_l(qb * P, TILE);
    GPK_TRY(launch_se_tiles(xq + q0 * d, (int)qb, h->x, n, d, h->hyp, h->G, (long)P * npad, (int)qb, npad,
                            noise_mode(h->kind, false), 0, 0, h->st));
    GradArgs a;
    a.xT = h->xT; a.ldxt = npad; a.xq = xq + q0 * d;
    a.n = n; a.npad = npad; a.d = d; a.P = P; a.Q = (int)qb;
    a.G = h->G; a.ldg = npad; a.rows_pad = (int)rows;
    grad_build_kernel<<<dim3((npad + 255) / 256, (unsigned)(qb + (rows - qb * P))), 256, 0, h->st>>>(a, h->hyp);
    GPK_LAUNCH_OK();
    rows_dot_kernel<<<(unsigned)((qb * P + 7) / 8), 256, 0, h->st>>>(h->G, npad, (int)(qb * P), npad, h->alpha, h->dots);
    GPK_LAUNCH_OK();
    if (var) {
      GPK_TRY(quad_forms(h, rows, h->V));
      group_dots_kernel<<<dim3((unsigned)nbi, (unsigned)qb), 256, 0, h->st>>>(h->V, npad, P, h->colsq, rows);
      GPK_LAUNCH_OK();
    }
    grad_finalize_kernel<<<(unsigned)((qb * P + 255) / 256), 256, 0, h->st>>>(
        h->dots, var ? h->colsq : nullptr, rows, nbi, (int)qb, d, meant, h->hyp.v + h->hyp.vt, mean + q0, dmean + q0 * d,
        var ? var + q0 : nullptr, dvar ? dvar + q0 * d : nullptr);
    GPK_LAUNCH_OK();
  }
  return 0;
}

int gpk_predict_grad(gpk_handle h, const double* xs, int64_t m, double meant, double* mean, double* var, double* dmean,
                     double* dvar) {
  H_OR_FAIL(h);
  if (!hh->factored || hh->matrix_state) { snprintf(g_err, sizeof(g_err), "not factored from theta"); return -2; }
  if (m < 0) { snprintf(g_err, sizeof(g_err), "gpk_predict_grad: negative query count"); return -2; }
  if (m == 0) return 0;
  if (!xs || !mean || !dmean || (var == nullptr) != (dvar == nullptr)) {
    snprintf(g_err, sizeof(g_err), "gpk_predict_grad: bad query or output argument (var and dvar go together)");
    return -2;
  }
  return predict_grad_impl(hh, xs, m, meant, mean, var, dmean, dvar);
}

static int propagate_impl(gpk_handle h, const double* U, const double* S, int64_t Q, int sigma_full, double meant,
                          double* mean, double* var, double* sigma2, double* rest) {
  H_OR_FAIL(h);
  if (!hh->factored || hh->matrix_state) { snprintf(g_err, sizeof(g_err), "not factored from theta"); return -2; }
  if (hh->kind != KIND_SE) { snprintf(g_err, sizeof(g_err), "propagation needs the Gaussian covariance"); return -2; }
  if (Q <= 0) return 0;
  const int npad = hh->npad, n = hh->n, d = hh->d;
  const int P = (d + 2 + 1) / 2 * 2;  // rows per query, even so (C,tr) form an aligned pair
  const long rows_cap = batch_rows_for(hh, Q * (long)P);
  long qb_max = rows_cap / P;
  if (qb_max < 1) qb_max = 1;
  const long rows_max = round_up_l(qb_max * P, TILE);
  GPK_TRY(ensure_query_ws(hh, rows_max));
  const int nbi = npad / TILE;
  const long sstride = sigma_full ? (long)d * d : d;
  for (int64_t q0 = 0; q0 < Q; q0 += qb_max) {
    const long qb = (Q - q0) < qb_max ? (long)(Q - q0) : qb_max;
    const long rows = round_up_l(qb * P, TILE);
    GAArgs a;
    a.xT = hh->xT; a.ldxt = npad; a.n = n; a.npad = npad; a.d = d; a.P = P;
    a.U = U + q0 * d; a.S = S + q0 * sstride; a.sigma_full = sigma_full;
    a.G = hh->G; a.ldg = npad; a.rows_pad = (int)rows; a.Q = (int)qb;
    dim3 grid((npad + 255) / 256, (unsigned)(qb + (rows - qb * P)));
    ga_build_kernel<<<grid, 256, 0, hh->st>>>(a, hh->hyp);
    GPK_LAUNCH_OK();
    rows_dot_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, hh->st>>>(hh->G, npad, (int)rows, npad, hh->alpha, hh->dots);
    GPK_LAUNCH_OK();
    GPK_TRY(quad_forms(hh, rows));
    ga_finalize_kernel<<<(unsigned)((qb + 255) / 256), 256, 0, hh->st>>>(hh->colsq, hh->pairdot, rows, nbi, hh->dots,
                                                                          a.S, sigma_full, (int)qb, d, P, hh->hyp.v,
                                                                          hh->hyp.vt, meant, mean ? mean + q0 : nullptr,
                                                                          var ? var + q0 : nullptr,
                                                                          sigma2 ? sigma2 + q0 : nullptr,
                                                                          rest ? rest + q0 : nullptr);
    GPK_LAUNCH_OK();
  }
  return 0;
}

int gpk_propagate_exact(gpk_handle h, const double* U, const double* Lam, const double* Dinv, const double* norms,
                        int64_t Q, double meant, double* mean, double* var) {
  H_OR_FAIL(h);
  if (!hh->factored || hh->matrix_state) { snprintf(g_err, sizeof(g_err), "not factored from theta"); return -2; }
  if (hh->d > 32) { snprintf(g_err, sizeof(g_err), "exact propagation supports d <= 32"); return -2; }
  if (hh->kind != KIND_SE) { snprintf(g_err, sizeof(g_err), "propagation needs the Gaussian covariance"); return -2; }
  if (Q <= 0) return 0;
  GPK_TRY(do_lauum(hh));
  const int nt = hh->npad / TILE, d = hh->d;
  const int64_t qb_max = Q < 4096 ? Q : 4096;
  GPK_TRY(ensure(&hh->part, &hh->part_elems, (size_t)qb_max * nt + (size_t)qb_max + (size_t)qb_max * hh->npad));
  double* mu = hh->part + (size_t)qb_max * nt;
  double* gq = mu + qb_max;
  for (int64_t q0 = 0; q0 < Q; q0 += qb_max) {
    const int qb = (int)((Q - q0) < qb_max ? (Q - q0) : qb_max);
    ExactArgs a;
    a.xT = hh->xT; a.ldxt = hh->npad; a.alpha = hh->alpha; a.Kinv = hh->W; a.ld = hh->npad;
    a.n = hh->n; a.npad = hh->npad; a.d = d; a.Q = qb;
    a.U = U + q0 * d; a.Lam = Lam + q0 * d * d; a.Dinv = Dinv + q0 * d; a.norms = norms + q0 * 2;
    exact_mean_kernel<<<qb, 256, 0, hh->st>>>(a, hh->hyp, mu);
    GPK_LAUNCH_OK();
    dim3 ggrid((hh->npad + 255) / 256, qb);
    exact_g_kernel<<<ggrid, 256, 0, hh->st>>>(a, hh->hyp, gq);
    GPK_LAUNCH_OK();
    dim3 grid(qb, nt);
    GPK_TRY(dispatch_pass_dim<32>(d, [&](auto dp) {
      exact_pair_kernel<decltype(dp)::value><<<grid, 256, 0, hh->st>>>(a, gq, hh->part);
      GPK_LAUNCH_OK();
      return 0;
    }));
    exact_finalize_kernel<<<(qb + 255) / 256, 256, 0, hh->st>>>(hh->part, nt, mu, a.norms, qb, hh->hyp.v + hh->hyp.vt,
                                                                 meant, mean + q0, var + q0);
    GPK_LAUNCH_OK();
  }
  return 0;
}

int gpk_propagate_ga(gpk_handle h, const double* U, const double* S, int64_t Q, int sigma_full, double meant,
                     double* mean, double* var) {
  return propagate_impl(h, U, S, Q, sigma_full, meant, mean, var, nullptr, nullptr);
}

int gpk_propagate_ga_parts(gpk_handle h, const double* U, const double* S, int64_t Q, int sigma_full,
                           double* sigma2, double* rest) {
  return propagate_impl(h, U, S, Q, sigma_full, 0.0, nullptr, nullptr, sigma2, rest);
}

// ---- test / measurement hooks --------------------------------------------------------------
int gpk_test_potrf_inv(double* A, double* X, int64_t ld, int64_t npad, double* dL, int* info_host, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (npad % TILE) { snprintf(g_err, sizeof(g_err), "npad must be a multiple of 128"); return -2; }
  int* info_dev = nullptr;
  GPK_CUDA_OK(cudaMalloc((void**)&info_dev, sizeof(int)));
  set_int_kernel<<<1, 1, 0, st>>>(info_dev, INT_MAX);
  FactorCtx c{A, X, (long)ld, dL, info_dev, st};
  int rc = potrf_inv_node(c, 0, (int)npad);
  int info = 0;
  cudaError_t e = cudaMemcpyAsync(&info, info_dev, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(info_dev);
  if (rc < 0) return rc;
  if (e != cudaSuccess) { snprintf(g_err, sizeof(g_err), "potrf_inv: %s", cudaGetErrorString(e)); return -1; }
  *info_host = (info == INT_MAX) ? 0 : info;
  return 0;
}

int gpk_test_oz_residues(const double* src, int64_t ld, int64_t rows, int64_t K, int trans, int lower, int moduli,
                         void* planes_out, double* scales_out, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  oz::Operand op;
  op.sl = reinterpret_cast<int8_t*>(planes_out); op.sc = scales_out;
  op.rows = (int)rows; op.K = (int)K; op.S = moduli;
  unsigned long long* mx = nullptr;
  GPK_CUDA_OK(cudaMalloc((void**)&mx, (size_t)rows * sizeof(unsigned long long)));
  int rc = oz::slice_operand(src, ld, trans, lower, op, mx, st);
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(mx);
  if (rc < 0) return rc;
  if (e != cudaSuccess) { snprintf(g_err, sizeof(g_err), "oz_residues: %s", cudaGetErrorString(e)); return -1; }
  return 0;
}

int gpk_test_oz_gemm(const double* A, int64_t lda, int transA, int lowerA, const double* B, int64_t ldb, int transB,
                     int lowerB, double* C, int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha, double beta,
                     int krange, int lower_only, int moduli, int64_t panel_rows, int reps, float* ms_out, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  oz::Operand a, b;
  a.rows = (int)M; a.K = (int)K; a.S = moduli;
  b.rows = (int)N; b.K = (int)K; b.S = moduli;
  unsigned long long* mx = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr;
  int rc = 0;
  auto cleanup = [&]() {
    cudaFree(a.sl); cudaFree(a.sc); cudaFree(b.sl); cudaFree(b.sc); cudaFree(mx); cudaFree(a.out);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (e2) cudaEventDestroy(e2);
  };
#define OZ_OK(expr)                                                                         \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      snprintf(g_err, sizeof(g_err), "oz_gemm: %s -> %s", #expr, cudaGetErrorString(_e));   \
      cleanup();                                                                            \
      return -1;                                                                            \
    }                                                                                       \
  } while (0)
  OZ_OK(cudaMalloc((void**)&a.sl, oz::Operand::slice_bytes(a.rows, a.K, a.S)));
  OZ_OK(cudaMalloc((void**)&b.sl, oz::Operand::slice_bytes(b.rows, b.K, b.S)));
  OZ_OK(cudaMalloc((void**)&a.sc, (size_t)M * sizeof(double)));
  OZ_OK(cudaMalloc((void**)&b.sc, (size_t)N * sizeof(double)));
  OZ_OK(cudaMalloc((void**)&mx, (size_t)(M > N ? M : N) * sizeof(unsigned long long)));
  {
    // residue planes of the product: whole product, or `panel_rows` rows at a time (exercises the panel loop)
    const long prow = panel_rows > 0 ? round_up_l((long)panel_rows, 256) : round_up_l((long)M, 256);
    size_t want_out = (size_t)a.S * prow * round_up_l((long)N, 256);
    if (want_out > ((size_t)16 << 30)) want_out = (size_t)16 << 30;
    OZ_OK(cudaMalloc((void**)&a.out, want_out));
    a.out_cap = want_out;
  }
  OZ_OK(cudaEventCreate(&e0));
  OZ_OK(cudaEventCreate(&e1));
  OZ_OK(cudaEventCreate(&e2));
  OZ_OK(cudaEventRecord(e0, st));
  rc = oz::slice_operand(A, lda, transA, lowerA, a, mx, st);
  if (rc == 0) rc = oz::slice_operand(B, ldb, transB, lowerB, b, mx, st);
  if (rc < 0) { cleanup(); return rc; }
  OZ_OK(cudaEventRecord(e1, st));
  if (reps < 1) reps = 1;
  for (int r = 0; r < reps && rc == 0; ++r) rc = oz::gemm_sliced(a, b, C, ldc, alpha, beta, krange, lower_only, st);
  if (rc < 0) { cleanup(); return rc; }
  OZ_OK(cudaEventRecord(e2, st));
  OZ_OK(cudaStreamSynchronize(st));
  if (ms_out) {
    OZ_OK(cudaEventElapsedTime(&ms_out[0], e0, e1));
    OZ_OK(cudaEventElapsedTime(&ms_out[1], e1, e2));
    ms_out[1] /= reps;
  }
#undef OZ_OK
  cleanup();
  return 0;
}

int gpk_test_position_lock(int on) {
  if (on >= 0 && on <= 2) oz::g_position_lock = on;
  return oz::g_position_lock;
}

int gpk_test_poison(int byte) {
  const size_t kib = g_poison_bytes >> 10;
  g_poison_bytes = 0;
  g_poison = byte & 0xff;
  int*& spill = oz::g_spill_dev[current_device_slot()];
  if (spill) GPK_CUDA_OK(poison_fill(spill, oz::SPILL_BYTES));
  g_poison_bytes = 0;   // the count covers allocations only
  return kib > INT_MAX ? INT_MAX : (int)kib;
}

int gpk_test_overlap(int on) {
  if (on == 0 || on == 1) g_overlap_T = on;
  return g_overlap_T;
}

int gpk_profile(int on) {
  g_prof_on = on != 0;
  return 0;
}

int gpk_profile_read(double* gemm_ms, int64_t* gemm_launches, int64_t* all_launches, double* max_gemm_ms) {
  double total = 0.0, longest = 0.0;
  for (auto& p : g_prof) {
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(p.b);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, p.a, p.b);
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
    if (e != cudaSuccess) {
      snprintf(g_err, sizeof(g_err), "gpk_profile_read: %s", cudaGetErrorString(e));
      g_prof.clear();
      return -1;
    }
    total += ms;
    if (ms > longest) longest = ms;
  }
  if (max_gemm_ms) *max_gemm_ms = longest;
  if (gemm_ms) *gemm_ms = total;
  if (gemm_launches) *gemm_launches = (int64_t)g_prof.size();
  if (all_launches) *all_launches = (int64_t)g_launch_count;
  g_prof.clear();
  g_launch_count = 0;
  return 0;
}

int gpk_microbench_i8(int64_t iters, double seconds, double* out_host) {
  int nsm = 0, dev = 0;
  GPK_CUDA_OK(cudaGetDevice(&dev));
  GPK_CUDA_OK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
  const int smem = 2 * oz::TILE_BYTES + 1024 + 64;
  GPK_CUDA_OK(cudaFuncSetAttribute(mb_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  const int pairs = nsm / 2;
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = nullptr;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaEvent_t e0, e1;
  GPK_CUDA_OK(cudaEventCreate(&e0));
  GPK_CUDA_OK(cudaEventCreate(&e1));
  const double ops_per_launch = (double)pairs * (double)iters * 4.0 * 256.0 * 256.0 * 32.0 * 2.0;
  long it = iters;
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    GPK_CUDA_OK(cudaEventRecord(e0));
    GPK_CUDA_OK(cudaLaunchKernelEx(&cfg, mb_i8_kernel, it));
    GPK_LAUNCH_OK();
    GPK_CUDA_OK(cudaEventRecord(e1));
    GPK_CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0.f;
    GPK_CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    const double tops = ops_per_launch / (ms * 1e-3) / 1e12;
    if (rep > 0 && tops > best) best = tops;
  }
  out_host[0] = best;
  out_host[1] = 0.0;
  if (seconds > 0.0) {
    const double per_launch_s = ops_per_launch / (best * 1e12);
    long launches = (long)(seconds / per_launch_s) + 1;
    GPK_CUDA_OK(cudaEventRecord(e0));
    for (long l = 0; l < launches; ++l) {
      GPK_CUDA_OK(cudaLaunchKernelEx(&cfg, mb_i8_kernel, it));
      GPK_LAUNCH_OK();
    }
    GPK_CUDA_OK(cudaEventRecord(e1));
    GPK_CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0.f;
    GPK_CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    out_host[1] = ops_per_launch * launches / (ms * 1e-3) / 1e12;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return 0;
}

}  // extern "C"
