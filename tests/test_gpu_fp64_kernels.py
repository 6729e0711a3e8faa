"""Kernel-level tests of the hand-written FP64 kernels against same-operand extended-precision references.

The end-to-end parity tests compare with the reference's LU-inverse numbers at 1e-9, which mixes the kernel's own error
with the conditioning of K. Here every check reads back what the kernel consumed (the matrix handed to the leaf, K^-1
from the lower triangle of W through `Engine.inverse_device`, alpha, x and theta) and recomputes the kernel's own
operation in numpy longdouble (64-bit significand, tests/arbiter.py). Factorisation and conditioning error drop out, so
the tolerances sit at the kernel's rounding: a sum is compared relative to the sum of the absolute values of its terms
("mag"), and the factorisation relative to the error of host FP64 computations on the same input. Every check prints its
observed ratio to the bound, so the margin is in the log (run with -s).

  A  leaf_blocked_kernel + the sub-2048 DMMA recursion (gpk_test_potrf_inv): X = L^-1, diag L, first bad pivot
  B  grad_trace_kernel<4|8|16|32> (one and two passes), trace_enqueue / trace_unpack, periodic_trace_kernel<4|8|16>
  C  exact_pair_kernel<4|8|16|32> through UncertaintyPropagationExact
  D  non-positive-definite K through gpk_factorize_matrix on the DMMA and INT8 routes
"""
import ctypes
import functools

import numpy as np
import pytest
import scipy.linalg as sla

from arbiter import LD, DenseArbiter, chol_ld, kernel_ld, solve_lower_ld
from oracle import gp_oracle as O

pytestmark = pytest.mark.gpu

TILE = 128


@pytest.fixture(scope="module")
def gpk():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import skgpuppy.Covariance as C
    import skgpuppy.GaussianProcess as G
    import skgpuppy.UncertaintyPropagation as U
    from skgpuppy import _engine, _native
    C.VERBOSE = False

    class NS:
        Cov = C
        GP = G
        UP = U
        eng = _engine
        nat = _native
        lib = _native.load()
    NS.torch = torch
    return NS


def report(what, ratio):
    """Print the observed error over its bound (a check passes at ratio <= 1)."""
    print("%-64s ratio %.3e" % (what, ratio))
    return ratio


def _synthetic(n, d, seed):
    """Inputs of the end-to-end parity tests (tests/test_gpu_parity.py): vt = 0.09, length scales ~ sqrt(d / 4)."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 1, (n, d))
    a = rng.uniform(0.5, 1.5, d)
    t = np.sin(2 * np.pi * a * x).sum(1) + 0.5 * np.prod(np.cos(np.pi * x[:, :2]), 1) + 0.3 * rng.standard_normal(n)
    theta = np.concatenate([[0.0, np.log(0.09)], np.log((4.0 / d) * np.linspace(0.75, 1.25, d))])
    return x, t, theta, rng


# ==== A. leaf and sub-2048 recursion ===================================================================================
def _se_matrix(n, cond, seed):
    """SE kernel matrix of n points in [0,1]^2 with the noise chosen so that cond(K) is about `cond`."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 1, (n, 2))
    Knl = np.asarray(kernel_ld(x, x, [0.0, 0.0, np.log(10.0), np.log(10.0)]), dtype=np.float64)
    lmax = float(np.linalg.eigvalsh(Knl)[-1])
    return Knl + (lmax / cond) * np.eye(n)


def _bbt_matrix(n, seed):
    rng = np.random.default_rng(seed)
    B = rng.standard_normal((n, n))
    return B @ B.T / n + np.eye(n)


@functools.lru_cache(maxsize=None)
def _leaf_input(kind, npad):
    """The FP64 matrix handed to the leaf recursion (order npad)."""
    if kind == "bbt":
        return _bbt_matrix(npad, npad)
    if kind.startswith("se"):
        return _se_matrix(npad, float(kind[2:]), npad + 1)
    # "embed300": K of order 300 with the identity padding load_matrix_kernel writes
    A = np.eye(npad)
    A[:300, :300] = _se_matrix(300, 1e4, 300)
    return A


@functools.lru_cache(maxsize=None)
def _leaf_chol_ld(kind, npad):
    return chol_ld(_leaf_input(kind, npad))


def _potrf_inv(gpk, A):
    """gpk_test_potrf_inv on a copy of A (host FP64, order npad): (X = L^-1, diag L, info) as host arrays. X starts
    at 7.0 everywhere so that a tile the kernel fails to write shows up."""
    torch, nat = gpk.torch, gpk.nat
    npad = A.shape[0]
    W = torch.as_tensor(np.ascontiguousarray(A), device="cuda").clone()
    X = torch.full_like(W, 7.0)
    dL = torch.zeros(npad, dtype=torch.float64, device="cuda")
    info = ctypes.c_int(-1)
    nat.check(gpk.lib.gpk_test_potrf_inv(nat.ptr(W), nat.ptr(X), npad, npad, nat.ptr(dL), ctypes.byref(info),
                                         nat.current_stream_ptr()), "gpk_test_potrf_inv")
    torch.cuda.synchronize()
    return X.cpu().numpy(), dL.cpu().numpy(), info.value


def _diag_tiles_upper_zero(X):
    for b in range(X.shape[0] // TILE):
        blk = X[b * TILE:(b + 1) * TILE, b * TILE:(b + 1) * TILE]
        assert np.all(np.triu(blk, 1) == 0.0), "tile %d: upper part of a diagonal tile of X is not zero" % b


def _recursion_fp64(A):
    """The recursion of factor.cuh in numpy FP64, leaves by LAPACK: L21 = A21 X11^T through the explicit inverse,
    A22 -= L21 L21^T, X21 = -X22 (L21 X11). Returns (X, diag L)."""
    A = A.copy()
    n = A.shape[0]
    X, dL = np.zeros_like(A), np.zeros(n)

    def node(r0, s):
        if s <= TILE:
            L = np.linalg.cholesky(A[r0:r0 + s, r0:r0 + s])
            dL[r0:r0 + s] = np.diag(L)
            X[r0:r0 + s, r0:r0 + s] = sla.solve_triangular(L, np.eye(s), lower=True)
            return
        h1 = (s // TILE // 2) * TILE
        r1, r2 = r0 + h1, r0 + s
        node(r0, h1)
        L21 = A[r1:r2, r0:r1] @ X[r0:r1, r0:r1].T
        T21 = L21 @ X[r0:r1, r0:r1]
        A[r1:r2, r1:r2] -= L21 @ L21.T
        node(r1, s - h1)
        X[r1:r2, r0:r1] = -X[r1:r2, r1:r2] @ T21
    node(0, n)
    return X, dL


def _block_rel(X, Xr):
    """max |X - Xr| / max |Xr| per 128-row block."""
    out = []
    for b in range(0, Xr.shape[0], TILE):
        ref = Xr[b:b + TILE]
        out.append(float(np.max(np.abs(np.asarray(X[b:b + TILE], dtype=LD) - ref)) / np.max(np.abs(ref))))
    return np.array(out)


@pytest.mark.parametrize("npad,kind", [(128, "se1e2"), (128, "bbt"), (256, "se1e5"), (384, "se1e8"), (384, "embed300"),
                                       (640, "se1e6"), (1152, "bbt")])
def test_leaf_recursion_vs_longdouble(gpk, npad, kind):
    """X = L^-1 and diag L of the DMMA recursion (leaves of 128, uneven splits at 384 / 640 / 1152) against the
    longdouble factor of the same FP64 matrix, per 128-row block, under 4 x the error of a host FP64 peer + 1e-15; the
    strict upper part of every diagonal tile of X is exactly zero.

    The peer error is the larger of two host computations: numpy/scipy `cholesky` + `solve_triangular`, and the same
    recursion in numpy FP64 (`_recursion_fp64`). The second is needed at high condition numbers: the recursion solves
    for L21 through the explicit inverse X11 instead of by substitution, and that alone costs accuracy. At cond(A) = 1e8
    (npad 384), in the blocks below the first leaf, the FP64 host recursion is up to 15x (X) and 20x (diag L) less
    accurate than substitution, the device recursion 14x and 16x (B200). Up to cond 1e6 the two host peers agree within
    2x."""
    A = _leaf_input(kind, npad)
    X, dL, info = _potrf_inv(gpk, A)
    assert info == 0
    _diag_tiles_upper_zero(X)
    Lr = _leaf_chol_ld(kind, npad)
    Xr = solve_lower_ld(Lr, np.eye(npad, dtype=LD))
    dr = np.diag(Lr)
    Lp = np.linalg.cholesky(A)
    Xp = sla.solve_triangular(Lp, np.eye(npad), lower=True)
    Xq, dq = _recursion_fp64(A)

    def d_rel(d):
        return np.array([float(np.max(np.abs(d[b:b + TILE] - dr[b:b + TILE]) / dr[b:b + TILE]))
                         for b in range(0, npad, TILE)])
    e_gpu, e_lapack, e_rec = _block_rel(np.tril(X), Xr), _block_rel(Xp, Xr), _block_rel(Xq, Xr)
    d_gpu, d_lapack, d_rec = d_rel(dL), d_rel(np.diag(Lp)), d_rel(dq)
    print("cond(A) = %.2e; per block error / substitution peer: device %s, host recursion %s" % (
        np.linalg.cond(A), np.array2string(e_gpu / e_lapack, precision=2), np.array2string(e_rec / e_lapack, precision=2)))
    rx = report("leaf npad=%d %s: X per block vs 4 x FP64 peer + 1e-15" % (npad, kind),
                float(np.max(e_gpu / (4 * np.maximum(e_lapack, e_rec) + 1e-15))))
    rd = report("leaf npad=%d %s: diag L per block vs 4 x FP64 peer + 1e-15" % (npad, kind),
                float(np.max(d_gpu / (4 * np.maximum(d_lapack, d_rec) + 1e-15))))
    assert rx <= 1.0 and rd <= 1.0


@pytest.mark.parametrize("kind", ["bbt", "se1e6"])
def test_leaf_recursion_npad2048_residual(gpk, kind):
    """npad = 2048, the largest all-DMMA block of the production recursion: max |X A X^T - I| against the same
    residual of the FP64 host factor (both evaluated with the same device matmul)."""
    torch = gpk.torch
    A = _bbt_matrix(2048, 2048) if kind == "bbt" else _se_matrix(2048, 1e6, 2049)
    X, dL, info = _potrf_inv(gpk, A)
    assert info == 0
    _diag_tiles_upper_zero(X)
    Lp = np.linalg.cholesky(A)
    Xp = sla.solve_triangular(Lp, np.eye(2048), lower=True)
    Ad = torch.as_tensor(A, device="cuda")
    I = torch.eye(2048, dtype=torch.float64, device="cuda")

    def resid(Xh):
        Xd = torch.as_tensor(np.tril(Xh), device="cuda")
        return float((Xd @ Ad @ Xd.T - I).abs().max())
    r_gpu, r_peer = resid(X), resid(Xp)
    # a pivot's relative error grows with A_jj / L_jj^2, the cancellation in its Schur complement
    amp = np.diag(A) / np.diag(Lp) ** 2
    dl = float(np.max(np.abs(dL - np.diag(Lp)) / np.diag(Lp) / amp))
    rr = report("leaf npad=2048 %s: max|X A X^T - I| %.2e vs 4 x peer %.2e + 1e-15" % (kind, r_gpu, r_peer),
                r_gpu / (4 * r_peer + 1e-15))
    rd = report("leaf npad=2048 %s: diag L vs FP64 host factor, 64 eps x A_jj / L_jj^2" % kind, dl / (64 * 2.2e-16))
    assert rr <= 1.0 and rd <= 1.0


@pytest.mark.parametrize("npad,kind", [(384, "se1e5"), (2048, "bbt")])
def test_leaf_recursion_power_of_4_scaling_is_exact(gpk, npad, kind):
    """D = diag(4^k_i), k_i in [-8, 8]: in exact arithmetic X(DAD) = X(A) D^-1 and diag L(DAD) = D diag L(A). Every
    FP64 operation of the recursion (DMMA included) commutes with power-of-two scalings, and so do the rcp.approx /
    rsqrt.approx seeds of the leaf with their Newton steps: the results are equal bit for bit."""
    A = _leaf_input(kind, npad) if npad < 2048 else _bbt_matrix(2048, 2048)
    rng = np.random.default_rng(npad)
    D = 4.0 ** rng.integers(-8, 9, npad)
    X, dL, info = _potrf_inv(gpk, A)
    Xs, dLs, info_s = _potrf_inv(gpk, D[:, None] * A * D[None, :])
    assert info == 0 and info_s == 0
    Xe, Xse = np.tril(X) / D[None, :], np.tril(Xs)
    ulps = np.abs(Xe.view(np.int64) - Xse.view(np.int64))
    print("npad=%d: max ulp distance X %d, diag L %d" % (npad, int(ulps.max()),
                                                          int(np.max(np.abs((dL * D).view(np.int64) - dLs.view(np.int64))))))
    assert np.array_equal(Xe, Xse)
    assert np.array_equal(dL * D, dLs)


def _with_pivot(A, L, k):
    """A with pivot k (1-based) moved to -0.5: A[k-1,k-1] -= p_k + 0.5, p_k = L[k-1,k-1]^2 from the longdouble factor.
    The leading minors of order < k are unchanged and stay positive definite."""
    B = A.copy()
    B[k - 1, k - 1] = float(LD(A[k - 1, k - 1]) - (L[k - 1, k - 1] ** 2 + LD(0.5)))
    return B


@pytest.mark.parametrize("npad,k", [(256, 1), (256, 16), (256, 17), (256, 128), (256, 129), (256, 256),
                                    (1152, 1000), (1152, 1152)])
def test_leaf_recursion_first_bad_pivot(gpk, npad, k):
    """info is exactly k: the first pivot of a chain-warp panel (17), the first pivot after a DMMA SYRK (129), the
    last row, and row 1000 of the 1152 recursion."""
    A = _leaf_input("bbt", npad)
    _, _, info = _potrf_inv(gpk, _with_pivot(A, _leaf_chol_ld("bbt", npad), k))
    print("npad=%d pivot %d: info %d" % (npad, k, info))
    assert info == k


@pytest.mark.parametrize("npad,j", [(256, 0), (256, 200), (1152, 700)])
def test_leaf_recursion_nan_diagonal(gpk, npad, j):
    A = _leaf_input("bbt", npad).copy()
    A[j, j] = np.nan
    _, _, info = _potrf_inv(gpk, A)
    print("npad=%d NaN at row %d: info %d" % (npad, j, info))
    assert 0 < info <= j + 1


# ==== B. gradient traces ===============================================================================================
class SETraceRef(object):
    """Same-operand longdouble reference of gpk_grad_trace_partial. Per row i: sum over columns j <= i, weight 2 below
    the diagonal and 1 on it, of M_ij Knl_ij (entry 0) and M_ij Knl_ij (x_ik - x_jk)^2 (entry 1 + k), with
    M = K^-1 - alpha alpha^T; entry d + 1 is K^-1_ii and d + 2 is alpha_i^2. The per-row absolute sums are the mags."""

    def __init__(self, x, theta, Kinv, alpha):
        n, d = x.shape
        self.n, self.d = n, d
        M = np.asarray(Kinv, dtype=LD) - np.outer(alpha, alpha).astype(LD)
        wt = np.tril(np.full((n, n), 2.0), -1) + np.eye(n)
        P = wt.astype(LD) * M * kernel_ld(x, x, theta)
        aP = np.abs(P)
        xl = x.astype(LD)
        self.rows = np.zeros((n, d + 3), dtype=LD)
        self.mags = np.zeros((n, d + 3), dtype=LD)
        self.rows[:, 0], self.mags[:, 0] = P.sum(1), aP.sum(1)
        for k in range(d):
            D2 = (xl[:, k][:, None] - xl[:, k][None, :]) ** 2
            self.rows[:, 1 + k], self.mags[:, 1 + k] = (P * D2).sum(1), (aP * D2).sum(1)
        kd = np.diag(np.asarray(Kinv)).astype(LD)
        a2 = np.asarray(alpha).astype(LD) ** 2
        self.rows[:, d + 1], self.mags[:, d + 1] = kd, np.abs(kd)
        self.rows[:, d + 2], self.mags[:, d + 2] = a2, a2

    def sums(self, b, e):
        r0, r1 = max(b, 0) * TILE, min(e * TILE, self.n)
        if r1 <= r0:
            return np.zeros(self.d + 3, dtype=LD), np.zeros(self.d + 3, dtype=LD)
        return self.rows[r0:r1].sum(0), self.mags[r0:r1].sum(0)


def _se_engine(gpk, n, d, seed, route=None):
    x, t, theta, _ = _synthetic(n, d, seed)
    tc = t - t.mean()
    eng = gpk.eng.Engine(x, tc, route=route)
    eng.factorize(theta, want_inverse=True)
    return eng, x, tc, theta


SE_CASES = [(300, d) for d in (1, 4, 5, 8, 9, 16, 17, 31, 32, 33, 64)] + [(1, 3), (128, 9), (129, 33)]


def _se_case_id(c):
    n, d = c
    dp = 4 if d <= 4 else 8 if d <= 8 else 16 if d <= 16 else 32
    return "n%d-d%d-DP%dx%d" % (n, d, dp, (d + dp - 1) // dp)


@pytest.mark.parametrize("n,d", SE_CASES, ids=[_se_case_id(c) for c in SE_CASES])
def test_se_trace_partial_vs_longdouble(gpk, n, d):
    """grad_trace_kernel<DP> (DP = 4 / 8 / 16 / 32, one pass and two at d = 33 / 64 = GPK_MAX_D) and the diag / alpha
    sums over tile-row ranges, against the same-operand reference at 1e-12 x mag; clamped ranges equal the full range,
    a 3-way partition sums to it; then the whole gradient."""
    eng, x, tc, theta = _se_engine(gpk, n, d, 1000 + 7 * n + d)
    Kinv = eng.inverse_device().cpu().numpy()
    alpha = eng.alpha_device().cpu().numpy()
    ref = SETraceRef(x, theta, Kinv, alpha)
    nt = eng.npad // TILE
    full = eng.grad_trace_partial(0, nt)
    worst = 0.0
    for b, e in sorted({(0, nt), (0, 1), (1, nt), (nt - 1, nt)}):
        raw = eng.grad_trace_partial(b, e)
        r, m = ref.sums(b, e)
        if e <= b:
            assert np.all(raw == 0.0)
            continue
        ratio = float(np.max(np.abs(raw.astype(LD) - r) / (1e-12 * m + 1e-300)))
        worst = max(worst, ratio)
        assert ratio <= 1.0, "tiles [%d, %d)" % (b, e)
    report("SE trace n=%d d=%d: ranges vs longdouble at 1e-12 mag" % (n, d), worst)
    assert np.all(eng.grad_trace_partial(nt, nt) == 0.0) and np.all(eng.grad_trace_partial(nt, 0) == 0.0)
    assert np.array_equal(eng.grad_trace_partial(-1, nt + 5), full)
    cuts = [0, nt // 3, (2 * nt) // 3, nt]
    part = sum(eng.grad_trace_partial(cuts[i], cuts[i + 1]).astype(LD) for i in range(3))
    _, m = ref.sums(0, nt)
    rp = report("SE trace n=%d d=%d: 3-way partition vs full at 1e-14 mag" % (n, d),
                float(np.max(np.abs(part - full.astype(LD)) / (1e-14 * m + 1e-300))))
    assert rp <= 1.0
    # whole gradient: closed form on the reference sums, and the longdouble arbiter
    _, g = eng.nll_grad(theta, want_grad=True)
    r, m = ref.sums(0, nt)
    vt, w = np.exp(LD(theta[1])), np.exp(theta[2:].astype(LD))
    g_ref = np.concatenate([[r[0] / 2, vt * (r[d + 1] - r[d + 2]) / 2], -w * r[1:d + 1] / 4])
    g_mag = np.concatenate([[m[0] / 2, vt * (m[d + 1] + m[d + 2]) / 2], w * m[1:d + 1] / 4])
    rg = report("SE gradient n=%d d=%d: closed form on reference sums at 1e-12 mag" % (n, d),
                float(np.max(np.abs(g.astype(LD) - g_ref) / (1e-12 * g_mag + 1e-300))))
    assert rg <= 1.0
    ga = DenseArbiter(x, tc, theta).gradient()
    ra = report("SE gradient n=%d d=%d: vs DenseArbiter at 1e-9" % (n, d),
                float(np.max(np.abs(g.astype(LD) - ga)) / np.max(np.abs(ga)) / 1e-9))
    assert ra <= 1.0
    # the prefetch path (want_grad = 2): same kernels and sum layout, copied to the pinned buffer and unpacked later
    eng.nll_grad(theta + 1e-3, want_grad=False)
    eng.nll_grad(theta, want_grad=False, prefetch_grad=True)
    _, g2 = eng.nll_grad(theta, want_grad=True)
    assert np.array_equal(g2, g)
    eng.close()


def test_se_trace_int8_route_n2200(gpk):
    """n = 2200, d = 17 on the production route: K^-1 comes from the INT8 planes kernel, the trace is unchanged."""
    eng, x, tc, theta = _se_engine(gpk, 2200, 17, 2217)
    assert eng.route()[0]
    Kinv = eng.inverse_device().cpu().numpy()
    alpha = eng.alpha_device().cpu().numpy()
    ref = SETraceRef(x, theta, Kinv, alpha)
    nt = eng.npad // TILE
    worst = 0.0
    for b, e in ((0, nt), (5, 11), (nt - 1, nt)):
        raw = eng.grad_trace_partial(b, e)
        r, m = ref.sums(b, e)
        worst = max(worst, float(np.max(np.abs(raw.astype(LD) - r) / (1e-12 * m))))
    report("SE trace n=2200 d=17 INT8 route: ranges vs longdouble at 1e-12 mag", worst)
    assert worst <= 1.0
    _, g = eng.nll_grad(theta, want_grad=True)
    eng.nll_grad(theta, want_grad=False, prefetch_grad=True)
    eng.nll_grad(theta + 1e-3, want_grad=False)
    eng.nll_grad(theta, want_grad=False, prefetch_grad=True)
    assert np.array_equal(eng.nll_grad(theta, want_grad=True)[1], g)
    eng.close()


def _periodic_inputs(n, d, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 1, (n, d))
    t = np.sin(2 * np.pi * x).sum(1) + 0.2 * rng.standard_normal(n)
    theta = np.concatenate([[0.0, np.log(0.09)], np.log((2.0 / d) * np.linspace(0.75, 1.25, d)),
                            np.log(np.linspace(0.6, 1.4, d)), np.log((1.0 / d) * np.linspace(1.25, 0.75, d))])
    return x, t - t.mean(), theta


@pytest.mark.parametrize("d", [1, 4, 5, 8, 9, 16], ids=lambda d: "d%d-DPp%d" % (d, 4 if d <= 4 else 8 if d <= 8 else 16))
def test_periodic_gradient_vs_longdouble(gpk, d):
    """periodic_trace_kernel<4|8|16> (full and partial pads) through the 2 + 3d gradient, against the same-operand
    longdouble gradient from the handle's K^-1 and alpha at 1e-12 x mag."""
    n = 300
    x, tc, theta = _periodic_inputs(n, d, 500 + d)
    eng = gpk.eng.Engine(x, tc, kind=1)
    eng.factorize(theta, want_inverse=True)
    Kinv = eng.inverse_device().cpu().numpy()
    alpha = eng.alpha_device().cpu().numpy()
    _, g = eng.nll_grad(theta, want_grad=True)
    v, vt = np.exp(LD(theta[0])), np.exp(LD(theta[1]))
    w, p, w2 = (np.exp(theta[2 + i * d:2 + (i + 1) * d].astype(LD)) for i in range(3))
    pf = (np.pi / np.exp(theta[2 + d:2 + 2 * d])).astype(LD)      # pi / p_k rounded in FP64, as the host does
    M = np.asarray(Kinv, dtype=LD) - np.outer(alpha, alpha).astype(LD)
    xl = x.astype(LD)
    Dk = [xl[:, k][:, None] - xl[:, k][None, :] for k in range(d)]
    Sk = [np.sin(pf[k] * Dk[k]) for k in range(d)]
    K = v * np.exp(LD(-0.5) * sum(w2[k] * Sk[k] ** 2 + w[k] * Dk[k] ** 2 for k in range(d)))
    P = M * K
    aP = np.abs(P)
    same = (x[:, None, :] == x[None, :, :]).all(-1)
    g_ref, g_mag = [P.sum() / 2, vt * M[same].sum() / 2], [aP.sum() / 2, vt * np.abs(M[same]).sum() / 2]
    for k in range(d):
        g_ref.append(-w[k] * (P * Dk[k] ** 2).sum() / 4)
        g_mag.append(w[k] * (aP * Dk[k] ** 2).sum() / 4)
    for k in range(d):
        sc = Dk[k] * Sk[k] * np.cos(pf[k] * Dk[k])
        g_ref.append(pf[k] * w2[k] * (P * sc).sum() / 2)
        g_mag.append(pf[k] * w2[k] * (aP * np.abs(sc)).sum() / 2)
    for k in range(d):
        g_ref.append(-w2[k] * (P * Sk[k] ** 2).sum() / 4)
        g_mag.append(w2[k] * (aP * Sk[k] ** 2).sum() / 4)
    g_ref, g_mag = np.array(g_ref, dtype=LD), np.array(g_mag, dtype=LD)
    r = report("periodic gradient n=%d d=%d: vs longdouble at 1e-12 mag" % (n, d),
               float(np.max(np.abs(g.astype(LD) - g_ref) / (1e-12 * g_mag))))
    assert r <= 1.0
    if d in (8, 16):
        go = O.periodic_d_nll_d_theta(x, tc, theta)
        ro = report("periodic gradient n=%d d=%d: vs oracle at 1e-9" % (n, d),
                    float(np.max(np.abs(g - go)) / np.max(np.abs(go)) / 1e-9))
        assert ro <= 1.0
    eng.close()


# ==== C. Girard exact moments ==========================================================================================
@pytest.mark.parametrize("d", [1, 5, 8, 12, 17, 24, 32],
                         ids=lambda d: "d%d-DP%d" % (d, 4 if d <= 4 else 8 if d <= 8 else 16 if d <= 16 else 32))
def test_exact_moments_vs_oracle(gpk, d):
    """exact_pair_kernel<DP> through UncertaintyPropagationExact against the oracle at 1e-9, diagonal and full Sigma,
    one query on a training point; a batch equals the same queries one by one, bit for bit."""
    n = 300
    x, t, theta, rng = _synthetic(n, d, 3000 + d)
    gp = gpk.GP.GaussianProcess(x, t, gpk.Cov.GaussianCovariance(), theta_min=theta.copy())
    up = gpk.UP.UncertaintyPropagationExact(gp)
    ogp = O.OracleGP(x, t, theta_min=theta)
    v = float(np.exp(theta[0]))
    U = rng.uniform(0.1, 0.9, (6, d))
    U[2] = x[17]                                            # query on a training point: the equality quirk of C
    Sd = rng.uniform(1e-4, 1e-2, (6, d))
    G = rng.standard_normal((6, d, d)) * 0.03
    Sf = G @ G.transpose(0, 2, 1) + np.stack([np.diag(s) for s in Sd])
    for name, S in (("diag", Sd), ("full", Sf)):
        mean, var = up.propagate_GA_many(U, S)
        one = np.array([up.propagate_GA_many(U[q:q + 1], S[q:q + 1]) for q in range(6)])[:, :, 0]
        assert np.array_equal(mean, one[:, 0]) and np.array_equal(var, one[:, 1])
        ref = np.array([O.propagate_exact(ogp, U[q], np.diag(S[q]) if S.ndim == 2 else S[q]) for q in range(6)])
        rm = float(np.max(np.abs(mean - ref[:, 0]) / np.maximum(np.abs(ref[:, 0]), 1.0)))
        rv = float(np.max(np.abs(var - ref[:, 1]) / np.maximum(np.abs(ref[:, 1]), 1e-3 * v)))
        r = report("exact moments d=%d %s Sigma: vs oracle at 1e-9" % (d, name), max(rm, rv) / 1e-9)
        assert r <= 1.0


def test_exact_moments_d33_is_refused(gpk):
    x, t, theta, _ = _synthetic(130, 33, 33)
    gp = gpk.GP.GaussianProcess(x, t, gpk.Cov.GaussianCovariance(), theta_min=theta.copy())
    with pytest.raises(gpk.nat.GpkError, match="d <= 32"):
        gpk.UP.UncertaintyPropagationExact(gp).propagate_GA_many(x[:2], np.full((2, 33), 1e-3))


# ==== D. non-positive-definite K through the product entry point =======================================================
@functools.lru_cache(maxsize=None)
def _npd_base(n):
    """SPD K = B B^T / n + I (cond ~ 5) and its FP64 Cholesky factor: with this conditioning the FP64 pivots are
    accurate to a few ulps, far inside the 0.5 margin of the placed pivot."""
    A = _bbt_matrix(n, 7 * n)
    return A, np.linalg.cholesky(A)


NPD_CASES = [("dmma", 900, k) for k in (5, 257, 900)] + [("int8_256", 900, k) for k in (5, 257, 900)] + \
            [("int8", 4200, k) for k in (5, 2049, 4200)]
ROUTES = {"dmma": {"int8": False}, "int8_256": {"int8": True, "min_dim": 256}, "int8": None}


@pytest.mark.parametrize("route,n,k", NPD_CASES, ids=["%s-n%d-k%d" % c for c in NPD_CASES])
def test_factorize_matrix_not_positive_definite(gpk, route, n, k):
    """The failing minor in the first leaf (NaN / Inf downstream, through the INT8 residue conversion too), at the
    first pivot after an INT8 SYRK (257 at min_dim 256, 2049 at npad 4224 = 2048 + 2176) and at the last row:
    LinAlgError naming exactly k, also through inv_cov_matrix; the same handle then factors an SPD K to the same bits
    as a fresh handle (no stale info, residues or workspace)."""
    torch = gpk.torch
    A, L = _npd_base(n)
    Kbad = A.copy()
    Kbad[k - 1, k - 1] -= L[k - 1, k - 1] ** 2 + 0.5
    rng = np.random.default_rng(n + k)
    t = rng.standard_normal(n)
    eng = gpk.eng.Engine(np.zeros((n, 1)), t, route=ROUTES[route])
    assert eng.route()[0] == (route != "dmma")
    with pytest.raises(np.linalg.LinAlgError, match=r"leading minor %d of K is not" % k):
        eng.factorize_matrix(Kbad, want_inverse=True)
    torch.cuda.synchronize()
    with pytest.raises(np.linalg.LinAlgError, match=r"leading minor %d of K is not" % k):
        gpk.Cov.GaussianCovariance().inv_cov_matrix(None, None, cov_matrix=Kbad)
    eng.factorize_matrix(A, want_inverse=True)
    fresh = gpk.eng.Engine(np.zeros((n, 1)), t, route=ROUTES[route])
    fresh.factorize_matrix(A, want_inverse=True)
    assert eng.logdet() == fresh.logdet()
    assert torch.equal(eng.alpha_device(), fresh.alpha_device())
    assert torch.equal(eng.inverse_device(), fresh.inverse_device())
    print("route %s n=%d: pivot %d reported exactly; handle reusable, logdet %.17g" % (route, n, k, eng.logdet()))
    eng.close()
    fresh.close()
