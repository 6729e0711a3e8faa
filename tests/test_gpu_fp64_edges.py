"""Both GEMM routes at the edges of FP64: extreme exponents, edge rows, non-finite operands and unwritten memory.

On the DMMA route every product is IEEE FP64 arithmetic. The INT8 route (csrc/oz_gemm.cuh) rebuilds FP64 semantics by
hand: a per-row exponent from the row maximum, clamped at -900; a conversion of the scaled operand to int64; a rescale
of the reconstructed integer by scA * p_scaled * scB. These tests check each step where it differs from plain FP64, and
what a user of the engine sees. Every bounded check prints its ratio to the bound (run with -s).

  A  exponent range of the INT8 GEMM: power-of-two equivariance (bitwise), edge rows, the -900 clamp
  B  NaN / +Inf / -Inf operands in valid tiles, masked tiles and outside a tile's k range, every k range
  C  one non-finite query (or input) through predict / cross / propagate / cov / grad, a NaN in a caller matrix, on
     the DMMA route, the INT8 route forced from 256 and the production INT8 route at npad = 4224 = 2048 + 2176
  D  gpk_test_poison: every buffer the library allocates, and the caller's X and W, filled with 0xFF or 0x7F bytes
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K_FULL, K_UPTO_BJ, K_FROM_BJ, K_UPTO_BI, K_FROM_BI = range(5)
BOUND = 2e-14                       # componentwise, relative to |A||B| (tests/test_gpu_oz.py)
DBL_MIN = 2.0 ** -1022


@pytest.fixture(scope="module")
def env():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import skgpuppy.Covariance as Cov
    from skgpuppy import _engine, _native
    Cov.VERBOSE = False
    lib = _native.load()

    class E:
        pass
    e = E()
    e.torch, e.nat, e.lib, e.dev, e.eng, e.Cov = torch, _native, lib, torch.device("cuda:0"), _engine, Cov
    e.P = lambda t: ctypes.c_void_p(t.data_ptr())
    e.stream = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def gemm(A, tA, lA, B, tB, lB, C, M, N, K, alpha, beta, kr, lo, moduli, panel_rows=0):
        ms = (ctypes.c_float * 2)()
        _native.check(lib.gpk_test_oz_gemm(e.P(A), A.stride(0), tA, lA, e.P(B), B.stride(0), tB, lB, e.P(C), C.stride(0),
                                           M, N, K, alpha, beta, kr, lo, moduli, panel_rows, 1, ms, e.stream()),
                      "oz_gemm")
        torch.cuda.synchronize()
    e.gemm = gemm
    return e


def report(what, ratio):
    """Print the observed error over its bound (a check passes at ratio <= 1)."""
    print("%-72s ratio %.3e" % (what, ratio))
    return ratio


def _tile_lower(env, rows, cols):
    t = env.torch
    r = t.arange(rows, device=env.dev)[:, None] // 128
    c = t.arange(cols, device=env.dev)[None, :] // 128
    return c <= r


# ==== helpers: operands as the kernel sees them ========================================================================
def _op_valid(env, rows, K, trans, lower):
    """Validity of operand element (r, k) (oz_valid): with `lower`, source tiles above the diagonal read as zero."""
    t = env.torch
    if not lower:
        return t.ones(rows, K, dtype=t.bool, device=env.dev)
    src = _tile_lower(env, K, rows) if trans else _tile_lower(env, rows, K)
    return src.t() if trans else src


def _krange_mask(env, M, N, K, kr):
    """(M or N, K) mask of the k-blocks each output row (BI) or column (BJ) sums over, and which side it applies to."""
    t = env.torch
    k = t.arange(K, device=env.dev)[None, :]
    if kr in (K_UPTO_BJ, K_FROM_BJ):
        n = t.arange(N, device=env.dev)[:, None] // 128
        return "b", (k < (n + 1) * 128) if kr == K_UPTO_BJ else (k >= n * 128)
    if kr in (K_UPTO_BI, K_FROM_BI):
        m = t.arange(M, device=env.dev)[:, None] // 128
        return "a", (k < (m + 1) * 128) if kr == K_UPTO_BI else (k >= m * 128)
    return None, None


def _operands(env, A, tA, lA, B, tB, lB, M, N, K, kr):
    """Masked operands a (M, K), b (N, K) of the reference, with the k range folded in (torch.where: NaN * 0 is NaN)."""
    t = env.torch
    a = A.t() if tA else A
    b = B.t() if tB else B
    a = t.where(_op_valid(env, M, K, tA, lA), a, t.zeros((), dtype=a.dtype, device=env.dev))
    b = t.where(_op_valid(env, N, K, tB, lB), b, t.zeros((), dtype=b.dtype, device=env.dev))
    side, rm = _krange_mask(env, M, N, K, kr)
    zero = t.zeros((), dtype=a.dtype, device=env.dev)
    if side == "a":
        a = t.where(rm, a, zero)
    elif side == "b":
        b = t.where(rm, b, zero)
    return a, b


def _lower_flags(kr):
    return (1 if kr in (K_UPTO_BI, K_FROM_BI) else 0), (1 if kr in (K_UPTO_BJ, K_FROM_BJ) else 0)


def _randn_wide(env, shape, seed):
    t = env.torch
    g = t.Generator(device=env.dev)
    g.manual_seed(seed)
    A = t.randn(shape, dtype=t.float64, device=env.dev, generator=g)
    return A * t.exp(2 * t.randn(shape, dtype=t.float64, device=env.dev, generator=g))


# ==== A. exponent range =================================================================================================
# -510 with -510: scA p_scaled scB underflows to 0 (eA + eB about -1000) while most results are normal and some subnormal
SHIFTS = [-600, -510, -490, -470, 0, 300, 490, 600]
# (name, M, N, K, tA, tB, krange, lower_only)
EXP_CASES = [("full", 512, 384, 640, 0, 0, K_FULL, 0), ("lower_trans", 640, 640, 640, 1, 1, K_FROM_BI, 1)]
MOD_PANEL = [(16, 0), (17, 0), (16, 256)]


@pytest.mark.parametrize("case", EXP_CASES, ids=[c[0] for c in EXP_CASES])
@pytest.mark.parametrize("moduli,panel", MOD_PANEL, ids=["m16", "m17", "m16_panels"])
def test_power_of_two_equivariance(env, case, moduli, panel):
    """C(A 2^s, B 2^t) = 2^(s+t) C(A, B) bit for bit wherever the result is a normal number: the residues are the same,
    and the reconstruction must not lose bits when scA p_scaled scB is subnormal or 0 (eA + eB below about -940) while the
    product itself is normal. Elements whose scaled value is subnormal are held to the componentwise bound instead."""
    t = env.torch
    name, M, N, K, tA, tB, kr, lo = case
    lA, lB = _lower_flags(kr)
    A = _randn_wide(env, (K, M) if tA else (M, K), 31 * M + K)
    B = _randn_wide(env, (K, N) if tB else (N, K), 37 * N + K + 1)
    a, b = _operands(env, A, tA, lA, B, tB, lB, M, N, K, kr)
    ref = a @ b.t()
    mag = a.abs() @ b.abs().t()
    mask = _tile_lower(env, M, N) if lo else t.ones(M, N, dtype=t.bool, device=env.dev)
    C0 = t.zeros(M, N, dtype=t.float64, device=env.dev)
    env.gemm(A, tA, lA, B, tB, lB, C0, M, N, K, 1.0, 0.0, kr, lo, moduli, panel)
    lg = float(t.log2(C0.abs().max()))
    worst = 0.0
    pairs = subnormal = 0
    for s in SHIFTS:
        for u in SHIFTS:
            if s + u + lg >= 1023 or s + u + lg < -1022:       # keep the pairs with no overflow and normal results
                continue
            As, Bs = A * 2.0 ** s, B * 2.0 ** u
            assert t.equal(As * 2.0 ** -s, A) and t.equal(Bs * 2.0 ** -u, B)   # the operands scale exactly
            C = t.zeros(M, N, dtype=t.float64, device=env.dev)
            env.gemm(As, tA, lA, Bs, tB, lB, C, M, N, K, 1.0, 0.0, kr, lo, moduli, panel)
            assert bool((C[~mask] == 0.0).all())
            Cu = C * 2.0 ** -(s + u)                           # exact: no overflow, subnormals scale up exactly
            normal = (C0.abs() * 2.0 ** (s + u) >= DBL_MIN) & mask
            bad = int(((Cu != C0) & normal).sum())
            assert bad == 0, "s=%d t=%d: %d normal elements are not 2^(s+t) C(A, B)" % (s, u, bad)
            rest = mask & ~normal
            if bool(rest.any()):
                tol = BOUND * mag + 2.0 ** (-1073 - (s + u))   # one subnormal ulp of the final rounding
                worst = max(worst, float(((Cu - ref).abs() / tol)[rest].max()))
                subnormal += int(rest.sum())
            pairs += 1
    assert pairs >= 30 and subnormal > 0
    print("%s m%d panel %d: %d elements with subnormal results checked" % (name, moduli, panel, subnormal))
    assert report("%s m%d panel %d: %d shift pairs bitwise; subnormal elements" % (name, moduli, panel, pairs),
                  worst) <= 1.0


@pytest.mark.parametrize("moduli", [16, 12])
def test_edge_rows(env, moduli):
    """Zero rows and columns, one nonzero per row, -0.0, subnormal entries inside normal rows, a row maximum just below a
    power of two (at 12 moduli, bits < 53, it rounds to -2^bits: the balanced residues of the extreme value), and a
    row whose maximum is far below the clamp at 2^-900: it is quantised on the grid 2^(-900 - bits) and comes out 0."""
    t = env.torch
    M, N, K = 384, 256, 512
    g = t.Generator(device=env.dev)
    g.manual_seed(4242 + moduli)
    A = t.randn(M, K, dtype=t.float64, device=env.dev, generator=g)
    B = t.randint(-100, 101, (N, K), device=env.dev, generator=g).double()
    B[:, 0] = 128.0                                          # row maxima of B are powers of two: B' = B 2^(bits - 8)
    A[0] = 0.0                                               # zero row
    B[3] = 0.0                                               # zero column of C
    A[1] = 0.0
    A[1, 17] = 3.0                                           # one nonzero
    A[2] = 0.0
    A[2, 300] = -0.0
    A[2, 301] = 2.0 ** -3                                    # one nonzero, a power of two, next to -0.0
    A[4] = 0.0
    A[4, 0] = -(2.0 - 2.0 ** -52)                            # rounds to -2^bits when bits < 53
    A[4, 5:9] = 1.0
    A[5, 40] = 8.0                                           # row maximum exactly a power of two
    A[6] = -0.0                                              # negative zero row
    A[7, ::7] = 5e-320                                       # subnormals inside a normal row
    A[8] *= 2.0 ** -1000                                     # whole row far below 2^-900
    B[10, ::5] = -0.0
    sl = t.zeros(moduli, M, K, dtype=t.int8, device=env.dev)
    sc = t.zeros(M, dtype=t.float64, device=env.dev)
    env.nat.check(env.lib.gpk_test_oz_residues(env.P(A), K, M, K, 0, 0, moduli, env.P(sl), env.P(sc), env.stream()),
                  "oz_residues")
    bits = 1 - int(round(float(t.log2(sc[4]))))              # e = 1 for row 4: sc = 2^(1 - bits)
    assert float(sc[8]) == 2.0 ** (-900 - bits)              # the clamp
    C = t.full((M, N), 7.0, dtype=t.float64, device=env.dev)
    env.gemm(A, 0, 0, B, 0, 0, C, M, N, K, 1.0, 0.0, K_FULL, 0, moduli, 0)
    for r in (0, 6, 8):
        assert bool((C[r] == 0.0).all()), "row %d" % r
    assert bool((C[:, 3] == 0.0).all())
    # row 4: exact value of the quantised row (a rounded to -2 when bits < 53), in longdouble
    a0 = -2.0 if bits < 53 else -(2.0 - 2.0 ** -52)
    Bh = B.cpu().numpy().astype(np.longdouble)
    exact4 = np.longdouble(a0) * Bh[:, 0] + Bh[:, 5:9].sum(1)
    err4 = float(np.max(np.abs((C[4].cpu().numpy() - exact4) / np.maximum(np.abs(exact4), 1.0))))
    assert report("m%d (bits %d) row 4, maximum rounding to -2^bits: relative to exact" % (moduli, bits),
                  err4 / 4.5e-16) <= 1.0
    if moduli >= 16:                                         # FP64-level operands: the componentwise bound
        ref = A @ B.t()
        mag = A.abs() @ B.abs().t()
        rows = [r for r in range(M) if r not in (0, 6, 8)]
        worst = float(((C[rows] - ref[rows]).abs() / (BOUND * mag[rows]).clamp_min(1e-300)).max())
        assert report("m%d edge rows: componentwise" % moduli, worst) <= 1.0


# ==== B. non-finite operands ============================================================================================
# (name, tA, tB, krange, lower_only): both orientations, all five k ranges
# (the lower operand's orientation goes with its k range, as in the factorisation: UPTO = non-transposed, FROM = transposed)
NF_CASES = [("full", 0, 0, K_FULL, 0), ("full_tt", 1, 1, K_FULL, 0), ("full_lower_only", 0, 1, K_FULL, 1),
            ("upto_bj", 0, 0, K_UPTO_BJ, 0), ("upto_bj_t", 1, 0, K_UPTO_BJ, 0),
            ("from_bj", 0, 1, K_FROM_BJ, 0), ("from_bj_t", 1, 1, K_FROM_BJ, 0),
            ("upto_bi", 0, 1, K_UPTO_BI, 0), ("upto_bi_n", 0, 0, K_UPTO_BI, 0),
            ("from_bi", 1, 1, K_FROM_BI, 1), ("from_bi_n", 1, 0, K_FROM_BI, 0)]


def _pick(mask, frac):
    idx = mask.nonzero()
    assert idx.shape[0] > 0
    i, k = idx[int(frac * (idx.shape[0] - 1))].tolist()
    return i, k


def _put(src, trans, r, k, v):
    if trans:
        src[k, r] = v
    else:
        src[r, k] = v


@pytest.mark.parametrize("case", NF_CASES, ids=[c[0] for c in NF_CASES])
@pytest.mark.parametrize("moduli,panel", [(16, 0), (16, 256)], ids=["m16", "m16_panels"])
def test_non_finite_operands(env, case, moduli, panel):
    """NaN, +Inf, -Inf in the operands. In masked-out tiles they change nothing (bitwise). Where they enter the sum, an
    element whose FP64 reference is non-finite is non-finite; an element whose reference is finite is within the
    componentwise bound, or NaN if its A row or B row holds a non-finite value in a valid tile (a row's scale covers
    every k range). No element is finite and wrong."""
    t = env.torch
    name, tA, tB, kr, lo = case
    M, N, K = 512, 384, 640
    lA, lB = _lower_flags(kr)
    A0 = _randn_wide(env, (K, M) if tA else (M, K), 1000 + kr * 7 + tA)
    g = t.Generator(device=env.dev)
    g.manual_seed(2000 + kr * 11 + tB)
    B0 = t.randn((K, N) if tB else (N, K), dtype=t.float64, device=env.dev, generator=g)   # wide A only, as test_gpu_oz
    vA, vB = _op_valid(env, M, K, tA, lA), _op_valid(env, N, K, tB, lB)
    omask = _tile_lower(env, M, N) if lo else t.ones(M, N, dtype=t.bool, device=env.dev)

    def run(A, B):
        C = t.zeros(M, N, dtype=t.float64, device=env.dev)
        env.gemm(A, tA, lA, B, tB, lB, C, M, N, K, 1.0, 0.0, kr, lo, moduli, panel)
        return C
    base = run(A0, B0)
    worst = 0.0
    for v in (float("nan"), float("inf"), float("-inf")):
        if lA or lB:                                         # masked tiles: nothing changes
            A, B = A0.clone(), B0.clone()
            for f in (0.1, 0.5, 0.9):
                if lA:
                    _put(A, tA, *_pick(~vA, f), v)
                if lB:
                    _put(B, tB, *_pick(~vB, f), v)
            assert t.equal(run(A, B), base), "%s: a non-finite value in a masked tile changed the product" % v
        A, B = A0.clone(), B0.clone()
        for f in (0.15, 0.6):
            _put(A, tA, *_pick(vA, f), v)
        for f in (0.3, 0.85):
            _put(B, tB, *_pick(vB, f), v)
        C = run(A, B)
        a, b = _operands(env, A, tA, lA, B, tB, lB, M, N, K, kr)
        ref = a @ b.t()
        rowbad = ~t.isfinite(t.where(vA, A.t() if tA else A, 0.0)).all(1)
        colbad = ~t.isfinite(t.where(vB, B.t() if tB else B, 0.0)).all(1)
        a0, b0 = t.nan_to_num(a, 0.0, 0.0, 0.0), t.nan_to_num(b, 0.0, 0.0, 0.0)
        ref0, mag = a0 @ b0.t(), a0.abs() @ b0.abs().t()
        refnf = ~t.isfinite(ref) & omask
        assert int(refnf.sum()) > 0
        assert bool((~t.isfinite(C))[refnf].all()), "%s: a non-finite reference element came out finite" % v
        fin = t.isfinite(ref) & omask
        may_nan = rowbad[:, None] | colbad[None, :]
        nan_ok = t.isnan(C) & may_nan
        assert not bool((fin & ~t.isfinite(C) & ~nan_ok).any()), "%s: a finite reference element came out Inf" % v
        chk = fin & t.isfinite(C)
        if bool(chk.any()):
            worst = max(worst, float(((C - ref0).abs() / (BOUND * mag).clamp_min(1e-300))[chk].max()))
    assert report("%s m%d panel %d: finite elements next to NaN / Inf operands" % (name, moduli, panel), worst) <= 1.0


# ==== C. what users see =================================================================================================
ROUTES = {"dmma": {"int8": False}, "int8_256": {"int8": True, "min_dim": 256}, "int8": None}
ROUTE_N = {"dmma": 900, "int8_256": 900, "int8": 4200}
ROUTE_SPLIT = {"dmma": 512, "int8_256": 512, "int8": 2048}


def _synthetic(n, d, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 1, (n, d))
    t = np.sin(2 * np.pi * x).sum(1) + 0.3 * rng.standard_normal(n)
    theta = np.concatenate([[0.0, np.log(0.09)], np.log((4.0 / d) * np.linspace(0.75, 1.25, d))])
    return x, t - t.mean(), theta, rng


_ENGINES = {}


def _fitted(env, route):
    if route not in _ENGINES:
        x, tt, theta, rng = _synthetic(ROUTE_N[route], 3, 77 + ROUTE_N[route])
        eng = env.eng.Engine(x, tt, route=ROUTES[route])
        assert eng.route()[0] == (route != "dmma")
        eng.factorize(theta)
        _ENGINES[route] = (eng, x, theta, rng)
    return _ENGINES[route]


def _same_elsewhere(what, got, ref, bad):
    """Entries outside `bad` are bitwise those of the finite call."""
    keep = np.ones(got.shape, dtype=bool)
    keep[bad] = False
    assert np.array_equal(got[keep], ref[keep]), "%s: entries of the other queries changed" % what


@pytest.mark.parametrize("route", list(ROUTES))
def test_non_finite_queries(env, route):
    """One non-finite query among m = 300 makes that query's outputs NaN (non-finite for +Inf in a caller row) and
    leaves every other output bitwise that of the same call with the query replaced by a finite one."""
    t = env.torch
    eng, x, theta, rng = _fitted(env, route)
    m, d = 300, 3
    xs = rng.uniform(0, 1, (m, d))
    bad = [5, 290]                                           # 290: in the last, ragged batch of 128 rows
    xs_nan = xs.copy()
    xs_nan[bad, 1] = np.nan
    env.nat.check(env.lib.gpk_set_batch_rows(eng.h, 128), "gpk_set_batch_rows")
    try:
        dv = lambda a: eng.to_device(a)
        mean, var = [u.cpu().numpy() for u in eng.predict_device(dv(xs_nan), 0.25)]
        mref, vref = [u.cpu().numpy() for u in eng.predict_device(dv(xs), 0.25)]
        assert np.isnan(mean[bad]).all() and np.isnan(var[bad]).all()
        _same_elsewhere("predict mean", mean, mref, bad)
        _same_elsewhere("predict var", var, vref, bad)

        Ks = env.eng.kernel_matrix(xs, x, theta)
        prior = t.full((m,), float(np.exp(theta[0]) + np.exp(theta[1])), dtype=t.float64, device=env.dev)
        Ksb = Ks.clone()
        Ksb[bad[0], 17] = float("inf")
        Ksb[bad[1], ROUTE_N[route] - 1] = float("inf")
        mean, var = [u.cpu().numpy() for u in eng.predict_cross_device(Ksb, prior, 0.0)]
        mref, vref = [u.cpu().numpy() for u in eng.predict_cross_device(Ks, prior, 0.0)]
        assert not np.isfinite(mean[bad]).any() and not np.isfinite(var[bad]).any()
        _same_elsewhere("cross mean", mean, mref, bad)
        _same_elsewhere("cross var", var, vref, bad)

        S = rng.uniform(1e-3, 1e-2, (m, d))
        U_nan = xs.copy()
        U_nan[bad[0], 0] = np.nan
        S_inf = S.copy()
        S_inf[bad[1], 2] = np.inf
        mean, var = [u.cpu().numpy() for u in eng.propagate_device(dv(U_nan), dv(S_inf), False, 0.0)]
        mref, vref = [u.cpu().numpy() for u in eng.propagate_device(dv(xs), dv(S), False, 0.0)]
        assert np.isnan(mean[bad[0]]) and np.isnan(var[bad[0]])
        assert not np.isfinite(mean[bad[1]]) and not np.isfinite(var[bad[1]])
        _same_elsewhere("propagate mean", mean, mref, bad)
        _same_elsewhere("propagate var", var, vref, bad)

        C = eng.predict_cov_device(dv(xs_nan)).cpu().numpy()
        Cref = eng.predict_cov_device(dv(xs)).cpu().numpy()
        assert np.isnan(C[bad, :]).all() and np.isnan(C[:, bad]).all()
        keep = np.ones(m, dtype=bool)
        keep[bad] = False
        assert np.array_equal(C[np.ix_(keep, keep)], Cref[np.ix_(keep, keep)]), "cov: other entries changed"

        got = [u.cpu().numpy() for u in eng.predict_grad_device(dv(xs_nan), 0.25)]
        ref = [u.cpu().numpy() for u in eng.predict_grad_device(dv(xs), 0.25)]
        for key, a, b in zip(("mean", "var", "dmean", "dvar"), got, ref):
            assert np.isnan(a[bad]).all(), "grad %s of the NaN query" % key
            _same_elsewhere("grad " + key, a, b, bad)
    finally:
        env.nat.check(env.lib.gpk_set_batch_rows(eng.h, 0), "gpk_set_batch_rows")
    print("route %s: NaN / Inf queries isolated in predict, cross, propagate, cov, grad" % route)


def _spd(env, n, seed):
    t = env.torch
    g = t.Generator(device=env.dev)
    g.manual_seed(seed)
    Bm = t.randn(n, n, dtype=t.float64, device=env.dev, generator=g)
    A = Bm @ Bm.t() / n
    A.diagonal().add_(1.0)
    return A


@pytest.mark.parametrize("route", list(ROUTES))
def test_factorize_matrix_with_nan(env, monkeypatch, route):
    """A NaN at (i, j) with j before and i after the first split of the recursion (so on the INT8 routes it enters
    through an INT8 product): LinAlgError naming the same pivot as the DMMA route, the 1e20 sentinel of the NLL for a
    host-built covariance class, and the handle then factors an SPD K to the same bits as a fresh handle."""
    t = env.torch
    n = ROUTE_N[route]
    i, j = ROUTE_SPLIT[route] + 37, 100
    A = _spd(env, n, 5 * n)
    Kbad = A.clone()
    Kbad[i, j] = Kbad[j, i] = float("nan")
    tt = np.random.default_rng(n).standard_normal(n)
    minor = r"leading minor %d of K is not" % (i + 1)
    ref = env.eng.Engine(np.zeros((n, 1)), tt, route=ROUTES["dmma"])
    with pytest.raises(np.linalg.LinAlgError, match=minor):
        ref.factorize_matrix(Kbad)
    ref.close()
    eng = env.eng.Engine(np.zeros((n, 1)), tt, route=ROUTES[route])
    assert eng.route()[0] == (route != "dmma")
    with pytest.raises(np.linalg.LinAlgError, match=minor):
        eng.factorize_matrix(Kbad, want_inverse=True)
    t.cuda.synchronize()

    Kbad_host = Kbad.cpu().numpy()

    class FixedMatrix(env.Cov.Covariance):
        def cov_matrix(self, x, theta):
            return Kbad_host

    monkeypatch.setattr(env.eng, "ROUTE", dict(env.eng.ROUTE, **(ROUTES[route] or {})))
    cov = FixedMatrix()
    assert cov._KIND is None
    assert cov._negativeloglikelihood(np.zeros((n, 1)), tt, np.zeros(2)) == 1.0e20
    assert cov._engine_for(np.zeros((n, 1)), tt).route()[0] == (route != "dmma")
    cov._session.engine.close()

    eng.factorize_matrix(A, want_inverse=True)
    fresh = env.eng.Engine(np.zeros((n, 1)), tt, route=ROUTES[route])
    fresh.factorize_matrix(A, want_inverse=True)
    assert eng.logdet() == fresh.logdet()
    assert t.equal(eng.alpha_device(), fresh.alpha_device())
    assert t.equal(eng.inverse_device(), fresh.inverse_device())
    print("route %s n=%d: NaN at (%d, %d) -> pivot %d on DMMA and here; NLL 1e20; handle reusable" % (route, n, i, j, i + 1))
    eng.close()
    fresh.close()


# ==== D. unwritten memory ===============================================================================================
def _exact_constants(theta, d, S):
    """Per-query Lambda, diag(Delta^-1), normalisers of UncertaintyPropagationExact for diagonal S (Q, d)."""
    w = np.exp(np.asarray(theta)[2:2 + d])
    dinv = w[None, :] - w[None, :] / (1.0 + w[None, :] * S)
    n1 = 1.0 / np.sqrt(np.prod(1.0 + w[None, :] * S, axis=1))
    n2 = 1.0 / np.sqrt(np.prod(1.0 + 2.0 * w[None, :] * S, axis=1))
    Sfull = np.zeros((S.shape[0], d, d))
    Sfull[:, np.arange(d), np.arange(d)] = S
    lam = 2.0 * np.diag(w)[None, :, :] - np.linalg.inv(0.5 * np.diag(1.0 / w)[None, :, :] + Sfull)
    return np.ascontiguousarray(lam), np.ascontiguousarray(dinv), np.ascontiguousarray(np.stack([n1, n2], axis=1))


def _poison_run(env, route, byte):
    """Every output of the engine's entry points on one route, with the library's allocations and X, W filled with
    `byte` (0: poisoning off and zero-filled X, W)."""
    t = env.torch
    n, d = ROUTE_N[route], 3
    x, tt, theta, rng = _synthetic(n, d, 4321)
    assert env.lib.gpk_test_poison(byte) >= 0
    out = {}
    try:
        eng = env.eng.Engine(x, tt, route=ROUTES[route])
        eng.X.view(t.uint8).fill_(byte)
        eng.W.view(t.uint8).fill_(byte)
        out["nll"], out["grad"] = eng.nll_grad(theta)
        th2 = theta + 0.01
        out["nll_pf"], _ = eng.nll_grad(th2, want_grad=False, prefetch_grad=True)
        out["nll_pf2"], out["grad_pf"] = eng.nll_grad(th2)
        out["inv"] = eng.inverse_device()
        out["res"] = np.array(eng.solve_residual())
        env.nat.check(env.lib.gpk_set_batch_rows(eng.h, 128), "gpk_set_batch_rows")
        xs = eng.to_device(rng.uniform(0, 1, (300, d)))
        out["pred"] = eng.predict_device(xs, 0.5)
        out["cov"] = eng.predict_cov_device(xs[:200])
        out["pgrad"] = eng.predict_grad_device(xs, 0.5)
        S = rng.uniform(1e-3, 1e-2, (300, d))
        out["ga"] = eng.propagate_device(xs, eng.to_device(S), False, 0.5)
        lam, dinv, norms = _exact_constants(th2, d, S[:40])
        out["exact"] = eng.propagate_exact_device(xs[:40], eng.to_device(lam), eng.to_device(dinv),
                                                  eng.to_device(norms), 0.5)
        t.cuda.synchronize()
        eng.close()
    finally:
        kib = env.lib.gpk_test_poison(0)
    npad = (n + 127) // 128 * 128
    if byte:   # the fill took place: at least one 128-row query batch of the scratch (and, on DMMA, little else)
        assert kib >= 128 * npad * 8 // 1024, "only %d KiB were filled" % kib
    flat = {}
    for k, v in out.items():
        for idx, a in enumerate(v if isinstance(v, tuple) else (v,)):
            flat["%s.%d" % (k, idx)] = a.cpu().numpy() if isinstance(a, t.Tensor) else np.asarray(a)
    return flat


@pytest.mark.parametrize("route", list(ROUTES))
def test_unwritten_memory_is_never_read(env, route):
    """0xFF makes every double a NaN and every residue -1, 0x7F every double 1.4e306 and every residue 127 (a read
    multiplied by zero or entering a row maximum shows). Every output is bitwise that of the clean run."""
    clean = _poison_run(env, route, 0)
    for byte in (0xFF, 0x7F):
        got = _poison_run(env, route, byte)
        diff = [k for k in clean if not np.array_equal(clean[k], got[k], equal_nan=True)]
        assert not diff, "route %s, byte 0x%02X: outputs %s differ from the clean run" % (route, byte, diff)
        assert all(np.isfinite(clean[k]).all() for k in clean)
    print("route %s: %d outputs bitwise equal under 0xFF and 0x7F poisoning" % (route, len(clean)))
