"""Joint predictive covariance on the B200: gpk_predict_cov / gpk_predict_cov_cross through GaussianProcess.estimate_many_cov,
estimate_cross_cov and the Engine.

  1  against the matrix the reference forms inside estimate_many (kss - kv Kinv kv^T, oracle/gp_oracle.py), golden fixtures
  2  against the same operands in numpy longdouble: X read back from the handle, prior - (G X^T)(G X^T)^T
  3  structure: exact symmetry, positive semi-definiteness, cross blocks == blocks of the joint matrix
  4  batch panels (gpk_set_batch_rows) against the unsplit call
  5  periodic family and a host-built user covariance (gpk_predict_cov_cross, in place)
  6  production route: n = 4224 at the default INT8 threshold, ragged m = 2500
  7  refusals

Every check prints its error and its ratio to the bound (run with -s).
"""
import numpy as np
import pytest

from arbiter import LD, kernel_ld
from oracle import gp_oracle as O

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
SYN = ["syn_n200_d3", "syn_n512_d8", "syn_n384_d16", "syn_n130_d33"]


@pytest.fixture(autouse=True, params=["dmma", "int8_crt"])
def gemm_path(request, monkeypatch):
    """Every test runs twice: with the O(n^3) contractions on the FP64 DMMA kernel only, and with the INT8
    tcgen05 CRT route (oz_gemm.cuh) forced on from 256-blocks upwards (production threshold 2048), so that the small
    reference fixtures exercise the kernels the large shapes run on. The route is per handle (gpk_set_route); the
    tests set the default of new engines."""
    from skgpuppy import _engine
    if request.param == "dmma":
        monkeypatch.setitem(_engine.ROUTE, "int8", False)
    else:
        monkeypatch.setitem(_engine.ROUTE, "int8", True)
        monkeypatch.setitem(_engine.ROUTE, "min_dim", 256)
    return request.param


@pytest.fixture(scope="module")
def sk():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import skgpuppy.Covariance as C
    import skgpuppy.GaussianProcess as G
    from skgpuppy import _engine, _native
    C.VERBOSE = False

    class NS:
        Cov = C
        GP = G
        eng = _engine
        nat = _native
        lib = _native.load()
    NS.torch = torch
    return NS


def report(what, err, bound):
    """Print the observed error and its ratio to the bound; a check passes at ratio <= 1."""
    ratio = float(err) / float(bound)
    print("%-66s err %.3e ratio %.3e" % (what, float(err), ratio))
    return ratio


def _synthetic(n, d, seed):
    """Inputs of the end-to-end parity tests: vt = 0.09, length scales ~ sqrt(d / 4)."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 1, (n, d))
    a = rng.uniform(0.5, 1.5, d)
    t = np.sin(2 * np.pi * a * x).sum(1) + 0.5 * np.prod(np.cos(np.pi * x[:, :2]), 1) + 0.3 * rng.standard_normal(n)
    theta = np.concatenate([[0.0, np.log(0.09)], np.log((4.0 / d) * np.linspace(0.75, 1.25, d))])
    return x, t, theta, rng


def _vpvt(theta):
    return float(np.exp(theta[0]) + np.exp(theta[1]))


# ==== 1. against the reference's own matrix ============================================================================
@pytest.mark.parametrize("name", SYN + ["c1_readme"])
def test_cov_vs_reference_matrix(sk, golden, gemm_path, name):
    g = golden(name)
    if name == "c1_readme":
        x, t, theta = g["x"], g["t"], g["theta_min"]
        xs = np.vstack([g["x_new"][::5], g["x"][5:6]])          # 80 grid points and one training point
    else:
        x, t, theta, xs = g["x"], g["t"], g["theta"], g["xs"]    # xs[5] sits on a training point
    vt = float(np.exp(theta[1]))
    gp = sk.GP.GaussianProcess(x, t, sk.Cov.GaussianCovariance(), theta_min=theta.copy())
    m, C = gp.estimate_many_cov(xs)
    me, ve = gp.estimate_many(xs)
    assert m.shape == (len(xs),) and C.shape == (len(xs), len(xs))
    assert np.array_equal(m, me)
    ogp = O.OracleGP(x, t, theta_min=theta)
    kv = O.cov_matrix_ij(xs, x, theta)
    ref = O.cov_matrix(xs, theta) - kv @ ogp.Kinv @ kv.T
    err = float(np.max(np.abs(C - ref) / np.maximum(np.abs(ref), vt)))
    assert report("%s %s: cov vs reference, rel to max(|ref|, vt)" % (gemm_path, name), err, 1e-9) <= 1.0
    derr = float(np.max(np.abs(np.diag(C) - ve))) / _vpvt(theta)
    assert report("%s %s: diag vs estimate_many, rel to v + vt" % (gemm_path, name), derr, 1e-13) <= 1.0


# ==== 2. same operands in extended precision ===========================================================================
def _kernel_err(K, theta, d):
    """Rounding of a covariance element built in FP64 by the tile kernel (or read back from longdouble): the exponent
    acc = sum_k w_k diff_k^2 carries (d + 3) eps relative error, exp(-acc / 2) turns it into 0.5 (d + 3) eps acc, and exp
    and the factor v add a few ulps."""
    K = np.abs(np.asarray(K, dtype=np.float64))
    v = float(np.exp(theta[0]))
    acc = -2.0 * np.log(np.clip(K / v, 1e-300, 1.0))
    return EPS * (4.0 + 0.5 * (d + 3) * acc) * K


def _cov_bound(X, Ga, Gb, Va, Vb, prior, theta, d, gemm_path, host_fp64=False):
    """Element-wise rounding bound of prior - Va^T Vb with V = X G^T, from the actual magnitudes of the operands.

    First product (n terms), error E of V:
      DMMA  n eps |X||G|^T                       (FP64 dot products)
      INT8  eps/4 (max_k|G_q| |X_j|_1 + max_k|X_j| |G_q|_1) + 3 eps |X||G|^T   (54-bit operands relative to their row
            maxima, exact integer sums, three roundings in the reconstruction)
      both  |X| dG^T for the rounding dG of G itself (_kernel_err)
    Second product (npad terms), with E carried through as E_a^T |V_b| + |V_a|^T E_b:
      DMMA  npad eps |V_a|^T |V_b|
      INT8  eps/4 (max_j|V_a| |V_b|_1 + |V_a|_1 max_j|V_b|) + 3 eps |V_a|^T |V_b|
      both  eps (|prior| + |V_a|^T |V_b|) for the final subtraction, and the rounding of the prior
    host_fp64: the reference V and product are themselves FP64 (DMMA-like terms added). The sum is doubled."""
    n, npad = X.shape[1], X.shape[0]
    aX = np.abs(X)
    aVa, aVb = np.abs(np.asarray(Va, dtype=np.float64)), np.abs(np.asarray(Vb, dtype=np.float64))

    def first(G):
        aG = np.abs(G)
        A = aX @ aG.T
        if gemm_path == "dmma":
            E = n * EPS * A
        else:
            E = EPS / 4 * (np.outer(aX.sum(1), aG.max(1)) + np.outer(aX.max(1), aG.sum(1))) + 3 * EPS * A
        if host_fp64:
            E = E + n * EPS * A
        return E + aX @ _kernel_err(G, theta, d).T

    VV = aVa.T @ aVb
    if gemm_path == "dmma":
        P = npad * EPS * VV
    else:
        P = EPS / 4 * (np.outer(aVa.max(0), aVb.sum(0)) + np.outer(aVa.sum(0), aVb.max(0))) + 3 * EPS * VV
    if host_fp64:
        P = P + npad * EPS * VV
    Ea, Eb = first(Ga), first(Gb)
    tail = EPS * (np.abs(prior) + VV) + _kernel_err(prior, theta, d)
    return 2 * (Ea.T @ aVb + aVa.T @ Eb + P + tail)


def _check_same_operand(what, out, X, Ga, Gb, prior, theta, d, gemm_path):
    Xl = X.astype(LD)
    Va, Vb = Xl @ Ga.astype(LD).T, Xl @ Gb.astype(LD).T
    ref = np.asarray(prior, dtype=LD) - Va.T @ Vb
    bound = _cov_bound(X, Ga, Gb, Va, Vb, prior, theta, d, gemm_path)
    err = np.abs(out.astype(LD) - ref).astype(np.float64)
    r = float(np.max(err / bound))
    print("%-66s err %.3e ratio %.3e (largest bound %.2e, largest |entry| %.2e)"
          % (what, float(err.max()), r, float(bound.max()), float(np.abs(out).max())))
    assert r <= 1.0


@pytest.mark.parametrize("n", [129, 300])
@pytest.mark.parametrize("d", [1, 8, 33, 64])
def test_cov_vs_longdouble_same_operands(sk, gemm_path, n, d):
    x, t, theta, rng = _synthetic(n, d, 7000 + 13 * n + d)
    eng = sk.eng.Engine(x, t - t.mean())
    eng.factorize(theta)
    X = np.tril(eng.X.cpu().numpy())[:, :n]                       # lower tiles; padding columns meet zero G columns
    for ma in (1, 127, 129):
        xa = rng.uniform(0, 1, (ma, d))
        xa[0] = x[min(3, n - 1)]
        C = eng.predict_cov_device(eng.to_device(xa)).cpu().numpy()
        assert np.array_equal(C, C.T)
        Ga = np.asarray(kernel_ld(xa, x, theta), dtype=np.float64)
        prior = np.asarray(kernel_ld(xa, xa, theta, noise_diag=True), dtype=np.float64)
        _check_same_operand("%s n=%d d=%d sym %d" % (gemm_path, n, d, ma), C, X, Ga, Ga, prior, theta, d, gemm_path)
    xa, xb = rng.uniform(0, 1, (77, d)), rng.uniform(0, 1, (300, d))
    xb[10] = xa[3]                                                # equal points: the Gaussian cross block adds no noise
    C = eng.predict_cov_device(eng.to_device(xa), eng.to_device(xb)).cpu().numpy()
    assert C.shape == (77, 300)
    Ga = np.asarray(kernel_ld(xa, x, theta), dtype=np.float64)
    Gb = np.asarray(kernel_ld(xb, x, theta), dtype=np.float64)
    prior = np.asarray(kernel_ld(xa, xb, theta), dtype=np.float64)
    _check_same_operand("%s n=%d d=%d cross 77x300" % (gemm_path, n, d), C, X, Ga, Gb, prior, theta, d, gemm_path)


# ==== 3. structure ===================================================================================================
def test_symmetry_psd_and_cross_blocks(sk, gemm_path):
    x, t, theta, rng = _synthetic(300, 2, 4242)
    vpvt = _vpvt(theta)
    gp = sk.GP.GaussianProcess(x, t, sk.Cov.GaussianCovariance(), theta_min=theta.copy())
    g1 = np.linspace(0.05, 0.95, 10)
    grid = np.array([[a, b] for a in g1 for b in g1])             # 100 well-separated queries
    _, C = gp.estimate_many_cov(grid)
    assert np.array_equal(C, C.T)
    lmin = float(np.linalg.eigvalsh(C)[0])
    print("%s smallest eigenvalue %.3e (v + vt = %.3f)" % (gemm_path, lmin, vpvt))
    assert lmin >= -1e-10 * vpvt
    A, B = rng.uniform(0, 1, (40, 2)), rng.uniform(0, 1, (50, 2))
    B[7] = A[2]
    _, U = gp.estimate_many_cov(np.vstack([A, B]))
    CAB = gp.estimate_cross_cov(A, B)
    CBA = gp.estimate_cross_cov(B, A)
    assert CAB.shape == (40, 50) and CBA.shape == (50, 40)
    e1 = float(np.max(np.abs(CAB - U[:40, 40:]))) / vpvt
    e2 = float(np.max(np.abs(CBA - U[:40, 40:].T))) / vpvt
    print("%s cross blocks: bitwise-equal entries %d / %d and %d / %d" % (
        gemm_path, int((CAB == U[:40, 40:]).sum()), CAB.size, int((CBA == U[40:, :40]).sum()), CBA.size))
    assert report("%s cross(A,B) vs block of joint(A u B)" % gemm_path, e1, 1e-13) <= 1.0
    assert report("%s cross(B,A) vs its transpose" % gemm_path, e2, 1e-13) <= 1.0
    if gemm_path != "dmma":          # exact integer products, per-row scales: the entries do not depend on the call
        assert np.array_equal(CAB, U[:40, 40:]) and np.array_equal(CBA, U[:40, 40:].T)


# ==== 4. batch panels ==================================================================================================
def test_batch_panels_match_unsplit_call(sk, gemm_path):
    x, t, theta, rng = _synthetic(400, 5, 515)
    eng = sk.eng.Engine(x, t - t.mean())
    eng.factorize(theta)
    xs = eng.to_device(rng.uniform(0, 1, (300, 5)))
    xb = eng.to_device(rng.uniform(0, 1, (200, 5)))
    full = eng.predict_cov_device(xs).cpu().numpy()
    full_x = eng.predict_cov_device(xs, xb).cpu().numpy()
    sk.nat.check(eng.lib.gpk_set_batch_rows(eng.h, 128), "gpk_set_batch_rows")
    split = eng.predict_cov_device(xs).cpu().numpy()
    split_x = eng.predict_cov_device(xs, xb).cpu().numpy()
    sk.nat.check(eng.lib.gpk_set_batch_rows(eng.h, 0), "gpk_set_batch_rows")
    vpvt = _vpvt(theta)
    for what, a, b in (("sym 300", split, full), ("cross 300x200", split_x, full_x)):
        print("%s batch rows 128, %s: bitwise-equal entries %d / %d" % (gemm_path, what, int((a == b).sum()), a.size))
        if gemm_path != "dmma":
            assert np.array_equal(a, b)
        else:
            assert report("%s batch rows 128, %s" % (gemm_path, what), np.max(np.abs(a - b)) / vpvt, 1e-14) <= 1.0


# ==== 5. periodic family and host-built covariances ====================================================================
@pytest.mark.parametrize("name", ["periodic_n48", "periodic_n90"])
def test_periodic_vs_class_formula(sk, golden, gemm_path, name):
    g = golden(name)
    x, t, theta = g["x"], g["t"], g["theta"]
    vt = float(np.exp(theta[1]))
    cov = sk.Cov.PeriodicCovariance()
    gp = sk.GP.GaussianProcess(x, t, cov, theta_min=theta.copy())
    xs = np.vstack([g["xs"], x[3:4]])                             # the last query equals a training point
    m, C = gp.estimate_many_cov(xs)
    me, ve = gp.estimate_many(xs)
    assert np.array_equal(m, me) and np.array_equal(C, C.T)
    Kinv = gp.Kinv
    kv = np.asarray(cov.cov_matrix_ij(xs, x, theta))
    ref = np.asarray(cov.cov_matrix_ij(xs, xs, theta)) - kv @ Kinv @ kv.T
    err = float(np.max(np.abs(C - ref) / np.maximum(np.abs(ref), vt)))
    assert report("%s %s: cov vs class formula" % (gemm_path, name), err, 1e-9) <= 1.0
    derr = float(np.max(np.abs(np.diag(C) - ve))) / _vpvt(theta)
    assert report("%s %s: diag vs estimate_many" % (gemm_path, name), derr, 1e-13) <= 1.0
    A, B = xs[:12], xs[6:]                                         # overlapping rows: the equality noise applies
    CAB = gp.estimate_cross_cov(A, B)
    kb = np.asarray(cov.cov_matrix_ij(B, x, theta))
    ref = np.asarray(cov.cov_matrix_ij(A, B, theta)) - kv[:12] @ Kinv @ kb.T
    err = float(np.max(np.abs(CAB - ref) / np.maximum(np.abs(ref), vt)))
    assert report("%s %s: cross cov vs class formula" % (gemm_path, name), err, 1e-9) <= 1.0


def test_host_built_covariance_and_in_place(sk, gemm_path):
    class RationalQuadratic(sk.Cov.Covariance):
        def __call__(self, xi, xj, theta):
            v, vt, a, ell = np.exp(theta)
            r2 = float(np.sum((np.asarray(xi) - np.asarray(xj)) ** 2))
            return v * (1.0 + r2 / (2 * a * ell ** 2)) ** (-a) + (vt if (np.asarray(xi) == np.asarray(xj)).all() else 0)

        def get_theta(self, x, t):
            return np.log([np.var(t), np.var(t) / 10, 1.0, 0.5])

    rng = np.random.default_rng(31)
    n, d = 48, 2
    x = rng.uniform(0, 2, (n, d))
    t = np.sin(2 * x).sum(1) + 0.1 * rng.standard_normal(n)
    theta = np.log([1.3, 0.02, 1.5, 0.6])
    cov = RationalQuadratic()
    assert cov._KIND is None
    gp = sk.GP.GaussianProcess(x, t, cov, theta_min=theta.copy())
    xs = rng.uniform(0, 2, (9, d))
    xs[4] = x[7]
    m, C = gp.estimate_many_cov(xs)
    me, ve = gp.estimate_many(xs)
    assert np.array_equal(m, me) and np.array_equal(C, C.T)
    K = np.array([[cov(a, b, theta) for b in x] for a in x])
    kv = np.array([[cov(a, b, theta) for b in x] for a in xs])
    ref = np.array([[cov(a, b, theta) for b in xs] for a in xs]) - kv @ np.linalg.inv(K) @ kv.T
    err = float(np.max(np.abs(C - ref) / np.maximum(np.abs(ref), 0.02)))
    assert report("%s rational quadratic: cov vs numpy" % gemm_path, err, 1e-9) <= 1.0
    assert report("%s rational quadratic: diag vs estimate_many" % gemm_path,
                  np.max(np.abs(np.diag(C) - ve)) / _vpvt(theta), 1e-13) <= 1.0
    xb = rng.uniform(0, 2, (5, d))
    xb[1] = xs[2]
    CAB = gp.estimate_cross_cov(xs, xb)
    kb = np.array([[cov(a, b, theta) for b in x] for a in xb])
    ref = np.array([[cov(a, b, theta) for b in xb] for a in xs]) - kv @ np.linalg.inv(K) @ kb.T
    err = float(np.max(np.abs(CAB - ref) / np.maximum(np.abs(ref), 0.02)))
    assert report("%s rational quadratic: cross cov vs numpy" % gemm_path, err, 1e-9) <= 1.0
    # cov_dev == prior_dev: the same bits as a separate output
    eng = gp._engine()
    Ka, Kb = eng.to_device(kv), eng.to_device(kb)
    for Kb_dev, xcols in ((None, xs), (Kb, xb)):
        mb = len(xcols)
        P = eng.to_device(np.array([[cov(a, b, theta) for b in xcols] for a in xs]))
        out = eng.predict_cov_cross_device(Ka, Kb_dev, P).cpu().numpy()
        rc = eng.lib.gpk_predict_cov_cross(eng.h, sk.nat.ptr(Ka), n, 9, sk.nat.ptr(Kb_dev), n, mb, sk.nat.ptr(P), mb,
                                           sk.nat.ptr(P), mb)
        sk.nat.check(rc, "gpk_predict_cov_cross in place")
        assert np.array_equal(P.cpu().numpy(), out)


# ==== 6. production route ==============================================================================================
def test_production_route_n4224_ragged_m(sk, gemm_path):
    from skgpuppy import _engine
    if gemm_path != "dmma":
        _engine.ROUTE["min_dim"] = 0                   # production threshold instead of the forced 256 (monkeypatch restores)
    n, d, m = 4224, 4, 2500
    x, t, theta, rng = _synthetic(n, d, 4224)
    gp = sk.GP.GaussianProcess(x, t, sk.Cov.GaussianCovariance(), theta_min=theta.copy())
    eng = gp._engine()
    on, moduli, min_dim, _ = eng.route()
    assert on == (gemm_path != "dmma") and min_dim == 2048 and (not on or moduli == 16)
    xs = rng.uniform(0, 1, (m, d))
    xs[100] = x[5]
    mean, C = gp.estimate_many_cov(xs)
    me, ve = gp.estimate_many(xs)
    assert np.array_equal(mean, me) and np.array_equal(C, C.T)
    vpvt = _vpvt(theta)
    assert report("%s n=4224 m=2500: diag vs estimate_many" % gemm_path, np.max(np.abs(np.diag(C) - ve)) / vpvt,
                  1e-13) <= 1.0
    X = np.tril(eng.X.cpu().numpy())[:, :n]
    worst, widest = 0.0, 0.0
    for _ in range(10):
        a0, b0 = int(rng.integers(0, m - 64)), int(rng.integers(0, m - 64))
        ia, ib = np.arange(a0, a0 + 64), np.arange(b0, b0 + 64)
        Ga = np.asarray(kernel_ld(xs[ia], x, theta), dtype=np.float64)      # direct differences, like the tile kernel
        Gb = np.asarray(kernel_ld(xs[ib], x, theta), dtype=np.float64)
        Va, Vb = X @ Ga.T, X @ Gb.T
        prior = np.asarray(kernel_ld(xs[ia], xs[ib], theta), dtype=np.float64) + \
            np.exp(theta[1]) * (ia[:, None] == ib[None, :])
        ref = prior - Va.T @ Vb
        bound = _cov_bound(X, Ga, Gb, Va, Vb, prior, theta, d, gemm_path, host_fp64=True)
        worst = max(worst, float(np.max(np.abs(C[np.ix_(ia, ib)] - ref) / bound)))
        widest = max(widest, float(bound.max()))
    print("%-66s ratio %.3e (largest bound %.2e of v + vt)"
          % ("%s n=4224 m=2500: 10 blocks 64x64 vs host FP64 V" % gemm_path, worst, widest / vpvt))
    assert worst <= 1.0
    assert widest <= 1e-8 * vpvt           # the check resolves errors far below the entries (|Sigma_ab| ~ 1e-3 off the diagonal)


# ==== 7. refusals ======================================================================================================
def test_refusals(sk, golden, gemm_path):
    x, t, theta, rng = _synthetic(200, 3, 77)
    eng = sk.eng.Engine(x, t - t.mean())
    xs = eng.to_device(rng.uniform(0, 1, (5, 3)))
    with pytest.raises(sk.nat.GpkError):
        eng.predict_cov_device(xs)                                # not factored
    K = O.cov_matrix(x, theta)
    eng.factorize_matrix(K)
    out = sk.torch.empty((5, 5), dtype=sk.torch.float64, device=eng.device)
    rc = eng.lib.gpk_predict_cov(eng.h, sk.nat.ptr(xs), 5, None, 5, sk.nat.ptr(out), 5)
    assert rc == -2                                               # a matrix state has no theta to build k(A, x) from
    eng.factorize(theta)
    rc = eng.lib.gpk_predict_cov(eng.h, sk.nat.ptr(xs), 5, None, 5, sk.nat.ptr(out), 4)
    assert rc == -2                                               # ldc < mb
    gp = sk.GP.GaussianProcess(x, t, sk.Cov.GaussianCovariance(), theta_min=theta.copy())
    with pytest.raises(ValueError):
        gp.estimate_many_cov(np.zeros((3, 4)))
    with pytest.raises(ValueError):
        gp.estimate_cross_cov(np.zeros((3, 3)), np.zeros((2, 2)))
    e = gp._engine()
    with pytest.raises(TypeError):
        e.predict_cov_device(sk.torch.zeros((3, 3), dtype=sk.torch.float32, device=e.device))
    with pytest.raises(TypeError):
        e.predict_cov_device(sk.torch.zeros((3, 3), dtype=sk.torch.float64))            # host tensor
    with pytest.raises(ValueError):
        e.predict_cov_device(sk.torch.zeros((3, 4), dtype=sk.torch.float64, device=e.device))
    m, C = gp.estimate_many_cov(np.zeros((0, 3)))
    assert m.shape == (0,) and C.shape == (0, 0)
    assert gp.estimate_cross_cov(np.zeros((0, 3)), np.zeros((4, 3))).shape == (0, 4)
    g = golden("spgp_n120")
    sp = sk.GP.GaussianProcess(g["x"], g["t"], sk.Cov.SPGPCovariance(int(g["m"])), theta_min=g["theta"].copy())
    with pytest.raises(NotImplementedError):
        sp.estimate_many_cov(g["xs"])
    with pytest.raises(NotImplementedError):
        sp.estimate_cross_cov(g["xs"], g["xs"])
