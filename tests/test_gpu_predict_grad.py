"""Gradients of the predictive mean and variance with respect to the query points on the B200: gpk_predict_grad through
GaussianProcess.estimate_many_grad and the Engine.

  1  against the reference's quantities on the golden fixtures: -sum_i beta_i J_ik with the reference's get_Jacobian
     (opposite sign) and -2 k*^T K^-1 D_k with K^-1 of inv_cov_matrix (oracle/gp_oracle.py)
  2  against the same operands in numpy longdouble: X and alpha read back from the handle, k* and D built in longdouble;
     with it the consistency with estimate_many (bitwise means, variances within the bound) and want_var=False
  3  central finite differences of estimate_many
  4  batch panels (gpk_set_batch_rows) against the unsplit call
  5  periodic family against the class formula, including a query equal to a training point
  6  production route: n = 4224 at the default INT8 threshold, d = 8, ragged m = 1500
  7  imported state (gpk_import_state) gives the same bits
  8  refusals

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
    NS.torch = torch
    return NS


def report(what, err, bound):
    """Print the observed error and its ratio to the bound; a check passes at ratio <= 1."""
    ratio = float(np.max(np.asarray(err, dtype=np.float64) / np.asarray(bound, dtype=np.float64)))
    print("%-70s err %.3e ratio %.3e" % (what, float(np.max(err)), ratio))
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


def _grad(eng, xs, want_var=True):
    out = eng.predict_grad_device(eng.to_device(xs), 0.0, want_var=want_var)
    return tuple(None if o is None else o.cpu().numpy() for o in out)


# ==== rows and bounds ==================================================================================================
def _rows_ld(xs, x, theta):
    """Gaussian k* (m, n) and D (m, d, n), D_k,i = -w_k (x*_k - x_ik) k*_i, in longdouble."""
    w = np.exp(np.asarray(theta[2:], dtype=np.float64).astype(LD))
    K = kernel_ld(xs, x, theta)
    diff = np.asarray(xs, dtype=np.float64).astype(LD)[:, :, None] - np.asarray(x, dtype=np.float64).astype(LD).T[None]
    return K, -w[None, :, None] * diff * K[:, None, :]


def _row_err(K, theta, d):
    """Relative rounding of a covariance element built in FP64 (or read back from longdouble): the exponent
    acc = sum_k w_k diff_k^2 carries (d + 3) eps relative error, exp(-acc / 2) turns it into 0.5 (d + 3) eps acc, and exp
    and the factor v add a few ulps. A derivative row adds three roundings (the difference, w_k times it, times E)."""
    K = np.abs(np.asarray(K, dtype=np.float64))
    v = float(np.exp(theta[0]))
    acc = -2.0 * np.log(np.clip(K / v, 1e-300, 1.0))
    return EPS * (4.0 + 0.5 * (d + 3) * acc)


def _stack(K, D):
    """Rows of G as the device orders them: k*_q, then D_1 .. D_d of each query; (m (d + 1), n)."""
    return np.concatenate([np.asarray(K)[:, None, :], np.asarray(D)], axis=1).reshape(-1, K.shape[1])


def _check_grad(what, out, X, alpha, K, D, theta, gemm_path, host_fp64=False):
    """Compare (mean, var, dmean, dvar) of the device (meant = 0) with the same operands: FP64 rows G = [k*, D] rounded
    from K, D (longdouble), X and alpha read back from the handle; the reference products in longdouble (host_fp64:
    in FP64, with their own rounding added to the bound). Bounds from the actual magnitudes, with separate terms for
      row rounding      |dG| = |G| (_row_err (+ 3 eps on D rows)), carried through |dG| |alpha| and |X| |dG|^T
      the product       V = G X^T: DMMA n eps |G||X|^T; INT8 eps/4 (max_i|G_r| |X_j|_1 + |G_r|_1 max_i|X_j|) + 3 eps
                        |G||X|^T (54-bit operands relative to their row maxima, exact integer sums, three roundings)
      the dots          npad eps |G||alpha| and npad eps |V_0||V_r| (group dot), plus eps of the final operations
    carried through as E_0 |V_r| + |V_0| E_r. The sum is doubled."""
    mean, var, dmean, dvar = out
    m, d, n = D.shape
    P = d + 1
    npad = X.shape[0]
    G = _stack(np.asarray(K, dtype=np.float64), np.asarray(D, dtype=np.float64))
    rel = _row_err(K, theta, d)
    Gerr = np.abs(G) * _stack(rel, np.repeat(rel[:, None, :], d, axis=1) + 3 * EPS)
    aX, aG, aa = np.abs(X), np.abs(G), np.abs(alpha)
    if host_fp64:
        dots, V = G @ alpha, G @ X.T
    else:
        Gl = G.astype(LD)
        dots, V = Gl @ alpha.astype(LD), Gl @ X.astype(LD).T
    A = aG @ aX.T
    if gemm_path == "dmma":
        E = n * EPS * A
    else:
        E = EPS / 4 * (np.outer(aG.max(1), aX.sum(1)) + np.outer(aG.sum(1), aX.max(1))) + 3 * EPS * A
    E = E + Gerr @ aX.T + (n * EPS * A if host_fp64 else 0)
    V3 = V.reshape(m, P, npad)
    aV, E3 = np.abs(np.asarray(V3, dtype=np.float64)), E.reshape(m, P, npad)
    vv = np.einsum("qj,qrj->qr", V3[:, 0], V3)                          # V_0 . V_r
    avv = np.einsum("qj,qrj->qr", aV[:, 0], aV)
    evv = np.einsum("qj,qrj->qr", E3[:, 0], aV) + np.einsum("qj,qrj->qr", aV[:, 0], E3)
    gdot = (npad * EPS * (2 if host_fp64 else 1)) * avv
    dbound = (npad * EPS * (2 if host_fp64 else 1)) * (aG @ aa) + Gerr @ aa
    dbound = 2 * (dbound + EPS * np.abs(np.asarray(dots, dtype=np.float64))).reshape(m, P)
    dots = dots.reshape(m, P)
    vpvt = _vpvt(theta)
    refs = {"mean": dots[:, 0], "dmean": dots[:, 1:], "var": vpvt - vv[:, 0], "dvar": -2 * vv[:, 1:]}
    bounds = {"mean": dbound[:, 0], "dmean": dbound[:, 1:],
              "var": 2 * (evv[:, 0] + gdot[:, 0] + EPS * (vpvt + avv[:, 0])),
              "dvar": 2 * (2 * (evv[:, 1:] + gdot[:, 1:]) + EPS * 2 * avv[:, 1:])}
    got = {"mean": mean, "dmean": dmean, "var": var, "dvar": dvar}
    for key in ("mean", "dmean", "var", "dvar"):
        if got[key] is None:
            continue
        err = np.abs(np.asarray(got[key], dtype=LD) - refs[key]).astype(np.float64)
        b = bounds[key]
        r = float(np.max(err / b))
        scale = float(np.max(np.abs(np.asarray(refs[key], dtype=np.float64))))
        print("%-70s err %.3e ratio %.3e (largest bound %.2e, largest |value| %.2e)"
              % ("%s %s" % (what, key), float(err.max()), r, float(b.max()), scale))
        assert r <= 1.0
        assert float(b.max()) <= 1e-6 * max(scale, 1e-3 * vpvt)         # a wrong tile would show far above the bound
    return bounds


# ==== 1. against the reference's own quantities ========================================================================
@pytest.mark.parametrize("name", SYN + ["c1_readme"])
def test_grad_vs_reference(sk, golden, gemm_path, name):
    g = golden(name)
    if name == "c1_readme":
        x, t, theta = g["x"], g["t"], g["theta_min"]
        xs = np.vstack([g["x_new"][::5], g["x"][5:6]])          # 80 grid points and one training point
    else:
        x, t, theta, xs = g["x"], g["t"], g["theta"], g["xs"]    # xs[5] sits on a training point
    m, d = xs.shape
    gp = sk.GP.GaussianProcess(x, t, sk.Cov.GaussianCovariance(), theta_min=theta.copy())
    mean, var, dmean, dvar = gp.estimate_many_grad(xs)
    assert mean.shape == (m,) and var.shape == (m,) and dmean.shape == (m, d) and dvar.shape == (m, d)
    me, ve = gp.estimate_many(xs)
    assert np.array_equal(mean, me)
    ogp = O.OracleGP(x, t, theta_min=theta)
    beta = ogp.beta()
    Kinv = O.inv_cov_matrix(x, theta)
    J = np.array([[O.get_jacobian(u, xi, theta)[:, 0] for xi in x] for u in xs])   # (m, n, d), reference sign
    ks = O.cov_matrix_ij(xs, x, theta)
    dm_ref = -np.einsum("i,qik->qk", beta, J)
    dv_ref = 2 * np.einsum("qi,ij,qjk->qk", ks, Kinv, J, optimize=True)
    dm_mag = np.einsum("i,qik->qk", np.abs(beta), np.abs(J))
    dv_mag = 2 * np.einsum("qi,ij,qjk->qk", np.abs(ks), np.abs(Kinv), np.abs(J), optimize=True)
    assert report("%s %s: dmean vs -beta.J, rel to sum |beta||J|" % (gemm_path, name),
                  np.abs(dmean - dm_ref) / dm_mag, 1e-9) <= 1.0
    assert report("%s %s: dvar vs -2 k* Kinv D, rel to sum |k*||Kinv||D|" % (gemm_path, name),
                  np.abs(dvar - dv_ref) / dv_mag, 1e-9) <= 1.0
    assert report("%s %s: var vs estimate_many, rel to v + vt" % (gemm_path, name),
                  np.abs(var - ve) / _vpvt(theta), 1e-13) <= 1.0


# ==== 2. same operands in extended precision, consistency with estimate_many ==========================================
@pytest.mark.parametrize("n", [129, 300])
@pytest.mark.parametrize("d", [1, 8, 33, 64])
def test_grad_vs_longdouble_same_operands(sk, gemm_path, n, d):
    x, t, theta, rng = _synthetic(n, d, 9000 + 13 * n + d)
    eng = sk.eng.Engine(x, t - t.mean())
    eng.factorize(theta)
    X = np.tril(eng.X.cpu().numpy())[:, :n]                       # lower tiles; padding columns meet zero G columns
    alpha = eng.alpha_device().cpu().numpy()
    m = 19                                                        # 19 (d + 1) rows: groups straddle the 128-row tiles
    xs = rng.uniform(0, 1, (m, d))
    xs[0] = x[min(3, n - 1)]
    out = _grad(eng, xs)
    K, D = _rows_ld(xs, x, theta)
    bounds = _check_grad("%s n=%d d=%d" % (gemm_path, n, d), out, X, alpha, K, D, theta, gemm_path)
    me, ve = (o.cpu().numpy() for o in eng.predict_device(eng.to_device(xs), 0.0, want_var=True))
    assert np.array_equal(out[0], me)
    assert report("%s n=%d d=%d: var vs estimate_many, rel to twice the bound" % (gemm_path, n, d),
                  np.abs(out[1] - ve), 2 * bounds["var"]) <= 1.0
    mean2, var2, dmean2, dvar2 = _grad(eng, xs, want_var=False)
    assert var2 is None and dvar2 is None
    assert np.array_equal(mean2, out[0]) and np.array_equal(dmean2, out[2])


# ==== 3. finite differences ============================================================================================
def test_grad_vs_finite_differences(sk, gemm_path):
    x, t, theta, rng = _synthetic(300, 4, 1234)
    w = np.exp(theta[2:])
    gp = sk.GP.GaussianProcess(x, t, sk.Cov.GaussianCovariance(), theta_min=theta.copy())
    xs = rng.uniform(0.1, 0.9, (12, 4))
    xs[3] = x[17]                                                  # on a training point: the noise is a jump, not a slope
    mean, var, dmean, dvar = gp.estimate_many_grad(xs)
    m, d = xs.shape
    h = 1e-4 / np.sqrt(w)
    steps = np.concatenate([xs[None] + (s * h[k]) * np.eye(d)[k][None, None] for k in range(d) for s in (1, -1)])
    fm, fv = gp.estimate_many(steps.reshape(-1, d))
    fm, fv = fm.reshape(d, 2, m), fv.reshape(d, 2, m)
    fd_m = ((fm[:, 0] - fm[:, 1]) / (2 * h[:, None])).T
    fd_v = ((fv[:, 0] - fv[:, 1]) / (2 * h[:, None])).T
    assert report("%s central differences vs dmean, rel to max |dmean|" % gemm_path,
                  np.abs(dmean - fd_m) / np.abs(dmean).max(), 1e-5) <= 1.0
    assert report("%s central differences vs dvar, rel to max |dvar|" % gemm_path,
                  np.abs(dvar - fd_v) / np.abs(dvar).max(), 1e-5) <= 1.0


# ==== 4. batch panels ==================================================================================================
def test_batch_panels_match_unsplit_call(sk, gemm_path):
    x, t, theta, rng = _synthetic(400, 5, 515)
    eng = sk.eng.Engine(x, t - t.mean())
    eng.factorize(theta)
    xs = rng.uniform(0, 1, (300, 5))
    full = _grad(eng, xs)
    sk.nat.check(eng.lib.gpk_set_batch_rows(eng.h, 128), "gpk_set_batch_rows")   # 21 queries of 6 rows per batch
    split = _grad(eng, xs)
    sk.nat.check(eng.lib.gpk_set_batch_rows(eng.h, 0), "gpk_set_batch_rows")
    for key, a, b in zip(("mean", "var", "dmean", "dvar"), split, full):
        print("%s batch rows 128, %s: bitwise-equal entries %d / %d" % (gemm_path, key, int((a == b).sum()), a.size))
    assert np.array_equal(split[0], full[0]) and np.array_equal(split[2], full[2])   # rows and dots do not see the batch
    if gemm_path != "dmma":          # exact integer products, per-row scales: the entries do not depend on the call
        assert np.array_equal(split[1], full[1]) and np.array_equal(split[3], full[3])
    else:
        X = np.tril(eng.X.cpu().numpy())[:, :400]
        alpha = eng.alpha_device().cpu().numpy()
        K, D = _rows_ld(xs[:40], x, theta)
        bounds = _check_grad("%s batch rows 128 (first 40 queries)" % gemm_path,
                             tuple(o[:40] for o in split), X, alpha, K, D, theta, gemm_path)
        assert report("%s batch rows 128 vs unsplit: var" % gemm_path,
                      np.abs(split[1][:40] - full[1][:40]), 2 * bounds["var"]) <= 1.0
        assert report("%s batch rows 128 vs unsplit: dvar" % gemm_path,
                      np.abs(split[3][:40] - full[3][:40]), 2 * bounds["dvar"]) <= 1.0


# ==== 5. periodic family ===============================================================================================
@pytest.mark.parametrize("name", ["periodic_n48", "periodic_n90"])
def test_periodic_vs_class_formula(sk, golden, gemm_path, name):
    g = golden(name)
    x, t, theta = g["x"], g["t"], g["theta"]
    d = x.shape[1]
    cov = sk.Cov.PeriodicCovariance()
    gp = sk.GP.GaussianProcess(x, t, cov, theta_min=theta.copy())
    xs = np.vstack([g["xs"], x[3:4]])                             # the last query equals a training point
    mean, var, dmean, dvar = gp.estimate_many_grad(xs)
    me, ve = gp.estimate_many(xs)
    assert np.array_equal(mean, me)
    v, vt, w, p, w2 = O.periodic_split(theta, d)
    ks = O.periodic_cov_matrix_ij(xs, x, theta)                   # vt at the coincident pair, as estimate_many builds it
    E = O.periodic_cov_matrix_ij(xs, x, theta, noise=False)
    diff = xs[:, None, :] - x[None, :, :]                         # (m, n, d)
    a = np.pi / p * diff
    D = -E[:, :, None] * (w * diff + w2 * (np.pi / p) * np.sin(a) * np.cos(a))
    K = O.periodic_cov_matrix_ij(x, x, theta)
    Kinv = np.linalg.inv(K)
    beta = Kinv @ (t - t.mean())
    dm_ref = np.einsum("i,qik->qk", beta, D)
    dv_ref = -2 * np.einsum("qi,ij,qjk->qk", ks, Kinv, D, optimize=True)
    dm_mag = np.einsum("i,qik->qk", np.abs(beta), np.abs(D))
    dv_mag = 2 * np.einsum("qi,ij,qjk->qk", np.abs(ks), np.abs(Kinv), np.abs(D), optimize=True)
    assert report("%s %s: dmean vs class formula, rel to sum |beta||D|" % (gemm_path, name),
                  np.abs(dmean - dm_ref) / dm_mag, 1e-9) <= 1.0
    assert report("%s %s: dvar vs class formula, rel to sum |k*||Kinv||D|" % (gemm_path, name),
                  np.abs(dvar - dv_ref) / dv_mag, 1e-9) <= 1.0
    assert report("%s %s: var vs estimate_many, rel to v + vt" % (gemm_path, name),
                  np.abs(var - ve) / _vpvt(theta), 1e-13) <= 1.0


# ==== 6. production route ==============================================================================================
def test_production_route_n4224_ragged_m(sk, gemm_path):
    from skgpuppy import _engine
    if gemm_path != "dmma":
        _engine.ROUTE["min_dim"] = 0                   # production threshold instead of the forced 256 (monkeypatch restores)
    n, d, m = 4224, 8, 1500
    x, t, theta, rng = _synthetic(n, d, 4224)
    gp = sk.GP.GaussianProcess(x, t, sk.Cov.GaussianCovariance(), theta_min=theta.copy())
    eng = gp._engine()
    on, moduli, min_dim, _ = eng.route()
    assert on == (gemm_path != "dmma") and min_dim == 2048 and (not on or moduli == 16)
    xs = rng.uniform(0, 1, (m, d))
    xs[100] = x[5]
    out = _grad(eng, xs)
    me, _ = eng.predict_device(eng.to_device(xs), 0.0, want_var=False)
    assert np.array_equal(out[0], me.cpu().numpy())
    X = np.tril(eng.X.cpu().numpy())[:, :n]
    alpha = eng.alpha_device().cpu().numpy()
    pick = np.concatenate([[100], rng.choice(m, 47, replace=False)])
    K, D = _rows_ld(xs[pick], x, theta)
    _check_grad("%s n=4224 d=8 m=1500: 48 queries vs host FP64 V" % gemm_path, tuple(o[pick] for o in out), X, alpha,
                K, D, theta, gemm_path, host_fp64=True)


# ==== 7. imported state ================================================================================================
def test_imported_state_same_bits(sk, gemm_path):
    x, t, theta, rng = _synthetic(300, 6, 808)
    src = sk.eng.Engine(x, t - t.mean())
    src.factorize(theta)
    dst = sk.eng.Engine(x, t - t.mean())
    dst.X.copy_(src.X)
    dst.import_state(theta, src.alpha_device(), have_inverse=False)
    xs = rng.uniform(0, 1, (50, 6))
    xs[7] = x[2]
    a, b = _grad(src, xs), _grad(dst, xs)
    for key, u, v in zip(("mean", "var", "dmean", "dvar"), a, b):
        print("%s imported state, %s: bitwise-equal entries %d / %d" % (gemm_path, key, int((u == v).sum()), u.size))
        assert np.array_equal(u, v)


# ==== 8. refusals ======================================================================================================
def test_refusals(sk, golden, gemm_path):
    x, t, theta, rng = _synthetic(200, 3, 77)
    eng = sk.eng.Engine(x, t - t.mean())
    xs = eng.to_device(rng.uniform(0, 1, (5, 3)))
    with pytest.raises(sk.nat.GpkError):
        eng.predict_grad_device(xs, 0.0)                          # not factored
    K = O.cov_matrix(x, theta)
    eng.factorize_matrix(K)
    f64 = dict(dtype=sk.torch.float64, device=eng.device)
    mean, var = sk.torch.empty((5,), **f64), sk.torch.empty((5,), **f64)
    dmean, dvar = sk.torch.empty((5, 3), **f64), sk.torch.empty((5, 3), **f64)
    P = sk.nat.ptr
    rc = eng.lib.gpk_predict_grad(eng.h, P(xs), 5, 0.0, P(mean), P(var), P(dmean), P(dvar))
    assert rc == -2                                               # a matrix state has no theta to build k* and D from
    eng.factorize(theta)
    assert eng.lib.gpk_predict_grad(eng.h, P(xs), 5, 0.0, P(mean), P(var), P(dmean), None) == -2
    assert eng.lib.gpk_predict_grad(eng.h, P(xs), 5, 0.0, P(mean), None, P(dmean), P(dvar)) == -2
    assert eng.lib.gpk_predict_grad(eng.h, P(xs), 5, 0.0, None, P(var), P(dmean), P(dvar)) == -2
    assert eng.lib.gpk_predict_grad(eng.h, P(xs), 5, 0.0, P(mean), P(var), None, P(dvar)) == -2
    assert eng.lib.gpk_predict_grad(eng.h, P(xs), 0, 0.0, None, None, None, None) == 0
    gp = sk.GP.GaussianProcess(x, t, sk.Cov.GaussianCovariance(), theta_min=theta.copy())
    with pytest.raises(ValueError):
        gp.estimate_many_grad(np.zeros((3, 4)))
    e = gp._engine()
    with pytest.raises(TypeError):
        e.predict_grad_device(sk.torch.zeros((3, 3), dtype=sk.torch.float32, device=e.device), 0.0)
    with pytest.raises(ValueError):
        e.predict_grad_device(sk.torch.zeros((3, 4), dtype=sk.torch.float64, device=e.device), 0.0)
    mean, var, dmean, dvar = gp.estimate_many_grad(np.zeros((0, 3)))
    assert mean.shape == (0,) and var.shape == (0,) and dmean.shape == (0, 3) and dvar.shape == (0, 3)
    mean, var, dmean, dvar = gp.estimate_many_grad(np.zeros((0, 3)), want_var=False)
    assert mean.shape == (0,) and var is None and dmean.shape == (0, 3) and dvar is None

    class RationalQuadratic(sk.Cov.Covariance):
        def __call__(self, xi, xj, theta):
            v, vt, a, ell = np.exp(theta)
            r2 = float(np.sum((np.asarray(xi) - np.asarray(xj)) ** 2))
            return v * (1.0 + r2 / (2 * a * ell ** 2)) ** (-a) + (vt if (np.asarray(xi) == np.asarray(xj)).all() else 0)

        def get_theta(self, x, t):
            return np.log([np.var(t), np.var(t) / 10, 1.0, 0.5])

    hb = sk.GP.GaussianProcess(x[:40], t[:40], RationalQuadratic(), theta_min=np.log([1.3, 0.02, 1.5, 0.6]))
    with pytest.raises(NotImplementedError):
        hb.estimate_many_grad(x[:3])
    with pytest.raises(NotImplementedError):
        hb.estimate_many_grad_device(hb._engine().to_device(x[:3]))
    g = golden("spgp_n120")
    sp = sk.GP.GaussianProcess(g["x"], g["t"], sk.Cov.SPGPCovariance(int(g["m"])), theta_min=g["theta"].copy())
    with pytest.raises(NotImplementedError):
        sp.estimate_many_grad(g["xs"])
