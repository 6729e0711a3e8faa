"""Device-side state of one Gaussian process: a gpk handle plus the torch tensors it works on.

torch is plumbing here (device memory, pinned staging buffers, streams, torch.distributed);
every number is produced by libgpk.so. No CPU fallback: construction fails without CUDA.
"""
import ctypes

import numpy as np

from . import _native as nat


# Default tensor-pipe route of new engines (include/gpk.h, gpk_set_route): "int8" None keeps the library default (exact
# INT8 CRT products on tcgen05 for blocks of order >= 2048, FP64 DMMA below), False selects FP64 DMMA everywhere, True
# forces the INT8 route from `min_dim` upwards. The tests set min_dim = 256 to push the small reference fixtures through
# the INT8 kernels. There is no silent fallback: if the INT8 workspace does not fit, the first factorisation raises
# GpkError and the caller may rebuild the engine with route={"int8": False}.
ROUTE = {"int8": None, "min_dim": 0, "moduli": 0, "plane_cap_bytes": 0}


def _as_f64(a, ndim=None):
    arr = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if ndim is not None and arr.ndim != ndim:
        raise ValueError("expected a %d-d array, got shape %s" % (ndim, arr.shape))
    return arr


class Engine(object):
    """Owns the padded n x n factor buffers (X = L^-1, W = K / K^-1) and the gpk handle."""

    def __init__(self, x, t, device=None, kind=0, route=None):
        torch = nat.require_cuda()
        if kind not in (0, 1):
            raise NotImplementedError("no device kernels for covariance kind %r" % (kind,))
        self.torch = torch
        self.lib = nat.load()
        x = _as_f64(x, 2)
        t = _as_f64(t, 1)
        if x.shape[0] != t.shape[0]:
            raise ValueError("x has %d rows but t has %d entries" % (x.shape[0], t.shape[0]))
        self.n, self.d = x.shape
        self.kind = int(kind)                      # 0 = GaussianCovariance, 1 = PeriodicCovariance
        self.ntheta = 2 + 3 * x.shape[1] if self.kind == 1 else 2 + x.shape[1]
        if self.d > 64:
            raise ValueError("this build supports d <= 64 (GPK_MAX_D)")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.npad = int(self.lib.gpk_npad(self.n))
        with torch.cuda.device(self.device):
            self.X = torch.empty((self.npad, self.npad), dtype=torch.float64, device=self.device)
            self.W = torch.empty((self.npad, self.npad), dtype=torch.float64, device=self.device)
            self.x_dev = self.to_device(x)
            self.t_dev = self.to_device(t)
            self.h = ctypes.c_void_p()
            nat.check(self.lib.gpk_create(self.n, self.d, nat.ptr(self.X), nat.ptr(self.W), ctypes.byref(self.h)),
                      "gpk_create")
            self._bind_stream()
            if self.kind:
                nat.check(self.lib.gpk_set_kernel(self.h, self.kind), "gpk_set_kernel")
            r = dict(ROUTE)
            r.update(route or {})
            if r["int8"] is not None or r["min_dim"] or r["moduli"] or r["plane_cap_bytes"]:
                want = (self.npad >= 2048) if r["int8"] is None else bool(r["int8"])
                nat.check(self.lib.gpk_set_route(self.h, int(want), int(r["min_dim"]), int(r["moduli"]),
                                                 int(r["plane_cap_bytes"])), "gpk_set_route")
            nat.check(self.lib.gpk_set_data(self.h, nat.ptr(self.x_dev), nat.ptr(self.t_dev)), "gpk_set_data")
        self.theta = None
        self.launches = 0

    # -- plumbing ---------------------------------------------------------------------------
    def to_device(self, a):
        """Pinned host staging + async copy on the current stream."""
        torch = self.torch
        src = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
        if src.numel() == 0:
            return torch.empty(src.shape, dtype=torch.float64, device=self.device)
        return src.pin_memory().to(self.device, non_blocking=True)

    def _bind_stream(self):
        nat.check(self.lib.gpk_set_stream(self.h, nat.current_stream_ptr()), "gpk_set_stream")

    def route(self):
        """(int8 route requested, moduli, smallest block order on it, operand bits at K = npad) of this handle."""
        out = (ctypes.c_int * 4)()
        nat.check(self.lib.gpk_get_route(self.h, out), "gpk_get_route")
        return bool(out[0]), int(out[1]), int(out[2]), int(out[3])

    def _dev_arg(self, t, shape, what):
        """Validate a caller-supplied device tensor before its raw pointer goes to libgpk: a wrong shape, dtype or
        device would make a kernel read past the buffer."""
        torch = self.torch
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != torch.float64:
            raise TypeError("%s must be a CUDA float64 tensor" % what)
        if t.device != self.device:
            raise ValueError("%s lives on %s but the engine on %s" % (what, t.device, self.device))
        if tuple(t.shape) != tuple(shape):
            raise ValueError("%s must have shape %s, got %s" % (what, tuple(shape), tuple(t.shape)))
        return t if t.is_contiguous() else t.contiguous()

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            self.lib.gpk_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def update_data(self, x, t):
        """Upload new training data of the same shape (host -> pinned -> device) into this handle."""
        x = _as_f64(x, 2)
        t = _as_f64(t, 1)
        if x.shape != (self.n, self.d) or t.shape != (self.n,):
            raise ValueError("update_data needs the shapes the engine was created with")
        with self.torch.cuda.device(self.device):
            self._bind_stream()
            self.x_dev = self.to_device(x)
            self.t_dev = self.to_device(t)
            nat.check(self.lib.gpk_set_data(self.h, nat.ptr(self.x_dev), nat.ptr(self.t_dev)), "gpk_set_data")
        self.theta = None

    # -- fit --------------------------------------------------------------------------------
    def factorize(self, theta, want_inverse=False):
        th, thp = nat.theta_ptr(theta)
        if th.shape[0] != self.ntheta:
            raise ValueError("theta must have %d entries" % self.ntheta)
        with self.torch.cuda.device(self.device):
            self._bind_stream()
            nat.check(self.lib.gpk_factorize(self.h, thp, int(want_inverse)), "gpk_factorize")
        self.theta = th.copy()

    def factorize_matrix(self, K, want_inverse=False):
        """Factor a caller-supplied SPD matrix (host array or CUDA tensor, n x n) with the same device stack
        (gpk_factorize_matrix): afterwards logdet / nll_matrix / alpha_device / inverse_device / solve_device apply."""
        torch = self.torch
        if not isinstance(K, torch.Tensor):
            K = self.to_device(_as_f64(K, 2))
        K = self._dev_arg(K, (self.n, self.n), "K")
        with torch.cuda.device(self.device):
            self._bind_stream()
            nat.check(self.lib.gpk_factorize_matrix(self.h, nat.ptr(K), self.n, int(want_inverse)),
                      "gpk_factorize_matrix")
        self.theta = None

    def nll_matrix(self):
        out = ctypes.c_double()
        nat.check(self.lib.gpk_nll_matrix(self.h, ctypes.byref(out)), "gpk_nll_matrix")
        return out.value

    def nll_grad(self, theta, want_grad=True, prefetch_grad=False):
        """(nll, grad). prefetch_grad (with want_grad False): the device goes on with K^-1 and the gradient sums while
        the host returns nll; the gradient call at the same theta collects them."""
        th, thp = nat.theta_ptr(theta)
        if th.shape[0] != self.ntheta:
            raise ValueError("theta must have %d entries" % self.ntheta)
        nll = ctypes.c_double()
        grad = np.zeros(self.ntheta)
        with self.torch.cuda.device(self.device):
            self._bind_stream()
            rc = self.lib.gpk_nll_grad(self.h, thp, ctypes.byref(nll), grad.ctypes.data_as(nat.c_double_p),
                                       1 if want_grad else (2 if prefetch_grad else 0))
        nat.check(rc, "gpk_nll_grad")
        self.theta = th.copy()
        return nll.value, (grad if want_grad else None)

    def logdet(self):
        out = ctypes.c_double()
        nat.check(self.lib.gpk_logdet(self.h, ctypes.byref(out)), "gpk_logdet")
        return out.value

    def grad_trace_partial(self, tile_row_begin, tile_row_end):
        out = np.zeros(self.d + 3)
        with self.torch.cuda.device(self.device):
            self._bind_stream()
            nat.check(self.lib.gpk_grad_trace_partial(self.h, int(tile_row_begin), int(tile_row_end),
                                                      out.ctypes.data_as(nat.c_double_p)), "gpk_grad_trace_partial")
        return out

    def inverse_device(self):
        """Dense symmetric n x n K^-1 as a CUDA tensor."""
        torch = self.torch
        with torch.cuda.device(self.device):
            self._bind_stream()
            out = torch.empty((self.n, self.n), dtype=torch.float64, device=self.device)
            nat.check(self.lib.gpk_inverse(self.h, nat.ptr(out), self.n), "gpk_inverse")
        return out

    def solve_residual(self):
        """(max |K alpha - t|, max |alpha|, max |t|) of the cached factorisation (gpk_solve_residual)."""
        out = (ctypes.c_double * 3)()
        with self.torch.cuda.device(self.device):
            self._bind_stream()
            nat.check(self.lib.gpk_solve_residual(self.h, out), "gpk_solve_residual")
        return float(out[0]), float(out[1]), float(out[2])

    def alpha_device(self):
        torch = self.torch
        with torch.cuda.device(self.device):
            self._bind_stream()
            out = torch.empty((self.n,), dtype=torch.float64, device=self.device)
            nat.check(self.lib.gpk_get_alpha(self.h, nat.ptr(out)), "gpk_get_alpha")
        return out

    def solve_device(self, b_dev):
        """K^-1 b for b of shape (n,) or (nrhs, n) (rows are right-hand sides)."""
        torch = self.torch
        if b_dev.shape[-1] != self.n:
            raise ValueError("right-hand sides must have %d entries" % self.n)
        b2 = self._dev_arg(b_dev.reshape(-1, self.n), (b_dev.numel() // self.n, self.n), "b")
        out = torch.empty_like(b2)
        with torch.cuda.device(self.device):
            self._bind_stream()
            nat.check(self.lib.gpk_solve(self.h, nat.ptr(b2), b2.shape[0], nat.ptr(out)), "gpk_solve")
        return out.reshape(b_dev.shape)

    def import_state(self, theta, alpha_dev, have_inverse):
        th, thp = nat.theta_ptr(theta)
        if th.shape[0] != self.ntheta:
            raise ValueError("theta must have %d entries" % self.ntheta)
        alpha_dev = self._dev_arg(alpha_dev, (self.n,), "alpha")
        with self.torch.cuda.device(self.device):
            self._bind_stream()
            nat.check(self.lib.gpk_import_state(self.h, thp, nat.ptr(alpha_dev), int(have_inverse)),
                      "gpk_import_state")
        self.theta = th.copy()

    # -- queries ----------------------------------------------------------------------------
    def predict_device(self, xs_dev, meant, want_var=True):
        torch = self.torch
        if xs_dev.dim() != 2:
            raise ValueError("queries must be a (m, %d) tensor" % self.d)
        m = int(xs_dev.shape[0])
        xs_dev = self._dev_arg(xs_dev, (m, self.d), "queries")
        mean = torch.empty((m,), dtype=torch.float64, device=self.device)
        var = torch.empty((m,), dtype=torch.float64, device=self.device)
        if m:
            with torch.cuda.device(self.device):
                self._bind_stream()
                nat.check(self.lib.gpk_predict(self.h, nat.ptr(xs_dev), m, float(meant), nat.ptr(mean), nat.ptr(var),
                                               int(want_var)), "gpk_predict")
        return mean, var

    def predict_cross_device(self, Ks_dev, prior_dev, meant, want_var=True):
        """Prediction from a caller-built m x n cross covariance and the m prior variances (gpk_predict_cross).
        want_var False: means only (prior_dev may be None, the variance GEMM is skipped) and None for the variances."""
        torch = self.torch
        if Ks_dev.dim() != 2:
            raise ValueError("the cross covariance must be a (m, %d) tensor" % self.n)
        m = int(Ks_dev.shape[0])
        Ks_dev = self._dev_arg(Ks_dev, (m, self.n), "cross covariance")
        mean = torch.empty((m,), dtype=torch.float64, device=self.device)
        var = None
        if want_var:
            prior_dev = self._dev_arg(prior_dev, (m,), "prior variances")
            var = torch.empty((m,), dtype=torch.float64, device=self.device)
        if m:
            with torch.cuda.device(self.device):
                self._bind_stream()
                nat.check(self.lib.gpk_predict_cross(self.h, nat.ptr(Ks_dev), self.n, m,
                                                     nat.ptr(prior_dev) if want_var else None, float(meant),
                                                     nat.ptr(mean), nat.ptr(var)), "gpk_predict_cross")
        return mean, var

    def _rows_arg(self, t, ncols, what):
        """A caller-supplied (m, ncols) device tensor and its m."""
        if not isinstance(t, self.torch.Tensor) or t.dim() != 2:
            raise ValueError("%s must be a 2-d (m, %d) tensor" % (what, ncols))
        m = int(t.shape[0])
        return self._dev_arg(t, (m, ncols), what), m

    def predict_cov_device(self, xa_dev, xb_dev=None):
        """Joint predictive covariance k(A, B) + noise - k(A, x) K^-1 k(x, B) as an (ma, mb) CUDA tensor
        (gpk_predict_cov). xb_dev None: B = A, exactly symmetric, with the noise of cov_matrix(A)."""
        torch = self.torch
        xa_dev, ma = self._rows_arg(xa_dev, self.d, "queries A")
        mb = ma
        if xb_dev is not None:
            xb_dev, mb = self._rows_arg(xb_dev, self.d, "queries B")
        out = torch.empty((ma, mb), dtype=torch.float64, device=self.device)
        if ma and mb:
            with torch.cuda.device(self.device):
                self._bind_stream()
                nat.check(self.lib.gpk_predict_cov(self.h, nat.ptr(xa_dev), ma, nat.ptr(xb_dev), mb, nat.ptr(out), mb),
                          "gpk_predict_cov")
        return out

    def predict_cov_cross_device(self, Ka_dev, Kb_dev, prior_dev):
        """Joint predictive covariance from caller-built cross covariances Ka (ma, n), Kb (mb, n) or None for B = A,
        and the prior block k(A, B) with its noise (ma, mb) (gpk_predict_cov_cross); an (ma, mb) CUDA tensor."""
        torch = self.torch
        Ka_dev, ma = self._rows_arg(Ka_dev, self.n, "cross covariance A")
        mb = ma
        if Kb_dev is not None:
            Kb_dev, mb = self._rows_arg(Kb_dev, self.n, "cross covariance B")
        prior_dev = self._dev_arg(prior_dev, (ma, mb), "prior covariance")
        out = torch.empty((ma, mb), dtype=torch.float64, device=self.device)
        if ma and mb:
            with torch.cuda.device(self.device):
                self._bind_stream()
                nat.check(self.lib.gpk_predict_cov_cross(self.h, nat.ptr(Ka_dev), self.n, ma, nat.ptr(Kb_dev), self.n, mb,
                                                         nat.ptr(prior_dev), mb, nat.ptr(out), mb),
                          "gpk_predict_cov_cross")
        return out

    def predict_grad_device(self, xs_dev, meant, want_var=True):
        """(mean (m,), var (m,), dmean (m, d), dvar (m, d)) as CUDA tensors (gpk_predict_grad): the predictive moments
        and their derivatives with respect to the query points. want_var False: var and dvar are None and the variance
        product is skipped."""
        torch = self.torch
        xs_dev, m = self._rows_arg(xs_dev, self.d, "queries")
        mean = torch.empty((m,), dtype=torch.float64, device=self.device)
        dmean = torch.empty((m, self.d), dtype=torch.float64, device=self.device)
        var = dvar = None
        if want_var:
            var = torch.empty((m,), dtype=torch.float64, device=self.device)
            dvar = torch.empty((m, self.d), dtype=torch.float64, device=self.device)
        if m:
            with torch.cuda.device(self.device):
                self._bind_stream()
                nat.check(self.lib.gpk_predict_grad(self.h, nat.ptr(xs_dev), m, float(meant), nat.ptr(mean), nat.ptr(var),
                                                    nat.ptr(dmean), nat.ptr(dvar)), "gpk_predict_grad")
        return mean, var, dmean, dvar

    def _ga_args(self, U_dev, S_dev, sigma_full):
        if U_dev.dim() != 2:
            raise ValueError("U must be a (Q, %d) tensor" % self.d)
        Q = int(U_dev.shape[0])
        U_dev = self._dev_arg(U_dev, (Q, self.d), "U")
        S_dev = self._dev_arg(S_dev, (Q, self.d, self.d) if sigma_full else (Q, self.d), "Sigma")
        return Q, U_dev, S_dev

    def propagate_device(self, U_dev, S_dev, sigma_full, meant):
        torch = self.torch
        Q, U_dev, S_dev = self._ga_args(U_dev, S_dev, sigma_full)
        mean = torch.empty((Q,), dtype=torch.float64, device=self.device)
        var = torch.empty((Q,), dtype=torch.float64, device=self.device)
        if Q:
            with torch.cuda.device(self.device):
                self._bind_stream()
                nat.check(self.lib.gpk_propagate_ga(self.h, nat.ptr(U_dev), nat.ptr(S_dev), Q, int(sigma_full),
                                                    float(meant), nat.ptr(mean), nat.ptr(var)), "gpk_propagate_ga")
        return mean, var


def _propagate_parts_device(self, U_dev, S_dev, sigma_full):
    """(sigma2, variance_rest) per query as CUDA tensors (gpk_propagate_ga_parts)."""
    torch = self.torch
    Q, U_dev, S_dev = self._ga_args(U_dev, S_dev, sigma_full)
    s2 = torch.empty((Q,), dtype=torch.float64, device=self.device)
    rest = torch.empty((Q,), dtype=torch.float64, device=self.device)
    if Q:
        with torch.cuda.device(self.device):
            self._bind_stream()
            nat.check(self.lib.gpk_propagate_ga_parts(self.h, nat.ptr(U_dev), nat.ptr(S_dev), Q, int(sigma_full),
                                                      nat.ptr(s2), nat.ptr(rest)), "gpk_propagate_ga_parts")
    return s2, rest


Engine.propagate_parts_device = _propagate_parts_device


def _propagate_exact_device(self, U_dev, Lam_dev, Dinv_dev, norms_dev, meant):
    """Exact SE-kernel moments per query as CUDA tensors (gpk_propagate_exact)."""
    torch = self.torch
    if U_dev.dim() != 2:
        raise ValueError("U must be a (Q, %d) tensor" % self.d)
    Q = int(U_dev.shape[0])
    U_dev = self._dev_arg(U_dev, (Q, self.d), "U")
    Lam_dev = self._dev_arg(Lam_dev, (Q, self.d, self.d), "Lam")
    Dinv_dev = self._dev_arg(Dinv_dev, (Q, self.d), "Dinv")
    norms_dev = self._dev_arg(norms_dev, (Q, 2), "norms")
    mean = torch.empty((Q,), dtype=torch.float64, device=self.device)
    var = torch.empty((Q,), dtype=torch.float64, device=self.device)
    if Q:
        with torch.cuda.device(self.device):
            self._bind_stream()
            nat.check(self.lib.gpk_propagate_exact(self.h, nat.ptr(U_dev), nat.ptr(Lam_dev), nat.ptr(Dinv_dev),
                                                   nat.ptr(norms_dev), Q, float(meant), nat.ptr(mean), nat.ptr(var)),
                      "gpk_propagate_exact")
    return mean, var


Engine.propagate_exact_device = _propagate_exact_device


def kernel_matrix(x1, x2, theta, add_noise=False, kind=0):
    """cov_matrix_ij on the device (n1 x n2 CUDA tensor). kind 0 = Gaussian (add_noise: + vt on the diagonal),
    kind 1 = periodic (add_noise: 0 none, 1 diagonal, 2 wherever the two points are equal element-wise)."""
    torch = nat.require_cuda()
    lib = nat.load()
    a = _as_f64(x1, 2)
    b = _as_f64(x2, 2)
    if a.shape[1] != b.shape[1]:
        raise ValueError("dimension mismatch: %s vs %s" % (a.shape, b.shape))
    th, thp = nat.theta_ptr(theta)
    need = 2 + 3 * a.shape[1] if kind == 1 else a.shape[1] + 2
    if th.shape[0] != need:
        raise ValueError("theta must have %d entries" % need)
    n1, n2, d = a.shape[0], b.shape[0], a.shape[1]
    out = torch.empty((n1, n2), dtype=torch.float64, device="cuda")
    if n1 and n2:
        a_dev = torch.from_numpy(a).pin_memory().to("cuda", non_blocking=True)
        b_dev = a_dev if x2 is x1 else torch.from_numpy(b).pin_memory().to("cuda", non_blocking=True)
        if kind == 1:
            nat.check(lib.gpk_kernel_matrix_periodic(nat.ptr(a_dev), n1, nat.ptr(b_dev), n2, d, thp, int(add_noise),
                                                     nat.ptr(out), n2, nat.current_stream_ptr()),
                      "gpk_kernel_matrix_periodic")
        else:
            nat.check(lib.gpk_kernel_matrix(nat.ptr(a_dev), n1, nat.ptr(b_dev), n2, d, thp, int(add_noise),
                                            nat.ptr(out), n2, nat.current_stream_ptr()), "gpk_kernel_matrix")
    return out
