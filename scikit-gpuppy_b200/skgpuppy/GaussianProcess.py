"""Drop-in `skgpuppy.GaussianProcess` (reference skgpuppy/GaussianProcess.py:11-191), B200 back end.

Same constructor, methods, attributes (x, n, d, t, meant, theta_min, Kinv, cov) and return types.
Device state lives in an `_engine.Engine`; `Kinv` is materialised on the host only when it is read.
"""
import numpy as np

from . import _engine
from . import _native as nat


# Backward-error guard of GaussianProcess._engine (see _check_residual): relative tolerance on max |K alpha - t|.
RESIDUAL_CHECK = True
RESIDUAL_RTOL = 1e-8


class GaussianProcess(object):
    """GP regression after Girard (2004); the heavy lifting is in the covariance / libgpk.so."""

    def __init__(self, x, t, cov, theta_min=None, _factorize=True):
        """x: (n,d) inputs; t: (n,) noisy responses; cov: covariance object; theta_min: skip the ML-II fit
        (reference GaussianProcess.py:19-41). `_factorize=False` (an addition) defers the factorisation,
        for ranks that receive the factor through broadcast_state()."""
        self.x = x
        self.n, self.d = np.shape(x)
        self.meant = np.mean(t)
        self.t = t - self.meant
        self.cov = cov
        self._eng = None
        self._Kinv_host = None
        self._beta_host = None
        self._state_theta = None
        if theta_min is not None:
            self.theta_min = theta_min
        else:
            self.theta_min = self.cov.ml_estimate(self.x, self.t)
        if _factorize and not hasattr(self.cov, "_sparse_predict"):
            self._engine()  # factorise at theta_min now, like the reference computes Kinv in the constructor

    # -- device state -------------------------------------------------------------------------
    def _engine(self):
        """Engine factorised at the current theta_min (re-factorises if theta_min was mutated). Covariance classes with
        device kernels (`cov._KIND` 0 / 1) build K on the GPU; any other `Covariance` subclass (the reference's extension
        point) builds K on the host through its own cov_matrix and only the factorisation runs on the device."""
        theta = np.array(self.theta_min, dtype=np.float64)
        kind = getattr(self.cov, "_KIND", None)
        if self._eng is None:
            sess = getattr(self.cov, "_session", None)
            if sess is not None and sess.matches(self.x, self.t):
                self._eng = sess.engine      # reuse the fit's device buffers
                self.cov._session = None     # the GP owns them from here on
            else:
                self._eng = _engine.Engine(self.x, self.t, kind=kind if kind is not None else 0)
        if self._state_theta is None or not np.array_equal(self._state_theta, theta):
            if kind is None:
                self._eng.factorize_matrix(np.asarray(self.cov.cov_matrix(self.x, theta), dtype=np.float64))
            else:
                self._eng.factorize(theta, want_inverse=False)
                if RESIDUAL_CHECK:
                    self._check_residual(theta)
            self._state_theta = theta
            self._Kinv_host = None
            self._beta_host = None
        return self._eng

    def _check_residual(self, theta):
        """Backward-error guard of the factorisation the object will answer queries from (gpk_solve_residual, one extra
        K build): max |K alpha - t| must stay within RESIDUAL_RTOL of the scale of the terms it cancels. The exact INT8
        route rounds operands to 54 bits relative to the ROW maximum; if that (or anything else) ever left a residual
        above the bound, the factorisation is redone on the FP64 DMMA kernels -- loudly, with a RuntimeWarning -- and a
        matrix that fails there too is reported as numerically singular."""
        import warnings
        res, amax, tmax = self._eng.solve_residual()
        vpvt = float(np.exp(theta[0]) + np.exp(theta[1]))
        limit = RESIDUAL_RTOL * (tmax + vpvt * amax)
        self.solve_residual = res
        if res <= limit or not np.isfinite(limit):
            return
        if self._eng.route()[0]:
            warnings.warn("factorisation residual %.3e exceeds %.3e on the INT8 route; refactorising on FP64 DMMA"
                          % (res, limit), RuntimeWarning)
            self._eng.close()
            self._eng = _engine.Engine(self.x, self.t, kind=getattr(self.cov, "_KIND", 0), route={"int8": False})
            self._eng.factorize(theta, want_inverse=False)
            res, amax, tmax = self._eng.solve_residual()
            self.solve_residual = res
            if res <= RESIDUAL_RTOL * (tmax + vpvt * amax):
                return
        raise np.linalg.LinAlgError("K is numerically singular at theta_min: max |K alpha - t| = %.3e" % res)

    @property
    def Kinv(self):
        """Dense n x n inverse covariance as a host array (reference attribute, GaussianProcess.py:41)."""
        if self._Kinv_host is None:
            if hasattr(self.cov, "_sparse_predict"):
                self._Kinv_host = self.cov.inv_cov_matrix(self.x, self.theta_min)     # Woodbury form of the class
            else:
                self._Kinv_host = self._engine().inverse_device().cpu().numpy()
        return self._Kinv_host

    @Kinv.setter
    def Kinv(self, value):
        self._Kinv_host = value

    def Kinv_device(self):
        """K^-1 as a CUDA tensor (no host copy)."""
        return self._engine().inverse_device()

    def __getstate__(self):
        return {"x": self.x, "n": self.n, "d": self.d, "meant": self.meant, "t": self.t, "cov": self.cov,
                "theta_min": self.theta_min}

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._eng = None
        self._Kinv_host = None
        self._beta_host = None
        self._state_theta = None

    # -- sampling -----------------------------------------------------------------------------
    @staticmethod
    def get_realisation(x, cov, theta):
        """One draw of the GP at x (reference GaussianProcess.py:44-57). K is built on the GPU; the
        draw itself is numpy's multivariate_normal on the host, consuming the global RandomState
        exactly like the reference (n normals, then the SVD transform)."""
        n, d = np.shape(x)
        K = cov.cov_matrix(x, theta)
        return np.random.multivariate_normal(np.zeros(n), K)

    # -- prediction ---------------------------------------------------------------------------
    def __call__(self, x_star):
        return self.estimate(x_star)

    def _queries(self, x_stars):
        xs = np.asarray(x_stars, dtype=np.float64)
        if xs.ndim == 1 and xs.size == self.d:
            xs = xs.reshape(1, self.d)
        if xs.ndim != 2 or xs.shape[1] != self.d:
            raise ValueError("x_stars must have shape (m, %d), got %s" % (self.d, xs.shape))
        return np.ascontiguousarray(xs)

    def estimate_many(self, x_stars):
        """Means and variances (noise included) at the rows of x_stars (reference GaussianProcess.py:68-80)."""
        if np.size(x_stars) == 0:
            return np.zeros(0), np.zeros(0)
        xs = self._queries(x_stars)
        if hasattr(self.cov, "_sparse_predict"):
            # sparse pseudo-input covariance: low-rank algebra, no n x n factor (SPGPCovariance)
            mean, var = self.cov._sparse_predict(self.x, self.t, self.theta_min, xs)
            return mean + self.meant, var
        eng = self._engine()
        if getattr(self.cov, "_KIND", None) is None:
            # host-built covariance: cross covariance and prior variances from the subclass, the products on the device
            kv = np.asarray(self.cov.cov_matrix_ij(xs, self.x, self.theta_min), dtype=np.float64)
            prior = np.array([np.asarray(self.cov.cov_matrix(xs[i:i + 1], self.theta_min))[0, 0]
                              for i in range(xs.shape[0])], dtype=np.float64)
            mean, var = eng.predict_cross_device(eng.to_device(kv), eng.to_device(prior), self.meant)
        else:
            mean, var = eng.predict_device(eng.to_device(xs), self.meant, want_var=True)
        return mean.cpu().numpy(), var.cpu().numpy()

    def estimate_many_device(self, xs_dev, want_var=True):
        """Same on device-resident queries; returns CUDA tensors."""
        return self._engine().predict_device(xs_dev, self.meant, want_var=want_var)

    # -- joint predictive covariance (an addition: the matrix the reference forms inside estimate_many,
    #    GaussianProcess.py:75-80, of which it returns only the diagonal) ------------------------------------------------
    def _no_sparse(self, what):
        if hasattr(self.cov, "_sparse_predict"):
            raise NotImplementedError("%s: the low-rank predictive covariance of %s is not implemented"
                                      % (what, type(self.cov).__name__))

    def estimate_many_cov(self, x_stars):
        """Means (m,) and the joint predictive covariance (m, m), noise included, at the rows of x_stars. The means are
        those of estimate_many, the diagonal of the covariance its variances; the matrix is exactly symmetric."""
        self._no_sparse("estimate_many_cov")
        if np.size(x_stars) == 0:
            return np.zeros(0), np.zeros((0, 0))
        xs = self._queries(x_stars)
        eng = self._engine()
        if getattr(self.cov, "_KIND", None) is None:
            kv = eng.to_device(np.asarray(self.cov.cov_matrix_ij(xs, self.x, self.theta_min), dtype=np.float64))
            prior = eng.to_device(np.asarray(self.cov.cov_matrix(xs, self.theta_min), dtype=np.float64))
            mean, _ = eng.predict_cross_device(kv, None, self.meant, want_var=False)
            cov = eng.predict_cov_cross_device(kv, None, prior)
        else:
            mean, cov = self.estimate_many_cov_device(eng.to_device(xs))
        return mean.cpu().numpy(), cov.cpu().numpy()

    def estimate_many_cov_device(self, xs_dev):
        """Same on device-resident queries (covariance classes with device kernels); returns CUDA tensors."""
        self._no_sparse("estimate_many_cov_device")
        eng = self._engine()
        mean, _ = eng.predict_device(xs_dev, self.meant, want_var=False)
        return mean, eng.predict_cov_device(xs_dev)

    def estimate_cross_cov(self, x_a, x_b):
        """Predictive covariance (ma, mb) between the rows of x_a and those of x_b, with the noise term of
        cov_matrix_ij(x_a, x_b) of the covariance class."""
        self._no_sparse("estimate_cross_cov")
        xa = self._queries(x_a) if np.size(x_a) else np.zeros((0, self.d))
        xb = self._queries(x_b) if np.size(x_b) else np.zeros((0, self.d))
        if not xa.shape[0] or not xb.shape[0]:
            return np.zeros((xa.shape[0], xb.shape[0]))
        eng = self._engine()
        if getattr(self.cov, "_KIND", None) is None:
            ka = eng.to_device(np.asarray(self.cov.cov_matrix_ij(xa, self.x, self.theta_min), dtype=np.float64))
            kb = eng.to_device(np.asarray(self.cov.cov_matrix_ij(xb, self.x, self.theta_min), dtype=np.float64))
            prior = eng.to_device(np.asarray(self.cov.cov_matrix_ij(xa, xb, self.theta_min), dtype=np.float64))
            cov = eng.predict_cov_cross_device(ka, kb, prior)
        else:
            cov = eng.predict_cov_device(eng.to_device(xa), eng.to_device(xb))
        return cov.cpu().numpy()

    # -- gradients with respect to the query points (an addition: the reference differentiates its mean numerically) ---
    def _grad_kind(self, what):
        self._no_sparse(what)
        if getattr(self.cov, "_KIND", None) is None:
            raise NotImplementedError("%s: %s is built on the host and has no derivative in x on the device"
                                      % (what, type(self.cov).__name__))

    def estimate_many_grad(self, x_stars, want_var=True):
        """Means (m,), variances (m,) and their gradients with respect to the query points, dmean (m, d) and dvar (m, d),
        at the rows of x_stars. Means and variances are those of estimate_many (noise included); the gradients are the
        true derivatives of the smooth part (the noise added where a query equals a training point is a jump). want_var
        False: the variances and their gradients are None and the variance product is skipped."""
        self._grad_kind("estimate_many_grad")
        if np.size(x_stars) == 0:
            dz = np.zeros((0, self.d))
            return np.zeros(0), (np.zeros(0) if want_var else None), dz, (dz.copy() if want_var else None)
        xs = self._queries(x_stars)
        out = self.estimate_many_grad_device(self._engine().to_device(xs), want_var=want_var)
        return tuple(None if o is None else o.cpu().numpy() for o in out)

    def estimate_many_grad_device(self, xs_dev, want_var=True):
        """Same on device-resident queries; returns CUDA tensors (mean, var, dmean, dvar)."""
        self._grad_kind("estimate_many_grad_device")
        return self._engine().predict_grad_device(xs_dev, self.meant, want_var=want_var)

    def estimate(self, x_star):
        """Mean and variance at one point (reference GaussianProcess.py:94-111)."""
        m, v = self.estimate_many(self._queries(np.atleast_2d(np.asarray(x_star, dtype=np.float64))))
        return m[0], v[0]

    # -- accessors used by the propagation classes (reference GaussianProcess.py:114-191) -------
    def _get_beta(self):
        eng = self._engine()
        if self._beta_host is None:
            self._beta_host = eng.alpha_device().cpu().numpy()
        return self._beta_host

    def _get_W_inv(self):
        return np.diag(np.exp(np.asarray(self.theta_min, dtype=np.float64)[2:self.d + 2]))

    def _get_v(self):
        return np.exp(self.theta_min[0])

    def _get_vt(self):
        return np.exp(self.theta_min[1])

    def _covariance(self, xi, xj, v=None, w=None):
        """Scalar covariance; like the reference, v / w overwrite theta_min in place (:133-149)."""
        theta = self.theta_min
        if v is not None:
            theta[0] = np.log(v)
        if w is not None:
            theta[2:] = np.log(w)
        return self.cov(xi, xj, theta)

    def _inv_cov_matrix(self):
        return self.Kinv

    def _get_mean_t(self):
        return self.meant

    def _get_Hessian(self, u, xi):
        return self.cov.get_Hessian(u, xi, self.theta_min)

    def _get_Jacobian(self, u, xi):
        return self.cov.get_Jacobian(u, xi, self.theta_min)

    # -- multi-GPU: query sharding (SURVEY.md 8e) ------------------------------------------------
    def broadcast_state(self, src=0, group=None):
        """Broadcast X = L^-1 and alpha from rank `src` to all ranks (NCCL over NVLink); afterwards every
        rank can run estimate_many / propagate_GA on its own shard of the queries. The factorisation
        itself stays on one GPU."""
        import torch.distributed as dist
        kind = getattr(self.cov, "_KIND", None)
        if kind is None:
            raise NotImplementedError("query sharding needs a covariance class with device kernels")
        eng = self._eng if self._eng is not None else _engine.Engine(self.x, self.t, kind=kind)
        self._eng = eng
        theta = np.array(self.theta_min, dtype=np.float64)
        if dist.get_rank(group) == src:
            self._engine()
            alpha = eng.alpha_device()
        else:
            alpha = eng.torch.empty((self.n,), dtype=eng.torch.float64, device=eng.device)
        dist.broadcast(eng.X, src=src, group=group)
        dist.broadcast(alpha, src=src, group=group)
        if dist.get_rank(group) != src:
            eng.import_state(theta, alpha, have_inverse=False)
            self._state_theta = theta
            self._Kinv_host = None
            self._beta_host = None
        return self
