"""bench.py -- headline benchmark of the dense-GP hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W                     (our arm, libgpk.so on B200)
    python bench.py --impl reference --gpus N --steps K --warmup W    (the reference's own CPU path on the host cores)

metric  : fit s/iter (K build + Cholesky/inverse + NLL + gradient) at n=32768, d=16, FP64 (BASELINE.json configs[2]);
          estimate_many at 1 M points, propagate_GA at 100 k queries (configs[2], [3]), the n=4096 ML-II fit
          (configs[1]) and the n=65536 d=32 fit iteration (configs[4]) ride along in `extra`.
step    : one fit iteration = one evaluation of NLL and its d+2 gradient at a fresh theta (what SciPy L-BFGS-B asks
          for per iteration), inputs resident in HBM. `e2e` is the same step through the reference-facing API
          (GaussianCovariance._negativeloglikelihood + ._d_nll_d_theta) with HOST arrays: x, t are uploaded and the
          scalars read back inside the timed region, every step.
N > 1   : the factorisation does not shard (SURVEY.md 8e) -> "replicas only": every rank runs its own fit iteration;
          `value` is the max-over-ranks time of ONE replica's iteration (weak scaling: constant = ideal), the replica
          throughput is in `replicas_iters_per_s`. The paths that do shard (estimate_many, propagate_GA by query; the
          gradient trace by tile rows) are measured across the N ranks in `extra.sharded`, weak and strong.
reference arm: the UNMODIFIED reference (baseline/_ref, import shims only) through its own API on the host cores, timed
          at n in {1024, 2048, 4096, 8192}, fitted a n^3 + b n^2 and evaluated at n=32768 -- labelled extrapolated
          (a direct run is ~18 min and ~45 GB per evaluation, SURVEY 6); the oracle port if baseline/_ref is absent.
One JSON line on stdout (rank 0). --dump-outputs DIR: rank 0 also writes the NLL and gradient of its last timed step as
          DIR/nll.npy and DIR/grad.npy (float64); the inputs are seeded, so runs with the same arguments compare directly.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "scikit-gpuppy_b200")
REF_INSTALL = os.path.join(ROOT, "baseline", "_ref")


def synthetic(n, d, seed):
    """SURVEY.md 8d: x ~ U(0,1)^{n x d}, smooth latent + 0.3 N(0,1); theta fixed (v=1, vt=0.09, s=4)."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 1, (n, d))
    a = rng.uniform(0.5, 1.5, d)
    t = np.sin(2 * np.pi * a * x).sum(1) + 0.5 * np.prod(np.cos(np.pi * x[:, :2]), 1) + 0.3 * rng.standard_normal(n)
    theta = np.concatenate([[0.0, np.log(0.09)], np.log((4.0 / d) * np.linspace(0.75, 1.25, d))])
    return x, t - t.mean(), theta


def fit_flops(n, d):
    """Algorithmic work of one fit iteration (SURVEY.md 8d): n^3 (potrf n^3/3 + explicit inverse 2n^3/3)
    + K build n^2(3d+2) + gradient trace n^2(2d+6) + alpha 2n^2."""
    return float(n) ** 3 + float(n) ** 2 * ((3 * d + 2) + (2 * d + 6) + 2)


class ClockSampler(object):
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        for line in self.f.read().splitlines():
            c = [s.strip() for s in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
                pw.append(float(c[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            load = [s for s, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
            out.update(sm_mhz=float(np.median(load)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm), power_w_max=float(max(pw)))
        return out


# ---------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the fit iteration
# ---------------------------------------------------------------------------------------------------------------------
def _reference_callables():
    """(f, g, kind): NLL and gradient of the reference. kind "reference": the unmodified package installed in
    baseline/_ref by `pip install --target` (DESIGN.md 6), imported with the three import shims of SURVEY 8c;
    kind "port": oracle/gp_oracle.py, the function-by-function numpy/scipy restatement, when the install is absent."""
    if os.path.isdir(os.path.join(REF_INSTALL, "skgpuppy")):
        import types
        import scipy.integrate
        import scipy.special
        if not hasattr(np, "Inf"):
            np.Inf = np.inf
        if not hasattr(scipy.integrate, "romberg"):
            scipy.integrate.romberg = lambda *a, **k: (_ for _ in ()).throw(NotImplementedError("romberg"))
        if "scipy.misc" not in sys.modules or not hasattr(sys.modules["scipy.misc"], "derivative"):
            misc = types.ModuleType("scipy.misc")
            misc.derivative = lambda func, x0, dx=1.0, n=1, args=(), order=3: (func(x0 + dx, *args) - func(x0 - dx, *args)) / (2.0 * dx)
            misc.factorial, misc.factorial2, misc.comb = scipy.special.factorial, scipy.special.factorial2, scipy.special.comb
            sys.modules["scipy.misc"] = misc
            import scipy
            scipy.misc = misc
        sys.path.insert(0, REF_INSTALL)
        try:
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                import skgpuppy.Covariance as RC
        finally:
            sys.path.remove(REF_INSTALL)
        assert os.path.realpath(RC.__file__).startswith(os.path.realpath(REF_INSTALL)), RC.__file__
        cov = RC.GaussianCovariance()
        return cov._negativeloglikelihood, cov._d_nll_d_theta, "reference"
    sys.path.insert(0, ROOT)
    from oracle import gp_oracle as O
    return O.negativeloglikelihood, O.d_nll_d_theta, "port"


def reference_query_rates(kind):
    """BASELINE.md 4: the reference's estimate_many (chunks of <= 2048 points: it builds m x m temporaries,
    GaussianProcess.py:75,78) and its Cython propagate_GA, at the largest training sizes that run in seconds on the
    host (the reference stores a dense LU inverse: n = 32768 is out of its reach)."""
    out = {}
    if kind == "reference":
        sys.path.insert(0, REF_INSTALL)
        try:
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                import contextlib
                import io
                import skgpuppy.Covariance as RC
                import skgpuppy.GaussianProcess as RG
                import skgpuppy.UncertaintyPropagation as RU
        finally:
            sys.path.remove(REF_INSTALL)
        make_gp = lambda x, t, th: RG.GaussianProcess(x, t, RC.GaussianCovariance(), theta_min=th.copy())
        make_up = lambda gp: RU.UncertaintyPropagationApprox(gp)
        prop = lambda up, u, S: up.propagate_GA(u, np.diag(S))
        out["propagate_impl"] = "Cython" if getattr(RU, "cython", False) else "pure Python twin"
    else:
        from oracle import gp_oracle as O
        make_gp = lambda x, t, th: O.OracleGP(x, t, theta_min=th)
        make_up = lambda gp: gp
        prop = lambda gp, u, S: O.propagate_ga(gp, u, np.diag(S))
        out["propagate_impl"] = "oracle port (C loops)"
    rng = np.random.default_rng(3)
    x, t, th = synthetic(4096, 16, 11)
    gp = make_gp(x, t, th)
    xs = rng.uniform(0, 1, (4096, 16))
    t0 = time.perf_counter()
    for c0 in range(0, 4096, 2048):
        gp.estimate_many(xs[c0:c0 + 2048])
    out["estimate_many_pts_per_s"] = 4096 / (time.perf_counter() - t0)
    out["estimate_many_at"] = "n=4096 d=16, 4096 points in chunks of 2048"
    x, t, th = synthetic(2048, 8, 12)
    up = make_up(make_gp(x, t, th))
    U, S = rng.uniform(0.1, 0.9, (6, 8)), rng.uniform(1e-4, 1e-2, (6, 8))
    prop(up, U[0], S[0])
    t0 = time.perf_counter()
    for q in range(1, 6):
        prop(up, U[q], S[q])
    out["propagate_GA_queries_per_s"] = 5 / (time.perf_counter() - t0)
    out["propagate_GA_at"] = "n=2048 d=8, 5 queries one by one"
    return out


def _time_fg(f, g, n, d, reps=1):
    x, t, theta = synthetic(n, d, 7)
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        f(x, t, theta)
        g(x, t, theta)
        best = min(best, time.perf_counter() - t0)
    return best


def fit_cubic_quadratic(ns, ts):
    """Non-negative least squares of T(n) = a n^3 + b n^2 (LAPACK terms + the single-threaded O(n^2 d) numpy terms that
    dominate below n ~ 8192, SURVEY 6), relative residuals."""
    from scipy.optimize import nnls
    ns, ts = np.asarray(ns, dtype=np.float64), np.asarray(ts, dtype=np.float64)
    A = np.stack([ns ** 3, ns ** 2], axis=1) / ts[:, None]
    coef, _ = nnls(A, np.ones(len(ns)))
    return float(coef[0]), float(coef[1])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, d = args.n, args.d
    f, g, kind = _reference_callables()
    sizes = [int(s) for s in args.ref_sizes.split(",")] if args.ref_sizes else [1024, 2048, 4096, 8192]
    sizes = sorted(set(sizes))
    # per step: the two smallest sizes (a few seconds); the larger ones once per run, shared by every step's fit
    per_step = sizes[:2] if len(sizes) > 2 else sizes
    once = [s for s in sizes if s not in per_step]
    _time_fg(f, g, 256, d)                                  # imports, BLAS thread pool: not part of any timing
    t_once = {s: _time_fg(f, g, s, d) for s in once}
    cores = os.cpu_count()
    vals, coefs, t_small = [], [], []
    for i in range(args.steps + args.warmup):
        ts = {s: _time_fg(f, g, s, d) for s in per_step}
        ts.update(t_once)
        if len(sizes) >= 2:
            a, b = fit_cubic_quadratic(sizes, [ts[s] for s in sizes])
        else:
            a, b = ts[sizes[0]] / float(sizes[0]) ** 3, 0.0
        if i >= args.warmup:
            vals.append(a * float(n) ** 3 + b * float(n) ** 2)
            coefs.append((a, b))
            t_small.append([ts[s] for s in sizes])
    val = float(np.mean(vals))
    a, b = np.mean(coefs, axis=0)
    tm = np.mean(t_small, axis=0)
    impl = ("unmodified reference (baseline/_ref) GaussianCovariance._negativeloglikelihood + ._d_nll_d_theta"
            if kind == "reference" else "oracle port of Covariance._negativeloglikelihood + _d_nll_d_theta")
    sample = ("%s, numpy/scipy on %d host cores, timed at n=%s d=%d: %s s; fitted T(n) = a n^3 + b n^2 with a=%.3e b=%.3e; "
              "value = T(%d) [extrapolated: a direct run is ~18 min and ~45 GB per evaluation]" % (
                  impl, cores, "/".join(str(s) for s in sizes), d, "/".join("%.2f" % v for v in tm), a, b, n))
    line = {
        "impl": "reference", "metric": "fit_s_per_iter", "value": val, "unit": "s/iter", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": val * 1e3, "higher_is_better": False,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C3 fit iteration: K build + Cholesky/inverse + NLL + gradient, n=%d d=%d" % (n, d),
                   "n": n, "d": d},
        "extrapolated": True, "n_sample": sizes, "fit": {"a_n3": float(a), "b_n2": float(b),
                                                          "measured_s": {str(s): float(v) for s, v in zip(sizes, tm)}},
        "cpu_baseline": {"value": val, "unit": "s/iter", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "s/iter", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_ref_queries:
        try:
            line["extra"] = {"reference_query_paths": reference_query_rates(kind)}
        except Exception as exc:
            line["extra"] = {"reference_query_paths": {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}}
    emit(line)


def cpu_baseline_subprocess(n, d, sizes):
    """The reference arm on a bounded sample, in its own process (its package is also called `skgpuppy`)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--no-ref-queries", "--n", str(n), "--d", str(d), "--ref-sizes", ",".join(str(s) for s in sizes)]
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, env=env)
    lines = [l for l in res.stdout.splitlines() if l.strip().startswith("{")]
    if res.returncode != 0 or not lines:
        return {"value": None, "unit": "s/iter", "cores": os.cpu_count(), "kind": "port",
                "sample": "reference arm failed: %s" % res.stderr[-300:]}
    return json.loads(lines[-1])["cpu_baseline"]


# ---------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import ctypes
    from skgpuppy import _engine, _native as nat, _shard
    import skgpuppy.Covariance as C
    from skgpuppy.GaussianProcess import GaussianProcess
    C.VERBOSE = False
    lib = nat.load()
    n, d = args.n, args.d
    K, Wm = args.steps, args.warmup

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(v):
        if world == 1:
            return v
        tt = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def gather_obj(obj):
        if world == 1:
            return [obj]
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    def timed(fn, reps=2):
        fn()
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(reps):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            fn()
            a1.record()
            torch.cuda.synchronize()
            best = min(best, a0.elapsed_time(a1) * 1e-3)
        return best

    # ---- tensor peaks of this box, measured in this run ----------------------------------------------------------
    # FP64: cuBLAS dgemm 8192^3 (MEASURED_PEAKS.json has no FP64 entry). INT8: tcgen05.mma.kind::i8 probe from resident
    # shared-memory tiles (gpk_microbench_i8): burst = best single launch, sustained = 4 s back to back.
    a = torch.randn(8192, 8192, device="cuda", dtype=torch.float64)
    b = torch.randn(8192, 8192, device="cuda", dtype=torch.float64)
    c = torch.empty_like(a)
    peak_tf = 0.0
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        peak_tf = max(peak_tf, 2.0 * 8192 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b, c
    torch.cuda.empty_cache()
    i8 = (ctypes.c_double * 2)()
    nat.check(lib.gpk_microbench_i8(20000, args.i8_seconds, i8), "gpk_microbench_i8")
    i8_burst, i8_sustained = float(i8[0]), float(i8[1]) or float(i8[0])
    time.sleep(1.0)                                         # let the power state settle before the timed region

    x, t, theta0 = synthetic(n, d, 3000 + rank)           # each replica fits its own GP
    eng = _engine.Engine(x, t)
    thetas = [theta0 + 1e-4 * (i + 1) for i in range(K + Wm + K + Wm + 2)]   # fresh theta per step: no cache hits

    sampler = ClockSampler(local)
    for i in range(Wm):
        eng.nll_grad(thetas[i])
    barrier()
    sampler.start()
    nat.check(lib.gpk_profile(1), "profile on")
    lib.gpk_profile_read(None, None, None, None)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for i in range(K):
        last = eng.nll_grad(thetas[Wm + i])
    e1.record()
    barrier()
    gemm_ms, gemm_l, all_l, max_ms = ctypes.c_double(), ctypes.c_int64(), ctypes.c_int64(), ctypes.c_double()
    nat.check(lib.gpk_profile_read(ctypes.byref(gemm_ms), ctypes.byref(gemm_l), ctypes.byref(all_l),
                                   ctypes.byref(max_ms)), "profile read")
    nat.check(lib.gpk_profile(0), "profile off")
    clocks_rank = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"nll": np.array([last[0]], dtype=np.float64), "grad": last[1]})
    clocks_all = gather_obj(clocks_rank)
    clocks = clocks_all[0]
    t_dev = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    s_per_iter = t_dev / K                                  # one replica's iteration, max over ranks

    # ---- e2e through the reference-facing API: host arrays in, host scalars out, every step -------------------
    int8_on, moduli, int8_min, int8_bits = eng.route()
    npad_main = eng.npad
    eng.close()
    del eng
    torch.cuda.empty_cache()
    cov = C.GaussianCovariance()
    t_steps = [t + 1e-9 * (i + 1) for i in range(K + Wm)]   # new host data per step: the API uploads x, t again
    for i in range(Wm):
        cov._negativeloglikelihood(x, t_steps[i], thetas[K + Wm + i])
        cov._d_nll_d_theta(x, t_steps[i], thetas[K + Wm + i])
    barrier()
    w0 = time.perf_counter()
    for i in range(K):
        nll_e = cov._negativeloglikelihood(x, t_steps[Wm + i], thetas[K + 2 * Wm + i])
        g_e = cov._d_nll_d_theta(x, t_steps[Wm + i], thetas[K + 2 * Wm + i])
    torch.cuda.synchronize()
    e2e_val = max_over_ranks((time.perf_counter() - w0) / K)
    h2d = int(x.nbytes + t.nbytes)
    d2h = int(8 * (d + 3))
    eng = cov._fit_session(x, t_steps[-1]).engine          # keep using these device buffers for the query legs
    eng.update_data(x, t)

    # ---- query paths at BASELINE sizes: estimate_many over 1 M points, propagate_GA over 100 k queries ----------
    extra = {}
    eng.nll_grad(theta0)
    rng = np.random.default_rng(99 + rank)
    m = args.predict_m
    xs = rng.uniform(0, 1, (m, d))
    xs_dev = eng.to_device(xs)
    tp = timed(lambda: eng.predict_device(xs_dev, 0.0, True), reps=1)
    gp_api = GaussianProcess(x, t, cov, theta_min=theta0.copy(), _factorize=False)
    gp_api._eng = eng
    gp_api._state_theta = np.array(theta0, dtype=np.float64)
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    mm, vv = gp_api.estimate_many(xs)                       # public API: host array in, host arrays out
    tp_e2e = time.perf_counter() - w0
    extra["predict"] = {"n": n, "d": d, "m": m, "pts_per_s": m / tp, "e2e_pts_per_s": m / tp_e2e,
                        "tflops_of_n2_per_pt": float(n) ** 2 * m / tp / 1e12,
                        "frac_of_dgemm_peak": float(n) ** 2 * m / tp / 1e12 / peak_tf,
                        "var_min": float(vv.min()), "var_max": float(vv.max())}
    del xs_dev
    pn, pd_, Q = args.prop_n, args.prop_d, args.prop_q
    px, pt, ptheta = synthetic(pn, pd_, 4000 + rank)
    from skgpuppy.UncertaintyPropagation import UncertaintyPropagationApprox, UncertaintyPropagationExact
    pgp1 = GaussianProcess(px, pt, C.GaussianCovariance(), theta_min=ptheta.copy())
    peng = pgp1._engine()
    U = rng.uniform(0.1, 0.9, (Q, pd_))
    S = rng.uniform(1e-4, 1e-2, (Q, pd_))
    U_dev, S_dev = peng.to_device(U), peng.to_device(S)
    tq = timed(lambda: peng.propagate_device(U_dev, S_dev, False, 0.0))
    upa = UncertaintyPropagationApprox(pgp1)
    upa.propagate_GA_many(U[:1024], S[:1024])
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    pm, pv = upa.propagate_GA_many(U, S)                    # public batched API with host arrays
    tq_e2e = time.perf_counter() - w0
    extra["propagate_GA"] = {"n": pn, "d": pd_, "Q": Q, "queries_per_s": Q / tq, "e2e_queries_per_s": Q / tq_e2e,
                             "tflops_of_(d+2)n2_per_q": (pd_ + 2) * float(pn) ** 2 * Q / tq / 1e12,
                             "frac_of_dgemm_peak": (pd_ + 2) * float(pn) ** 2 * Q / tq / 1e12 / peak_tf}
    # exact (Girard) propagation, SURVEY 8f #1: O(n^2 d) exp-bound pair kernel per query
    upe = UncertaintyPropagationExact(pgp1)
    Qe = min(Q, 1024)
    lam, dinv, norms = upe._constants(S[:Qe])
    args_e = [peng.to_device(U[:Qe]), peng.to_device(lam), peng.to_device(dinv), peng.to_device(norms)]
    te = timed(lambda: peng.propagate_exact_device(args_e[0], args_e[1], args_e[2], args_e[3], 0.0))
    extra["propagate_exact"] = {"n": pn, "d": pd_, "Q": Qe, "queries_per_s": Qe / te,
                                "gflops_of_n2_(d+30)_over_2_per_q": float(pn) ** 2 / 2 * (pd_ + 30) * Qe / te / 1e9}
    del U_dev, S_dev, args_e

    # BASELINE configs[1]: ML-II fit at n=4096, d=8 (one L-BFGS evaluation = NLL + gradient), through the public API
    if rank == 0 and not args.no_c2:
        import scipy.optimize  # noqa: F401  (its first import costs ~0.3 s; keep it out of the timed fit)
        cx, ct, ctheta = synthetic(4096, 8, 2000)
        ccov = C.GaussianCovariance()
        ccov._negativeloglikelihood(cx, ct, ctheta)
        ccov._d_nll_d_theta(cx, ct, ctheta)
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        for i in range(5):
            th = ctheta + 1e-4 * (i + 1)
            ccov._negativeloglikelihood(cx, ct, th)
            ccov._d_nll_d_theta(cx, ct, th)
        torch.cuda.synchronize()
        per_eval = (time.perf_counter() - w0) / 5
        evals = {"f": 0, "g": 0, "f_s": 0.0, "g_s": 0.0}
        f0, g0 = ccov._negativeloglikelihood, ccov._d_nll_d_theta

        def f_count(x_, t_, th_):
            evals["f"] += 1
            c0 = time.perf_counter()
            r = f0(x_, t_, th_)
            evals["f_s"] += time.perf_counter() - c0
            return r

        def g_count(x_, t_, th_):
            evals["g"] += 1
            c0 = time.perf_counter()
            r = g0(x_, t_, th_)
            evals["g_s"] += time.perf_counter() - c0
            return r
        ccov._negativeloglikelihood, ccov._d_nll_d_theta = f_count, g_count
        w0 = time.perf_counter()
        th_min = ccov.ml_estimate(cx, ct)
        torch.cuda.synchronize()
        t_fit = time.perf_counter() - w0
        extra["c2_ml2_fit_n4096_d8"] = {"s_per_lbfgs_evaluation": per_eval, "full_fit_s": t_fit, "nll_evals": evals["f"],
                                        "grad_evals": evals["g"], "s_in_nll_calls": evals["f_s"], "s_in_grad_calls": evals["g_s"],
                                        "tflops_of_n3_per_evaluation": fit_flops(4096, 8) / per_eval / 1e12,
                                        "nll_min": float(f0(cx, ct, th_min))}
        ccov._session.engine.close()
        del ccov

    # ---- sharded paths across ranks (factor broadcast once, queries split, no data-path collective) ---------------
    if world > 1:
        x0, t0, th0 = synthetic(n, d, 3000)                 # rank 0's GP, identical inputs on all ranks
        gp = GaussianProcess(x0, t0, C.GaussianCovariance(), theta_min=th0.copy(), _factorize=False)
        gp._eng = eng                                       # reuse this rank's buffers for the shared GP
        eng.update_data(x0, t0)
        barrier()
        warm = torch.zeros(1 << 20, dtype=torch.float64, device="cuda")
        dist.broadcast(warm, src=0)                         # NCCL channel set-up outside the timed broadcast
        if rank == 0:
            gp._engine()                                    # factorise on rank 0 before timing the broadcast itself
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        gp.broadcast_state(src=0)
        b1.record()
        barrier()
        t_bcast = max_over_ranks(b0.elapsed_time(b1) * 1e-3)
        sh = {"broadcast_s": t_bcast, "broadcast_bytes": int(gp._eng.X.numel() * 8 + n * 8)}

        def sharded_time(total, make_args, run):
            lo, hi = _shard.my_shard(total, rank, world)
            dev_args = make_args(lo, hi)
            run(*dev_args)
            barrier()
            b0.record()
            out = run(*dev_args)
            b1.record()
            barrier()
            return max_over_ranks(b0.elapsed_time(b1) * 1e-3), out, (lo, hi)

        # estimate_many: weak (m per GPU) and strong (the same m in total, BASELINE configs[2]: 1 M points)
        xs_all = np.random.default_rng(5).uniform(0, 1, (m, d))
        ts_strong, out_s, (lo, hi) = sharded_time(m, lambda lo, hi: (gp._eng.to_device(xs_all[lo:hi]),),
                                                  lambda q: gp._eng.predict_device(q, 0.0, True))
        sh["predict_strong"] = {"m_total": m, "pts_per_s": m / ts_strong, "s": ts_strong,
                                "s_incl_broadcast": ts_strong + t_bcast,
                                "speedup_vs_this_run_1gpu_rate": (m / ts_strong) / (m / tp)}
        # sharded == single-GPU, bitwise: rank 0 recomputes the first 4096/N rows of every shard on its own
        cnt = 4096 // world
        if m // world >= cnt:                               # the same decision on every rank (no collective mismatch)
            bnd = _shard.shard_bounds(m, world)
            sub = np.concatenate([np.arange(bnd[r], bnd[r] + cnt) for r in range(world)])
            part = torch.stack([out_s[0][:cnt], out_s[1][:cnt]], dim=1).contiguous()
            parts = [torch.empty_like(part) for _ in range(world)] if rank == 0 else None
            dist.gather(part, parts, dst=0)
            if rank == 0:
                ref_m, ref_v = gp._eng.predict_device(gp._eng.to_device(xs_all[sub]), 0.0, True)
                got = torch.cat(parts, dim=0)
                sh["sharded_parity"] = bool(torch.equal(got[:, 0], ref_m) and torch.equal(got[:, 1], ref_v))
        tw, _, _ = sharded_time(m * world, lambda lo, hi: (gp._eng.to_device(
            np.random.default_rng(50 + rank).uniform(0, 1, (hi - lo, d))),), lambda q: gp._eng.predict_device(q, 0.0, True))
        sh["predict_weak"] = {"m_total": m * world, "pts_per_s": m * world / tw, "s": tw}
        # gradient trace sharded by tile rows: row panels of K^-1 to their ranks + partial traces + one all-reduce
        barrier()
        _shard.sharded_gradient(gp, src=0)                  # first call: NCCL point-to-point channel set-up
        barrier()
        tim = {}
        g_sh = _shard.sharded_gradient(gp, src=0, timings=tim)
        sh["gradient"] = {k: max_over_ranks(v) if k.endswith("_s") else v for k, v in tim.items()}
        tot = gather_obj(tim.get("bytes_moved", 0))
        sh["gradient"]["bytes_sent_by_rank0"] = int(tot[0])
        if rank == 0:
            tt = timed(lambda: eng.grad_trace_partial(0, eng.npad // 128))
            sh["gradient"]["single_gpu_trace_s"] = tt
            g1 = eng.nll_grad(th0)[1]
            sh["gradient"]["max_rel_diff_vs_single_gpu"] = float(np.max(np.abs(g_sh - g1)) / np.max(np.abs(g1)))
        # propagate_GA sharded by query (BASELINE configs[3]: 100 k queries in total = strong; Q per GPU = weak)
        px0, pt0, pth0 = synthetic(pn, pd_, 4000)
        pgp = GaussianProcess(px0, pt0, C.GaussianCovariance(), theta_min=pth0.copy(), _factorize=(rank == 0))
        pgp.broadcast_state(src=0)
        U_all = np.random.default_rng(6).uniform(0.1, 0.9, (Q * world, pd_))
        S_all = np.random.default_rng(7).uniform(1e-4, 1e-2, (Q * world, pd_))
        for key, total in (("propagate_strong", Q), ("propagate_weak", Q * world)):
            tq_s, _, _ = sharded_time(total, lambda lo, hi: (pgp._eng.to_device(U_all[lo:hi]), pgp._eng.to_device(S_all[lo:hi])),
                                      lambda u, s: pgp._eng.propagate_device(u, s, False, 0.0))
            sh[key] = {"Q_total": total, "queries_per_s": total / tq_s, "s": tq_s}
        sh["propagate_strong"]["speedup_vs_this_run_1gpu_rate"] = sh["propagate_strong"]["queries_per_s"] / (Q / tq)
        sh["clocks_per_rank"] = [{"rank": r, "sm_mhz": cr.get("sm_mhz"), "power_w_max": cr.get("power_w_max"),
                                  "reasons": cr.get("reasons")} for r, cr in enumerate(clocks_all)]
        extra["sharded"] = sh
        pgp._eng.close()
    peng.close()
    del pgp1, peng, upa, upe
    torch.cuda.empty_cache()

    # ---- the same fit iteration with every contraction on the FP64 DMMA kernel, for comparison --------------------
    if rank == 0 and world == 1 and int8_on and not args.no_dmma:
        nll_int8 = eng.nll_grad(thetas[1])[0]
        eng.close()
        cov._session = None
        del eng, gp_api
        torch.cuda.empty_cache()
        deng = _engine.Engine(x, t, route={"int8": False})
        deng.nll_grad(thetas[0])
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        dl = deng.nll_grad(thetas[1])
        a1.record()
        torch.cuda.synchronize()
        ds = a0.elapsed_time(a1) * 1e-3
        extra["fit_fp64_dmma_only"] = {"s_per_iter": ds, "tflops_of_n3": fit_flops(n, d) / ds / 1e12,
                                       "nll_rel_diff_vs_int8_route": abs(dl[0] - nll_int8) / abs(nll_int8)}
        deng.close()
        del deng
    else:
        try:
            eng.close()
        except Exception:
            pass
        cov._session = None
    torch.cuda.empty_cache()

    # ---- BASELINE configs[4]: n=65536, d=32 fit iteration + a prediction batch on one GPU -------------------------
    if rank == 0 and world == 1 and not args.no_c5:
        try:
            n5, d5 = args.c5_n, args.c5_d
            x5, t5, th5 = synthetic(n5, d5, 5000)
            e5 = _engine.Engine(x5, t5)
            e5.nll_grad(th5)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            nll5, g5 = e5.nll_grad(th5 + 1e-4)
            a1.record()
            torch.cuda.synchronize()
            s5 = a0.elapsed_time(a1) * 1e-3
            a0.record()
            e5.nll_grad(th5 + 3e-4, want_grad=False)
            a1.record()
            torch.cuda.synchronize()
            s5f = a0.elapsed_time(a1) * 1e-3
            e5.nll_grad(th5 + 1e-4)
            m5 = 16384
            xs5 = e5.to_device(np.random.default_rng(1).uniform(0, 1, (m5, d5)))
            tp5 = timed(lambda: e5.predict_device(xs5, 0.0, True), reps=1)
            free_b, total_b = torch.cuda.mem_get_info()
            extra["c5_n65536_d32"] = {"n": n5, "d": d5, "fit_s_per_iter": s5, "fit_tflops_of_n3": fit_flops(n5, d5) / s5 / 1e12,
                                      "factor_plus_triangular_inverse_s": s5f,
                                      "tflops_of_2n3_over_3": 2.0 / 3.0 * float(n5) ** 3 / s5f / 1e12,
                                      "predict_pts_per_s": m5 / tp5, "predict_m": m5,
                                      "predict_tflops_of_n2_per_pt": float(n5) ** 2 * m5 / tp5 / 1e12,
                                      "device_mem_used_GB": (total_b - free_b) / 1e9, "nll": nll5,
                                      "route": list(e5.route())}
            e5.close()
            del e5, xs5
        except Exception as exc:                            # e.g. a smaller-memory device: report, do not hide
            extra["c5_n65536_d32"] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:300])}
        torch.cuda.empty_cache()

    # ---- CPU baseline (rank 0, N == 1): bounded sample of the same workload through the reference arm --------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu_baseline = cpu_baseline_subprocess(n, d, [int(s) for s in args.cpu_sizes.split(",")])

    if rank == 0:
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            traffic = tr.get("%s_n%d" % ("oz_planes_lauum" if int8_on else "dmma_lauum", n))
        except Exception:
            pass
        gemm_s_per_iter = gemm_ms.value * 1e-3 / K
        # dominant kernel = the largest launch of the step: K^-1 = X^T X, n^3/3 algorithmic FP64 flops in a single
        # launch pair (planes GEMM + reconstruction), timed by CUDA events on its own stream inside the timed region
        achieved = float(n) ** 3 / 3.0 / (max_ms.value * 1e-3) / 1e12
        i8_tops = achieved * moduli if int8_on else None       # n^3/6 MACs x moduli x 2 ops = n^3/3 x moduli
        line = {
            "metric": "fit_s_per_iter", "value": s_per_iter, "unit": "s/iter", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": s_per_iter * 1e3, "higher_is_better": False, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C3 fit iteration: K build + Cholesky/inverse + NLL + gradient, n=%d d=%d" % (n, d),
                       "n": n, "d": d,
                       "parallelism": "replicas only (fit does not shard): value = one replica's s/iter, max over ranks; "
                                      "queries shard by row, the gradient trace by tile rows (extra.sharded)",
                       "l2": "inputs larger than L2 (two %.1f GB matrices per step), no flush needed" % (
                           8.0 * npad_main ** 2 / 1e9),
                       "theta": "v=1 vt=0.09 w=(4/d)*linspace(.75,1.25,d), perturbed per step",
                       "contractions": ("exact INT8 CRT products on tcgen05 (%d coprime moduli, %d-bit operands, int32 "
                                        "accumulation in TMEM, exact reconstruction to FP64) for blocks >= %d, FP64 DMMA "
                                        "below" % (moduli, int8_bits, int8_min)) if int8_on else "FP64 DMMA"},
            "replicas_iters_per_s": world / s_per_iter,
            "fit_tflops_of_n3": fit_flops(n, d) / s_per_iter / 1e12,
            "roofline": {"bound": "tensor",
                         "kernel": ("oz_crt_planes_kernel + oz_crt_reconstruct_kernel<STORE> (K^-1 = X^T X on the INT8 "
                                    "tcgen05 pipe: largest launch, n^3/3 FP64 flops = %d int8 products of n^3/6 MACs)" % moduli
                                    if int8_on else
                                    "dgemm_dmma_kernel<MC,MC,STORE> (K^-1 = X^T X: largest launch, n^3/3 flops)"),
                         # On the INT8 route the pipe that bounds the launch is the int8 tensor pipe: achieved / peak are
                         # int8 operations (2 per multiply-add); the FP64 view of the same launch is in `fp64_equivalent`.
                         "achieved": (i8_tops if int8_on else achieved), "peak": (i8_sustained if int8_on else peak_tf),
                         "unit": "TFLOP/s", "frac": (i8_tops / i8_sustained if int8_on else achieved / peak_tf),
                         "traffic": traffic, "launch_ms": max_ms.value,
                         "frac_of_burst_peak": (i8_tops / i8_burst if int8_on else None),
                         "peak_source": ("int8 tensor pipe measured in this run by gpk_microbench_i8 (tcgen05.mma.cta_group::2"
                                         ".kind::i8 M=256 N=256 K=32 from resident shared-memory tiles on every SM pair): "
                                         "sustained %.0f TOP/s over %.0f s back to back (used: this launch sits inside a long "
                                         "power-capped step), burst %.0f TOP/s; ops = 2 x int8 multiply-adds" % (
                                             i8_sustained, args.i8_seconds, i8_burst)
                                         if int8_on else
                                         "cuBLAS dgemm 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry)"),
                         "fp64_equivalent": {"achieved_tflops": achieved, "fp64_tensor_peak_tflops": peak_tf,
                                             "ratio": achieved / peak_tf,
                                             "peak_source": "cuBLAS dgemm 8192^3 measured in this run"},
                         "algorithmic_flops_per_launch": float(n) ** 3 / 3.0,
                         "all_tensor_launches": {"sum_ms_per_iter": gemm_s_per_iter * 1e3,
                                                 "tflops_of_n3": float(n) ** 3 / gemm_s_per_iter / 1e12,
                                                 "launches_per_iter": gemm_l.value / K},
                         "share_of_step": max_ms.value * 1e-3 / s_per_iter},
            "e2e": {"value": e2e_val, "unit": "s/iter", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "GaussianCovariance._negativeloglikelihood + ._d_nll_d_theta with host arrays"},
            "gpu_launches": int(all_l.value),
            "clocks": clocks,
            "extra": extra,
            "nll": last[0] if last else None,
        }
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """What the timed path returned in its last step, one DIR/<name>.npy per array, so that two builds run with the
    same arguments (hence the same seeded inputs) can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


_RESULT_FD = None


def _reserve_stdout():
    """The contract is ONE JSON line on stdout. Libraries print there too (NCCL's version banner at N > 1), so the
    process-level stdout is pointed at stderr for the whole run and the result line goes to the saved descriptor."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=32768)
    ap.add_argument("--d", type=int, default=16)
    ap.add_argument("--predict-m", type=int, default=1048576, help="estimate_many points (BASELINE configs[2]: 1 M)")
    ap.add_argument("--prop-n", type=int, default=8192)
    ap.add_argument("--prop-d", type=int, default=8)
    ap.add_argument("--prop-q", type=int, default=100000, help="propagate_GA queries (BASELINE configs[3]: 100 k)")
    ap.add_argument("--c5-n", type=int, default=65536)
    ap.add_argument("--c5-d", type=int, default=32)
    ap.add_argument("--i8-seconds", type=float, default=4.0, help="duration of the sustained INT8 tensor-peak probe")
    ap.add_argument("--cpu-sizes", default="1024,2048,4096", help="sizes of the bounded cpu_baseline sample (our arm)")
    ap.add_argument("--ref-sizes", default="", help="sizes timed by the reference arm (default 1024,2048,4096,8192)")
    ap.add_argument("--no-ref-queries", action="store_true", help="reference arm: skip the estimate_many / propagate_GA rates")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-c2", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the n=65536 d=32 leg (needs ~165 GB of HBM)")
    ap.add_argument("--no-dmma", action="store_true", help="skip the FP64-DMMA-only comparison leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's NLL and gradient as DIR/nll.npy, DIR/grad.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    _reserve_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
