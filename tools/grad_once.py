"""Gradients of the predictive mean and variance (gpk_predict_grad) on the flagship inputs: ms per call and points/s,
with and without the variances, and estimate_many and propagate_GA at the same number of points beside it.

    python tools/grad_once.py [--out FILE] [--reps R]

Inputs: bench.synthetic at n = 32768, d = 16 (the fit state of the default bench, m = 4096 points) and at n = 8192,
d = 8 (m = 16384), on the INT8 route (the default at these sizes) and on FP64 DMMA. Call times are CUDA events around
single calls after a warm-up of the same shape (median of --reps). Work (flops) of the variance path: (d + 1) m n^2
(one row of V = X G^T per row of G, X triangular); propagate_GA runs d + 2 rows per query. Card name and power limit
are read in the same run.
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scikit-gpuppy_b200"))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from bench import synthetic
from skgpuppy import _engine


def card():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                              "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = "power limit not readable (%s)" % e
    return "%s, %s" % (name, out)


def timed(fn, reps):
    fn()                                              # warm-up of this shape
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms))


def run(n, d, m, route, reps, log):
    x, t, theta = synthetic(n, d, 3000 if n == 32768 else 4000)
    eng = _engine.Engine(x, t, route=route)
    eng.factorize(theta)
    tag = "INT8" if eng.route()[0] else "DMMA"
    rng = np.random.default_rng(9)
    xs = eng.to_device(rng.uniform(0, 1, (m, d)))
    S = eng.to_device(np.full((m, d), 1e-3))
    g_ms = timed(lambda: eng.predict_grad_device(xs, 0.0, want_var=True), reps)
    gm_ms = timed(lambda: eng.predict_grad_device(xs, 0.0, want_var=False), reps)
    em_ms = timed(lambda: eng.predict_device(xs, 0.0, True), reps)
    ga_ms = timed(lambda: eng.propagate_device(xs, S, False, 0.0), reps)
    work = float(d + 1) * m * n * n
    log("%s n=%d d=%d m=%d: grad %9.2f ms (%.0f points/s, %.1f TFLOP/s of (d+1) m n^2) | grad want_var=False %8.2f ms "
        "(%.0f points/s) | estimate_many %8.2f ms (%.0f points/s) | propagate_GA %8.2f ms (%.0f queries/s)"
        % (tag, n, d, m, g_ms, m / g_ms * 1e3, work / g_ms / 1e9, gm_ms, m / gm_ms * 1e3, em_ms, m / em_ms * 1e3,
           ga_ms, m / ga_ms * 1e3))
    eng.close()
    del eng
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "grad_once.py measures on a CUDA device"
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log("card: " + card())
    for n, d, m in ((32768, 16, 4096), (8192, 8, 16384)):
        for route in (None, {"int8": False}):
            run(n, d, m, route, a.reps, log)
    log("card: " + card())
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
