"""Joint predictive covariance (gpk_predict_cov) on the flagship inputs: ms per call split into the V step and the product,
rates against the algorithmic work, and estimate_many at the same m beside it.

    python tools/cov_once.py [--out FILE] [--reps R]

Inputs: bench.synthetic at n = 32768, d = 16 (the fit state of the default bench) and at n = 8192, d = 8; symmetric
m in {2048, 8192, 16384} and one 8192 x 8192 cross case, on the INT8 route (the default at these sizes) and on FP64
DMMA. Call times are CUDA events around single calls after a warm-up of the same shape (median of --reps). The split
comes from one extra call under torch.profiler: the V step is every kernel before the last se_tile_kernel launch (the
prior block), the product is that launch and everything after it (residues of V, the product, copy-out).
Work (flops): V = X k(x, Q) for each query set is ma n^2 (X is triangular); the product is 2 ma mb n, half of it when
symmetric (lower tiles only). Card name and power limit are read in the same run.
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


def split(fn):
    """(V step ms, product ms) as kernel spans of one profiled call."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ks = sorted((e for e in prof.events() if e.device_type.name == "CUDA" and "Memcpy" not in e.name
                 and "Memset" not in e.name), key=lambda e: e.time_range.start)
    cut = max(i for i, e in enumerate(ks) if "se_tile_kernel" in e.name)
    v = (ks[cut - 1].time_range.end - ks[0].time_range.start) / 1e3
    p = (ks[-1].time_range.end - ks[cut].time_range.start) / 1e3
    return v, p


def run(n, d, route, sizes, cross, reps, log):
    x, t, theta = synthetic(n, d, 3000 if n == 32768 else 4000)
    eng = _engine.Engine(x, t, route=route)
    eng.factorize(theta)
    on = eng.route()[0]
    rng = np.random.default_rng(9)
    tag = "INT8" if on else "DMMA"
    for ma, mb in [(m, None) for m in sizes] + [cross]:
        xa = eng.to_device(rng.uniform(0, 1, (ma, d)))
        xb = None if mb is None else eng.to_device(rng.uniform(0, 1, (mb, d)))
        nb = ma if mb is None else mb
        ms = timed(lambda: eng.predict_cov_device(xa, xb), reps)
        try:
            v_ms, p_ms = split(lambda: eng.predict_cov_device(xa, xb))
        except Exception as e:           # the call time above stands without the split
            log("split not available: %r" % (e,))
            v_ms = p_ms = float("nan")
        v_work = float(ma) * n * n + (0.0 if mb is None else float(mb) * n * n)
        p_work = (1.0 if mb is None else 2.0) * ma * nb * n
        em = timed(lambda: eng.predict_device(xa, 0.0, True), reps)
        log("%s n=%d d=%d %s %5d x %5d: %9.2f ms/call (V step %8.2f ms, %6.1f TFLOP/s; product %8.2f ms, %6.1f TFLOP/s; "
            "whole call %6.1f TFLOP/s) | estimate_many m=%d %8.2f ms, %.0f points/s"
            % (tag, n, d, "sym  " if mb is None else "cross", ma, nb, ms, v_ms, v_work / v_ms / 1e9, p_ms,
               p_work / p_ms / 1e9, (v_work + p_work) / ms / 1e9, ma, em, ma / em * 1e3))
    eng.close()
    del eng
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "cov_once.py measures on a CUDA device"
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log("card: " + card())
    for n, d in ((32768, 16), (8192, 8)):
        for route in (None, {"int8": False}):
            run(n, d, route, (2048, 8192, 16384), (8192, 8192), a.reps, log)
    log("card: " + card())
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
