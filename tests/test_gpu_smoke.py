"""The driver's smoke entry point must stay green on the default route (it asserts that the INT8 route is active)."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_graft_entry_smoke():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as entry
    entry.smoke()


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs writes the NLL / gradient of the last of --steps timed steps: the oracle's values at that
    step's theta, which a second run with the same arguments (same seeded inputs) reproduces."""
    import json
    import subprocess
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from oracle import gp_oracle as O
    n, d, steps, warmup = 2304, 8, 3, 2                   # npad 2304: the INT8 route, like the default n = 32768
    small = ["--n", str(n), "--d", str(d), "--predict-m", "4096", "--prop-n", "1024", "--prop-q", "2048",
             "--i8-seconds", "0", "--no-cpu", "--no-c2", "--no-c5", "--no-dmma"]
    outs = []
    for run in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                              "--warmup", str(warmup), "--dump-outputs", str(tmp_path / run)] + small,
                             capture_output=True, text=True, timeout=900)
        assert res.returncode == 0, res.stderr[-3000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["warmup"] == warmup
        nll, grad = np.load(tmp_path / run / "nll.npy"), np.load(tmp_path / run / "grad.npy")
        assert nll.dtype == np.float64 and nll.shape == (1,) and grad.dtype == np.float64 and grad.shape == (d + 2,)
        assert nll[0] == line["nll"]
        outs.append((nll[0], grad))
    x, t, theta0 = bench.synthetic(n, d, 3000)
    theta = theta0 + 1e-4 * (warmup + steps)               # bench.py: step i evaluates theta0 + 1e-4 (i + 1)
    nll_o, grad_o = O.negativeloglikelihood(x, t, theta), O.d_nll_d_theta(x, t, theta)
    for nll, grad in outs:
        assert abs(nll - nll_o) < 1e-9 * abs(nll_o)
        assert np.max(np.abs(grad - grad_o)) < 1e-9 * np.max(np.abs(grad_o))
    assert abs(outs[0][0] - outs[1][0]) <= 1e-12 * abs(outs[0][0])
    assert np.max(np.abs(outs[0][1] - outs[1][1])) <= 1e-12 * np.max(np.abs(outs[0][1]))
