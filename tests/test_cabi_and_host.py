"""CPU-only checks: the C-ABI library loads and exports every symbol include/gpk.h declares, the host
layer mirrors the reference's scalar functions, and the product path fails loudly without CUDA."""
import ctypes
import os
import pickle
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import PKG, ROOT
from oracle import gp_oracle as O

HEADER = os.path.join(ROOT, "include", "gpk.h")            # the drop-in boundary
TEST_HEADER = os.path.join(ROOT, "include", "gpk_test.h")  # measurement / test hooks, not part of the boundary


@pytest.fixture(scope="module")
def native():
    sys.path.insert(0, PKG)
    import build_native
    build_native.build()
    from skgpuppy import _native
    _native.load()
    return _native


def declared_functions(header=HEADER):
    src = open(header).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gpk_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported_and_bound(native):
    names = declared_functions()
    assert len(names) >= 20
    lib = ctypes.CDLL(native.lib_path())
    for nm in names:
        assert hasattr(lib, nm), "libgpk.so does not export %s" % nm
        assert nm in native.SIGNATURES, "%s has no ctypes prototype in _native.SIGNATURES" % nm
    assert set(native.SIGNATURES) == set(names)
    hooks = declared_functions(TEST_HEADER)
    for nm in hooks:
        assert hasattr(lib, nm), "libgpk.so does not export %s" % nm
    assert set(native.TEST_SIGNATURES) == set(hooks)
    assert not set(hooks) & set(names)
    # the product layer binds the hooks (one loader) but never calls them
    for root, _, files in os.walk(os.path.join(PKG, "skgpuppy")):
        for f in files:
            if f.endswith(".py") and f != "_native.py":
                src = open(os.path.join(root, f)).read()
                for nm in hooks:
                    assert nm not in src, "%s uses the test hook %s" % (f, nm)
    assert native.load().gpk_version() >= 100
    assert native.load().gpk_npad(100) == 128 and native.load().gpk_npad(129) == 256


def test_library_is_sm100a_with_dmma(native):
    out = subprocess.run(["cuobjdump", "-lelf", native.lib_path()], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run(["cuobjdump", "-sass", native.lib_path()], capture_output=True, text=True).stdout
    assert "DMMA.8x8x4" in sass and "LDGSTS" in sass
    # the INT8 route: tcgen05 int8 MMA on CTA pairs, TMEM loads, 5-D TMA loads, dp4a residues, dp2a reconstruction
    for mnemonic in ("UTCIMMA.2CTA", "LDTM", "UTMALDG.5D", "IDP.4A", "IDP.2A"):
        assert mnemonic in sass, mnemonic
    # ONE route: the CRT kernels (256x256 pair tiles + reconstruction pass); the round-1 variants are gone
    for kernel in ("oz_crt_planes_kernel", "oz_crt_reconstruct_kernel", "oz_residue_rows_kernel"):
        assert kernel in sass, kernel
    for kernel in ("oz_crt_pair_kernel", "oz_gemm_pair_kernel", "oz_slice_rows_kernel", "mb_dmma_kernel",
                   "mb_dfma_kernel"):
        assert kernel not in sass, kernel
    # one reconstruction kernel per epilogue (store, row sums) and group of 4 moduli (8..18 moduli: 2..5 groups)
    functions = set(re.findall(r"Function : (\S+)", sass))
    assert len([f for f in functions if "oz_crt_reconstruct_kernel" in f]) == 8


def test_library_reads_no_environment_variables(native):
    """Route selection is per handle (gpk_set_route), never an environment switch (SURVEY 5: no multi-backend dispatch)."""
    for f in os.listdir(os.path.join(PKG, "csrc")):
        if f.endswith((".cu", ".cuh", ".h")):
            assert "getenv" not in open(os.path.join(PKG, "csrc", f)).read(), f


def test_no_cpu_fallback(native):
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from skgpuppy.Covariance import GaussianCovariance
    from skgpuppy.GaussianProcess import GaussianProcess
    x = np.random.rand(10, 2)
    t = np.random.rand(10)
    with pytest.raises(native.GpkError):
        GaussianProcess(x, t, GaussianCovariance(), theta_min=np.zeros(4))
    with pytest.raises(native.GpkError):
        GaussianCovariance().cov_matrix(x, np.zeros(4))


def test_product_does_not_import_oracle():
    for root, _, files in os.walk(os.path.join(PKG, "skgpuppy")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), f


def test_scalar_host_functions_match_oracle(native):
    from skgpuppy.Covariance import GaussianCovariance, tracedot
    rng = np.random.default_rng(5)
    cov = GaussianCovariance()
    for d in (1, 3, 8):
        theta = rng.normal(size=d + 2)
        u, xi = rng.normal(size=d), rng.normal(size=d)
        assert cov(u, xi, theta) == pytest.approx(O.cov_scalar(u, xi, theta), rel=1e-15)
        assert cov(u, u.copy(), theta) == pytest.approx(np.exp(theta[0]) + np.exp(theta[1]), rel=1e-15)
        np.testing.assert_allclose(cov.get_Jacobian(u, xi, theta), O.get_jacobian(u, xi, theta), rtol=1e-14)
        np.testing.assert_allclose(cov.get_Hessian(u, xi, theta), O.get_hessian(u, xi, theta), rtol=1e-14, atol=1e-300)
        assert cov.get_Jacobian(u, xi, theta).shape == (d, 1)
        x = rng.normal(size=(20, d))
        t = rng.normal(size=20)
        np.testing.assert_array_equal(cov.get_theta(x, t), O.get_theta(x, t))
        A, B = rng.normal(size=(d, d)), rng.normal(size=(d, d))
        assert tracedot(A, B) == pytest.approx(np.trace(A @ B), rel=1e-13)
        for j in range(d + 2):
            eps = 1e-6
            e = np.zeros(d + 2)
            e[j] = eps
            fd = (cov(u, xi, theta + e) - cov(u, xi, theta - e)) / (2 * eps)
            assert cov._d_cov_d_theta(u, xi, theta, j) == pytest.approx(fd, rel=1e-5, abs=1e-9)


def test_minimize_mirror_on_quadratic(native):
    from skgpuppy.Utilities import minimize
    f = lambda th: float(np.sum((th - np.array([1.0, -2.0, 0.5])) ** 2))
    g = lambda th: 2 * (th - np.array([1.0, -2.0, 0.5]))
    for method in (["l_bfgs_b"], "bfgs", "cg", "tnc"):
        th = minimize(f, np.zeros(3), None, None, fprime=g, method=method, verbose=False)
        np.testing.assert_allclose(th, [1.0, -2.0, 0.5], atol=1e-4)


def test_covariance_object_pickles_without_device_state(native):
    from skgpuppy.Covariance import GaussianCovariance
    c = GaussianCovariance()
    c2 = pickle.loads(pickle.dumps(c, protocol=0))
    assert isinstance(c2, GaussianCovariance) and c2._session is None


def test_crt_tables_are_current_and_self_consistent(tmp_path):
    """The committed csrc/oz_crt_tables.h equals what tools/gen_crt_tables.py generates (whose self-check replays the
    sloppy-Barrett / 96-bit fixed-point CRT reconstruction and the dp4a residue path with exact integers)."""
    import shutil
    hdr = os.path.join(PKG, "csrc", "oz_crt_tables.h")
    keep = tmp_path / "oz_crt_tables.h"
    shutil.copy2(hdr, keep)
    try:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_crt_tables.py")], capture_output=True,
                             text=True)
        assert out.returncode == 0 and "CRT self-check ok" in out.stdout, out.stdout + out.stderr
        assert open(hdr).read() == open(keep).read(), "oz_crt_tables.h is stale: run tools/gen_crt_tables.py"
    finally:
        shutil.copy2(keep, hdr)    # with its mtime, or build_native would take libgpk.so for stale and rebuild it
    # moduli: pairwise coprime, <= 256, and 17 of them carry 58-bit operands at K = 32768
    from math import gcd, log2
    mods = [256, 255, 253, 251, 247, 241, 239, 233, 229, 227, 223, 217, 211, 199, 197, 193, 191, 181]
    assert all(gcd(a, b) == 1 for i, a in enumerate(mods) for b in mods[i + 1:]) and max(mods) <= 256
    log2P = sum(log2(m) for m in mods[:17])
    assert int((log2P - 1 - 15 - 1e-6) // 2) == 58


def test_build_dependency_list_covers_every_source():
    """build_native skips the rebuild when libgpk.so is newer than its dependencies: every file under csrc/ must be one."""
    sys.path.insert(0, os.path.join(ROOT, "scikit-gpuppy_b200"))
    import build_native
    listed = {os.path.basename(d) for d in build_native.DEPS}
    for f in os.listdir(build_native.CSRC):
        if f.endswith((".cu", ".cuh", ".h")):
            assert f in listed, f


def test_bench_reference_arm_prints_one_json_line():
    """The reference arm of bench.py (CPU only) keeps the driver's contract: exactly one JSON line on stdout with the
    required keys; everything else (library banners, warnings) goes to stderr."""
    import json
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-sizes", "256,384,512"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout[-2000:]
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["higher_is_better"] is False
    # the unmodified reference from baseline/_ref when it is installed (DESIGN.md 6), the oracle port otherwise
    installed = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "skgpuppy"))
    assert line["cpu_baseline"]["kind"] == ("reference" if installed else "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["extrapolated"] is True and line["n_sample"] == [256, 384, 512] and set(line["fit"]) >= {"a_n3", "b_n2"}
    assert line["value"] == pytest.approx(line["fit"]["a_n3"] * 32768.0 ** 3 + line["fit"]["b_n2"] * 32768.0 ** 2, rel=1e-9)
    # non-zero ranks of a torchrun launch exit 0 without work or output
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-sizes", "256,384"], capture_output=True, text=True, timeout=600, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_reference_arm_port_and_install_agree(golden):
    """Whichever `kind` the reference arm uses (the oracle port, or the installed reference in baseline/_ref), it gives
    the unmodified reference's NLL / gradient on the bench workload: tests/golden/syn_*.npz hold the reference's own
    values on the inputs bench.synthetic draws for these seeds (oracle/make_golden.py)."""
    import json
    sys.path.insert(0, ROOT)
    import bench
    cases = [("syn_n512_d8", 512, 8, 2003), ("syn_n384_d16", 384, 16, 2004)]
    for name, n, d, seed in cases:
        g = golden(name)
        x, t, th = bench.synthetic(n, d, seed)
        assert np.array_equal(x, g["x"]) and np.array_equal(t, g["t"] - g["t"].mean()) and np.array_equal(th, g["theta"])
    code = ("import sys, json; sys.path.insert(0, %r); import bench; import numpy as np\n"
            "f, g, kind = bench._reference_callables()\n"
            "out = [kind]\n"
            "for n, d, seed in %r:\n"
            "    x, t, th = bench.synthetic(n, d, seed)\n"
            "    out.append([float(f(x, t, th)), [float(v) for v in g(x, t, th)]])\n"
            "print(json.dumps(out))" % (ROOT, [c[1:] for c in cases]))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    installed = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "skgpuppy"))
    assert out[0] == ("reference" if installed else "port")
    for (name, _, _, _), (nll, grad) in zip(cases, out[1:]):
        g = golden(name)
        assert nll == pytest.approx(float(g["nll"]), rel=1e-12), name
        np.testing.assert_allclose(grad, g["grad"], rtol=1e-10, err_msg=name)
