"""One K^-1 = X^T X shaped product (for ncu): python tools/probes/lauum_once.py [n] [position_lock]"""
import ctypes, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "scikit-gpuppy_b200"))
import torch
from skgpuppy import _native as nat
lib = nat.load()
n = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
lib.gpk_test_position_lock(int(sys.argv[2]) if len(sys.argv) > 2 else 2)
dev = torch.device("cuda:0")
g = torch.Generator(device=dev); g.manual_seed(0)
X = torch.randn(n, n, dtype=torch.float64, device=dev, generator=g).tril_()
C = torch.zeros(n, n, dtype=torch.float64, device=dev)
P = lambda t: ctypes.c_void_p(t.data_ptr())
ms = (ctypes.c_float * 2)()
nat.check(lib.gpk_test_oz_gemm(P(X), n, 1, 1, P(X), n, 1, 1, P(C), n, n, n, n, 1.0, 0.0, 4, 1, 16, 0, 1, ms,
                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "oz_gemm")
torch.cuda.synchronize()
print("n=%d residues %.2f ms gemm+reconstruction %.2f ms" % (n, ms[0], ms[1]))
