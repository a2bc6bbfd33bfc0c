"""Launch one configuration a few times (for ncu).  usage: profile_one.py {gemv|gemm|skinny|imma} K N M [tune0 tune1 tune2]"""
import sys, os
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from autogptq_b200 import _lib
from tools.microbench import Layers

kind, K, N, M = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
tune = [int(v) for v in sys.argv[5:8]] + [0] * (3 - len(sys.argv[5:8]))
lib = _lib.load()
L = Layers(K, N, 128, 6, "cuda")
x = torch.randn(M, K, dtype=torch.float16, device="cuda")
y = torch.empty(M, N, dtype=torch.float16, device="cuda")
for it in range(2):
    for c in range(L.copies):
        rc = lib.agb200_w4a16_forward_ex(x.data_ptr(), L.qw[c].data_ptr(), L.qw_tc[c].data_ptr(), L.qz[c].data_ptr(), L.sc[c].data_ptr(), None, None,
                                         y.data_ptr(), M, K, N, 128, 0, None, 0, None, {"gemv": 1, "gemm": 2, "skinny": 3, "imma": 6}[kind], *tune)
        assert rc == 0, lib.agb200_last_error()
torch.cuda.synchronize()
print("ok")
