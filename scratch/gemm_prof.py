"""clock64 phase accounting of the persistent tcgen05 GEMM (CTA medians) on a few of the C5 step's shapes."""
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arreau_b200 import _lib  # noqa: E402

dev = torch.device("cuda")
lib = _lib.load()
lib.arreau_debug_set_gemm_prof.argtypes = [C.c_void_p]
partial = torch.empty(8 << 20, device=dev)
s = torch.cuda.current_stream().cuda_stream
prof = torch.zeros(148, 16, dtype=torch.int64, device=dev)
Re, Rn = 284928, 35616
shapes = [("z1 = mono W1^T", Re, 128, 128, 1, 1), ("kernels = kb Wk^T", Re, 640, 256, 1, 1), ("dWk = dkern^T kb", 640, 256, Re, 0, 0),
          ("dz2 = dkern Wk", Re, 256, 640, 1, 0), ("dW1 = dz1^T mono", 128, 128, Re, 0, 0), ("MLP z = y W1^T", Rn, 512, 128, 1, 1)]
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
names = ["P:wait empty", "P:issue", "P:slabs", "M:wait tmem", "M:wait full", "M:issue", "E:wait acc", "E:store"]
for name, M, N, K, ak, bk in shapes:
    A = torch.randn((M, K) if ak else (K, M), device=dev)
    B = torch.randn((N, K) if bk else (K, N), device=dev)
    Cm = torch.zeros(M, N, device=dev)
    for it in range(2):
        flush.zero_()
        prof.zero_()
        lib.arreau_debug_set_gemm_prof(prof.data_ptr() if it else None)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.call("arreau_sgemm", ak | 2, bk, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), Cm.data_ptr(), N, M, N, K,
                  C.c_float(1.0), None, 0, partial.data_ptr(), partial.numel(), s)
        e1.record()
        torch.cuda.synchronize()
    lib.arreau_debug_set_gemm_prof(None)
    med = prof.double().median(dim=0).values.tolist()
    print(f"{name}: {e0.elapsed_time(e1) * 1e3:.0f} us; CTA medians (cycles): " +
          ", ".join(f"{n} {int(v)}" for n, v in zip(names, med)), flush=True)
