"""tcgen05 kind::tf32 GEMM on the C5 training step's shapes: correctness of the four operand orders (ragged sizes), then
time and the HBM bandwidth of the algorithmic bytes (read A, read B, write C once)."""
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arreau_b200 import _lib  # noqa: E402

dev = torch.device("cuda")
partial = torch.empty(8 << 20, device=dev)
s = torch.cuda.current_stream().cuda_stream


def run(ak, bk, A, B, Cm, M, N, K, tf32=1):
    _lib.call("arreau_sgemm", ak | (2 * tf32), bk, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), Cm.data_ptr(), N, M, N, K,
              C.c_float(1.0), None, 0, partial.data_ptr(), partial.numel(), s)


def check(M, N, K, ak, bk):
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    A = torch.randn((M, K) if ak else (K, M), generator=g).to(dev)
    B = torch.randn((N, K) if bk else (K, N), generator=g).to(dev)
    ref = (A.double() if ak else A.double().T) @ (B.double().T if bk else B.double())
    Cm = torch.zeros(M, N, device=dev)
    run(ak, bk, A, B, Cm, M, N, K)
    torch.cuda.synchronize()
    return f"{float((Cm.double() - ref).abs().max() / ref.abs().max()):.2e}"


for (M, N, K) in ((256, 256, 512), (300, 128, 96), (76, 132, 100), (128, 16, 36), (1000, 512, 8), (640, 256, 20000)):
    print(f"M={M} N={N} K={K}: " + ", ".join(f"({ak},{bk}) {check(M, N, K, ak, bk)}" for ak in (1, 0) for bk in (1, 0)), flush=True)
# how the operands reach TF32: 1 + 0.75 * 2^-10 rounds to 1 + 2^-10 (nearest) or 1 (truncation)
for ak, bk in ((1, 1), (1, 0), (0, 1), (0, 0)):
    M, N, K = 128, 128, 64
    A = torch.full((M, K) if ak else (K, M), 1.0 + 0.75 * 2.0 ** -10, device=dev)
    B = torch.ones((N, K) if bk else (K, N), device=dev)
    Cm = torch.zeros(M, N, device=dev)
    run(ak, bk, A, B, Cm, M, N, K)
    torch.cuda.synchronize()
    print(f"rounding probe ({ak},{bk}): C[0,0] / K = {float(Cm[0, 0]) / K:.8f} (nearest {1 + 2.0 ** -10:.8f}, truncation 1.0), uniform {bool((Cm == Cm[0, 0]).all())}", flush=True)
Re, Rn = 284928, 35616
shapes = [("z1 = mono W1^T", Re, 128, 128, 1, 1), ("z2 = a1 W2^T", Re, 256, 128, 1, 1), ("kernels = kb Wk^T (5 layers)", Re, 640, 256, 1, 1),
          ("dWk = dkern^T kb", 640, 256, Re, 0, 0), ("dz2 = dkern Wk", Re, 256, 640, 1, 0), ("dW2 = dz2^T a1", 256, 128, Re, 0, 0),
          ("dz1 = dz2 W2", Re, 128, 256, 1, 0), ("dW1 = dz1^T mono", 128, 128, Re, 0, 0), ("MLP z = y W1^T", Rn, 512, 128, 1, 1),
          ("MLP m = a W2^T", Rn, 128, 512, 1, 1), ("MLP dz = dm W2", Rn, 512, 128, 1, 0), ("MLP dy = dz W1", Rn, 128, 512, 1, 0),
          ("MLP dW2 = dm^T a", 128, 512, Rn, 0, 0), ("MLP dW1 = dz^T y", 512, 128, Rn, 0, 0)]
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
tot = 0.0
for name, M, N, K, ak, bk in shapes:
    A = torch.randn((M, K) if ak else (K, M), device=dev)
    B = torch.randn((N, K) if bk else (K, N), device=dev)
    Cm = torch.zeros(M, N, device=dev)
    run(ak, bk, A, B, Cm, M, N, K)
    ts = []
    for _ in range(5):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(ak, bk, A, B, Cm, M, N, K)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = sorted(ts)[len(ts) // 2]
    gb = 4.0 * (M * K + N * K + M * N) / 1e9
    tot += ms
    print(f"{name:32s} M={M:6d} N={N:4d} K={K:6d}: {ms * 1e3:6.0f} us  {gb / ms:6.2f} TB/s  {2.0 * M * N * K / ms / 1e9:5.0f} TFLOP/s", flush=True)
print(f"sum {tot * 1e3:.0f} us")
