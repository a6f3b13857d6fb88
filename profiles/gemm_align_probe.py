"""Does the row pitch of the operands (multiple of 128 B or not) change the tcgen05 GEMM's k-block rate?"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import gic_b200
from gic_b200 import _lib as L
L.require_cuda(); lib = L.lib(); dev = torch.device("cuda:0")

def bench(M, N, K, lda, ldb, ldc, tB=1, beta=0.0, iters=100):
    A = torch.randn(M, lda, device=dev)
    B = torch.randn(N if tB else K, ldb, device=dev)
    C = torch.zeros(M, ldc, device=dev)
    s = L.stream()
    def run():
        L.check(lib.gic_gemm(1, 0, tB, M, N, K, 1.0, L.ptr(A), lda, L.ptr(B), ldb, beta, L.ptr(C), ldc, None, s), "gemm")
    for _ in range(5): run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters): run()
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    print(f"M{M} N{N} K{K} lda{lda} ldb{ldb} ldc{ldc} tB{tB} beta{beta}: {us:8.2f} us  {2.0*M*N*K/us/1e6:7.1f} TF/s", flush=True)

print("SK =", os.environ.get("GIC_SK"))
bench(18944, 1024, 1024, 1024, 1024, 1024)   # 148 x 4 tiles of 128 x 256: exactly 4 rounds
bench(18944, 1024, 4096, 4096, 4096, 1024)
