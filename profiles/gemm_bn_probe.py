"""Tile-width sweep of the persistent TF32 GEMM on one shape (option GIC_GEMM_BN)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import gic_b200
from gic_b200 import _lib as L
L.require_cuda(); lib = L.lib(); dev = torch.device("cuda:0")


def bench(mode, tA, tB, M, N, K, iters=100):
    A = torch.randn((K, M) if tA else (M, K), device=dev)
    B = torch.randn((N, K) if tB else (K, N), device=dev)
    C = torch.zeros(M, N, device=dev)
    s = L.stream()
    for bn in (0, 128, 192, 240, 256):
        L.set_option("GIC_GEMM_BN", bn)
        def run():
            L.check(lib.gic_gemm(mode, tA, tB, M, N, K, 1.0, L.ptr(A), A.shape[1], L.ptr(B), B.shape[1], 0.0, L.ptr(C), N, None, s), "gemm")
        for _ in range(5): run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters): run()
        e1.record(); torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / iters
        print(f"mode {mode} tA{tA} tB{tB} {M}x{N}x{K} BN {bn or 'auto':>4}: {us:7.1f} us", flush=True)
    L.clear_option("GIC_GEMM_BN")


bench(1, 0, 1, 10000, 2048, 512)
bench(1, 0, 1, 8192, 2048, 512)
bench(1, 0, 1, 8192, 8192, 512)
