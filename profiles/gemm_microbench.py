"""Back-to-back launches of one GEMM shape, CUDA-event timed: separates the per-launch fixed cost of the
tcgen05 kernel from its main loop.   python profiles/gemm_microbench.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import gic_b200  # noqa: E402
from gic_b200 import _lib as L  # noqa: E402

L.require_cuda()
lib = L.lib()
dev = torch.device("cuda:0")


def bench(mode, tA, tB, M, N, K, iters=200, beta=0.0):
    A = torch.randn((K, M) if tA else (M, K), device=dev)
    B = torch.randn((N, K) if tB else (K, N), device=dev)
    C = torch.zeros(M, N, device=dev)
    s = L.stream()

    def run():
        L.check(lib.gic_gemm(mode, tA, tB, M, N, K, 1.0, L.ptr(A), A.shape[1], L.ptr(B), B.shape[1], beta, L.ptr(C), N,
                             None, s), "gemm")
    for _ in range(10):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        run()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    tf = 2.0 * M * N * K / (us * 1e-6) / 1e12
    print(f"mode {mode} tA{tA} tB{tB} {M:6d}x{N:6d}x{K:6d} beta {beta}: {us:8.2f} us/launch  {tf:8.1f} TFLOP/s", flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "short":
        bench(1, 0, 0, 16384, 900, 900, beta=1.0)
        bench(1, 1, 0, 10000, 512, 5120)
        bench(1, 0, 0, 5120, 512, 10000)
        bench(1, 1, 0, 900, 900, 16384)
        bench(1, 0, 1, 16384, 900, 900)
        sys.exit(0)
    # decode
    bench(1, 0, 1, 256, 10000, 512)          # vocab projection, one step
    bench(1, 0, 1, 256, 2048, 512)           # gates, one operand
    bench(1, 0, 0, 256, 512, 2048)           # BPTT dh_rec = dG W_hh
    # discriminator
    bench(1, 0, 1, 16384, 900, 900)          # highway fwd
    bench(1, 0, 0, 16384, 900, 900, beta=1.0)  # dx += dh W_h
    bench(1, 1, 0, 900, 900, 16384)          # dW_h
    bench(1, 0, 1, 5120, 64, 10000)          # soft embedding
    bench(1, 1, 0, 64, 10000, 5120)          # dW_e
    bench(1, 0, 0, 5120, 10000, 64)          # dinp
    # generator backward
    bench(1, 1, 0, 10000, 512, 5120)         # dW_out
    bench(1, 0, 0, 5120, 512, 10000)         # dhtop
    bench(1, 1, 0, 2048, 512, 5120)          # dW_ih / dW_hh
    bench(1, 0, 0, 5120, 512, 2048)          # dX
    bench(1, 0, 1, 8192, 8192, 8192, iters=10)
    bench(1, 0, 1, 32768, 900, 900, iters=50)
