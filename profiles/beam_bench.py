"""Beam-search generation at the c2 inference shape (B 256, L 20, V 10 000, E = H = 512), layers 1 and 2, K in {1, 3, 5},
GEMM modes tf32 and fp32, in ONE process:

  * decode rate: captions/s and generated row-steps/s (B K L per decode), gic_decode_beam timed over >= 1 s of decodes after
    warm-up (host clock around work that ends in a device synchronise);
  * candidate producer: per-call time of gic_vocab_topk at M = B K with CUDA events over many launches, the fused
    tcgen05 kernel (vocab_topk_kernel) against the unfused path (tcgen05 GEMM to memory + row_topk_kernel, option
    GIC_FUSED_TOPK = 0), each against the tensor bound 2 M H V flop at the data-sheet dense TF32 rate;
  * the same decode built from torch ops on the same GPU (cuBLAS linear to HBM + log_softmax + topk + the same selection
    rule), run alternately with the library's in the same call, and the fraction of images whose best caption is identical;
  * the GPU name and power limit, read in the same call.
The working set (W_out 40 MB, h 2.6 MB) fits the 126 MB L2: the producer numbers are L2-resident steady state, as in a
decode loop.  Prints the results and writes them to beam_bench.json in $GIC_REPORT_DIR (default: the system's temporary
directory)."""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import gic_b200  # noqa: E402
from gic_b200 import _lib  # noqa: E402
from gic_b200.args import default_args  # noqa: E402
from gic_b200.generator import Decoder, decode_beam  # noqa: E402

B, L, V, E, H = 256, 20, 10000, 512, 512
TF32_PEAK = 1125e12            # NVIDIA HGX B200 data sheet, dense TF32, one GPU (1 000 W part)
MODES = {"tf32": gic_b200.GEMM_TF32, "fp32": gic_b200.GEMM_FP32}


def gpu_info():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else "unavailable"
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = "unavailable (%s)" % e
    return info


def make_decoder(layers):
    """U(-0.2, 0.2) weights (the reference's U(-0.05, 0.05) init, scaled so that the distributions are peaked as in a trained
    model) and a raised <E> bias, so that beams finish and freeze during the decode."""
    a = default_args(vocab_size=V, gen_embed_dim=E, gen_hidden_dim=H, gen_num_layers=layers, conditional_gan=0)
    dec = Decoder(a)
    g = torch.Generator().manual_seed(11 + layers)
    with torch.no_grad():
        for p in dec.parameters():
            p.copy_(torch.rand(p.shape, generator=g) * 0.4 - 0.2)
        dec.linear.bias[2] += 3.0
    return dec.cuda()


def torch_beam(dec, feats, K, eos=2):
    """The same search from torch ops: LSTM cell, cuBLAS vocab projection to memory, log_softmax, per-beam topk, the image's
    K best (stable sort: higher score, then lower parent, then lower token), frozen beams extended by PAD."""
    layers = dec.lstm.num_layers
    W = [(getattr(dec.lstm, f"weight_ih_l{l}"), getattr(dec.lstm, f"weight_hh_l{l}"), getattr(dec.lstm, f"bias_ih_l{l}"),
          getattr(dec.lstm, f"bias_hh_l{l}")) for l in range(layers)]
    BK = B * K
    hs = [feats.new_zeros(BK, H) for _ in range(layers)]
    cs = [feats.new_zeros(BK, H) for _ in range(layers)]
    x = feats.repeat_interleave(K, 0)
    score = torch.full((B, K), -float("inf"), device="cuda")
    score[:, 0] = 0
    fin = torch.zeros(B, K, dtype=torch.bool, device="cuda")
    trace_p, trace_t = [], []
    ar = torch.arange(B, device="cuda")[:, None]
    for t in range(L):
        inp = x
        for l in range(layers):
            g = F.linear(inp, W[l][0], W[l][2]) + F.linear(hs[l], W[l][1], W[l][3])
            i, f, gg, o = g.chunk(4, 1)
            cs[l] = torch.sigmoid(f) * cs[l] + torch.sigmoid(i) * torch.tanh(gg)
            hs[l] = torch.sigmoid(o) * torch.tanh(cs[l])
            inp = hs[l]
        logp = F.log_softmax(F.linear(inp, dec.linear.weight, dec.linear.bias), -1)
        v, w = torch.topk(logp, K, dim=1)
        cand = score[:, :, None] + v.view(B, K, K)
        tok = w.view(B, K, K)
        frozen_cand = torch.full_like(cand, -float("inf"))
        frozen_cand[:, :, 0] = score
        cand = torch.where(fin[:, :, None], frozen_cand, cand)
        tok = torch.where(fin[:, :, None], torch.zeros_like(tok), tok)
        order = torch.sort(cand.view(B, K * K), dim=1, descending=True, stable=True).indices[:, :K]
        par = order // K
        ntok = tok.view(B, K * K).gather(1, order)
        score = cand.view(B, K * K).gather(1, order)
        fin = fin.gather(1, par) | (ntok == eos)
        rows = (ar * K + par).reshape(-1)
        hs = [h[rows] for h in hs]
        cs = [c[rows] for c in cs]
        x = dec.embed.weight[ntok.reshape(-1)]
        trace_p.append(par)
        trace_t.append(ntok)
    best = score.argmax(1)          # length penalty 0: the best beam is the highest score (lowest slot on ties)
    ids = torch.zeros(B, L, dtype=torch.int64, device="cuda")
    slot = best
    for t in range(L - 1, -1, -1):
        ids[:, t] = trace_t[t].gather(1, slot[:, None])[:, 0]
        slot = trace_p[t].gather(1, slot[:, None])[:, 0]
    return ids


def timed(fn, min_s=1.0):
    fn()
    torch.cuda.synchronize()
    n, t0 = 0, time.perf_counter()
    while True:
        fn()
        n += 1
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        if el >= min_s:
            return el / n, n


def producer_ms(mode, h, dec, K, fused, iters=200):
    lib = _lib.lib()
    M = h.shape[0]
    logp = torch.empty(M, K, device="cuda")
    tok = torch.empty(M, K, dtype=torch.int64, device="cuda")
    ws = torch.empty(lib.gic_vocab_topk_workspace_floats(M, V, K), device="cuda")
    W, b = dec.linear.weight.detach(), dec.linear.bias.detach()

    def call():
        _lib.check(lib.gic_vocab_topk(mode, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), M, V, H, K, _lib.ptr(logp), _lib.ptr(tok),
                                      None, _lib.ptr(ws), _lib.stream()), "gic_vocab_topk")
    with _lib.options(GIC_FUSED_TOPK=1 if fused else 0):
        want = "vocab_topk_kernel" if fused else "row_topk_kernel"
        with _lib.expect_kernels(want):
            for _ in range(10):
                call()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            call()
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (logp.clone(), tok.clone())


def main():
    _lib.require_cuda()
    out = dict(gpu=gpu_info(), shape=dict(B=B, L=L, V=V, E=E, H=H), decode={}, producer={}, torch_ops={})
    torch.manual_seed(0)
    feats = torch.randn(B, E, device="cuda")
    with torch.no_grad():
        for layers in (1, 2):
            dec = make_decoder(layers)
            for mname, mode in MODES.items():
                torch.backends.cuda.matmul.allow_tf32 = (mname == "tf32")
                for K in (1, 3, 5):
                    key = "%s/layers%d/K%d" % (mname, layers, K)
                    # library decode and torch-ops decode, alternated three times in this call
                    lib_s, tor_s = [], []
                    for _ in range(3):
                        s, n = timed(lambda: decode_beam(dec, feats, K, L, 0.0, 2, mode=mode))
                        lib_s.append(s)
                        s2, _ = timed(lambda: torch_beam(dec, feats, K), min_s=0.5)
                        tor_s.append(s2)
                    s = min(lib_s)
                    out["decode"][key] = dict(ms_per_decode=1e3 * s, captions_per_s=B / s, row_steps_per_s=B * K * L / s,
                                              decodes_timed=n, ms_all=[1e3 * x for x in lib_s])
                    ids = decode_beam(dec, feats, K, L, 0.0, 2, mode=mode)[0][:, 0]
                    tids = torch_beam(dec, feats, K)
                    out["torch_ops"][key] = dict(ms_per_decode=1e3 * min(tor_s), ms_all=[1e3 * x for x in tor_s],
                                                 speedup=min(tor_s) / s,
                                                 identical_best_caption=float((ids == tids).all(1).float().mean()))
                    print(key, json.dumps(out["decode"][key]), json.dumps(out["torch_ops"][key]), flush=True)
            # candidate producer at M = B K on the decoder's own last hidden state shape (random rows)
            if layers == 1:
                for K in (1, 3, 5):
                    M = B * K
                    h = torch.randn(M, H, device="cuda").clamp(-1, 1)
                    bound_ms = 2.0 * M * H * V / TF32_PEAK * 1e3
                    fused_ms, a = producer_ms(gic_b200.GEMM_TF32, h, dec, K, True)
                    unfused_ms, b_ = producer_ms(gic_b200.GEMM_TF32, h, dec, K, False)
                    fused_ms2, _ = producer_ms(gic_b200.GEMM_TF32, h, dec, K, True)
                    fp32_ms, _ = producer_ms(gic_b200.GEMM_FP32, h, dec, K, False, iters=50)
                    out["producer"]["K%d" % K] = dict(
                        M=M, fused_tcgen05_us=1e3 * min(fused_ms, fused_ms2), unfused_tcgen05_gemm_plus_row_topk_us=1e3 * unfused_ms,
                        exact_fp32_gemm_plus_row_topk_us=1e3 * fp32_ms, tensor_bound_us=1e3 * bound_ms,
                        bound="tensor (2 M H V flop at 1125 TFLOP/s dense TF32)",
                        fused_share_of_tensor_bound=bound_ms / min(fused_ms, fused_ms2),
                        same_tokens_fused_vs_unfused=float((a[1] == b_[1]).float().mean()))
                    print("producer K%d" % K, json.dumps(out["producer"]["K%d" % K]), flush=True)
    rdir = os.environ.get("GIC_REPORT_DIR") or tempfile.gettempdir()
    os.makedirs(rdir, exist_ok=True)
    with open(os.path.join(rdir, "beam_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["gpu"]))


if __name__ == "__main__":
    main()
