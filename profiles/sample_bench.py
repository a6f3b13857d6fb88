"""Sampled caption generation (gic_sample_captions, Decoder.sample_captions) at the c2 inference shape (B 256, L 20,
V 10 000, E = H = 512), one and two layers, n = 1 and 5 captions per image, GEMM modes tf32 and fp32, in ONE process:

  * sampling rate: ms per call, captions/s (B n per call) and row-steps/s (B n L), for top_k = 0 (full vocabulary) and
    top_k = 16 with top_p = 0.9, timed over >= 0.3 s of calls after warm-up (host clock around work that ends in a device
    synchronise);
  * alternated with it, three runs each, at the same row count B n:
      - Decoder.sample(u=torch.rand(L, B n, V)) (the training sampler: Gumbel-softmax output [B n, L, V] in fp32, no EOS,
        no filter, temperature 1 on the ids), the torch.rand included; full-vocabulary rows only;
      - a torch-ops path: the LSTM with F.linear (cuBLAS), z = F.linear(h, W_out, b_out), softmax(z / T) (over the top 16
        and its nucleus when filtered), torch.multinomial, PAD after EOS;
  * one sampling step alone (gic_vocab_sample at M = B n, CUDA events over many launches): the Gumbel producer
    (top_k = 0: vocab_gumbel_kernel, or row_gumbel_kernel in fp32) against the plain producer at the same M (top_k = 1:
    vocab_topk_kernel<4>, or row_topk_kernel), each followed by the same sample_rows_kernel, alternated three times,
    against the tensor bound 2 M H V flop at the data-sheet dense TF32 rate (a bound, not a reached peak);
  * the GPU name, power limit and max SM clock, read in the same call.
The producer's working set (W_out 20.5 MB, h <= 2.6 MB) fits the 126 MB L2: its numbers are close to L2-resident.  Prints
the results and writes sample_bench.json in $GIC_REPORT_DIR (default: the system's temporary directory)."""
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import gic_b200  # noqa: E402
from gic_b200 import _lib  # noqa: E402
from gic_b200.args import default_args  # noqa: E402
from gic_b200.generator import Decoder, lstm_split, sample_captions  # noqa: E402

TF32_PEAK = 1125e12            # NVIDIA HGX B200 data sheet, dense TF32, one GPU (1 000 W part)
MODES = {"tf32": gic_b200.GEMM_TF32, "fp32": gic_b200.GEMM_FP32}
SHAPE = dict(B=256, L=20, V=10000, E=512, H=512)
FILTERS = {"top_k0": (0, 1.0), "top_k16_top_p0.9": (16, 0.9)}
EOS = 2


def make_decoder(layers):
    """U(-0.2, 0.2) weights: the reference's U(-0.05, 0.05) init scaled so that the distributions are peaked as in a trained
    model (score_bench.py uses the same)."""
    s = SHAPE
    a = default_args(vocab_size=s["V"], gen_embed_dim=s["E"], gen_hidden_dim=s["H"], gen_num_layers=layers,
                     conditional_gan=0)
    dec = Decoder(a)
    g = torch.Generator().manual_seed(11 + layers)
    with torch.no_grad():
        for p in dec.parameters():
            p.copy_(torch.rand(p.shape, generator=g) * 0.4 - 0.2)
    dec.temperature = 1.0
    return dec.cuda()


def timed(fn, min_s=0.3):
    fn()
    torch.cuda.synchronize()
    n, t0 = 0, time.perf_counter()
    while True:
        fn()
        n += 1
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        if el >= min_s:
            return el / n


def torch_ops_sample(dec, x, L, T, k, p):
    """The same definition with torch ops (a different random stream): cuBLAS linears, softmax, multinomial, PAD after EOS."""
    W_ih, W_hh, b_ih, b_hh = lstm_split([w.detach() for w in dec.lstm_params()])
    emb, W_out, b_out = dec.embed.weight.detach(), dec.linear.weight.detach(), dec.linear.bias.detach()
    M = x.shape[0]
    H = W_out.shape[1]
    hs = [x.new_zeros(M, H) for _ in W_ih]
    cs = [x.new_zeros(M, H) for _ in W_ih]
    fin = torch.zeros(M, dtype=torch.bool, device=x.device)
    ids = torch.zeros(M, L, dtype=torch.int64, device=x.device)
    for t in range(L):
        inp = x
        for l in range(len(W_ih)):
            i, f, g, o = (F.linear(inp, W_ih[l], b_ih[l]) + F.linear(hs[l], W_hh[l], b_hh[l])).chunk(4, 1)
            cs[l] = torch.sigmoid(f) * cs[l] + torch.sigmoid(i) * torch.tanh(g)
            hs[l] = torch.sigmoid(o) * torch.tanh(cs[l])
            inp = hs[l]
        z = F.linear(inp, W_out, b_out)
        if k:
            v, cols = z.topk(k, dim=1)
            q = torch.softmax(v / T, 1)
            if p < 1:
                excl = q.cumsum(1) - q
                q = torch.where(excl < p, q, torch.zeros_like(q))
            tok = cols.gather(1, torch.multinomial(q, 1))[:, 0]
        else:
            tok = torch.multinomial(torch.softmax(z / T, 1), 1)[:, 0]
        ids[:, t] = torch.where(fin, torch.zeros_like(tok), tok)
        fin |= tok == EOS
        x = emb[tok]
    return ids


def step_ms(mode, h, dec, k, iters=100):
    lib = _lib.lib()
    M, H = h.shape
    V = dec.linear.weight.shape[0]
    tok = torch.empty(M, dtype=torch.int64, device="cuda")
    logp = torch.empty(M, device="cuda")
    ws = torch.empty(lib.gic_vocab_sample_workspace_floats(M, V, k), device="cuda")
    W, b = dec.linear.weight.detach(), dec.linear.bias.detach()

    def call():
        _lib.check(lib.gic_vocab_sample(mode, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), M, V, H, 0, 1.0, k, 1.0, _lib.ptr(tok),
                                        _lib.ptr(logp), _lib.ptr(ws), _lib.stream()), "gic_vocab_sample")
    tensor = mode != gic_b200.GEMM_FP32
    want = ("vocab_gumbel_kernel" if tensor else "row_gumbel_kernel") if k == 0 else \
        ("vocab_topk_kernel" if tensor else "row_topk_kernel")
    with _lib.expect_kernels(want, "sample_rows_kernel"):
        for _ in range(5):
            call()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        call()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, want


def main():
    _lib.require_cuda()
    from beam_bench import gpu_info
    out = dict(gpu=gpu_info(), shape=SHAPE, sample={}, step={})
    B, L, V, E, H = SHAPE["B"], SHAPE["L"], SHAPE["V"], SHAPE["E"], SHAPE["H"]
    torch.manual_seed(0)
    with torch.no_grad():
        for layers in (1, 2):
            dec = make_decoder(layers)
            feats = torch.randn(B, E, device="cuda")
            for n in (1, 5):
                M = B * n
                rows = feats.repeat_interleave(n, 0)
                for mname, mode in MODES.items():
                    torch.backends.cuda.matmul.allow_tf32 = (mname == "tf32")
                    gic_b200.set_gemm_mode(mode)
                    for fname, (k, p) in FILTERS.items():
                        _lib.lib().gic_set_rng(1, 0, None)

                        def lib_call():
                            return sample_captions(dec, feats, n, L, 1.0, k, p, EOS, mode=mode)

                        def train_call():
                            return dec.sample(rows, max_caption_len=L, u=torch.rand(L, M, V, device="cuda"))

                        def torch_call():
                            return torch_ops_sample(dec, rows, L, 1.0, k, p)
                        lib_s, tr_s, to_s = [], [], []
                        for _ in range(3):
                            lib_s.append(timed(lib_call))
                            if k == 0:
                                tr_s.append(timed(train_call))
                            to_s.append(timed(torch_call))
                        t = min(lib_s)
                        ids, _, lengths = lib_call()
                        key = "layers%d/n%d/%s/%s" % (layers, n, mname, fname)
                        r = dict(ms_per_call=1e3 * t, captions_per_s=M / t, row_steps_per_s=M * L / t,
                                 ms_all=[1e3 * x for x in lib_s], torch_ops_ms=1e3 * min(to_s),
                                 torch_ops_ms_all=[1e3 * x for x in to_s], speedup_over_torch_ops=min(to_s) / t,
                                 mean_length=float(lengths.float().mean()),
                                 distinct_captions=len({tuple(c) for c in ids.view(M, L).tolist()}))
                        if tr_s:
                            r.update(decoder_sample_ms=1e3 * min(tr_s), decoder_sample_ms_all=[1e3 * x for x in tr_s],
                                     speedup_over_decoder_sample=min(tr_s) / t)
                        out["sample"][key] = r
                        print(key, json.dumps(r), flush=True)
                    _lib.lib().gic_set_rng(0, 0, None)
                if layers == 1:
                    h = torch.rand(M, H, device="cuda") * 2 - 1
                    bound_ms = 2.0 * M * H * V / TF32_PEAK * 1e3
                    for mname, mode in MODES.items():
                        gum, plain = [], []
                        for _ in range(3):
                            ms, gk = step_ms(mode, h, dec, 0, iters=100 if mname == "tf32" else 20)
                            gum.append(ms)
                            ms, pk = step_ms(mode, h, dec, 1, iters=100 if mname == "tf32" else 20)
                            plain.append(ms)
                        r = dict(M=M, gumbel_producer=gk, gumbel_step_us=1e3 * min(gum), gumbel_us_all=[1e3 * x for x in gum],
                                 plain_producer=pk, plain_step_us=1e3 * min(plain), plain_us_all=[1e3 * x for x in plain],
                                 gumbel_over_plain=min(gum) / min(plain), tensor_bound_us=1e3 * bound_ms,
                                 bound="tensor (2 M H V flop at 1125 TFLOP/s dense TF32)",
                                 gumbel_share_of_tensor_bound=bound_ms / min(gum), plain_share_of_tensor_bound=bound_ms / min(plain),
                                 note="each time is one gic_vocab_sample call: the producer plus the same sample_rows_kernel")
                        out["step"]["n%d/%s" % (n, mname)] = r
                        print("step", "n%d/%s" % (n, mname), json.dumps(r), flush=True)
    gic_b200.set_gemm_mode(gic_b200.GEMM_FP32)
    rdir = os.environ.get("GIC_REPORT_DIR") or tempfile.gettempdir()
    os.makedirs(rdir, exist_ok=True)
    with open(os.path.join(rdir, "sample_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["gpu"]))


if __name__ == "__main__":
    main()
