"""Teacher-forced caption scoring (gic_score_captions, Decoder.score) at the c2 shape (B 256, L 20, V 10 000, E = H = 512,
one and two layers) and the per-GPU shape of c4 (B 128, L 20, V 30 000, E 512, H 1 024), GEMM modes tf32 and fp32, in ONE
process:

  * scoring rate: ms per call, captions/s and tokens/s (B L per call), timed over >= 0.3 s of calls after warm-up (host
    clock around work that ends in a device synchronise);
  * the composed path a user would otherwise write -- Decoder.sample(pretrain=True, forced_ids=captions), which writes the
    [B, L, V] logits, then torch log_softmax + gather -- alternated with the scoring call, three runs each;
  * the target-logit producer alone (gic_vocab_target_logp at M = B L, CUDA events over many launches): the fused tcgen05
    kernel (vocab_topk_kernel with the target pick) against the unfused path (tcgen05 GEMM to memory + row_topk_kernel,
    option GIC_FUSED_TOPK = 0), alternated three times each, against the tensor bound 2 M H V flop at the data-sheet dense
    TF32 rate (a bound, not a reached peak);
  * with --beam, beam_bench.py's measurements in the same process (the producer is shared with beam search);
  * the GPU name, power limit and max SM clock, read in the same call.
Algorithmic work per call: c2 52.4 GF of projection + 21.5 GF of recurrence (one layer) and 205 MB of logits not written;
c4 157 GF of projection, 307 MB of logits.  The producer's working set (W_out 40 / 123 MB, h 10.5 MB) is at or below the
126 MB L2: its numbers are close to L2-resident.  Prints the results and writes score_bench.json in $GIC_REPORT_DIR (default:
the system's temporary directory)."""
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
from gic_b200.generator import Decoder, score_captions  # noqa: E402

TF32_PEAK = 1125e12            # NVIDIA HGX B200 data sheet, dense TF32, one GPU (1 000 W part)
MODES = {"tf32": gic_b200.GEMM_TF32, "fp32": gic_b200.GEMM_FP32}
SHAPES = {"c2/layers1": dict(B=256, L=20, V=10000, E=512, H=512, layers=1),
          "c2/layers2": dict(B=256, L=20, V=10000, E=512, H=512, layers=2),
          "c4/layers1": dict(B=128, L=20, V=30000, E=512, H=1024, layers=1)}


def make_decoder(s):
    """U(-0.2, 0.2) weights: the reference's U(-0.05, 0.05) init scaled so that the distributions are peaked as in a trained
    model."""
    a = default_args(vocab_size=s["V"], gen_embed_dim=s["E"], gen_hidden_dim=s["H"], gen_num_layers=s["layers"],
                     conditional_gan=0)
    dec = Decoder(a)
    g = torch.Generator().manual_seed(11 + s["layers"])
    with torch.no_grad():
        for p in dec.parameters():
            p.copy_(torch.rand(p.shape, generator=g) * 0.4 - 0.2)
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


def producer_ms(mode, h, tgt, dec, fused, iters=100):
    lib = _lib.lib()
    M, H = h.shape
    V = dec.linear.weight.shape[0]
    logp = torch.empty(M, device="cuda")
    ws = torch.empty(lib.gic_vocab_target_logp_workspace_floats(M, V), device="cuda")
    W, b = dec.linear.weight.detach(), dec.linear.bias.detach()

    def call():
        _lib.check(lib.gic_vocab_target_logp(mode, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), _lib.ptr(tgt), M, V, H,
                                             _lib.ptr(logp), None, None, _lib.ptr(ws), _lib.stream()), "gic_vocab_target_logp")
    with _lib.options(GIC_FUSED_TOPK=1 if fused else 0):
        want = "vocab_topk_kernel" if fused and mode != gic_b200.GEMM_FP32 else "row_topk_kernel"
        with _lib.expect_kernels(want):
            for _ in range(5):
                call()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            call()
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, logp.clone()


def main():
    _lib.require_cuda()
    from beam_bench import gpu_info
    out = dict(gpu=gpu_info(), shapes=SHAPES, score={}, producer={})
    torch.manual_seed(0)
    with torch.no_grad():
        for name, s in SHAPES.items():
            B, L, V, E, H = s["B"], s["L"], s["V"], s["E"], s["H"]
            dec = make_decoder(s)
            feats = torch.randn(B, E, device="cuda")
            caps = torch.randint(3, V, (B, L), device="cuda")
            for mname, mode in MODES.items():
                torch.backends.cuda.matmul.allow_tf32 = (mname == "tf32")
                gic_b200.set_gemm_mode(mode)

                def fused_call():
                    return score_captions(dec, feats, caps, None, mode=mode)

                def composed_call():
                    logits, _ = dec.sample(feats, pretrain=True, max_caption_len=L, forced_ids=caps)
                    return F.log_softmax(logits, -1).gather(2, caps[:, :, None])[:, :, 0]
                lib_s, comp_s = [], []
                for _ in range(3):
                    lib_s.append(timed(fused_call))
                    comp_s.append(timed(composed_call))
                t = min(lib_s)
                a, c = fused_call()[0], composed_call()
                key = "%s/%s" % (name, mname)
                out["score"][key] = dict(ms_per_call=1e3 * t, captions_per_s=B / t, tokens_per_s=B * L / t,
                                         ms_all=[1e3 * x for x in lib_s], composed_ms=1e3 * min(comp_s),
                                         composed_ms_all=[1e3 * x for x in comp_s], speedup_over_composed=min(comp_s) / t,
                                         max_abs_logp_diff_vs_composed=float((a - c).abs().max()))
                print(key, json.dumps(out["score"][key]), flush=True)
            gic_b200.set_gemm_mode(gic_b200.GEMM_FP32)
            if s["layers"] == 1:
                M = B * L
                h = (torch.rand(M, H, device="cuda") * 2 - 1)
                tgt = caps.reshape(-1).contiguous()
                bound_ms = 2.0 * M * H * V / TF32_PEAK * 1e3
                fz, un = [], []
                for _ in range(3):
                    ms, a = producer_ms(gic_b200.GEMM_TF32, h, tgt, dec, True)
                    fz.append(ms)
                    ms, b_ = producer_ms(gic_b200.GEMM_TF32, h, tgt, dec, False)
                    un.append(ms)
                fp32_ms, _ = producer_ms(gic_b200.GEMM_FP32, h, tgt, dec, False, iters=20)
                out["producer"][name] = dict(
                    M=M, fused_tcgen05_us=1e3 * min(fz), fused_us_all=[1e3 * x for x in fz],
                    unfused_tcgen05_gemm_plus_row_topk_us=1e3 * min(un), unfused_us_all=[1e3 * x for x in un],
                    exact_fp32_gemm_plus_row_topk_us=1e3 * fp32_ms, tensor_bound_us=1e3 * bound_ms,
                    bound="tensor (2 M H V flop at 1125 TFLOP/s dense TF32)", fused_share_of_tensor_bound=bound_ms / min(fz),
                    fused_over_unfused=min(fz) / min(un), max_abs_logp_diff_fused_vs_unfused=float((a - b_).abs().max()))
                print("producer", name, json.dumps(out["producer"][name]), flush=True)
    rdir = os.environ.get("GIC_REPORT_DIR") or tempfile.gettempdir()
    os.makedirs(rdir, exist_ok=True)
    with open(os.path.join(rdir, "score_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["gpu"]))
    if "--beam" in sys.argv:
        import beam_bench
        beam_bench.main()


if __name__ == "__main__":
    main()
