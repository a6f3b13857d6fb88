"""Constrained caption generation at the c2 inference shape (B 256, L 20, V 10 000, E = H = 512), one and two layers, TF32,
in ONE process:

  * per call (host clock around work that ends in a device synchronise, >= 0.3 s of calls after warm-up), three variants
    alternated three times:
      (a) the unconstrained call (gic_decode_beam_constrained / gic_sample_captions_constrained with NULL constraints, the
          path of gic_decode_beam / gic_sample_captions);
      (b) the constrained call with constraints that never bind (min_length 1, no_repeat_ngram_size L + 1, bad ids
          outside [0, V)): the ban bitmap is built and every producer is the masked one;
      (c) typical constraints: min_length 5, no_repeat_ngram_size 3, bad_ids {0, 1, 3};
    for beam search K = 1 / 3 / 5 and sampling n = 1 / 5 at top_k = 0 and at top_k = 16, top_p = 0.9;
  * one step alone at M = 1280 rows (CUDA events over many launches): the unmasked and the masked producer + consumer
    (gic_vocab_topk(_masked) at K = 5, gic_vocab_sample(_masked) at top_k = 0), alternated three times;
  * the mean ban_rows_kernel time per launch (torch.profiler, in a pass of its own after the timed ones);
  * the GPU name, power limit and max SM clock, read in the same call.
Prints the results and writes constrain_bench.json in $GIC_REPORT_DIR (default: the system's temporary directory)."""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import gic_b200  # noqa: E402
from gic_b200 import _lib  # noqa: E402
from gic_b200.args import default_args  # noqa: E402
from gic_b200.generator import Decoder, decode_beam, sample_captions  # noqa: E402

SHAPE = dict(B=256, L=20, V=10000, E=512, H=512)
MODE = gic_b200.GEMM_TF32
VARIANTS = {"a_unconstrained": {},
            "b_non_binding": dict(min_length=1, no_repeat_ngram_size=SHAPE["L"] + 1, bad_ids=[-1, SHAPE["V"]]),
            "c_typical": dict(min_length=5, no_repeat_ngram_size=3, bad_ids=[0, 1, 3])}
CALLS = [("beam_K%d" % K, dict(K=K)) for K in (1, 3, 5)] + \
        [("sample_n%d_%s" % (n, f), dict(n=n, k=k, p=p)) for n in (1, 5) for f, (k, p) in
         (("top_k0", (0, 1.0)), ("top_k16_top_p0.9", (16, 0.9)))]


def make_decoder(layers):
    """U(-0.2, 0.2) weights, as sample_bench.py and score_bench.py use (peaked distributions, as in a trained model)."""
    s = SHAPE
    a = default_args(vocab_size=s["V"], gen_embed_dim=s["E"], gen_hidden_dim=s["H"], gen_num_layers=layers,
                     conditional_gan=0)
    dec = Decoder(a)
    g = torch.Generator().manual_seed(11 + layers)
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


def call(dec, feats, c, cons):
    L = SHAPE["L"]
    if "K" in c:
        return lambda: decode_beam(dec, feats, c["K"], L, 0.0, 2, mode=MODE, **cons)
    return lambda: sample_captions(dec, feats, c["n"], L, 1.0, c["k"], c["p"], 2, mode=MODE, **cons)


def step_events(dec, reps=200):
    """ms per launch of one step's producer + consumer at M = B * 5 rows, unmasked vs masked (empty bitmap)."""
    lib = _lib.lib()
    M, V, H = SHAPE["B"] * 5, SHAPE["V"], SHAPE["H"]
    h = torch.randn(M, H, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)) * 0.5
    W, b = dec.linear.weight.detach(), dec.linear.bias.detach()
    ban = torch.zeros(M, (V + 31) // 32, dtype=torch.int32, device="cuda")
    ban[:, 0] = 0b1011                                       # PAD, <S>, <UNK>
    K = 5
    logp, tok = torch.empty(M, K, device="cuda"), torch.empty(M, K, dtype=torch.int64, device="cuda")
    wsk = torch.empty(lib.gic_vocab_topk_workspace_floats(M, V, K), device="cuda")
    wss = torch.empty(lib.gic_vocab_sample_workspace_floats(M, V, 0), device="cuda")
    P = lambda t: _lib.ptr(t)  # noqa: E731
    fns = {
        "topk_K5": lambda: lib.gic_vocab_topk(MODE, P(h), P(W), P(b), M, V, H, K, P(logp), P(tok), None, P(wsk), _lib.stream()),
        "topk_K5_masked": lambda: lib.gic_vocab_topk_masked(MODE, P(h), P(W), P(b), M, V, H, K, P(logp), P(tok), None, P(ban),
                                                            P(wsk), _lib.stream()),
        "sample_top_k0": lambda: lib.gic_vocab_sample(MODE, P(h), P(W), P(b), M, V, H, 0, 1.0, 0, 1.0, P(tok), P(logp),
                                                      P(wss), _lib.stream()),
        "sample_top_k0_masked": lambda: lib.gic_vocab_sample_masked(MODE, P(h), P(W), P(b), M, V, H, 0, 1.0, 0, 1.0, P(tok),
                                                                    P(logp), P(ban), P(wss), _lib.stream()),
    }
    out = {k: [] for k in fns}
    for _ in range(3):
        for k, f in fns.items():
            f()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                f()
            e1.record()
            torch.cuda.synchronize()
            out[k].append(e0.elapsed_time(e1) / reps)
    return out


def ban_rows_time(dec, feats):
    """Mean device time per launch of ban_rows_kernel and of the masked producers in a typical constrained beam (K = 5)
    and sampling (n = 5) call (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    fns = [call(dec, feats, dict(K=5), VARIANTS["c_typical"]), call(dec, feats, dict(n=5, k=0, p=1.0), VARIANTS["c_typical"])]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for f in fns:
            f()
        torch.cuda.synchronize()
    res = {}
    for ev in prof.key_averages():
        for name in ("ban_rows_kernel", "ban_base_kernel", "vocab_topk_ban_kernel", "vocab_gumbel_ban_kernel", "beam_merge_kernel",
                     "sample_rows_kernel"):
            if name in ev.key:
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                r = res.setdefault(name, dict(us_total=0.0, launches=0))
                r["us_total"] += t
                r["launches"] += ev.count
    for r in res.values():
        r["us_per_launch"] = r["us_total"] / max(r["launches"], 1)
    return res


def main():
    _lib.require_cuda()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = dict(gpu=gpu, shape=SHAPE, mode="tf32", calls={}, step_ms={}, ban_rows={})
    for layers in (1, 2):
        dec = make_decoder(layers)
        feats = dec.embed.weight.detach()[1].expand(SHAPE["B"], SHAPE["E"]).contiguous()
        for cname, c in CALLS:
            ms = {v: [] for v in VARIANTS}
            for _ in range(3):
                for v, cons in VARIANTS.items():
                    ms[v].append(1e3 * timed(call(dec, feats, c, cons)))
            rows = SHAPE["B"] * c.get("K", c.get("n"))
            key = "layers%d/%s" % (layers, cname)
            res["calls"][key] = {v: dict(ms=x, ms_min=min(x), captions_per_s=rows / (min(x) * 1e-3)) for v, x in ms.items()}
            a = min(ms["a_unconstrained"])
            print("%-32s " % key + "  ".join("%s %.3f ms (%+.1f%%)" % (v[0], min(x), 100 * (min(x) / a - 1))
                                             for v, x in ms.items()), flush=True)
        if layers == 1:
            res["step_ms"] = step_events(dec)
            res["ban_rows"] = ban_rows_time(dec, feats)
    for k, v in res["step_ms"].items():
        print("step %-22s %.4f ms (min of 3)" % (k, min(v)))
    for k, v in res["ban_rows"].items():
        print("profiler %-24s %.2f us/launch over %d launches" % (k, v["us_per_launch"], v["launches"]))
    print("gpu:", gpu)
    out = os.environ.get("GIC_REPORT_DIR") or tempfile.gettempdir()
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "constrain_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
