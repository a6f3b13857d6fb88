"""Beam-search caption generation (EXTENSION, parity unpinned by reference) on the GPU against oracle/ref_ext.py
beam_search: the vocab top-K producer against float64, the exact-fp32 decode against the oracle bit for bit, the
tensor-core decode at the c2 inference shape step by step through its trace (differences classified as tie / rounding /
real, real must be 0), greedy K = 1 against Decoder.sample(pretrain=True), GANInstructor.generate and CUDA-graph capture.
Counts go to beam_report.json in $GIC_REPORT_DIR (default: the system's temporary directory)."""
import json
import os
import tempfile

import pytest
import torch
import torch.nn.functional as F

from oracle import ref_beam as rx
from oracle import ref_port as rp

pytestmark = pytest.mark.gpu
REPORT = {}
MODES = {"fp32": 0, "tf32": 1, "bf16": 3}
U_TC = 2.0 ** -10                      # TF32 operand rounding


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    out = os.environ.get("GIC_REPORT_DIR") or tempfile.gettempdir()
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "beam_report.json"), "w") as f:
        json.dump(REPORT, f, indent=1, sort_keys=True)


def L_():
    import gic_b200  # noqa: F401
    from gic_b200 import _lib
    _lib.require_cuda()
    return _lib


def u_of(mode, H):
    # exact-fp32 mode: the FFMA sum of H products, ~sqrt(H) roundings of 2^-24 each
    return U_TC if mode else max(1e-6, 2.0 ** -24 * 2.0 * H ** 0.5)


def vocab_topk(mode, h, W, b, K):
    _lib = L_()
    lib = _lib.lib()
    M, H = h.shape
    V = W.shape[0]
    logp = torch.empty(M, K, device="cuda")
    tok = torch.empty(M, K, dtype=torch.int64, device="cuda")
    lse = torch.empty(M, device="cuda")
    ws = torch.empty(lib.gic_vocab_topk_workspace_floats(M, V, K), device="cuda")
    _lib.check(lib.gic_vocab_topk(mode, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), M, V, H, K, _lib.ptr(logp), _lib.ptr(tok),
                                  _lib.ptr(lse), _lib.ptr(ws), _lib.stream()), "gic_vocab_topk")
    return logp, tok, lse


@pytest.mark.parametrize("mode_name", list(MODES))
@pytest.mark.parametrize("M,V,H,K", [(7, 50, 32, 1), (128, 1000, 512, 5), (1280, 10000, 512, 5), (256, 30000, 1024, 16),
                                     (5, 60001, 64, 3)])
def test_vocab_topk_against_float64(mode_name, M, V, H, K):
    _lib = L_()
    mode = MODES[mode_name]
    g = torch.Generator(device="cuda").manual_seed(M + V + H + K)
    h = torch.randn(M, H, device="cuda", generator=g)
    W = torch.randn(V, H, device="cuda", generator=g) * (3.0 / H ** 0.5)
    b = torch.randn(V, device="cuda", generator=g) * 0.5
    aligned = V % 4 == 0 and H % 4 == 0
    want = "vocab_topk_kernel" if (mode != 0 and aligned) else "row_topk_kernel"
    with _lib.expect_kernels(want):
        logp, tok, lse = vocab_topk(mode, h, W, b, K)
        torch.cuda.synchronize()
    ref = h.double() @ W.double().t() + b.double()
    ref_lse = torch.logsumexp(ref, 1)
    ref_val, ref_tok = torch.topk(ref, K, dim=1)
    absprod = h.double().abs() @ W.double().abs().t()               # sum_k |h_k| |W[n,k]|
    scale = absprod.max(1).values + b.double().abs().max()
    u = u_of(mode, H)
    # token sets: a difference is rounding when the float64 gap at the K-th place is within the operand-rounding bound
    rounding = real = 0
    diff_rows = (torch.sort(tok, 1).values != torch.sort(ref_tok, 1).values).any(1).nonzero()[:, 0].tolist()
    for m in diff_rows:
        a = int(ref_tok[m, K - 1])
        for w in set(tok[m].tolist()) - set(ref_tok[m].tolist()):
            gap = float(ref[m, a] - ref[m, w])
            bound = 2 * u * float(absprod[m, a] + absprod[m, w]) + 1e-6 * float(scale[m])
            if gap <= bound:
                rounding += 1
            else:
                real += 1
    # logp of the tokens returned, and lse, within 4u of the scale
    ref_lp = (ref - ref_lse[:, None]).gather(1, tok)
    err_lp = float(((logp.double() - ref_lp).abs() / scale[:, None]).max())
    err_lse = float(((lse.double() - ref_lse).abs() / scale).max())
    REPORT["vocab_topk/%s/M%d_V%d_H%d_K%d" % (mode_name, M, V, H, K)] = dict(
        rows=M, rows_with_set_difference=len(diff_rows), rounding=rounding, real=real, logp_err_over_scale=err_lp,
        lse_err_over_scale=err_lse, kernel=want)
    assert real == 0
    assert err_lp <= 4 * u and err_lse <= 4 * u, (err_lp, err_lse)
    # descending, no repeated token
    assert bool((logp[:, :-1] >= logp[:, 1:]).all())
    assert all(len(set(r)) == K for r in tok.tolist())


def test_vocab_topk_rejects_bad_shapes():
    _lib = L_()
    lib = _lib.lib()
    h = torch.zeros(4, 8, device="cuda")
    W = torch.zeros(10, 8, device="cuda")
    b = torch.zeros(10, device="cuda")
    out = torch.zeros(4, 32, device="cuda")
    tok = torch.zeros(4, 32, dtype=torch.int64, device="cuda")
    ws = torch.zeros(lib.gic_vocab_topk_workspace_floats(4, 10, 16), device="cuda")
    for K in (0, 17, 11):
        rc = lib.gic_vocab_topk(1, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), 4, 10, 8, K, _lib.ptr(out), _lib.ptr(tok), None,
                                _lib.ptr(ws), _lib.stream())
        assert rc == 1, K


# ---------------------------------------------------------------------------------------------------------------------
def make_decoder(V, E, H, layers, seed, scale, eos_boost=0.0):
    from gic_b200.generator import Decoder
    cfg = dict(B=1, L=2, V=V, E=E, H=H, layers=layers, feat=0, filters=[4, 4, 4])
    a = rp.args_for(cfg)
    p = {k: v * scale for k, v in rp.make_params(rp.gen_param_shapes(a), seed).items()}
    p["decoder.linear.bias"][2] += eos_boost
    dec = Decoder(a)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in p.items() if k.startswith("decoder.")})
    return dec.cuda(), p


def run_beam(dec, feats, K, L, lp=0.0, mode=None, trace=None):
    from gic_b200.generator import decode_beam
    return decode_beam(dec, feats, K, L, lp, 2, mode=mode, trace=trace)


def check_invariants(ids, scores, lengths, lp, name):
    ids, scores, lengths = ids.cpu(), scores.cpu().double(), lengths.cpu()
    B, K, L = ids.shape
    bad = 0
    for b in range(B):
        norm = scores[b] / lengths[b].double() ** lp
        bad += int((norm[:-1] < norm[1:]).sum())
        rows = [tuple(r) for r in ids[b].tolist()]
        bad += len(rows) - len(set(rows))                      # a frozen beam is never duplicated
        for k in range(K):
            n = int(lengths[b, k])
            eos = (ids[b, k] == 2).nonzero()
            if len(eos):
                bad += int(int(eos[0]) + 1 != n) + int((ids[b, k, n:] != 0).sum())
            else:
                bad += int(n != L)
    REPORT["invariants/" + name] = dict(violations=bad)
    assert bad == 0


@pytest.mark.parametrize("V", [50, 1000])
@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("K", [1, 3, 5])
@pytest.mark.parametrize("lp", [0.0, 0.7])
def test_decode_beam_fp32_equals_oracle(V, layers, K, lp):
    _lib = L_()
    B, L, E, H = 4, 8, 16, 32
    for seed in range(40):
        dec, p = make_decoder(V, E, H, layers, 100 + seed, 40.0, eos_boost=2.0)
        feats = torch.randn(B, E, generator=torch.Generator().manual_seed(seed))
        ref = rx.beam_search(p, feats, K, L, eos_id=2, length_penalty=lp)
        if ref["margin"] > 1e-3:
            break
    assert ref["margin"] > 1e-3, "no seed gives a decisive oracle"
    trace = torch.empty(L, B, K, 2, dtype=torch.int32, device="cuda")
    with _lib.expect_kernels("row_topk_kernel", "beam_merge_kernel", "beam_finalize_kernel", absent=("vocab_topk_kernel",)):
        ids, scores, lengths = run_beam(dec, feats.cuda(), K, L, lp, mode=0, trace=trace)
        torch.cuda.synchronize()
    REPORT["fp32_exact/V%d_l%d_K%d_lp%g" % (V, layers, K, lp)] = dict(
        margin=ref["margin"], seed=seed, eos_beams=int((ref["lengths"] < L).sum()))
    assert torch.equal(ids.cpu(), ref["ids"])
    assert torch.equal(lengths.cpu(), ref["lengths"])
    assert torch.equal(trace.cpu().long(), ref["trace"])
    torch.testing.assert_close(scores.cpu().double(), ref["scores"], rtol=1e-5, atol=1e-5)
    check_invariants(ids, scores, lengths, lp, "fp32/V%d_l%d_K%d_lp%g" % (V, layers, K, lp))


@pytest.mark.parametrize("mode_name", ["tf32", "bf16"])
@pytest.mark.parametrize("layers", [1, 2])
def test_decode_beam_tensor_cores_c2_follows_oracle(mode_name, layers):
    """c2 inference shape: at every step the float64 oracle, following the GPU's own beams (trace), rescores every
    candidate; the GPU's K must be the oracle's K except within the accumulated rounding bound."""
    _lib = L_()
    mode = MODES[mode_name]
    B, K, L, V, E, H = 256, 5, 20, 10000, 512, 512
    dec, p = make_decoder(V, E, H, layers, 7 + layers, 4.0, eos_boost=1.5)
    feats = torch.randn(B, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    trace = torch.empty(L, B, K, 2, dtype=torch.int32, device="cuda")
    with _lib.expect_kernels("vocab_topk_kernel", "beam_merge_kernel", absent=("row_topk_kernel",)):
        ids, scores, lengths = run_beam(dec, feats, K, L, 0.0, mode=mode, trace=trace)
        torch.cuda.synchronize()
    P = {k: v.cuda().double() for k, v in p.items() if k.startswith("decoder.")}
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    hs = [torch.zeros(B * K, H, dtype=torch.float64, device="cuda") for _ in range(layers)]
    cs = [torch.zeros(B * K, H, dtype=torch.float64, device="cuda") for _ in range(layers)]
    x = feats.double().repeat_interleave(K, 0)
    score = torch.full((B, K), -float("inf"), dtype=torch.float64, device="cuda")
    score[:, 0] = 0
    fin = torch.zeros(B, K, dtype=torch.bool, device="cuda")
    bound = torch.zeros(B, K, dtype=torch.float64, device="cuda")
    tr = trace.long()
    counts = dict(same=0, tie=0, rounding=0, real=0)
    ar = torch.arange(B, device="cuda")
    for t in range(L):
        top = rx._lstm_stack(P, x, hs, cs)
        logits = top @ W_out.t() + b_out
        logp = F.log_softmax(logits, -1).view(B, K, V)
        step_b = (8 * U_TC * (top.abs() @ W_out.abs().t()).max(1).values).view(B, K)
        cand = score[:, :, None] + logp
        valid = ~fin[:, :, None].expand(B, K, V).clone()
        valid[:, :, 0] |= fin
        cand = torch.where(fin[:, :, None], score[:, :, None].expand(B, K, V), cand)
        cand = torch.where(valid, cand, torch.full_like(cand, -float("inf")))
        cb = torch.where(fin, bound, bound + step_b)                  # candidate's accumulated bound, per parent
        kth = torch.topk(cand.view(B, K * V), K, dim=1).values[:, K - 1]
        par, tok = tr[t, :, :, 0], tr[t, :, :, 1]
        got = cand[ar[:, None], par, tok]                            # [B,K] oracle score of the GPU's choices
        okv = valid[ar[:, None], par, tok]
        counts["real"] += int((~okv).sum())                          # a frozen beam extended by a token other than PAD
        gap = kth[:, None] - got
        gb = cb.gather(1, par) + cb.max(1, keepdim=True).values
        counts["same"] += int((gap <= 0).sum())
        counts["tie"] += int(((gap > 0) & (gap <= 1e-12)).sum())
        counts["rounding"] += int(((gap > 1e-12) & (gap <= gb)).sum())
        counts["real"] += int((gap > gb).sum())
        # follow the GPU's beams
        rows = (ar[:, None] * K + par).reshape(-1)
        hs = [h[rows] for h in hs]
        cs = [c[rows] for c in cs]
        bound = cb.gather(1, par)
        score = got
        fin = fin.gather(1, par) | (tok == 2)
        x = emb[tok.reshape(-1)]
    resc, sc = rx.beam_rescore({k: v.cuda() for k, v in p.items()}, feats, ids, lengths)
    score_err = (scores.double() - resc).abs()
    score_bad = int((score_err > 8 * U_TC * sc + 1e-4).sum())
    REPORT["tc_c2/%s/layers%d" % (mode_name, layers)] = dict(counts, score_bound_violations=score_bad,
                                                             max_score_err=float(score_err.max()),
                                                             eos_beams=int((lengths < L).sum()))
    assert counts["real"] == 0, counts
    assert score_bad == 0
    check_invariants(ids, scores, lengths, 0.0, "tc_c2/%s/layers%d" % (mode_name, layers))


@pytest.mark.parametrize("mode_name", list(MODES))
def test_k1_equals_greedy_sample(mode_name):
    _lib = L_()
    import gic_b200
    mode = MODES[mode_name]
    B, L, V, E, H = 64, 12, 1000, 64, 64
    dec, p = make_decoder(V, E, H, 1, 31, 10.0, eos_boost=1.0)
    feats = torch.randn(B, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    prev = gic_b200.get_gemm_mode()
    gic_b200.set_gemm_mode(mode)
    try:
        with torch.no_grad():
            _, sids = dec.sample(feats, pretrain=True, max_caption_len=L)
            ids, _, _ = dec.beam_search(feats, beam_size=1, max_caption_len=L)
    finally:
        gic_b200.set_gemm_mode(prev)
    ids, sids = ids[:, 0].cpu(), sids.cpu()
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    ties = real = 0
    for b in range(B):
        eos = (sids[b] == 2).nonzero()
        n = int(eos[0]) + 1 if len(eos) else L
        d = (ids[b, :n] != sids[b, :n]).nonzero()
        if not len(d):
            continue
        t = int(d[0])
        # float64 logits after the common prefix: the two argmaxes must be within rounding of each other
        hs = [torch.zeros(1, H, dtype=torch.float64)]
        cs = [torch.zeros(1, H, dtype=torch.float64)]
        x = feats[b:b + 1].double().cpu()
        for s in range(t + 1):
            top = rx._lstm_stack(P, x, hs, cs)
            x = P["decoder.embed.weight"][sids[b, s]][None]
        lg = (top @ P["decoder.linear.weight"].t() + P["decoder.linear.bias"])[0]
        sc = float((top.abs() @ P["decoder.linear.weight"].abs().t()).max())
        gap = abs(float(lg[ids[b, t]] - lg[sids[b, t]]))
        if gap <= 8 * u_of(mode, H) * sc * (t + 1):
            ties += 1
        else:
            real += 1
    REPORT["greedy/%s" % mode_name] = dict(rows=B, ties=ties, real=real)
    assert real == 0
    if mode == 0:
        assert ties == 0


def test_generate_matches_beam_search_and_leaves_state():
    _lib = L_()
    import gic_b200
    from gic_b200.generator import encoder_eval
    from gic_b200.training import GANInstructor
    cfg = dict(B=16, L=10, V=500, E=64, H=128, layers=2, feat=256, filters=[40, 40, 40])
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    a.device = "cuda"
    gic_b200.set_gemm_mode(gic_b200.GEMM_TF32)
    try:
        inst = GANInstructor(a, device="cuda:0")
        inst.pretrain_step(inp["captions"], pooled=inp["pooled"])     # optimizer state, BN running statistics, counters
        torch.cuda.synchronize()
        fg, fd = inst._flat_g, inst._flat_d
        snap = {n: t.clone() for n, t in (("g.flat", fg.flat), ("g.grad", fg.grad), ("g.m", fg.m), ("g.v", fg.v))}
        if fd is not None:
            snap.update({n: t.clone() for n, t in (("d.flat", fd.flat), ("d.grad", fd.grad), ("d.m", fd.m), ("d.v", fd.v))})
        bn = inst.gen.encoder.bn
        snap.update(rm=bn.running_mean.clone(), rv=bn.running_var.clone(), nb=bn.num_batches_tracked.clone())
        scal = (fg.step, fd.step if fd is not None else None, inst._rng_offset, inst.pretrain_steps, inst.gen_steps,
                inst.disc_steps, inst.gen.decoder.temperature)
        pooled = inp["pooled"].cuda()
        ids, scores, lengths = inst.generate(pooled=pooled, beam_size=4, max_caption_len=12, length_penalty=0.7)
        with inst._ctx:
            want = inst.gen.decoder.beam_search(encoder_eval(inst.gen.encoder, pooled, gic_b200.GEMM_TF32), beam_size=4,
                                                max_caption_len=12, length_penalty=0.7)
        torch.cuda.synchronize()
        assert torch.equal(ids, want[0]) and torch.equal(scores, want[1]) and torch.equal(lengths, want[2])
        for n, t in (("g.flat", fg.flat), ("g.grad", fg.grad), ("g.m", fg.m), ("g.v", fg.v)):
            assert torch.equal(t, snap[n]), n
        if fd is not None:
            for n, t in (("d.flat", fd.flat), ("d.grad", fd.grad), ("d.m", fd.m), ("d.v", fd.v)):
                assert torch.equal(t, snap[n]), n
        assert torch.equal(bn.running_mean, snap["rm"]) and torch.equal(bn.running_var, snap["rv"])
        assert torch.equal(bn.num_batches_tracked, snap["nb"])
        assert scal == (fg.step, fd.step if fd is not None else None, inst._rng_offset, inst.pretrain_steps, inst.gen_steps,
                        inst.disc_steps, inst.gen.decoder.temperature)
        check_invariants(ids, scores, lengths, 0.7, "generate")
    finally:
        gic_b200.set_gemm_mode(gic_b200.GEMM_FP32)


def test_decode_beam_cuda_graph_replay():
    _lib = L_()
    dec, p = make_decoder(1000, 64, 64, 2, 77, 10.0, eos_boost=1.0)
    feats = torch.randn(32, 64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    with torch.no_grad():
        eager = run_beam(dec, feats, 3, 10, 0.5, mode=1)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            with torch.cuda.graph(g):
                out = run_beam(dec, feats, 3, 10, 0.5, mode=1)
        torch.cuda.current_stream().wait_stream(s)
        for t in out:
            t.zero_()
        g.replay()
        torch.cuda.synchronize()
    for a_, b_ in zip(eager, out):
        assert torch.equal(a_, b_)
