"""Teacher-forced caption scoring (EXTENSION, parity unpinned by reference) on the GPU against oracle/ref_score.py
teacher_forced_logp: the target-logit producer against float64 in every mode (argmax differences classified as tie /
rounding / real, real must be 0), exact-fp32 scoring against the oracle, every mode against the composed path
Decoder.sample(pretrain=True, forced_ids) + float64 log_softmax, the tensor-core path at the c2 shape, lengths, out-of-range
ids, determinism, CUDA-graph capture and GANInstructor.evaluate_nll.  Counts go to score_report.json in $GIC_REPORT_DIR
(default: the system's temporary directory)."""
import json
import math
import os
import tempfile

import pytest
import torch
import torch.nn.functional as F

from oracle import ref_score as rs
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
    with open(os.path.join(out, "score_report.json"), "w") as f:
        json.dump(REPORT, f, indent=1, sort_keys=True)


def L_():
    import gic_b200  # noqa: F401
    from gic_b200 import _lib
    _lib.require_cuda()
    return _lib


def u_of(mode, H):
    # exact-fp32 mode: the FFMA sum of H products, ~sqrt(H) roundings of 2^-24 each
    return U_TC if mode else max(1e-6, 2.0 ** -24 * 2.0 * H ** 0.5)


def producer(mode, fused, V, H):
    """Kernels that must run: the fused producer in the tensor-core modes on TMA-friendly shapes, else row_topk_kernel."""
    if mode != 0 and fused and V % 4 == 0 and H % 4 == 0:
        return ("vocab_topk_kernel", "score_rows_kernel"), ("row_topk_kernel",)
    return ("row_topk_kernel", "score_rows_kernel"), ("vocab_topk_kernel",)


def target_logp(mode, h, W, b, tgt):
    _lib = L_()
    lib = _lib.lib()
    M, H = h.shape
    V = W.shape[0]
    logp = torch.empty(M, device="cuda")
    lse = torch.empty(M, device="cuda")
    am = torch.empty(M, dtype=torch.int64, device="cuda")
    ws = torch.empty(lib.gic_vocab_target_logp_workspace_floats(M, V), device="cuda")
    _lib.check(lib.gic_vocab_target_logp(mode, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), _lib.ptr(tgt), M, V, H, _lib.ptr(logp),
                                         _lib.ptr(lse), _lib.ptr(am), _lib.ptr(ws), _lib.stream()), "gic_vocab_target_logp")
    return logp, lse, am


@pytest.mark.parametrize("mode_name,fused", [("fp32", 1), ("tf32", 1), ("bf16", 1), ("tf32", 0)])
@pytest.mark.parametrize("M,V,H", [(7, 50, 32), (1280, 10000, 512), (5120, 10000, 512), (2560, 30000, 1024), (300, 6001, 64)])
def test_vocab_target_logp_against_float64(mode_name, fused, M, V, H):
    _lib = L_()
    mode = MODES[mode_name]
    g = torch.Generator(device="cuda").manual_seed(M + V + H)
    h = torch.randn(M, H, device="cuda", generator=g)
    W = torch.randn(V, H, device="cuda", generator=g) * (3.0 / H ** 0.5)
    b = torch.randn(V, device="cuda", generator=g) * 0.5
    tgt = torch.randint(0, V, (M,), device="cuda", generator=g)
    tgt[: M // 4] = (h.double() @ W.double().t() + b.double())[: M // 4].argmax(1)      # targets at the argmax too
    tgt[0], tgt[-1] = -3, V                                                               # outside [0, V): NaN, no fault
    want, absent = producer(mode, fused, V, H)
    with _lib.options(GIC_FUSED_TOPK=fused), _lib.expect_kernels(*want, absent=absent):
        logp, lse, am = target_logp(mode, h, W, b, tgt)
        torch.cuda.synchronize()
    ref = h.double() @ W.double().t() + b.double()
    ref_lse = torch.logsumexp(ref, 1)
    absprod = h.double().abs() @ W.double().abs().t()
    scale = absprod.max(1).values + b.double().abs().max()
    u = u_of(mode, H)
    ok = (tgt >= 0) & (tgt < V)
    assert bool(torch.isnan(logp[~ok]).all()) and bool(torch.isfinite(logp[ok]).all())
    ref_lp = ref.gather(1, tgt.clamp(0, V - 1)[:, None])[:, 0] - ref_lse
    err_lp = float(((logp.double() - ref_lp).abs() / scale)[ok].max())
    err_lse = float(((lse.double() - ref_lse).abs() / scale).max())
    # argmax: a difference is a tie when the float64 logits are equal, rounding when within the operand-rounding bound
    ref_am = ref.argmax(1)
    tie = rounding = real = 0
    for m in (am != ref_am).nonzero()[:, 0].tolist():
        a, w = int(ref_am[m]), int(am[m])
        gap = float(ref[m, a] - ref[m, w])
        bound = 2 * u * float(absprod[m, a] + absprod[m, w]) + 1e-6 * float(scale[m])
        if gap == 0:
            tie += 1
        elif gap <= bound:
            rounding += 1
        else:
            real += 1
    REPORT["target_logp/%s_fused%d/M%d_V%d_H%d" % (mode_name, fused, M, V, H)] = dict(
        rows=M, tie=tie, rounding=rounding, real=real, logp_err_over_scale=err_lp, lse_err_over_scale=err_lse, kernels=want)
    assert real == 0
    assert err_lp <= 4 * u and err_lse <= 4 * u, (err_lp, err_lse)


def test_vocab_target_logp_rejects_bad_shapes():
    _lib = L_()
    lib = _lib.lib()
    h = torch.zeros(4, 8, device="cuda")
    W = torch.zeros(10, 8, device="cuda")
    b = torch.zeros(10, device="cuda")
    t = torch.zeros(4, dtype=torch.int64, device="cuda")
    out = torch.zeros(4, device="cuda")
    ws = torch.zeros(lib.gic_vocab_target_logp_workspace_floats(4, 10), device="cuda")
    for M, V, H in ((-1, 10, 8), (4, 0, 8), (4, 10, 0)):
        rc = lib.gic_vocab_target_logp(1, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), _lib.ptr(t), M, V, H, _lib.ptr(out), None,
                                       None, _lib.ptr(ws), _lib.stream())
        assert rc == 1, (M, V, H)
    assert lib.gic_vocab_target_logp(1, None, None, None, None, 0, 10, 8, None, None, None, None, _lib.stream()) == 0
    assert lib.gic_vocab_target_logp(1, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), None, 4, 10, 8, _lib.ptr(out), None, None,
                                     _lib.ptr(ws), _lib.stream()) == 2


# ---------------------------------------------------------------------------------------------------------------------
def make_decoder(V, E, H, layers, seed, scale):
    from gic_b200.generator import Decoder
    cfg = dict(B=1, L=2, V=V, E=E, H=H, layers=layers, feat=0, filters=[4, 4, 4])
    a = rp.args_for(cfg)
    p = {k: v * scale for k, v in rp.make_params(rp.gen_param_shapes(a), seed).items()}
    dec = Decoder(a)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in p.items() if k.startswith("decoder.")})
    return dec.cuda(), {k: v.cuda() for k, v in p.items()}


def make_batch(B, L, V, E, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    feats = torch.randn(B, E, device="cuda", generator=g)
    caps = torch.randint(3, V, (B, L), device="cuda", generator=g)
    lengths = torch.randint(1, L + 1, (B,), device="cuda", generator=g, dtype=torch.int32)
    return feats, caps, lengths


def score(dec, feats, caps, lengths, mode):
    from gic_b200.generator import score_captions
    logp, total, corr = score_captions(dec, feats, caps, lengths, mode=mode)
    return logp, total, corr


@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("V", [50, 1003])
def test_score_captions_fp32_equals_oracle(layers, V):
    _lib = L_()
    B, L, E, H = 16, 9, 24, 40
    dec, p = make_decoder(V, E, H, layers, 40 + layers, 10.0)
    feats, caps, lengths = make_batch(B, L, V, E, V + layers)
    with _lib.expect_kernels("teacher_inputs_kernel", "row_topk_kernel", "score_rows_kernel", absent=("vocab_topk_kernel",)):
        logp, total, corr = score(dec, feats, caps, lengths, 0)
        torch.cuda.synchronize()
    ref = rs.teacher_forced_logp(p, feats, caps, lengths)
    torch.testing.assert_close(logp.double(), ref["logp"], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(total.double(), ref["total"], rtol=1e-5, atol=1e-5)
    live = torch.arange(L, device="cuda")[None] < lengths[:, None]
    want = live & (ref["argmax"] == caps)
    diff = (corr.bool() != want)
    near = diff & (ref["gap"] <= 1e-5 * ref["scale"])
    REPORT["fp32/V%d_l%d" % (V, layers)] = dict(correct=int(corr.sum()), differ=int(diff.sum()), near_ties=int(near.sum()))
    assert int((diff & ~near).sum()) == 0


@pytest.mark.parametrize("mode_name,fused", [("fp32", 1), ("tf32", 1), ("bf16", 1), ("tf32", 0)])
@pytest.mark.parametrize("layers", [1, 2])
def test_score_matches_composed_sample(mode_name, fused, layers):
    """Same hidden states as Decoder.sample(pretrain=True, forced_ids): only the projection differs."""
    _lib = L_()
    import gic_b200
    mode = MODES[mode_name]
    B, L, V, E, H = 64, 12, 4000, 128, 256
    dec, p = make_decoder(V, E, H, layers, 11 + layers, 6.0)
    feats, caps, _ = make_batch(B, L, V, E, 21)
    want, absent = producer(mode, fused, V, H)
    prev = gic_b200.get_gemm_mode()
    gic_b200.set_gemm_mode(mode)
    try:
        with torch.no_grad(), _lib.options(GIC_FUSED_TOPK=fused):
            logits, _ = dec.sample(feats, pretrain=True, max_caption_len=L, forced_ids=caps)
            with _lib.expect_kernels(*want, absent=absent):
                logp, total, corr = dec.score(feats, caps)
                torch.cuda.synchronize()
    finally:
        gic_b200.set_gemm_mode(prev)
    z = logits.double()
    lp = F.log_softmax(z, -1).gather(2, caps[:, :, None])[:, :, 0]
    ref = rs.teacher_forced_logp(p, feats, caps)
    u = u_of(mode, H)
    err = float(((logp.double() - lp).abs() / ref["scale"]).max())
    # correct: the composed path's first maximum, differences only between logits within rounding of each other
    am = z.argmax(2)
    zt = z.gather(2, caps[:, :, None])[:, :, 0]
    za = z.gather(2, am[:, :, None])[:, :, 0]
    diff = corr != (am == caps)
    real = int((diff & ((za - zt).abs() > 4 * u * ref["scale"])).sum())
    REPORT["composed/%s_fused%d/layers%d" % (mode_name, fused, layers)] = dict(
        logp_err_over_scale=err, correct_differ=int(diff.sum()), real=real, kernels=want)
    assert err <= 4 * u, err
    assert real == 0
    torch.testing.assert_close(total.double(), logp.double().sum(1), rtol=1e-6, atol=1e-4)


@pytest.mark.parametrize("mode_name", ["tf32", "bf16"])
@pytest.mark.parametrize("layers", [1, 2])
def test_score_tensor_cores_c2_follows_oracle(mode_name, layers):
    """c2 shape: caption totals within the accumulated bound of test_decode_beam_tensor_cores_c2_follows_oracle (8u of the
    logit scale per step), argmax differences only within rounding."""
    _lib = L_()
    mode = MODES[mode_name]
    B, L, V, E, H = 256, 20, 10000, 512, 512
    dec, p = make_decoder(V, E, H, layers, 7 + layers, 4.0)
    feats, caps, lengths = make_batch(B, L, V, E, 3 + layers)
    with _lib.expect_kernels("vocab_topk_kernel", "score_rows_kernel", absent=("row_topk_kernel",)):
        logp, total, corr = score(dec, feats, caps, lengths, mode)
        torch.cuda.synchronize()
    ref = rs.teacher_forced_logp(p, feats, caps, lengths)
    live = torch.arange(L, device="cuda")[None] < lengths[:, None]
    sc = torch.where(live, ref["scale"], torch.zeros_like(ref["scale"]))
    bound = 8 * U_TC * sc.cumsum(1)
    tok_bad = int(((logp.double() - ref["logp"]).abs() > bound + 1e-4).sum())
    tot_err = (total.double() - ref["total"]).abs()
    tot_bad = int((tot_err > 8 * U_TC * sc.sum(1) + 1e-4).sum())
    diff = corr.bool() != (live & (ref["argmax"] == caps))
    real = int((diff & (ref["gap"] > bound)).sum())
    REPORT["tc_c2/%s/layers%d" % (mode_name, layers)] = dict(
        token_bound_violations=tok_bad, score_bound_violations=tot_bad, max_score_err=float(tot_err.max()),
        correct_differ=int(diff.sum()), real=real)
    assert tok_bad == 0 and tot_bad == 0
    assert real == 0


def test_score_lengths_out_of_range_determinism_and_graph():
    _lib = L_()
    B, L, V, E, H = 32, 10, 1000, 64, 64
    dec, p = make_decoder(V, E, H, 2, 77, 10.0)
    feats, caps, lengths = make_batch(B, L, V, E, 9)
    lengths[0], lengths[1], lengths[2] = 0, L + 5, -3              # clamped to [0, L]
    mode = 1
    with torch.no_grad():
        a = score(dec, feats, caps, lengths, mode)
        b_ = score(dec, feats, caps, lengths, mode)
        torch.cuda.synchronize()
    for x, y in zip(a, b_):
        assert torch.equal(x, y)                                    # bit-identical calls
    n = lengths.clamp(0, L)
    live = torch.arange(L, device="cuda")[None] < n[:, None]
    assert bool((a[0][~live] == 0).all()) and bool((a[2][~live] == 0).all())
    # tokens past lengths change nothing
    caps2 = torch.where(live, caps, torch.randint(0, V, caps.shape, device="cuda"))
    c = score(dec, feats, caps2, lengths, mode)
    for x, y in zip(a, c):
        assert torch.equal(x, y)
    # out-of-range ids: NaN at their position (inside the length), no fault; captions without one are unchanged
    caps3 = caps.clone()
    caps3[3, 2], caps3[4, 0] = -7, V + 11
    lengths3 = lengths.clone()
    lengths3[3], lengths3[4] = L, L
    d = score(dec, feats, caps3, lengths3, mode)
    e = score(dec, feats, caps, lengths3, mode)
    torch.cuda.synchronize()
    assert bool(torch.isnan(d[0][3, 2])) and bool(torch.isnan(d[0][4, 0]))
    assert bool(torch.isnan(d[1][3])) and bool(torch.isnan(d[1][4]))
    assert torch.equal(d[0][3, :2], e[0][3, :2])
    keep = torch.ones(B, dtype=torch.bool, device="cuda")
    keep[3] = keep[4] = False
    assert torch.equal(d[0][keep], e[0][keep]) and torch.equal(d[1][keep], e[1][keep])
    with pytest.raises(ValueError):
        dec.score(feats, caps3, lengths3)
    # CUDA-graph replay equals the eager call
    with torch.no_grad():
        gr = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            with torch.cuda.graph(gr):
                out = score(dec, feats, caps, lengths, mode)
        torch.cuda.current_stream().wait_stream(s)
        for t in out:
            t.zero_()
        gr.replay()
        torch.cuda.synchronize()
    for x, y in zip(a, out):
        assert torch.equal(x, y)
    REPORT["lengths_oob_graph"] = dict(ok=True)


def test_evaluate_nll_matches_oracle_and_leaves_state():
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
        g = torch.Generator().manual_seed(5)
        pooled = [inp["pooled"].cuda(), torch.randn(12, inp["pooled"].shape[1], generator=g).cuda()]
        caps = [inp["captions"].cuda(), torch.randint(3, cfg["V"], (12, 14), generator=g).cuda()]
        caps[1][:5, 6] = 2                                               # <E> inside some captions of the second batch
        lengths0 = torch.randint(1, caps[0].shape[1] + 1, (caps[0].shape[0],), generator=g, dtype=torch.int32)
        batches = [(pooled[0], caps[0], lengths0), (pooled[1], caps[1])]
        with _lib.expect_kernels("lstm_step_tf32_kernel", "vocab_topk_kernel", "score_rows_kernel"):
            res = inst.evaluate_nll(batches)
            torch.cuda.synchronize()
        # oracle from the same start features (eval-mode encoder projection)
        p = {k: v.cuda() for k, v in inst.gen.state_dict().items() if k.startswith("decoder.")}
        lp = tok = hits = bound = near = 0.0
        for i, (pl, cp) in enumerate(zip(pooled, caps)):
            with inst._ctx:
                feats = encoder_eval(inst.gen.encoder, pl, gic_b200.GEMM_TF32)
            if i == 0:
                n = lengths0.cuda().long()
            else:
                eos = cp == 2
                n = torch.where(eos.any(1), eos.int().argmax(1) + 1, torch.full_like(cp[:, 0], cp.shape[1]))
            r = rs.teacher_forced_logp(p, feats, cp, n)
            live = torch.arange(cp.shape[1], device="cuda")[None] < n[:, None]
            lp += float(r["total"].sum())
            tok += float(n.sum())
            hits += float((live & (r["argmax"] == cp)).sum())
            bound += float((8 * U_TC * torch.where(live, r["scale"], torch.zeros_like(r["scale"])).sum(1)).sum())
            steps = torch.arange(1, cp.shape[1] + 1, device="cuda")[None]
            near += float((live & (r["gap"] <= 8 * U_TC * r["scale"] * steps)).sum())
        nll = -lp / tok
        REPORT["evaluate_nll"] = dict(res, ref_nll=nll, ref_token_accuracy=hits / tok)
        assert res["tokens"] == int(tok) and res["captions"] == 28
        assert abs(res["nll"] - nll) * tok <= bound + 1e-3
        assert res["perplexity"] == pytest.approx(math.exp(res["nll"]), rel=1e-12)
        assert abs(res["token_accuracy"] * tok - hits) <= near + 1e-6
        for n_, t in (("g.flat", fg.flat), ("g.grad", fg.grad), ("g.m", fg.m), ("g.v", fg.v)):
            assert torch.equal(t, snap[n_]), n_
        if fd is not None:
            for n_, t in (("d.flat", fd.flat), ("d.grad", fd.grad), ("d.m", fd.m), ("d.v", fd.v)):
                assert torch.equal(t, snap[n_]), n_
        assert torch.equal(bn.running_mean, snap["rm"]) and torch.equal(bn.running_var, snap["rv"])
        assert torch.equal(bn.num_batches_tracked, snap["nb"])
        assert scal == (fg.step, fd.step if fd is not None else None, inst._rng_offset, inst.pretrain_steps, inst.gen_steps,
                        inst.disc_steps, inst.gen.decoder.temperature)
    finally:
        gic_b200.set_gemm_mode(gic_b200.GEMM_FP32)
