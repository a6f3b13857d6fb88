"""GPU parity tests: the CUDA path (through the C ABI of libgic_b200.so) against the CPU oracle on the
same seeded inputs, and against the committed golden vectors from the reference.

Tolerances (BASELINE.json north_star): token ids bit-exact (mismatches must be ties: top-2 probability
gap < 1e-6, counted and reported); everything floating point within rtol 1e-3 in fp32, measured
against the tensor's own scale (max |reference|)."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_port as rp

pytestmark = pytest.mark.gpu

RTOL = 1e-3
REPORT = {}


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "parity_report.json"), "w") as f:
        json.dump(REPORT, f, indent=1, sort_keys=True)


def close(name, got, want, rtol=RTOL, atol=0.0, outlier_frac=0.0):
    """max |got - want| <= atol + rtol * max|want|.  outlier_frac > 0 (gradients downstream of the max-pool
    only): up to that fraction of entries may exceed the bound, by at most 50x -- a max-over-time whose top
    two candidates differ by <= 1 ulp (they exist in every config, see DESIGN.md "ties") can route its
    gradient to the other time step under a different summation order."""
    got = got.detach().double().cpu().reshape(-1) if isinstance(got, torch.Tensor) else torch.as_tensor(got).double().reshape(-1)
    want = want.detach().double().cpu().reshape(-1) if isinstance(want, torch.Tensor) else torch.as_tensor(want).double().reshape(-1)
    assert got.shape == want.shape, f"{name}: shape {tuple(got.shape)} vs {tuple(want.shape)}"
    scale = float(want.abs().max()) if want.numel() else 0.0
    diff = (got - want).abs()
    err = float(diff.max()) if want.numel() else 0.0
    rel = err / scale if scale > 0 else err
    bound = atol + rtol * max(scale, 1e-30)
    n_out = int((diff > bound).sum())
    REPORT[name] = dict(max_abs_err=err, scale=scale, rel=rel, outliers=n_out, numel=int(want.numel()))
    if outlier_frac > 0.0:
        assert n_out <= max(1, int(outlier_frac * want.numel())) and err <= 50 * bound, \
            f"{name}: {n_out} outliers, max err {err:.3e}, scale {scale:.3e}, rel {rel:.3e}"
    else:
        assert err <= bound, f"{name}: max err {err:.3e}, scale {scale:.3e}, rel {rel:.3e}"


GRAD = dict(atol=1e-9, outlier_frac=1e-3)     # gradient comparisons (see close())
ADAM_ATOL = 0.15 * 1e-4                      # Adam normalises g: where |g| <~ eps = 1e-8 (exact zeros in the reference) fp32 noise of 1e-9 in g moves the update by lr*noise/eps


def lib():
    import gic_b200
    from gic_b200 import _lib
    _lib.require_cuda()
    return _lib


def build_models(cfg, inp):
    """Our Generator/Discriminator loaded with the oracle's seeded weights."""
    import gic_b200.generator as G
    import gic_b200.discriminator as D
    a = inp["args"]
    a.device = "cuda"
    gen = G.Generator(a)
    sd = gen.state_dict()
    for k, v in inp["gen"].items():
        assert k in sd, k
        sd[k] = v.clone()
    gen.load_state_dict(sd)
    disc = D.Discriminator(a)
    disc.load_state_dict({k: v.clone() for k, v in inp["disc"].items()})
    return gen.to(dev()), disc.to(dev())


# ------------------------------------------------------------------------------------------------
# primitives
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tA", [0, 1])
@pytest.mark.parametrize("tB", [0, 1])
@pytest.mark.parametrize("M,N,K", [(8, 2048, 544), (37, 50, 19), (256, 1000, 512), (130, 900, 900), (1, 1, 1),
                                   (5120, 64, 1000)])
def test_gemm_fp32(tA, tB, M, N, K):
    L = lib()
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K + tA * 2 + tB)
    A = torch.randn((K, M) if tA else (M, K), generator=g)
    B = torch.randn((N, K) if tB else (K, N), generator=g)
    C0 = torch.randn(M, N, generator=g)
    bias = torch.randn(N, generator=g)
    want = 0.75 * ((A.t() if tA else A).double() @ (B.t() if tB else B).double()) + 0.5 * C0.double() + bias.double()
    Ad, Bd, Cd, bd = A.to(dev()), B.to(dev()), C0.clone().to(dev()), bias.to(dev())
    L.check(L.lib().gic_gemm(0, tA, tB, M, N, K, 0.75, L.ptr(Ad), A.shape[1], L.ptr(Bd), B.shape[1], 0.5, L.ptr(Cd), N,
                             L.ptr(bd), L.stream()), "gic_gemm")
    close(f"gemm_fp32/{M}x{N}x{K}/tA{tA}tB{tB}", Cd, want, rtol=2e-6 * max(1, K) ** 0.5)


def test_gemm_beta0_ignores_garbage():
    L = lib()
    A = torch.randn(33, 20).to(dev()); B = torch.randn(20, 17).to(dev())
    C = torch.full((33, 17), float("nan"), device=dev())
    L.check(L.lib().gic_gemm(0, 0, 0, 33, 17, 20, 1.0, L.ptr(A), 20, L.ptr(B), 17, 0.0, L.ptr(C), 17, None, L.stream()), "gemm")
    close("gemm_fp32/beta0", C, A.cpu().double() @ B.cpu().double(), rtol=1e-5)


@pytest.mark.parametrize("V,T,pretrain", [(50, 1.0, 0), (1000, 100.0, 0), (10000, 7.5, 0), (37, 1.0, 1), (60000, 2.0, 0)])
def test_sample_step(V, T, pretrain):
    L = lib()
    B, Lc, E, t = 6, 3, 8, 1
    g = torch.Generator().manual_seed(V)
    logits = torch.randn(B, V, generator=g)
    u = torch.rand(B, V, generator=g)
    emb = torch.randn(V, E, generator=g)
    if pretrain:
        want = logits
        pred = F.softmax(logits, -1)
    else:
        want = F.softmax((logits + rp.gumbel_noise(u)) * T, -1)
        pred = want
    tok = pred.max(1)[1]
    out = torch.zeros(B, Lc, V, device=dev())
    ids = torch.zeros(B, Lc, dtype=torch.int64, device=dev())
    xn = torch.zeros(B, E, device=dev())
    logits_d, u_d, emb_d = logits.to(dev()), u.to(dev()), emb.to(dev())      # keep the device copies alive
    L.check(L.lib().gic_sample_step(pretrain, L.ptr(logits_d), L.ptr(u_d), T, B, V, Lc, t, L.ptr(out),
                                    L.ptr(ids), None, L.ptr(emb_d), E, L.ptr(xn), L.stream()), "sample_step")
    close(f"sample_step/V{V}/probs", out[:, t], want)
    assert torch.equal(ids[:, t].cpu(), tok), "sampled ids differ"
    assert torch.equal(xn.cpu(), emb[tok]), "next-input gather differs"
    assert float(out[:, 0].abs().sum()) == 0.0 and float(out[:, 2].abs().sum()) == 0.0, "wrote outside row t"


def test_sample_step_tie_rule_lowest_index():
    L = lib()
    V = 64
    logits = torch.zeros(2, V)
    logits[0, [5, 9, 40]] = 3.0       # exact ties -> index 5
    logits[1, [63, 17]] = 1.0         # -> 17
    out = torch.zeros(2, 1, V, device=dev()); ids = torch.zeros(2, 1, dtype=torch.int64, device=dev())
    logits_d = logits.to(dev())
    L.check(L.lib().gic_sample_step(1, L.ptr(logits_d), None, 1.0, 2, V, 1, 0, L.ptr(out), L.ptr(ids), None,
                                    None, 0, None, L.stream()), "sample_step")
    assert ids.view(-1).tolist() == [5, 17]


# ------------------------------------------------------------------------------------------------
# decode forward (teacher-forced against the oracle), all configs with a CPU oracle that runs in seconds
# ------------------------------------------------------------------------------------------------
def classify_ids(name, ids_gpu, ids_ref, probs_ref):
    """Bit-exact token ids, except ties: the oracle's top-2 probabilities within 1e-6 (counted)."""
    mism = (ids_gpu.cpu() != ids_ref).nonzero()
    ties = 0
    for b, t in mism.tolist():
        top2 = probs_ref[b, t].topk(2)[0]
        assert float(top2[0] - top2[1]) < 1e-6, f"{name}: real token mismatch at (b={b}, t={t})"
        ties += 1
    REPORT[name + "/id_ties"] = dict(mismatches=int(mism.shape[0]), ties=ties, total=int(ids_ref.numel()))
    return ties


@pytest.mark.parametrize("cfg_name,T", [("c0", 1.0), ("c0", 100.0), ("c0_l2", 5.0), ("c1", 100.0), ("c1", 1.0)])
def test_decode_forward_vs_oracle(cfg_name, T):
    cfg = rp.CONFIGS[cfg_name]
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    gen, _ = build_models(cfg, inp)
    gen.train()
    B, Lc = inp["captions"].shape
    feats = rp.encoder_project(inp["gen"], inp["pooled"]) if a.conditional_gan else rp.start_features(inp["gen"], B)
    probs_ref, ids_ref, _ = rp.decoder_sample(inp["gen"], feats, inp["u"], T, Lc, a.gen_num_layers)
    gen.decoder.temperature = T
    with torch.no_grad():
        if a.conditional_gan:
            f_gpu = gen.encoder(inp["pooled"].to(dev()))
            close(f"decode/{cfg_name}/T{T}/features", f_gpu, feats)
        else:
            f_gpu = gen.decoder.embed.weight[1].expand(B, -1).contiguous()
        probs, ids = gen.decoder.sample(f_gpu, max_caption_len=Lc, u=inp["u"].to(dev()), forced_ids=ids_ref.to(dev()))
    classify_ids(f"decode/{cfg_name}/T{T}", ids, ids_ref, probs_ref)
    close(f"decode/{cfg_name}/T{T}/probs", probs, probs_ref)
    # free-running (no forcing) must reproduce the same captions when no tie occurred
    with torch.no_grad():
        probs2, ids2 = gen.decoder.sample(f_gpu, max_caption_len=Lc, u=inp["u"].to(dev()))
    if REPORT[f"decode/{cfg_name}/T{T}/id_ties"]["mismatches"] == 0:
        assert torch.equal(ids2.cpu(), ids_ref)


def test_decode_pretrain_mode_logits():
    cfg = rp.CONFIGS["c0_l2"]
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    gen, _ = build_models(cfg, inp)
    B, Lc = inp["captions"].shape
    feats = rp.encoder_project(inp["gen"], inp["pooled"])
    logits_ref, ids_ref, _ = rp.decoder_sample(inp["gen"], feats, None, 1.0, Lc, a.gen_num_layers, pretrain=True)
    with torch.no_grad():
        out, ids = gen.decoder.sample(feats.to(dev()), pretrain=True, max_caption_len=Lc, forced_ids=ids_ref.to(dev()))
    close("decode/pretrain/logits", out, logits_ref)
    assert torch.equal(ids.cpu(), ids_ref)


# ------------------------------------------------------------------------------------------------
# discriminator forward
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg_name", ["c0", "c0_l2", "c1"])
def test_disc_forward_vs_oracle(cfg_name):
    cfg = rp.CONFIGS[cfg_name]
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    _, disc = build_models(cfg, inp)
    B, Lc = inp["captions"].shape
    g = torch.Generator().manual_seed(5)
    soft = F.softmax(torch.randn(B, Lc, a.vocab_size, generator=g) * 3, -1)
    keep = inp["keep"]
    with torch.no_grad():
        disc.train()
        got_soft = disc(soft.to(dev()), keep=keep[1].to(dev()))
        got_ids = disc.forward_ids(inp["captions"].to(dev()), keep=keep[0].to(dev()))
        got_onehot = disc(F.one_hot(inp["captions"], a.vocab_size).float().to(dev()), keep=keep[0].to(dev()))
        disc.eval()
        got_eval = disc(soft.to(dev()))
    close(f"disc/{cfg_name}/soft", got_soft, rp.disc_forward(inp["disc"], soft, keep[1], a.disc_filter_sizes))
    close(f"disc/{cfg_name}/ids", got_ids, rp.disc_forward_ids(inp["disc"], inp["captions"], keep[0], a.disc_filter_sizes))
    close(f"disc/{cfg_name}/onehot_dense", got_onehot, got_ids.cpu(), rtol=1e-5)
    close(f"disc/{cfg_name}/eval", got_eval, rp.disc_forward(inp["disc"], soft, None, a.disc_filter_sizes))


def test_disc_generic_embed_dim_single_gt1():
    """disc_embed_dim != disc_num_rep (emb_dim_single = 2): the generic conv path."""
    cfg = dict(B=3, L=9, V=41, E=8, H=16, layers=1, feat=0, filters=[6, 5, 7])
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    a.disc_embed_dim, a.disc_num_rep = 16, 8
    inp["disc"] = rp.make_params(rp.disc_param_shapes(a), 77)
    import gic_b200.discriminator as D
    disc = D.Discriminator(a)
    disc.load_state_dict({k: v.clone() for k, v in inp["disc"].items()})
    disc = disc.to(dev()).eval()
    g = torch.Generator().manual_seed(9)
    soft = F.softmax(torch.randn(3, 9, 41, generator=g), -1)
    # oracle for es > 1: the reference's own ops (conv2d with kernel (f, es), stride (1, es))
    p = inp["disc"]
    emb = (soft @ p["embeddings.weight"].t()).unsqueeze(1)
    pools = [F.max_pool2d(F.relu(F.conv2d(emb, p[f"convs.{i}.weight"], p[f"convs.{i}.bias"], stride=(1, 2))),
                          (9 - f + 1, 1)).squeeze(2) for i, f in enumerate(a.disc_filter_sizes)]
    x = torch.cat(pools, 1).permute(0, 2, 1).contiguous().view(-1, 18)
    hw = F.linear(x, p["highway.weight"], p["highway.bias"])
    y = torch.sigmoid(hw) * F.relu(hw) + (1 - torch.sigmoid(hw)) * x
    want = F.linear(F.linear(y, p["feature2out.weight"], p["feature2out.bias"]), p["out2logits.weight"],
                    p["out2logits.bias"]).squeeze(1)
    with torch.no_grad():
        got = disc(soft.to(dev()))
    close("disc/es2/eval", got, want)


# ------------------------------------------------------------------------------------------------
# losses
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lt", ["standard", "JS", "KL", "hinge", "tv", "rsgan"])
def test_get_losses_and_seeds(lt):
    from gic_b200.utils import get_losses
    g = torch.Generator().manual_seed(11)
    xs = [(torch.randn(512, generator=g) * 2).requires_grad_(True) for _ in range(3)]
    gl_ref, dl_ref = rp.get_losses(*xs, lt)
    ys = [x.detach().to(dev()).requires_grad_(True) for x in xs]
    gl, dl = get_losses(*ys, lt)
    close(f"loss/{lt}/g", gl, gl_ref, rtol=1e-5)
    close(f"loss/{lt}/d", dl, dl_ref, rtol=1e-5)
    (dl_ref + 2 * gl_ref).backward() if gl_ref.requires_grad else dl_ref.backward()
    (dl + 2 * gl).backward()
    for i, (x, y) in enumerate(zip(xs, ys)):
        want = x.grad if x.grad is not None else torch.zeros_like(x)
        close(f"loss/{lt}/seed{i}", y.grad, want, rtol=1e-5, atol=1e-9)


def test_get_losses_unknown_type_raises():
    from gic_b200.utils import get_losses
    x = torch.zeros(4, device=dev())
    with pytest.raises(NotImplementedError):
        get_losses(x, x, x, "nope")


# ------------------------------------------------------------------------------------------------
# backward through the module interfaces (autograd.Function wrappers) vs oracle autograd
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg_name,T", [("c0", 1.0), ("c0_l2", 5.0), ("c1", 1.0)])
def test_decode_backward_vs_oracle(cfg_name, T):
    cfg = rp.CONFIGS[cfg_name]
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    gen, _ = build_models(cfg, inp)
    gen.train()
    B, Lc = inp["captions"].shape
    gw = torch.randn(B, Lc, a.vocab_size, generator=torch.Generator().manual_seed(3))
    gp = {k: v.clone().requires_grad_(True) for k, v in inp["gen"].items()}
    feats = rp.encoder_project(gp, inp["pooled"]) if a.conditional_gan else rp.start_features(gp, B)
    probs_ref, ids_ref, _ = rp.decoder_sample(gp, feats, inp["u"], T, Lc, a.gen_num_layers)
    (probs_ref * gw).sum().backward()
    gen.decoder.temperature = T
    if a.conditional_gan:
        f_gpu = gen.encoder(inp["pooled"].to(dev()))
    else:
        f_gpu = gen.decoder.embed(torch.ones(B, dtype=torch.long, device=dev()))
    probs, ids = gen.decoder.sample(f_gpu, max_caption_len=Lc, u=inp["u"].to(dev()), forced_ids=ids_ref.to(dev()))
    (probs * gw.to(dev())).sum().backward()
    got = dict(gen.named_parameters())
    for k, v in gp.items():
        if v.grad is None:
            assert got[k].grad is None or float(got[k].grad.abs().max()) == 0.0, k
            continue
        close(f"decode_bwd/{cfg_name}/{k}", got[k].grad, v.grad, atol=1e-9)


@pytest.mark.parametrize("cfg_name", ["c0", "c0_l2", "c1"])
def test_disc_backward_vs_oracle(cfg_name):
    cfg = rp.CONFIGS[cfg_name]
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    _, disc = build_models(cfg, inp)
    disc.train()
    B, Lc = inp["captions"].shape
    g = torch.Generator().manual_seed(5)
    soft = F.softmax(torch.randn(B, Lc, a.vocab_size, generator=g) * 3, -1)
    gw = torch.randn(B * a.disc_num_rep, generator=g)
    keep = inp["keep"]
    # oracle: loss = sum(w * D(soft)) + sum(w * D(ids))
    dp = {k: v.clone().requires_grad_(True) for k, v in inp["disc"].items()}
    s_ref = soft.clone().requires_grad_(True)
    l_ref = (rp.disc_forward(dp, s_ref, keep[1], a.disc_filter_sizes) * gw).sum() + \
            (rp.disc_forward_ids(dp, inp["captions"], keep[0], a.disc_filter_sizes) * gw).sum()
    l_ref.backward()
    s_gpu = soft.to(dev()).requires_grad_(True)
    l = (disc(s_gpu, keep=keep[1].to(dev())) * gw.to(dev())).sum() + \
        (disc.forward_ids(inp["captions"].to(dev()), keep=keep[0].to(dev())) * gw.to(dev())).sum()
    l.backward()
    close(f"disc_bwd/{cfg_name}/dinp", s_gpu.grad, s_ref.grad, **GRAD)
    got = dict(disc.named_parameters())
    for k, v in dp.items():
        close(f"disc_bwd/{cfg_name}/{k}", got[k].grad, v.grad, **GRAD)


# ------------------------------------------------------------------------------------------------
# full adversarial step: fused trainer vs the reference's golden vectors and vs the oracle
# ------------------------------------------------------------------------------------------------
def run_fused_step(cfg_name, T, loss, train=True, forced=None):
    from gic_b200.training import GANInstructor
    cfg = rp.CONFIGS[cfg_name]
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    a.device = "cuda"
    a.adv_loss_type = loss
    inst = GANInstructor(a, device="cuda:0")
    sd = inst.gen.state_dict()
    sd.update({k: v.clone() for k, v in inp["gen"].items()})
    inst.gen.load_state_dict(sd)
    inst.disc.load_state_dict({k: v.clone() for k, v in inp["disc"].items()})
    inst.gen.train(); inst.disc.train()
    inst.gen.decoder.temperature = T
    out = inst.adv_step(inp["captions"], pooled=inp["pooled"], u=inp["u"], keep=inp["keep"] if train else None,
                        train=train, forced_ids=forced)
    torch.cuda.synchronize()
    return inst, inp, out


@pytest.mark.parametrize("name,cfg_name,T,loss,train", [
    ("c0_T1_standard", "c0", 1.0, "standard", True), ("c0_T100_JS", "c0", 100.0, "JS", True),
    ("c0_T3_rsgan", "c0", 3.0, "rsgan", True), ("c0_T1_eval", "c0", 1.0, "standard", False),
    ("c0l2_T5_KL", "c0_l2", 5.0, "KL", True)])
def test_fused_step_vs_reference_golden(golden_dir, name, cfg_name, T, loss, train):
    gold = np.load(os.path.join(golden_dir, name + ".npz"))
    ids_ref = torch.from_numpy(gold["ids"])
    inst, inp, out = run_fused_step(cfg_name, T, loss, train, forced=ids_ref)
    classify_ids(f"golden/{name}", out["ids"], ids_ref, torch.from_numpy(gold["probs"]))
    close(f"golden/{name}/probs", out["probs"], gold["probs"])
    for k in ("d_real", "d_fake", "g_out", "g_loss", "d_loss"):
        close(f"golden/{name}/{k}", out[k], gold[k])
    if not train:
        return
    close(f"golden/{name}/d_norm", out["d_sqnorm"].sqrt(), gold["d_norm"])
    fd, fg = inst._flat_d, inst._flat_g
    for k, p in inst.disc.named_parameters():
        close(f"golden/{name}/d_grads/{k}", fd.g(p), gold[f"d_grads/{k}"], **GRAD)
        close(f"golden/{name}/new_disc/{k}", p, gold[f"new_disc/{k}"], rtol=1e-5, atol=ADAM_ATOL)
    if loss == "rsgan":
        for k, p in inst.gen.named_parameters():
            if k in inp["gen"]:
                close(f"golden/{name}/gen_unchanged/{k}", p, inp["gen"][k], rtol=0, atol=0)
        return
    close(f"golden/{name}/g_norm", out["g_sqnorm"].sqrt(), gold["g_norm"])
    for k, p in inst.gen.named_parameters():
        if f"g_grads/{k}" in gold.files:
            close(f"golden/{name}/g_grads/{k}", fg.g(p), gold[f"g_grads/{k}"], **GRAD)
            close(f"golden/{name}/new_gen/{k}", p, gold[f"new_gen/{k}"], rtol=1e-5, atol=ADAM_ATOL)


@pytest.mark.parametrize("T", [100.0, 1.0])
def test_fused_step_c1_vs_oracle(T):
    """BASELINE.json configs[0]: args.py defaults, batch 8, 2048-d pooled features, vocab 1000, len 16."""
    inp0 = rp.make_inputs(rp.CONFIGS["c1"])
    ref = rp.adversarial_step(inp0, T, "standard")
    inst, inp, out = run_fused_step("c1", T, "standard", True, forced=ref["ids"])
    classify_ids(f"step/c1/T{T}", out["ids"], ref["ids"], ref["probs"])
    for k in ("probs", "d_real", "d_fake", "g_out", "g_loss", "d_loss", "features"):
        close(f"step/c1/T{T}/{k}", out[k], ref[k])
    close(f"step/c1/T{T}/d_norm", out["d_sqnorm"].sqrt(), ref["d_norm"])
    close(f"step/c1/T{T}/g_norm", out["g_sqnorm"].sqrt(), ref["g_norm"])
    fd, fg = inst._flat_d, inst._flat_g
    for k, p in inst.disc.named_parameters():
        close(f"step/c1/T{T}/d_grads/{k}", fd.g(p), ref["d_grads"][k], **GRAD)
        close(f"step/c1/T{T}/new_disc/{k}", p, ref["new_disc"][k], rtol=1e-5, atol=ADAM_ATOL)
    for k, p in inst.gen.named_parameters():
        if k in ref["g_grads"]:
            close(f"step/c1/T{T}/g_grads/{k}", fg.g(p), ref["g_grads"][k], **GRAD)
            close(f"step/c1/T{T}/new_gen/{k}", p, ref["new_gen"][k], rtol=1e-5, atol=ADAM_ATOL)


def test_two_steps_adam_state_carries():
    """Second step uses the first step's Adam moments and updated weights (oracle run twice)."""
    inp = rp.make_inputs(rp.CONFIGS["c0"])
    st = {}
    r1 = rp.adversarial_step(inp, 2.0, "standard", adam_state=st, step=1)
    inp2 = dict(inp)
    inp2["gen"], inp2["disc"] = r1["new_gen"], r1["new_disc"]
    r2 = rp.adversarial_step(inp2, 2.0, "standard", adam_state=st, step=2)
    from gic_b200.training import GANInstructor
    a = inp["args"]; a.device = "cuda"
    inst = GANInstructor(a, device="cuda:0")
    sd = inst.gen.state_dict(); sd.update({k: v.clone() for k, v in inp["gen"].items()}); inst.gen.load_state_dict(sd)
    inst.disc.load_state_dict({k: v.clone() for k, v in inp["disc"].items()})
    inst.gen.train(); inst.disc.train(); inst.gen.decoder.temperature = 2.0
    inst.adv_step(inp["captions"], u=inp["u"], keep=inp["keep"], forced_ids=r1["ids"])
    inst.adv_step(inp["captions"], u=inp["u"], keep=inp["keep"], forced_ids=r2["ids"])
    for k, p in inst.disc.named_parameters():
        close(f"two_steps/disc/{k}", p, r2["new_disc"][k], rtol=1e-5, atol=2 * ADAM_ATOL)
    for k, p in inst.gen.named_parameters():
        if k in r2["g_grads"]:
            close(f"two_steps/gen/{k}", p, r2["new_gen"][k], rtol=1e-5, atol=2 * ADAM_ATOL)


def test_checkpoint_resume_continues_training(tmp_path):
    """save_checkpoint after two steps, load into a fresh instructor, take the third step on both: same parameters
    (the resumed run has the Adam moments, step counts and temperature of the original one)."""
    from gic_b200.training import GANInstructor
    inp = rp.make_inputs(rp.CONFIGS["c0"])
    a = inp["args"]; a.device = "cuda"

    def fresh(seed):
        torch.manual_seed(seed)
        inst = GANInstructor(a, device="cuda:0")
        inst.gen.train(); inst.disc.train()
        return inst
    inst = fresh(1)
    sd = inst.gen.state_dict(); sd.update({k: v.clone() for k, v in inp["gen"].items()}); inst.gen.load_state_dict(sd)
    inst.disc.load_state_dict({k: v.clone() for k, v in inp["disc"].items()})
    inst.gen.decoder.temperature = 3.0
    forced = inp["captions"]
    for _ in range(2):
        inst.adv_step(inp["captions"], u=inp["u"], keep=inp["keep"], forced_ids=forced)
    path = str(tmp_path / "adv_model.ckpt")
    inst.save_checkpoint(path)
    other = fresh(2)
    assert other.load_checkpoint(path) is True
    assert other.gen.decoder.temperature == 3.0 and other._flat_d.step == 2 and other._flat_g.step == 2
    inst.adv_step(inp["captions"], u=inp["u"], keep=inp["keep"], forced_ids=forced)
    other.adv_step(inp["captions"], u=inp["u"], keep=inp["keep"], forced_ids=forced)
    torch.cuda.synchronize()
    for (k, p), (_, q) in zip(inst.gen.named_parameters(), other.gen.named_parameters()):
        close(f"resume/gen/{k}", q, p, rtol=1e-6, atol=ADAM_ATOL)
    for (k, p), (_, q) in zip(inst.disc.named_parameters(), other.disc.named_parameters()):
        close(f"resume/disc/{k}", q, p, rtol=1e-6, atol=ADAM_ATOL)


def test_reference_style_loop_with_torch_optimizers():
    """Drop-in use exactly as src/training.py:144-169 writes it (Q1-fixed order), torch.optim.Adam on
    our modules' parameters, autograd driving our kernels."""
    import gic_b200.generator as G
    import gic_b200.discriminator as D
    from gic_b200.utils import get_losses
    cfg = rp.CONFIGS["c0"]
    inp = rp.make_inputs(cfg)
    ref = rp.adversarial_step(inp, 1.0, "standard")
    gen, disc = build_models(cfg, inp)
    gen.train(); disc.train()
    a = inp["args"]
    B, Lc = inp["captions"].shape
    gen.decoder.temperature = 1.0
    keep = inp["keep"].to(dev())
    gen_opt = torch.optim.Adam(gen.parameters(), lr=a.gen_lr)
    disc_opt = torch.optim.Adam(disc.parameters(), lr=a.disc_lr)
    features = gen.decoder.embed(torch.ones(B, 1, dtype=torch.long).squeeze(1).to(dev()))
    gen_captions, gen_ids = gen.decoder.sample(features, max_caption_len=Lc, u=inp["u"].to(dev()),
                                               forced_ids=ref["ids"].to(dev()))
    fake = gen_captions.detach()
    real = F.one_hot(inp["captions"].to(dev()), a.vocab_size).float()
    d_out_real = disc(real, keep=keep[0])
    d_out_fake = disc(fake, keep=keep[1])
    g_out = disc(gen_captions, keep=keep[2])
    g_loss, d_loss = get_losses(d_out_real, d_out_fake, g_out, "standard")
    close("loop/g_loss", g_loss, ref["g_loss"]); close("loop/d_loss", d_loss, ref["d_loss"])
    dgr = torch.autograd.grad(d_loss, list(disc.parameters()), retain_graph=True)
    ggr = torch.autograd.grad(g_loss, [p for p in gen.decoder.parameters()], allow_unused=True)
    for (k, p), g_ in zip(disc.named_parameters(), dgr):
        close(f"loop/d_grads/{k}", g_, ref["d_grads"][k], **GRAD)
        p.grad = g_
    for (k, p), g_ in zip(gen.decoder.named_parameters(), ggr):
        close(f"loop/g_grads/decoder.{k}", g_, ref["g_grads"]["decoder." + k], **GRAD)
        p.grad = g_
    torch.nn.utils.clip_grad_norm_(disc.parameters(), a.clip_norm); disc_opt.step()
    torch.nn.utils.clip_grad_norm_(gen.parameters(), a.clip_norm); gen_opt.step()
    for k, p in disc.named_parameters():
        close(f"loop/new_disc/{k}", p, ref["new_disc"][k], rtol=1e-5, atol=ADAM_ATOL)


def test_empty_batch_and_bad_shapes():
    L = lib()
    # B == 0 is a no-op
    L.check(L.lib().gic_sample_step(0, None, None, 1.0, 0, 10, 1, 0, None, None, None, None, 0, None, L.stream()), "empty")
    import gic_b200.discriminator as D
    a = rp.default_args(vocab_size=30, disc_num_filters=[4, 4, 4])
    disc = D.Discriminator(a).to(dev()).eval()
    with pytest.raises(Exception):
        disc(torch.rand(2, 4, 30, device=dev()))          # L=4 < max filter size 5 (reference also fails)
    with pytest.raises(ValueError):
        disc(torch.rand(2, 8, 31, device=dev()))          # wrong vocab


# ------------------------------------------------------------------------------------------------
# tensor-core mode (tcgen05 kind::tf32, fp32 accumulate): stated separately from the exact-fp32 mode
# ------------------------------------------------------------------------------------------------
MID = dict(B=64, L=16, V=2000, E=64, H=256, layers=1, feat=512, filters=[300, 300, 300])


@pytest.fixture
def tf32_mode():
    import gic_b200
    old = gic_b200.get_gemm_mode()
    gic_b200.set_gemm_mode(gic_b200.GEMM_TF32)
    yield
    gic_b200.set_gemm_mode(old)


# The oracle comparisons of the tensor-core modes (TF32 / BF16) live in tests/test_gpu_parity_modes.py: MID, c2, c4 per-GPU and
# a c5 slice, with every token mismatch classified and tolerances derived from the operand mantissa.


def test_graph_replay_matches_eager_steps():
    """CUDA-graph replay of the fused step (device-side temperature and Adam bias corrections) against the same
    three steps enqueued eagerly: identical inputs, a different temperature per step (update_temperature)."""
    from gic_b200.training import GANInstructor
    inp = rp.make_inputs(rp.CONFIGS["c1"])
    a = inp["args"]; a.device = "cuda"

    def fresh():
        inst = GANInstructor(a, device="cuda:0")
        sd = inst.gen.state_dict(); sd.update({k: v.clone() for k, v in inp["gen"].items()}); inst.gen.load_state_dict(sd)
        inst.disc.load_state_dict({k: v.clone() for k, v in inp["disc"].items()})
        inst.gen.train(); inst.disc.train()
        return inst
    temps = [1.0, 1.7, 3.1, 5.0]
    caps, pooled = inp["captions"].cuda(), inp["pooled"].cuda()
    u, keep = inp["u"].cuda(), inp["keep"].to(torch.uint8).cuda()
    eager, graphed = fresh(), fresh()
    outs_e, outs_g = [], []
    for T in temps:
        eager.gen.decoder.temperature = T
        r = eager.adv_step(caps, pooled=pooled, u=u, keep=keep)
        outs_e.append((r["g_loss"].item(), r["d_loss"].item(), r["ids"].clone()))
        graphed.gen.decoder.temperature = T
        r = graphed.adv_step(caps, pooled=pooled, u=u, keep=keep, graph=True)
        outs_g.append((r["g_loss"].item(), r["d_loss"].item(), r["ids"].clone()))
    torch.cuda.synchronize()
    assert graphed.graph_launches_per_step > 50
    for (ge, de, ie), (gg, dg, ig) in zip(outs_e, outs_g):
        assert abs(ge - gg) <= 1e-6 * max(1.0, abs(ge)) and abs(de - dg) <= 1e-6 * max(1.0, abs(de))
        assert torch.equal(ie, ig)
    for (k, pe), (_, pg) in zip(eager.disc.named_parameters(), graphed.disc.named_parameters()):
        close(f"graph/disc/{k}", pg, pe.detach().cpu(), rtol=1e-5, atol=len(temps) * ADAM_ATOL)   # atomics order differs run to run
    for (k, pe), (_, pg) in zip(eager.gen.named_parameters(), graphed.gen.named_parameters()):
        close(f"graph/gen/{k}", pg, pe.detach().cpu(), rtol=1e-5, atol=len(temps) * ADAM_ATOL)


@pytest.mark.parametrize("cfg_name", ["c0", "c1"])
def test_pretrain_step_vs_oracle(cfg_name):
    """Generator pre-training step (src/training.py:53-95): free-running greedy decode, CrossEntropyLoss over all
    positions (PAD included), gradients of every generator parameter vs autograd on the oracle."""
    import torch.nn.functional as F
    from gic_b200.training import GANInstructor
    inp = rp.make_inputs(rp.CONFIGS[cfg_name])
    a = inp["args"]
    gp = {k: v.clone().requires_grad_(True) for k, v in inp["gen"].items()}
    B, L = inp["captions"].shape
    feats = rp.encoder_project(gp, inp["pooled"]) if a.conditional_gan else rp.start_features(gp, B)
    logits, ids, _ = rp.decoder_sample(gp, feats, None, 1.0, L, layers=a.gen_num_layers, pretrain=True)
    loss = F.cross_entropy(logits.reshape(-1, logits.shape[-1]), inp["captions"].reshape(-1))      # :81-83
    names = [k for k in gp]
    grads = torch.autograd.grad(loss, [gp[k] for k in names], allow_unused=True)
    a.device = "cuda"
    inst = GANInstructor(a, device="cuda:0")
    sd = inst.gen.state_dict(); sd.update({k: v.clone() for k, v in inp["gen"].items()}); inst.gen.load_state_dict(sd)
    inst.gen.train()
    out = inst.pretrain_step(inp["captions"], pooled=inp["pooled"], update=False)
    torch.cuda.synchronize()
    assert torch.equal(out["ids"].cpu(), ids)
    close(f"pretrain/{cfg_name}/loss", out["loss"], loss.detach())
    close(f"pretrain/{cfg_name}/logits", out["logits"], logits.detach())
    fg = inst._flat_g
    ref = {k: g for k, g in zip(names, grads) if g is not None}
    for k, p in inst.gen.named_parameters():
        if k in ref:
            close(f"pretrain/{cfg_name}/grad/{k}", fg.g(p), ref[k], **GRAD)
    w0 = inst.gen.decoder.linear.weight.detach().clone()
    inst.pretrain_step(inp["captions"], pooled=inp["pooled"])
    assert not torch.equal(w0, inst.gen.decoder.linear.weight.detach())


def test_pretrain_step_refuses_an_eval_mode_encoder():
    """The encoder backward needs the batch statistics of a train-mode forward: a conditional pre-training step with
    gen.eval() raises, as adv_step does, instead of computing encoder gradients from stale statistics."""
    from gic_b200.training import GANInstructor
    inp = rp.make_inputs(rp.CONFIGS["c1"])
    a = inp["args"]
    a.device = "cuda"
    assert a.conditional_gan
    inst = GANInstructor(a, device="cuda:0")
    inst.gen.eval()
    with pytest.raises(NotImplementedError):
        inst.pretrain_step(inp["captions"], pooled=inp["pooled"])


# ------------------------------------------------------------------------------------------------
# full-size properties (BASELINE.json configs[1], c2): sizes the oracle cannot reach in seconds
# ------------------------------------------------------------------------------------------------
def test_full_size_c2_properties_and_row_locality():
    """One c2-shaped adversarial step (B 256, L 20, V 10 000, E = H = 512) in the bench's GEMM mode, checked through
    size-independent properties: every soft caption row is a probability vector, the sampled id is its first maximum,
    the losses are the BCE of the returned logits, and -- the premise of the data-parallel sharding -- the gradients
    of the full batch equal the mean of the gradients of its two half batches (every op is row-local; teacher-forced so
    that the halves decode the same tokens)."""
    import gic_b200
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    B, L, V = 256, 20, 10000
    a = default_args(vocab_size=V, gen_embed_dim=512, gen_hidden_dim=512, gen_num_layers=1, conditional_gan=0, device="cuda")
    old = gic_b200.get_gemm_mode()
    gic_b200.set_gemm_mode(gic_b200.GEMM_BF16)
    try:
        torch.manual_seed(1008)
        inst = GANInstructor(a, device="cuda:0")
        inst.gen.train(); inst.disc.train(); inst.gen.decoder.temperature = 1.0
        g = torch.Generator(device="cuda:0").manual_seed(5)
        caps = torch.randint(4, V, (B, L), generator=g, device="cuda:0"); caps[:, 0] = 1; caps[:, -1] = 2
        u = torch.rand(L, B, V, generator=g, device="cuda:0")
        keep = (torch.rand(3, B * 64, 900, generator=g, device="cuda:0") >= 0.2).to(torch.uint8)
        out = inst.adv_step(caps, u=u, keep=keep, update=False)
        torch.cuda.synchronize()
        probs, ids = out["probs"], out["ids"]
        rs = probs.sum(-1)
        assert float((rs - 1).abs().max()) < 2e-4 and float(probs.min()) >= 0.0
        assert torch.equal(ids, probs.argmax(-1))                      # first maximum (torch.argmax returns the first)
        assert int(ids.min()) >= 0 and int(ids.max()) < V
        d_loss = F.binary_cross_entropy_with_logits(out["d_real"], torch.ones_like(out["d_real"])) + \
            F.binary_cross_entropy_with_logits(out["d_fake"], torch.zeros_like(out["d_fake"]))
        g_loss = F.binary_cross_entropy_with_logits(out["g_out"], torch.ones_like(out["g_out"]))
        close("c2/d_loss", out["d_loss"], d_loss, rtol=1e-5)
        close("c2/g_loss", out["g_loss"], g_loss, rtol=1e-5)
        full_g, full_d = inst._flat_g.grad.clone(), inst._flat_d.grad.clone()
        assert bool(torch.isfinite(full_g).all()) and bool(torch.isfinite(full_d).all())
        forced = ids.clone()
        # same step teacher-forced (reference for the halves), then the two half batches
        inst.adv_step(caps, u=u, keep=keep, update=False, forced_ids=forced)
        ref_g, ref_d = inst._flat_g.grad.clone(), inst._flat_d.grad.clone()
        # (two runs of the same step differ by ~1e-3 of the scale: fp32 atomics order + max-over-time ties, DESIGN.md "Ties")
        close("c2/forced_equals_free/g", ref_g, full_g, rtol=5e-3, atol=1e-12, outlier_frac=1e-3)
        acc_g, acc_d = torch.zeros_like(ref_g), torch.zeros_like(ref_d)
        h = B // 2
        for lo in (0, h):
            kp = keep.view(3, B, 64, 900)[:, lo:lo + h].reshape(3, h * 64, 900).contiguous()
            inst.adv_step(caps[lo:lo + h], u=u[:, lo:lo + h].contiguous(), keep=kp, update=False, forced_ids=forced[lo:lo + h])
            acc_g += inst._flat_g.grad; acc_d += inst._flat_d.grad
        torch.cuda.synchronize()
        close("c2/row_locality/g", acc_g / 2, ref_g, rtol=2e-2, atol=1e-12, outlier_frac=1e-3)    # observed 4.5e-3 (bf16 dz, |g| ~ 2e-8)
        close("c2/row_locality/d", acc_d / 2, ref_d, rtol=5e-3, atol=1e-12, outlier_frac=1e-3)
    finally:
        gic_b200.set_gemm_mode(old)


def test_two_instructors_in_one_process_do_not_share_state():
    """The temperature pointer, prepared discriminator weights and Philox state are per library context (one per
    GANInstructor): two instructors stepping alternately -- different temperatures, graph replay, library-side draws -- give
    exactly what each gives alone."""
    from gic_b200.training import GANInstructor
    inp = rp.make_inputs(rp.CONFIGS["c1"])
    a = inp["args"]; a.device = "cuda"
    caps, pooled = inp["captions"].cuda(), inp["pooled"].cuda()

    def fresh(seed):
        torch.manual_seed(seed)
        inst = GANInstructor(a, device="cuda:0")
        sd = inst.gen.state_dict(); sd.update({k: v.clone() for k, v in inp["gen"].items()}); inst.gen.load_state_dict(sd)
        inst.disc.load_state_dict({k: v.clone() for k, v in inp["disc"].items()})
        inst.gen.train(); inst.disc.train()
        return inst

    def run(insts, temps, steps=4):
        outs = [[] for _ in insts]
        for s in range(steps):
            for k, (inst, T) in enumerate(zip(insts, temps)):
                inst.gen.decoder.temperature = T * (1 + s)
                r = inst.adv_step(caps, pooled=pooled, graph=True)          # u / keep drawn by the library (per-context Philox state)
                outs[k].append((r["ids"].clone(), float(r["g_loss"]), float(r["d_loss"])))
        torch.cuda.synchronize()
        return outs
    solo_a = run([fresh(11)], [1.0])[0]
    solo_b = run([fresh(22)], [3.0])[0]
    both = run([fresh(11), fresh(22)], [1.0, 3.0])
    for solo, mixed in ((solo_a, both[0]), (solo_b, both[1])):
        for (i0, g0, d0), (i1, g1, d1) in zip(solo, mixed):
            assert torch.equal(i0, i1)
            assert abs(g0 - g1) <= 1e-5 * max(1.0, abs(g0)) and abs(d0 - d1) <= 1e-5 * max(1.0, abs(d0))
