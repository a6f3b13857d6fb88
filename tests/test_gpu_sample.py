"""Sampled caption generation (EXTENSION, parity unpinned by reference) on the GPU against oracle/ref_sample.py: one
sampling step (gic_vocab_sample) against float64 in every mode, the exact-fp32 decode against the oracle bit for bit, the
tensor-core decode at the c2 inference shape step by step through the teacher-forced checker (differences classified as
tie / rounding / real, real must be 0), greedy and Decoder.sample cross-checks, the sampled distribution (chi-square),
determinism, CUDA-graph replay, GANInstructor.sample_captions and the argument checks.  Counts go to sample_report.json
in $GIC_REPORT_DIR (default: the system's temporary directory)."""
import json
import os
import tempfile

import pytest
import torch

from oracle import ref_beam as rx
from oracle import ref_port as rp
from oracle import ref_sample as rs

pytestmark = pytest.mark.gpu
REPORT = {}
MODES = {"fp32": 0, "tf32": 1, "bf16": 3}
U_TC = 2.0 ** -10                      # TF32 operand rounding
TAG = 0x53                             # GIC_RNG_TAG_SAMPLE


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    out = os.environ.get("GIC_REPORT_DIR") or tempfile.gettempdir()
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "sample_report.json"), "w") as f:
        json.dump(REPORT, f, indent=1, sort_keys=True)


def L_():
    import gic_b200  # noqa: F401
    from gic_b200 import _lib
    _lib.require_cuda()
    return _lib


def u_of(mode, H):
    # exact-fp32 mode: the FFMA sum of H products, ~sqrt(H) roundings of 2^-24 each
    return U_TC if mode else max(1e-6, 2.0 ** -24 * 2.0 * H ** 0.5)


def tf32(x, trunc):
    """float64 value of x rounded to a TF32 operand (10-bit mantissa): round to nearest even, or truncate."""
    b = x.float().view(torch.int32)
    if not trunc:
        b = b + 0x0FFF + ((b >> 13) & 1)
    return (b & ~0x1FFF).view(torch.float32).double()


def projection_error(h, W, b):
    """Per row of h[M,H] W^T + b: max over the columns of |logit from TF32-rounded operands - float64 logit|, the worse of
    round-to-nearest and truncation (the tensor-core modes' operand rounding, measured rather than bounded)."""
    z = h.double() @ W.double().t() + b.double()
    return torch.stack([(tf32(h, tr) @ tf32(W, tr).t() + b.double() - z).abs().max(1).values for tr in (False, True)]).max(0).values


def decode_logit_error(P, feats, n, ids):
    """Per (row, step) of a decode that follows ids[M,L]: max over the columns of |z_tc - z|, z_tc computed in float64
    from TF32-rounded operands in every contraction (each LSTM layer and the projection), z exactly; the worse of
    round-to-nearest and truncation.  It measures how far the operand rounding moves the logits, hidden-state drift included."""
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    layers = rx._decoder_layers(P)
    M, L = ids.shape
    H = W_out.shape[1]
    out = []
    for trunc in (False, True):
        def stack(x, hs, cs, rnd):
            for l in range(layers):
                f = (lambda v: tf32(v, trunc)) if rnd else (lambda v: v.double())
                hs[l], cs[l] = rp.lstm_cell(f(x), f(hs[l]), cs[l], f(P[f"decoder.lstm.weight_ih_l{l}"]),
                                            f(P[f"decoder.lstm.weight_hh_l{l}"]), P[f"decoder.lstm.bias_ih_l{l}"].double(),
                                            P[f"decoder.lstm.bias_hh_l{l}"].double())
                x = hs[l]
            return x
        z0 = [torch.zeros(M, H, dtype=torch.float64, device=ids.device) for _ in range(4 * layers)]
        he, ce, hx, cx = z0[:layers], z0[layers:2 * layers], z0[2 * layers:3 * layers], z0[3 * layers:]
        x = feats.double().repeat_interleave(n, 0)
        err = []
        for t in range(L):
            te, tx = stack(x, he, ce, True), stack(x, hx, cx, False)
            ze = tf32(te, trunc) @ tf32(W_out, trunc).t() + b_out.double()
            zx = tx @ W_out.double().t() + b_out.double()
            err.append((ze - zx).abs().max(1).values)
            x = emb[ids[:, t]].double()
        out.append(torch.stack(err, 1))
    return torch.maximum(out[0], out[1])


def set_rng(seed, offset=0, dev=None):
    _lib = L_()
    _lib.lib().gic_set_rng(seed, offset, None if dev is None else _lib.ptr(dev))


def uniforms(n):
    """The first n elements of the GIC_RNG_TAG_SAMPLE stream at the current gic_set_rng state (float32, cuda)."""
    _lib = L_()
    u = torch.empty(n, device="cuda")
    _lib.check(_lib.lib().gic_philox_uniform(TAG, n, _lib.ptr(u), _lib.stream()), "gic_philox_uniform")
    return u


def vocab_sample(mode, h, W, b, step, T, k, p):
    _lib = L_()
    lib = _lib.lib()
    M, H = h.shape
    V = W.shape[0]
    tok = torch.empty(M, dtype=torch.int64, device="cuda")
    logp = torch.empty(M, device="cuda")
    ws = torch.empty(lib.gic_vocab_sample_workspace_floats(M, V, k), device="cuda")
    _lib.check(lib.gic_vocab_sample(mode, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), M, V, H, step, float(T), k, float(p),
                                    _lib.ptr(tok), _lib.ptr(logp), _lib.ptr(ws), _lib.stream()), "gic_vocab_sample")
    return tok, logp


def producer(mode, V, H, k):
    tensor = mode != 0 and V % 4 == 0 and H % 4 == 0
    if k == 0:
        return "vocab_gumbel_kernel" if tensor else "row_gumbel_kernel"
    return "vocab_topk_kernel" if tensor else "row_topk_kernel"


FILTERS = [(0, 1.0), (1, 1.0), (5, 1.0), (5, 0.9), (16, 1.0), (16, 0.9), (1, 0.9)]


@pytest.mark.parametrize("mode_name", list(MODES))
@pytest.mark.parametrize("M,V,H", [(7, 50, 32), (256, 10000, 512), (130, 1003, 64)])
@pytest.mark.parametrize("k,p", FILTERS)
def test_vocab_sample_against_float64(mode_name, M, V, H, k, p):
    _vocab_sample_case(mode_name, M, V, H, k, p, True)


@pytest.mark.parametrize("k,p", [(0, 1.0), (5, 0.9)])
def test_vocab_sample_unfused_option(k, p):
    """GIC_FUSED_TOPK=0 also selects the unfused producer (tcgen05 GEMM to memory + row kernel) for sampling."""
    _vocab_sample_case("tf32", 256, 10000, 512, k, p, False)


def _vocab_sample_case(mode_name, M, V, H, k, p, fused):
    _lib = L_()
    mode = MODES[mode_name]
    T, step = 0.8, 3
    g = torch.Generator(device="cuda").manual_seed(M + V + H + k)
    h = torch.randn(M, H, device="cuda", generator=g)
    W = torch.randn(V, H, device="cuda", generator=g) * (3.0 / H ** 0.5)
    b = torch.randn(V, device="cuda", generator=g) * 0.5
    set_rng(1234 + k, 77)
    want = producer(mode if fused else 0, V, H, k)
    absent = [n for n in ("vocab_gumbel_kernel", "row_gumbel_kernel", "vocab_topk_kernel", "row_topk_kernel") if n != want]
    with _lib.options(GIC_FUSED_TOPK=1 if fused else 0), _lib.expect_kernels(want, "sample_rows_kernel", absent=absent):
        tok, logp = vocab_sample(mode, h, W, b, step, T, k, p)
        torch.cuda.synchronize()
    U = uniforms((step + 1) * M * V).view(step + 1, M, V)[step].double()
    set_rng(0, 0)
    z = h.double() @ W.double().t() + b.double()
    lse = torch.logsumexp(z, 1)
    absprod = h.double().abs() @ W.double().abs().t()
    scale = absprod.max(1).values + b.double().abs().max()
    u = u_of(mode, H)
    ref, key, S, cut = rs.draw(z, U, T, k, p)
    kgap = rs.top_k_gap(z, k)
    # per-row logit error: the measured TF32 operand rounding (tensor-core modes) plus fp32 accumulation, doubled
    eb = 2 * ((projection_error(h, W, b) if mode else 0.0) + 4e-6 * scale)
    counts = dict(same=0, tie=0, rounding=0, real=0)
    ref_l, tok_l = ref.tolist(), tok.tolist()
    for m in range(M):
        r, w = ref_l[m], tok_l[m]
        if r == w:
            counts["same"] += 1
            continue
        e = float(eb[m])
        kr = float(key[m, r])
        kw = float(z[m, w] / T + rp.gumbel_noise(U[m, w]))
        # the set is undecided when the top-k boundary or the nucleus cut lies within the logit error (the nucleus
        # masses move by at most ~2e / T when every logit moves by e)
        amb = float(kgap[m]) <= 2 * e or float(cut[m]) <= 2 * e / T + 1e-5
        if abs(kr - kw) <= 1e-6 * (1 + abs(kr)):
            counts["tie"] += 1
        elif (bool(S[m, w]) and kr - kw <= 2 * e / T + 1e-5 * (1 + abs(kr))) or amb:
            counts["rounding"] += 1
        else:
            counts["real"] += 1
    err_lp = float(((logp.double() - (z.gather(1, tok[:, None])[:, 0] - lse)).abs() / scale).max())
    REPORT["vocab_sample/%s%s/M%d_V%d_H%d/k%d_p%g" % (mode_name, "" if fused else "_unfused", M, V, H, k, p)] = dict(counts, logp_err_over_scale=err_lp,
                                                                                    kernel=want)
    assert counts["real"] == 0, counts
    assert err_lp <= 4 * u, err_lp
    assert bool(((tok >= 0) & (tok < V)).all())
    if k:
        # never outside the top k (beyond rounding of the k-th place)
        kth = torch.topk(z, k, dim=1).values[:, -1]
        zt = z.gather(1, tok[:, None])[:, 0]
        assert bool((zt >= kth - 2 * eb).all())


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


def run(dec, feats, n, L, T, k, p, mode, eos=2):
    from gic_b200.generator import sample_captions
    return sample_captions(dec, feats, n, L, T, k, p, eos, mode=mode)


def check_invariants(ids, lengths, name, eos=2):
    """PAD after every EOS; lengths = position of the first EOS + 1, or L."""
    ids, lengths = ids.reshape(-1, ids.shape[-1]).cpu(), lengths.reshape(-1).cpu()
    L = ids.shape[1]
    bad = 0
    for m in range(ids.shape[0]):
        e = (ids[m] == eos).nonzero()
        n = int(e[0]) + 1 if len(e) else L
        bad += int(int(lengths[m]) != n) + int((ids[m, n:] != 0).sum())
    REPORT["invariants/" + name] = dict(violations=bad, eos_rows=int((lengths < L).sum()))
    assert bad == 0


@pytest.mark.parametrize("V", [50, 1000])
@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("k,p", [(0, 1.0), (1, 1.0), (5, 0.9), (16, 1.0)])
def test_sample_captions_fp32_equals_oracle(V, layers, k, p):
    _lib = L_()
    B, n, L, E, H, T = 4, 3, 8, 16, 32, 0.9
    dec, prm = make_decoder(V, E, H, layers, 300 + layers, 10.0, eos_boost=2.0)
    feats = torch.randn(B, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(layers))
    M = B * n
    P = {kk: v.cuda() for kk, v in prm.items()}
    for seed in range(40):
        # a seed whose every decision is decisive at the fp32 bar: Gumbel keys and nucleus masses 1e-3 apart, the top-k
        # boundary 1e-4 of the logit scale apart (fp32 logits are within ~1e-6 of it)
        set_rng(seed, 5)
        U = uniforms(L * M * V).view(L, M, V).double()
        ref = rs.sample_captions(P, feats, n, L, T, k, p, 2, U)
        chk = rs.step_check(P, feats, n, ref["ids"], T, k, p, 2, U)
        live = chk["live"]
        margins = dict(key=float(chk["margin"][live].min()), cut=float(chk["cut"][live].min()),
                       kgap_over_scale=float((chk["kgap"] / chk["scale"])[live].min()))
        decisive = margins["key"] > 1e-3 and margins["cut"] > 1e-3 and margins["kgap_over_scale"] > 1e-4
        if decisive:
            break
    assert decisive, ("no seed gives a decisive oracle", margins)
    with _lib.expect_kernels(producer(0, V, H, k), "sample_rows_kernel", "sample_init_kernel"):
        ids, lp, lengths = run(dec, feats, n, L, T, k, p, 0)
        torch.cuda.synchronize()
    set_rng(0, 0)
    REPORT["fp32_exact/V%d_l%d_k%d_p%g" % (V, layers, k, p)] = dict(seed=seed, margins=margins,
                                                                     eos_rows=int((ref["lengths"] < L).sum()))
    assert torch.equal(ids.view(M, L), ref["ids"])
    assert torch.equal(lengths.view(M), ref["lengths"])
    torch.testing.assert_close(lp.view(M).double(), ref["caption_logp"], rtol=1e-5, atol=1e-4)
    check_invariants(ids, lengths, "fp32/V%d_l%d_k%d_p%g" % (V, layers, k, p))


@pytest.mark.parametrize("mode_name", ["tf32", "bf16"])
@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("k,p", [(0, 1.0), (16, 0.9)])
def test_sample_captions_tensor_cores_c2(mode_name, layers, k, p):
    """c2 inference shape, 5 captions per image: the float64 oracle follows the GPU's own ids step by step; every token
    differing from the oracle's must be a tie or within the operand-rounding bound."""
    _lib = L_()
    mode = MODES[mode_name]
    B, n, L, V, E, H, T = 256, 5, 20, 10000, 512, 512, 1.0
    M = B * n
    dec, prm = make_decoder(V, E, H, layers, 7 + layers, 4.0, eos_boost=1.5)
    feats = torch.randn(B, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    set_rng(99, 1)
    with _lib.expect_kernels(producer(mode, V, H, k), "sample_rows_kernel"):
        ids, lp, lengths = run(dec, feats, n, L, T, k, p, mode)
        torch.cuda.synchronize()
    U = uniforms(L * M * V).view(L, M, V)
    set_rng(0, 0)
    P = {kk: v.cuda() for kk, v in prm.items()}
    chk = rs.step_check(P, feats, n, ids.view(M, L), T, k, p, 2, U)
    live = chk["live"]
    diff = live & (chk["win"] != ids.view(M, L))
    # per (row, step) logit error: the measured effect of TF32 operand rounding on the whole decode, tripled (the
    # hardware's rounding instances differ from the emulation's), plus fp32 accumulation
    eb = 3 * decode_logit_error(P, feats, n, ids.view(M, L)) + 4e-6 * chk["scale"]
    kb = 2 * eb / T + 1e-5
    amb = (chk["kgap"] <= 2 * eb) | (chk["cut"] <= 2 * eb / T + 1e-5)
    tie = diff & (chk["gpu_gap"] <= 1e-6)
    by_key = diff & ~tie & chk["in_S"] & (chk["gpu_gap"] <= kb)
    by_set = diff & ~tie & ~by_key & amb
    rounding = by_key | by_set
    real = diff & ~tie & ~rounding
    counts = dict(steps=int(live.sum()), same=int((live & ~diff).sum()), tie=int(tie.sum()), rounding=int(rounding.sum()),
                  rounding_key_gap=int(by_key.sum()), rounding_set_boundary=int(by_set.sum()), real=int(real.sum()),
                  median_logit_error_bound=float(eb[live].median()), max_logit_error_bound=float(eb[live].max()),
                  median_cut_tolerance=float((2 * eb / T + 1e-5)[live].median()),
                  median_scale=float(chk["scale"][live].median()))
    resc, sc = rx.beam_rescore(P, feats.repeat_interleave(n, 0), ids.view(M, 1, L), lengths.view(M, 1))
    err = (lp.view(M, 1).double() - resc).abs()
    bad = int((err > 8 * U_TC * sc + 1e-4).sum())
    REPORT["tc_c2/%s/layers%d/k%d_p%g" % (mode_name, layers, k, p)] = dict(
        counts, logp_bound_violations=bad, max_logp_err=float(err.max()), eos_rows=int((lengths < L).sum()),
        distinct_captions=len({tuple(r) for r in ids.view(M, L).tolist()}))
    assert counts["real"] == 0, counts
    assert bad == 0
    check_invariants(ids, lengths, "tc_c2/%s/layers%d/k%d_p%g" % (mode_name, layers, k, p))


@pytest.mark.parametrize("mode_name", list(MODES))
def test_top_k_1_equals_greedy_beam(mode_name):
    L_()
    from gic_b200.generator import decode_beam
    mode = MODES[mode_name]
    B, L, V, E, H = 64, 12, 1000, 64, 64
    dec, prm = make_decoder(V, E, H, 2, 31, 10.0, eos_boost=1.0)
    feats = torch.randn(B, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    ids, _, lengths = run(dec, feats, 1, L, 1.7, 1, 1.0, mode)
    bids, _, blen = decode_beam(dec, feats, 1, L, 0.0, 2, mode=mode)
    torch.cuda.synchronize()
    ids, bids = ids[:, 0].cpu(), bids[:, 0].cpu()
    P = {k: v.double() for k, v in prm.items() if k.startswith("decoder.")}
    ties = real = 0
    for b in range(B):
        d = (ids[b] != bids[b]).nonzero()
        if not len(d):
            continue
        t = int(d[0])
        hs = [torch.zeros(1, H, dtype=torch.float64) for _ in range(2)]
        cs = [torch.zeros(1, H, dtype=torch.float64) for _ in range(2)]
        x = feats[b:b + 1].double().cpu()
        for s in range(t + 1):
            top = rx._lstm_stack(P, x, hs, cs)
            x = P["decoder.embed.weight"][ids[b, s]][None]
        lg = (top @ P["decoder.linear.weight"].t() + P["decoder.linear.bias"])[0]
        sc = float((top.abs() @ P["decoder.linear.weight"].abs().t()).max())
        if abs(float(lg[ids[b, t]] - lg[bids[b, t]])) <= 8 * u_of(mode, H) * sc * (t + 1):
            ties += 1
        else:
            real += 1
    REPORT["greedy_vs_beam/%s" % mode_name] = dict(rows=B, ties=ties, real=real)
    assert real == 0
    if mode == 0:
        assert ties == 0 and torch.equal(lengths[:, 0].cpu(), blen[:, 0].cpu())


@pytest.mark.parametrize("mode_name", ["fp32", "tf32"])
def test_full_vocabulary_at_t1_equals_decoder_sample(mode_name):
    """n = 1, temperature 1, top_k = 0 draws Decoder.sample's ids when Decoder.sample gets the GIC_RNG_TAG_SAMPLE stream as
    its uniforms (up to and including the first EOS; differences must be classified ties)."""
    import gic_b200
    L_()
    mode = MODES[mode_name]
    B, L, V, E, H = 128, 10, 1000, 64, 64
    dec, prm = make_decoder(V, E, H, 1, 41, 4.0, eos_boost=1.0)
    dec.temperature = 1.0
    feats = torch.randn(B, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    set_rng(2024, 3)
    ids, _, lengths = run(dec, feats, 1, L, 1.0, 0, 1.0, mode)
    U = uniforms(L * B * V).view(L, B, V)
    set_rng(0, 0)
    prev = gic_b200.get_gemm_mode()
    gic_b200.set_gemm_mode(mode)
    try:
        with torch.no_grad():
            _, sids = dec.sample(feats, max_caption_len=L, u=U)
        torch.cuda.synchronize()
    finally:
        gic_b200.set_gemm_mode(prev)
    ids = ids[:, 0]
    chk = rs.step_check({k: v.cuda() for k, v in prm.items()}, feats, 1, sids, 1.0, 0, 1.0, 2, U)
    ties = real = compared = 0
    for b in range(B):
        e = (sids[b] == 2).nonzero()
        n = int(e[0]) + 1 if len(e) else L
        d = (ids[b, :n] != sids[b, :n]).nonzero()
        compared += 1
        if not len(d):
            continue
        t = int(d[0])
        # the two implementations disagree at step t: the oracle's best two keys there must be within rounding
        if float(chk["margin"][b, t]) <= 2 * 8 * u_of(mode, H) * float(chk["scale"][b, t]) + 1e-5:
            ties += 1
        else:
            real += 1
    REPORT["decoder_sample/%s" % mode_name] = dict(rows=compared, ties=ties, real=real)
    assert real == 0


@pytest.mark.parametrize("mode_name,T,k,p", [("fp32", 1.0, 0, 1.0), ("fp32", 0.7, 0, 1.0), ("fp32", 1.5, 16, 1.0),
                                             ("fp32", 1.0, 16, 0.9), ("tf32", 1.0, 0, 1.0), ("tf32", 1.0, 16, 0.9)])
def test_step0_distribution_chi_square(mode_name, T, k, p):
    """One image repeated as n = 65536 rows: the step-0 tokens must follow the float64 filtered softmax(z / T)."""
    from scipy.stats import chisquare
    L_()
    mode = MODES[mode_name]
    n, V, E, H = 65536, 40, 64, 64
    dec, prm = make_decoder(V, E, H, 1, 55, 3.0)
    feats = torch.randn(1, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    set_rng(31337 + k, 0)
    with L_().expect_kernels(producer(mode, V, H, k), "sample_rows_kernel"):
        ids, _, _ = run(dec, feats, n, 1, T, k, p, mode)
        torch.cuda.synchronize()
    set_rng(0, 0)
    P = {kk: v.double().cuda() for kk, v in prm.items() if kk.startswith("decoder.")}
    top = rx._lstm_stack(P, feats.double(), [torch.zeros(1, H, dtype=torch.float64, device="cuda")],
                         [torch.zeros(1, H, dtype=torch.float64, device="cuda")])
    z = top @ P["decoder.linear.weight"].t() + P["decoder.linear.bias"]
    S, _ = rs.candidate_mask(z, T, k, p)
    q = torch.where(S, torch.softmax(z / T, 1), torch.zeros_like(z))[0]
    q = (q / q.sum()).cpu()
    obs = torch.bincount(ids.view(-1).cpu(), minlength=V).double()
    outside = int(obs[~S[0].cpu()].sum())
    exp_ = q * n
    big = exp_ >= 5
    f_obs = torch.cat([obs[big], obs[~big & S[0].cpu()].sum()[None]])
    f_exp = torch.cat([exp_[big], exp_[~big & S[0].cpu()].sum()[None]])
    if float(f_exp[-1]) < 5:                   # fold a small remainder into the last large bin
        f_obs = torch.cat([f_obs[:-2], (f_obs[-2] + f_obs[-1])[None]])
        f_exp = torch.cat([f_exp[:-2], (f_exp[-2] + f_exp[-1])[None]])
    pv = float(chisquare(f_obs.numpy(), f_exp.numpy() * float(f_obs.sum() / f_exp.sum())).pvalue) if len(f_obs) > 1 else 1.0
    REPORT["chi2/%s/T%g_k%d_p%g" % (mode_name, T, k, p)] = dict(bins=len(f_obs), p_value=pv, outside_S=outside,
                                                                support=int(S.sum()))
    assert outside == 0
    assert pv > 1e-6, pv


def test_determinism_and_offsets():
    L_()
    dec, _ = make_decoder(1000, 64, 64, 2, 61, 4.0, eos_boost=1.0)
    feats = torch.randn(32, 64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    outs = []
    for off in (7, 7, 8):
        set_rng(5, off)
        outs.append(run(dec, feats, 3, 12, 1.0, 0, 1.0, 1))
    set_rng(0, 0)
    torch.cuda.synchronize()
    for a_, b_ in zip(outs[0], outs[1]):
        assert torch.equal(a_, b_)
    assert not torch.equal(outs[0][0], outs[2][0])


@pytest.mark.parametrize("k,p", [(0, 1.0), (8, 0.9)])
def test_cuda_graph_replay_with_device_rng_state(k, p):
    L_()
    dec, _ = make_decoder(1000, 64, 64, 2, 77, 10.0, eos_boost=1.0)
    feats = torch.randn(32, 64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    state = torch.tensor([11, 4], dtype=torch.int64, device="cuda")
    with torch.no_grad():
        set_rng(0, 0, state)
        run(dec, feats, 2, 10, 0.8, k, p, 1)                 # warm-up outside the capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            with torch.cuda.graph(g):
                out = run(dec, feats, 2, 10, 0.8, k, p, 1)
        torch.cuda.current_stream().wait_stream(s)
        for off in (4, 9):
            state.copy_(torch.tensor([11, off]))
            for t in out:
                t.zero_()
            g.replay()
            set_rng(11, off)
            eager = run(dec, feats, 2, 10, 0.8, k, p, 1)
            torch.cuda.synchronize()
            for a_, b_ in zip(eager, out):
                assert torch.equal(a_, b_), off
    set_rng(0, 0)


def _instructor(cgan):
    from gic_b200.training import GANInstructor
    cfg = dict(B=16, L=10, V=500, E=64, H=128, layers=2, feat=256, filters=[40, 40, 40])
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    a.device = "cuda"
    a.conditional_gan = cgan
    return GANInstructor(a, device="cuda:0"), inp


def test_instructor_sample_captions_leaves_state_and_matches_decoder():
    L_()
    import gic_b200
    from gic_b200.generator import encoder_eval
    gic_b200.set_gemm_mode(gic_b200.GEMM_TF32)
    try:
        inst, inp = _instructor(1)
        inst.pretrain_step(inp["captions"], pooled=inp["pooled"])
        torch.cuda.synchronize()
        fg, fd = inst._flat_g, inst._flat_d
        snap = {nm: t.clone() for nm, t in (("g.flat", fg.flat), ("g.grad", fg.grad), ("g.m", fg.m), ("g.v", fg.v))}
        if fd is not None:
            snap.update({nm: t.clone() for nm, t in (("d.flat", fd.flat), ("d.grad", fd.grad), ("d.m", fd.m), ("d.v", fd.v))})
        bn = inst.gen.encoder.bn
        snap.update(rm=bn.running_mean.clone(), rv=bn.running_var.clone(), nb=bn.num_batches_tracked.clone())
        scal = (fg.step, fd.step if fd is not None else None, inst._rng_seed, inst._rng_offset, inst.pretrain_steps,
                inst.gen_steps, inst.disc_steps, inst.gen.decoder.temperature)
        pooled = inp["pooled"].cuda()
        ids, lp, lengths = inst.sample_captions(pooled=pooled, num_samples=3, max_caption_len=12, temperature=0.9, top_k=8,
                                                top_p=0.95, seed=17)
        with inst._ctx:
            set_rng(17, 0)
            want = inst.gen.decoder.sample_captions(encoder_eval(inst.gen.encoder, pooled, gic_b200.GEMM_TF32), num_samples=3,
                                                    max_caption_len=12, temperature=0.9, top_k=8, top_p=0.95)
            set_rng(0, 0)
        torch.cuda.synchronize()
        assert tuple(ids.shape) == (16, 3, 12)
        assert torch.equal(ids, want[0]) and torch.equal(lp, want[1]) and torch.equal(lengths, want[2])
        for nm, t in (("g.flat", fg.flat), ("g.grad", fg.grad), ("g.m", fg.m), ("g.v", fg.v)):
            assert torch.equal(t, snap[nm]), nm
        if fd is not None:
            for nm, t in (("d.flat", fd.flat), ("d.grad", fd.grad), ("d.m", fd.m), ("d.v", fd.v)):
                assert torch.equal(t, snap[nm]), nm
        assert torch.equal(bn.running_mean, snap["rm"]) and torch.equal(bn.running_var, snap["rv"])
        assert torch.equal(bn.num_batches_tracked, snap["nb"])
        assert scal == (fg.step, fd.step if fd is not None else None, inst._rng_seed, inst._rng_offset, inst.pretrain_steps,
                        inst.gen_steps, inst.disc_steps, inst.gen.decoder.temperature)
        check_invariants(ids, lengths, "instructor")
        # seed=None: one draw from torch's default generator
        torch.manual_seed(3)
        a1 = inst.sample_captions(pooled=pooled, num_samples=2, max_caption_len=8)
        torch.manual_seed(3)
        a2 = inst.sample_captions(pooled=pooled, num_samples=2, max_caption_len=8)
        torch.cuda.synchronize()
        assert all(torch.equal(x, y) for x, y in zip(a1, a2))
    finally:
        gic_b200.set_gemm_mode(gic_b200.GEMM_FP32)


def test_instructor_unconditional_rows_differ():
    L_()
    inst, _ = _instructor(0)
    ids, lp, lengths = inst.sample_captions(batch_size=4, num_samples=8, max_caption_len=10, seed=5)
    torch.cuda.synchronize()
    rows = {tuple(r) for r in ids.view(32, 10).tolist()}
    REPORT["unconditional"] = dict(rows=32, distinct=len(rows))
    assert len(rows) > 16
    check_invariants(ids, lengths, "unconditional")


def test_argument_checks():
    _lib = L_()
    lib = _lib.lib()
    dec, _ = make_decoder(10, 8, 8, 1, 1, 1.0)
    from gic_b200.generator import lstm_split
    W_ih, W_hh, b_ih, b_hh = lstm_split([w.detach().contiguous() for w in dec.lstm_params()])
    feats = torch.zeros(2, 8, device="cuda")
    ids = torch.zeros(2, 2, 4, dtype=torch.int64, device="cuda")
    lp = torch.zeros(4, device="cuda")
    ln = torch.zeros(4, dtype=torch.int32, device="cuda")
    ws = torch.zeros(lib.gic_sample_captions_workspace_floats(2, 2, 10, 8, 8, 1, 16) + 4096, device="cuda")
    ptr = _lib.ptr
    base = dict(B=2, n=2, L=4, layers=1, eos=2, T=1.0, k=0, p=1.0)

    def cap(**kw):
        a = dict(base, **kw)
        return lib.gic_sample_captions(1, ptr(feats), ptr(dec.embed.weight), _lib.ptr_array(W_ih), _lib.ptr_array(W_hh),
                                       _lib.ptr_array(b_ih), _lib.ptr_array(b_hh), ptr(dec.linear.weight),
                                       ptr(dec.linear.bias), a["B"], a["n"], a["L"], 10, 8, 8, a["layers"], a["eos"], a["T"],
                                       a["k"], a["p"], ptr(ids), ptr(lp), ptr(ln), ptr(ws), _lib.stream())

    def one(**kw):
        a = dict(base, **kw)
        return lib.gic_vocab_sample(1, ptr(feats), ptr(dec.linear.weight), ptr(dec.linear.bias), 2, 10, 8, 0, a["T"], a["k"],
                                    a["p"], ptr(ids), ptr(lp), ptr(ws), _lib.stream())

    shared = [dict(T=0.0), dict(T=-1.0), dict(T=float("inf")), dict(T=float("nan")), dict(p=0.0), dict(p=1.01),
              dict(p=float("nan")), dict(k=-1), dict(k=17), dict(k=11), dict(k=0, p=0.9)]
    for bad in shared:
        assert cap(**bad) == 1, bad
        assert one(**bad) == 1, bad
    for bad in (dict(n=0), dict(L=0), dict(eos=-1), dict(eos=10), dict(layers=0), dict(layers=9)):
        assert cap(**bad) == 1, bad
    assert cap(B=0) == 0
    assert cap() == 0 and one(k=10, p=0.5) == 0
    torch.cuda.synchronize()
