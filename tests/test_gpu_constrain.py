"""Constrained caption generation (min_length, no-repeat n-grams, banned tokens) on the GPU against the float64 oracle:
the masked producers (oracle/ref_constrain.py; gic_vocab_topk_masked, gic_vocab_sample_masked) in every mode with random masks, masks that ban
each row's true top K, a whole 128-column tile or half the vocabulary; constrained exact-fp32 beam search and sampling
against the oracle bit for bit; the c2 tensor-core decodes step by step; non-binding constraints bit-identical to the
unconstrained call; CUDA-graph replay, determinism, the instructor and the ABI error cases.  Counts go to
constrain_report.json in $GIC_REPORT_DIR (default: the system's temporary directory)."""
import ctypes as C
import json
import os
import tempfile

import pytest
import torch

from oracle import ref_beam as rx
from oracle import ref_constrain as rc
from oracle import ref_port as rp
from oracle import ref_sample as rs

pytestmark = pytest.mark.gpu
REPORT = {}
MODES = {"fp32": 0, "tf32": 1, "bf16": 3}
U_TC = 2.0 ** -10
TAG = 0x53
CONS = dict(min_length=5, no_repeat_ngram_size=3, bad_ids=[0, 1, 3])


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    out = os.environ.get("GIC_REPORT_DIR") or tempfile.gettempdir()
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "constrain_report.json"), "w") as f:
        json.dump(REPORT, f, indent=1, sort_keys=True)


def L_():
    import gic_b200  # noqa: F401
    from gic_b200 import _lib
    _lib.require_cuda()
    return _lib


def set_rng(seed, offset=0, dev=None):
    _lib = L_()
    _lib.lib().gic_set_rng(seed, offset, None if dev is None else _lib.ptr(dev))


def uniforms(n):
    _lib = L_()
    u = torch.empty(n, device="cuda")
    _lib.check(_lib.lib().gic_philox_uniform(TAG, n, _lib.ptr(u), _lib.stream()), "gic_philox_uniform")
    return u


def pack(ban):
    """bool [M, V] -> the uint32 bitmap [M, ceil(V / 32)] (as int32) of the masked entry points."""
    M, V = ban.shape
    W = (V + 31) // 32
    pad = torch.zeros(M, W * 32, dtype=torch.int64, device=ban.device)
    pad[:, :V] = ban.long()
    w = (pad.view(M, W, 32) << torch.arange(32, device=ban.device)).sum(-1)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32).contiguous()


def tf32(x, trunc):
    b = x.float().view(torch.int32)
    if not trunc:
        b = b + 0x0FFF + ((b >> 13) & 1)
    return (b & ~0x1FFF).view(torch.float32).double()


def logit_error(mode, h, W, b):
    """Per row: 2 x (the measured TF32 operand rounding in the tensor-core modes + fp32 accumulation)."""
    z = h.double() @ W.double().t() + b.double()
    scale = (h.double().abs() @ W.double().abs().t()).max(1).values + b.double().abs().max()
    e = 0.0
    if mode:
        e = torch.stack([(tf32(h, tr) @ tf32(W, tr).t() + b.double() - z).abs().max(1).values for tr in (False, True)]).max(0).values
    return z, 2 * (e + 4e-6 * scale)


def masks(kind, z, K, seed):
    M, V = z.shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    ban = torch.rand(M, V, device="cuda", generator=g) < (0.3 if kind == "random" else 0.05)
    if kind == "top":
        ban.scatter_(1, torch.topk(z, K, dim=1).indices, True)            # every row's true top K
    elif kind == "tile":
        ban[:, 128:256] = True
    elif kind == "half":
        ban[:, :V // 2] = True                                            # whole slices at V = 10 000
    return ban


def producers(mode, V, H, k, fused, gumbel):
    tensor = fused and mode != 0 and V % 4 == 0 and H % 4 == 0
    if gumbel:
        return "vocab_gumbel_ban_kernel" if tensor else "row_gumbel_ban_kernel"
    return "vocab_topk_ban_kernel" if tensor else "row_topk_ban_kernel"


PLAIN = ["vocab_topk_kernel", "vocab_gumbel_kernel", "row_topk_kernel", "row_gumbel_kernel"]
SHAPES = [(7, 50, 32), (256, 10000, 512), (130, 1003, 64)]


@pytest.mark.parametrize("mode_name", list(MODES))
@pytest.mark.parametrize("M,V,H", SHAPES)
@pytest.mark.parametrize("kind", ["random", "top", "tile", "half"])
@pytest.mark.parametrize("K", [1, 5, 16])
def test_vocab_topk_masked_against_float64(mode_name, M, V, H, kind, K):
    _topk_case(mode_name, M, V, H, kind, K, True)


@pytest.mark.parametrize("kind", ["random", "top"])
def test_vocab_topk_masked_unfused_option(kind):
    _topk_case("tf32", 256, 10000, 512, kind, 8, False)


def _topk_case(mode_name, M, V, H, kind, K, fused):
    _lib = L_()
    lib = _lib.lib()
    mode = MODES[mode_name]
    g = torch.Generator(device="cuda").manual_seed(M + V + H + K)
    h = torch.randn(M, H, device="cuda", generator=g)
    W = torch.randn(V, H, device="cuda", generator=g) * (3.0 / H ** 0.5)
    b = torch.randn(V, device="cuda", generator=g) * 0.5
    z, eb = logit_error(mode, h, W, b)
    ban = masks(kind, z, K, K + M)
    bits = pack(ban)
    logp = torch.empty(M, K, device="cuda")
    tok = torch.empty(M, K, dtype=torch.int64, device="cuda")
    lse = torch.empty(M, device="cuda")
    ws = torch.empty(lib.gic_vocab_topk_workspace_floats(M, V, K), device="cuda")
    want = producers(mode, V, H, K, fused, False)
    with _lib.options(GIC_FUSED_TOPK=1 if fused else 0), _lib.expect_kernels(want, absent=PLAIN):
        _lib.check(lib.gic_vocab_topk_masked(mode, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), M, V, H, K, _lib.ptr(logp),
                                             _lib.ptr(tok), _lib.ptr(lse), _lib.ptr(bits), _lib.ptr(ws), _lib.stream()),
                   "gic_vocab_topk_masked")
        torch.cuda.synchronize()
    lse64 = torch.logsumexp(z, 1)
    zm = z.masked_fill(ban, -float("inf"))
    want_v = torch.topk(zm, K, dim=1).values
    assert bool(((tok >= 0) & (tok < V)).all())
    assert not bool(ban.gather(1, tok).any()), "a banned column was returned"
    got_v = z.gather(1, tok)
    # a token that differs from the float64 order is within the logit error of the value it replaced (rounding)
    err = (got_v - want_v).abs().max(1).values
    real = int((err > 2 * eb).sum())
    same = int((tok == torch.topk(zm, K, dim=1).indices).all(1).sum())
    scale = eb.max()
    lp_err = float((logp.double() - (got_v - lse64[:, None])).abs().max() / scale)
    lse_err = float(((lse.double() - lse64).abs() / eb).max())
    REPORT["topk_masked/%s%s/M%d_V%d_H%d/%s/K%d" % (mode_name, "" if fused else "_unfused", M, V, H, kind, K)] = dict(
        rows=M, same=same, real=real, logp_err_over_bound=lp_err, lse_err_over_bound=lse_err, kernel=want)
    assert real == 0
    assert len(set(map(tuple, tok.sort(1).values.tolist()))) >= 1
    assert all(len(set(r)) == K for r in tok.tolist())
    assert lp_err <= 2 and lse_err <= 2


FILTERS = [(0, 1.0), (1, 1.0), (5, 0.9), (16, 1.0)]


@pytest.mark.parametrize("mode_name", list(MODES))
@pytest.mark.parametrize("M,V,H", SHAPES)
@pytest.mark.parametrize("kind", ["random", "top", "tile", "half"])
@pytest.mark.parametrize("k,p", FILTERS)
def test_vocab_sample_masked_against_float64(mode_name, M, V, H, kind, k, p):
    _sample_case(mode_name, M, V, H, kind, k, p, True)


@pytest.mark.parametrize("k,p", [(0, 1.0), (5, 0.9)])
def test_vocab_sample_masked_unfused_option(k, p):
    _sample_case("tf32", 256, 10000, 512, "random", k, p, False)


def _sample_case(mode_name, M, V, H, kind, k, p, fused):
    _lib = L_()
    lib = _lib.lib()
    mode = MODES[mode_name]
    T, step = 0.8, 3
    g = torch.Generator(device="cuda").manual_seed(M + V + H + k)
    h = torch.randn(M, H, device="cuda", generator=g)
    W = torch.randn(V, H, device="cuda", generator=g) * (3.0 / H ** 0.5)
    b = torch.randn(V, device="cuda", generator=g) * 0.5
    z, eb = logit_error(mode, h, W, b)
    ban = masks(kind, z, max(k, 1), k + M)
    bits = pack(ban)
    set_rng(4321 + k, 7)
    tok = torch.empty(M, dtype=torch.int64, device="cuda")
    logp = torch.empty(M, device="cuda")
    ws = torch.empty(lib.gic_vocab_sample_workspace_floats(M, V, k), device="cuda")
    want = producers(mode, V, H, k, fused, k == 0)
    with _lib.options(GIC_FUSED_TOPK=1 if fused else 0), _lib.expect_kernels(want, "sample_rows_kernel", absent=PLAIN):
        _lib.check(lib.gic_vocab_sample_masked(mode, _lib.ptr(h), _lib.ptr(W), _lib.ptr(b), M, V, H, step, float(T), k,
                                               float(p), _lib.ptr(tok), _lib.ptr(logp), _lib.ptr(bits), _lib.ptr(ws),
                                               _lib.stream()), "gic_vocab_sample_masked")
        torch.cuda.synchronize()
    U = uniforms((step + 1) * M * V).view(step + 1, M, V)[step].double()
    set_rng(0, 0)
    ref, key, S, cut = rc.draw(z, U, T, k, p, ban)
    kgap = rs.top_k_gap(z.masked_fill(ban, -float("inf")), k)
    counts = dict(same=0, tie=0, rounding=0, real=0)
    for m in range(M):
        r, w = int(ref[m]), int(tok[m])
        if r == w:
            counts["same"] += 1
            continue
        e = float(eb[m])
        kr = float(key[m, r])
        kw = float(z[m, w] / T + rp.gumbel_noise(U[m, w]))
        amb = float(kgap[m]) <= 2 * e or float(cut[m]) <= 2 * e / T + 1e-5
        if bool(ban[m, w]):
            counts["real"] += 1
        elif abs(kr - kw) <= 1e-6 * (1 + abs(kr)):
            counts["tie"] += 1
        elif (bool(S[m, w]) and kr - kw <= 2 * e / T + 1e-5 * (1 + abs(kr))) or amb:
            counts["rounding"] += 1
        else:
            counts["real"] += 1
    lse = torch.logsumexp(z, 1)
    lp_err = float(((logp.double() - (z.gather(1, tok[:, None])[:, 0] - lse)).abs() / eb).max())
    REPORT["sample_masked/%s%s/M%d_V%d_H%d/%s/k%d_p%g" % (mode_name, "" if fused else "_unfused", M, V, H, kind, k, p)] = dict(
        counts, logp_err_over_bound=lp_err, kernel=want)
    assert counts["real"] == 0, counts
    assert lp_err <= 2
    assert not bool(ban.gather(1, tok[:, None]).any())


# ---------------------------------------------------------------------------------------------------------------------
def make_decoder(V, E, H, layers, seed, scale, boost=()):
    from gic_b200.generator import Decoder
    cfg = dict(B=1, L=2, V=V, E=E, H=H, layers=layers, feat=0, filters=[4, 4, 4])
    a = rp.args_for(cfg)
    p = {k: v * scale for k, v in rp.make_params(rp.gen_param_shapes(a), seed).items()}
    for w, d in boost:
        p["decoder.linear.bias"][w] += d
    dec = Decoder(a)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in p.items() if k.startswith("decoder.")})
    return dec.cuda(), p


# EOS and PAD made likely, so that min_length and the ban bind
BOOST = ((2, 2.0), (0, 1.5), (3, 1.0))


def check_constraints(ids, lengths, L, min_length, n, bad, name, eos=2):
    ids, lengths = ids.reshape(-1, ids.shape[-1]).cpu(), lengths.reshape(-1).cpu()
    bad_rows = 0
    for m in range(ids.shape[0]):
        row, ln = ids[m].tolist(), int(lengths[m])
        live = row[:ln]
        e = [i for i, w in enumerate(row) if w == eos]
        ok = ln >= min(min_length, L) and not any(w in bad for w in live) and all(w == 0 for w in row[ln:])
        ok = ok and (ln == (e[0] + 1 if e else L))
        if n:
            grams = [tuple(live[s:s + n]) for s in range(len(live) - n + 1)]
            ok = ok and len(grams) == len(set(grams))
        bad_rows += not ok
    REPORT["constraints/" + name] = dict(rows=ids.shape[0], violations=bad_rows, eos_rows=int((lengths < L).sum()))
    assert bad_rows == 0


@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("K", [1, 3, 5])
@pytest.mark.parametrize("cons", [CONS, dict(no_repeat_ngram_size=1), dict(min_length=8, bad_ids=[0, 1, 3, 7, 1000])])
def test_decode_beam_fp32_equals_oracle(layers, K, cons):
    _lib = L_()
    from gic_b200.generator import decode_beam
    B, L, V, E, H = 6, 8, 40, 16, 32
    dec, prm = make_decoder(V, E, H, layers, 500 + layers, 8.0, BOOST)
    P = {k: v.cuda() for k, v in prm.items()}
    for seed in range(20):
        # inputs whose every decision is decisive at the fp32 bar
        feats = torch.randn(B, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
        ref = rc.beam_search(P, feats, K, L, eos_id=2, **cons)
        if ref["margin"] > 1e-4:
            break
    with _lib.expect_kernels("ban_rows_kernel", "ban_base_kernel", "row_topk_ban_kernel", absent=PLAIN):
        ids, scores, lengths = decode_beam(dec, feats, K, L, 0.0, 2, mode=0, **cons)
        torch.cuda.synchronize()
    REPORT["beam_fp32/l%d_K%d/%s" % (layers, K, sorted(cons.items()))] = dict(margin=ref["margin"])
    assert ref["margin"] > 1e-4
    assert torch.equal(ids.cpu(), ref["ids"].cpu())
    assert torch.equal(lengths.cpu(), ref["lengths"].cpu())
    torch.testing.assert_close(scores.double(), ref["scores"], rtol=1e-5, atol=1e-4)
    check_constraints(ids, lengths, L, cons.get("min_length", 0), cons.get("no_repeat_ngram_size", 0),
                      set(w for w in cons.get("bad_ids", ()) if w < V), "beam_fp32/l%d_K%d" % (layers, K))


@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("k,p", [(0, 1.0), (1, 1.0), (5, 0.9), (16, 1.0)])
def test_sample_captions_fp32_equals_oracle(layers, k, p):
    _lib = L_()
    from gic_b200.generator import sample_captions
    B, n, L, V, E, H, T = 4, 3, 8, 60, 16, 32, 0.9
    M = B * n
    dec, prm = make_decoder(V, E, H, layers, 300 + layers, 10.0, BOOST)
    feats = torch.randn(B, E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(layers))
    P = {kk: v.cuda() for kk, v in prm.items()}
    for seed in range(40):
        set_rng(seed, 5)
        U = uniforms(L * M * V).view(L, M, V).double()
        ref = rc.sample_captions(P, feats, n, L, T, k, p, 2, U, **CONS)
        chk = rc.step_check(P, feats, n, ref["ids"], T, k, p, 2, U, **CONS)
        live = chk["live"]
        margins = dict(key=float(chk["margin"][live].min()), cut=float(chk["cut"][live].min()),
                       kgap_over_scale=float((chk["kgap"] / chk["scale"])[live].min()))
        if margins["key"] > 1e-3 and margins["cut"] > 1e-3 and margins["kgap_over_scale"] > 1e-4:
            break
    else:
        pytest.fail("no seed gives a decisive oracle: %s" % margins)
    want = "row_gumbel_ban_kernel" if k == 0 else "row_topk_ban_kernel"
    with _lib.expect_kernels(want, "ban_rows_kernel", "sample_rows_kernel", absent=PLAIN):
        ids, lp, lengths = sample_captions(dec, feats, n, L, T, k, p, 2, mode=0, **CONS)
        torch.cuda.synchronize()
    set_rng(0, 0)
    REPORT["sample_fp32/l%d_k%d_p%g" % (layers, k, p)] = dict(seed=seed, margins=margins)
    assert torch.equal(ids.view(M, L), ref["ids"])
    assert torch.equal(lengths.view(M), ref["lengths"])
    torch.testing.assert_close(lp.view(M).double(), ref["caption_logp"], rtol=1e-5, atol=1e-4)
    check_constraints(ids, lengths, L, 5, 3, {0, 1, 3}, "sample_fp32/l%d_k%d_p%g" % (layers, k, p))


def c2_decoder(layers):
    return make_decoder(10000, 512, 512, layers, 7 + layers, 4.0, ((2, 1.5), (0, 1.0), (3, 1.0)))


@pytest.mark.parametrize("mode_name", ["tf32", "bf16"])
@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("k,p", [(0, 1.0), (16, 0.9)])
def test_sample_captions_tensor_cores_c2(mode_name, layers, k, p):
    """c2 shape, 5 captions per image: the oracle follows the GPU's ids step by step under the constraints; a token that
    differs from the oracle's must be a tie or within the measured operand-rounding bound; every caption obeys them."""
    _lib = L_()
    from gic_b200.generator import sample_captions
    from test_gpu_sample import decode_logit_error
    mode = MODES[mode_name]
    B, n, L, V, T = 256, 5, 20, 10000, 1.0
    M = B * n
    dec, prm = c2_decoder(layers)
    feats = torch.randn(B, 512, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    set_rng(99, 1)
    want = "vocab_gumbel_ban_kernel" if k == 0 else "vocab_topk_ban_kernel"
    with _lib.expect_kernels(want, "ban_rows_kernel", "sample_rows_kernel", absent=PLAIN):
        ids, lp, lengths = sample_captions(dec, feats, n, L, T, k, p, 2, mode=mode, **CONS)
        torch.cuda.synchronize()
    U = uniforms(L * M * V).view(L, M, V)
    set_rng(0, 0)
    P = {kk: v.cuda() for kk, v in prm.items()}
    chk = rc.step_check(P, feats, n, ids.view(M, L), T, k, p, 2, U, **CONS)
    live = chk["live"]
    diff = live & (chk["win"] != ids.view(M, L))
    eb = 3 * decode_logit_error(P, feats, n, ids.view(M, L)) + 4e-6 * chk["scale"]
    kb = 2 * eb / T + 1e-5
    amb = (chk["kgap"] <= 2 * eb) | (chk["cut"] <= 2 * eb / T + 1e-5)
    tie = diff & (chk["gpu_gap"] <= 1e-6)
    by_key = diff & ~tie & chk["in_S"] & (chk["gpu_gap"] <= kb)
    rounding = by_key | (diff & ~tie & ~by_key & amb)
    real = diff & ~tie & ~rounding
    counts = dict(steps=int(live.sum()), same=int((live & ~diff).sum()), tie=int(tie.sum()), rounding=int(rounding.sum()),
                  real=int(real.sum()), outside_S=int((live & ~chk["in_S"]).sum()))
    REPORT["sample_c2/%s/layers%d/k%d_p%g" % (mode_name, layers, k, p)] = counts
    assert counts["real"] == 0, counts
    check_constraints(ids, lengths, L, 5, 3, {0, 1, 3}, "sample_c2/%s/l%d/k%d" % (mode_name, layers, k))


@pytest.mark.parametrize("mode_name", ["tf32", "bf16"])
@pytest.mark.parametrize("layers", [1, 2])
def test_decode_beam_tensor_cores_c2_follows_oracle(mode_name, layers):
    """c2 shape, K = 5: at every step and image the oracle re-ranks the candidates of the GPU's own beams (scores carried
    from the GPU's choices) under the constraints; every chosen (parent, token) must be allowed, and the chosen set must
    equal the oracle's K best up to candidates within the rounding bound of the K-th score."""
    _lib = L_()
    from gic_b200.generator import decode_beam
    mode = MODES[mode_name]
    B, K, L, V = 64, 5, 20, 10000
    dec, prm = c2_decoder(layers)
    feats = torch.randn(B, 512, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
    trace = torch.empty(L, B, K, 2, dtype=torch.int32, device="cuda")
    with _lib.expect_kernels("vocab_topk_ban_kernel", "ban_rows_kernel", "beam_merge_kernel", absent=PLAIN):
        ids, scores, lengths = decode_beam(dec, feats, K, L, 0.0, 2, mode=mode, trace=trace, **CONS)
        torch.cuda.synchronize()
    P = {kk: v.double().cuda() for kk, v in prm.items() if kk.startswith("decoder.")}
    tr = trace.long()
    hs = [torch.zeros(B * K, 512, dtype=torch.float64, device="cuda") for _ in range(layers)]
    cs = [torch.zeros(B * K, 512, dtype=torch.float64, device="cuda") for _ in range(layers)]
    x = feats.double().repeat_interleave(K, 0)
    score = torch.full((B, K), -float("inf"), dtype=torch.float64, device="cuda")
    score[:, 0] = 0
    fin = torch.zeros(B, K, dtype=torch.bool, device="cuda")
    seq = torch.zeros(B, K, L, dtype=torch.int64, device="cuda")
    real = checked = near = 0
    for t in range(L):
        top = rx._lstm_stack(P, x, hs, cs)
        z = top @ P["decoder.linear.weight"].t() + P["decoder.linear.bias"]
        sc = (top.abs() @ P["decoder.linear.weight"].abs().t()).max(1).values
        logp = torch.log_softmax(z, 1).view(B, K, V)
        ban = rc.ban_mask(seq.view(B * K, L), t, V, 2, ~fin.view(-1), **CONS).view(B, K, V)
        cand = torch.where(ban | fin[:, :, None], torch.full_like(logp, -float("inf")), score[:, :, None] + logp)
        cand[:, :, 0] = torch.where(fin, score, cand[:, :, 0])
        par, tok = tr[t, :, :, 0], tr[t, :, :, 1]
        chosen = cand.view(B, K * V).gather(1, par * V + tok)
        kth = torch.topk(cand.view(B, K * V), K, dim=1).values[:, -1]
        tol = (16 * U_TC * (t + 1) * sc.view(B, K).max(1).values + 1e-4)
        bad = ~torch.isfinite(chosen) | (chosen < kth[:, None] - tol[:, None])
        real += int(bad.sum())
        near += int((chosen < kth[:, None]).sum())
        checked += B * K
        pf = fin.gather(1, par)
        score = chosen
        fin = pf | (tok == 2)
        seq = seq.gather(1, par[:, :, None].expand(B, K, L)).clone()
        seq[:, :, t] = tok
        rows = (torch.arange(B, device="cuda")[:, None] * K + par).reshape(-1)
        hs = [h[rows] for h in hs]
        cs = [c[rows] for c in cs]
        x = P["decoder.embed.weight"][tok.reshape(-1)]
    REPORT["beam_c2/%s/layers%d" % (mode_name, layers)] = dict(checked=checked, below_kth_within_rounding=near, real=real)
    assert real == 0
    check_constraints(ids, lengths, L, 5, 3, {0, 1, 3}, "beam_c2/%s/l%d" % (mode_name, layers))


NONBINDING = dict(min_length=1, no_repeat_ngram_size=21, bad_ids=[-5, 10000, 123456])     # L = 20, V = 10 000


@pytest.mark.parametrize("mode_name", list(MODES))
def test_non_binding_constraints_are_bit_identical(mode_name):
    _lib = L_()
    from gic_b200.generator import decode_beam, sample_captions
    mode = MODES[mode_name]
    B, L = 32, 20
    dec, _ = c2_decoder(1)
    feats = torch.randn(B, 512, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    a = decode_beam(dec, feats, 3, L, 0.0, 2, mode=mode)
    with _lib.expect_kernels("ban_rows_kernel"):
        b = decode_beam(dec, feats, 3, L, 0.0, 2, mode=mode, **NONBINDING)
        torch.cuda.synchronize()
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    for k, p in ((0, 1.0), (16, 0.9)):
        set_rng(5, 0)
        a = sample_captions(dec, feats, 2, L, 1.0, k, p, 2, mode=mode)
        set_rng(5, 0)
        b = sample_captions(dec, feats, 2, L, 1.0, k, p, 2, mode=mode, **NONBINDING)
        torch.cuda.synchronize()
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    set_rng(0, 0)


def test_graph_replay_and_determinism():
    _lib = L_()
    from gic_b200.generator import decode_beam, sample_captions
    B, L = 64, 20
    dec, _ = c2_decoder(1)
    feats = torch.randn(B, 512, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    eager = decode_beam(dec, feats, 3, L, 0.0, 2, mode=1, **CONS)
    again = decode_beam(dec, feats, 3, L, 0.0, 2, mode=1, **CONS)
    for x, y in zip(eager, again):
        assert torch.equal(x, y)
    set_rng(11, 0)
    s1 = sample_captions(dec, feats, 2, L, 1.0, 16, 0.9, 2, mode=1, **CONS)
    set_rng(11, 0)
    s2 = sample_captions(dec, feats, 2, L, 1.0, 16, 0.9, 2, mode=1, **CONS)
    for x, y in zip(s1, s2):
        assert torch.equal(x, y)
    # capture both constrained calls into one graph and replay it (bad ids already on the device: nothing to copy)
    dcons = dict(CONS, bad_ids=torch.tensor(CONS["bad_ids"], device="cuda"))
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        set_rng(11, 0)
        decode_beam(dec, feats, 3, L, 0.0, 2, mode=1, **dcons)          # warm-up on the capture stream
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            gb = decode_beam(dec, feats, 3, L, 0.0, 2, mode=1, **dcons)
            gs = sample_captions(dec, feats, 2, L, 1.0, 16, 0.9, 2, mode=1, **dcons)
    for o in list(gb) + list(gs):
        o.zero_()
    g.replay()
    torch.cuda.synchronize()
    set_rng(0, 0)
    for x, y in zip(gb, eager):
        assert torch.equal(x, y)
    for x, y in zip(gs, s1):
        assert torch.equal(x, y)


def test_instructor_state_untouched():
    L_()
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=500, gen_embed_dim=32, gen_hidden_dim=32, disc_num_filters=[4, 4, 4], conditional_gan=0,
                     device="cuda")
    inst = GANInstructor(a, device="cuda:0")
    before = {k: v.clone() for k, v in inst.gen.state_dict().items()}
    rng = torch.get_rng_state()
    ids, _, lengths = inst.generate(batch_size=8, beam_size=3, max_caption_len=12, **CONS)
    sids, _, slen = inst.sample_captions(batch_size=8, num_samples=2, max_caption_len=12, top_k=5, seed=3, **CONS)
    torch.cuda.synchronize()
    check_constraints(ids, lengths, 12, 5, 3, {0, 1, 3}, "instructor/beam")
    check_constraints(sids, slen, 12, 5, 3, {0, 1, 3}, "instructor/sample")
    for k, v in inst.gen.state_dict().items():
        assert torch.equal(v, before[k]), k
    assert torch.equal(torch.get_rng_state(), rng)


def test_abi_error_cases():
    _lib = L_()
    lib = _lib.lib()
    B, K, L, V, E, H = 2, 3, 6, 40, 8, 8
    dec, _ = make_decoder(V, E, H, 1, 1, 1.0)
    from gic_b200.generator import lstm_split
    W_ih, W_hh, b_ih, b_hh = lstm_split([w.detach().contiguous() for w in dec.lstm_params()])
    f = torch.zeros(B, E, device="cuda")
    bad = torch.tensor([0, 1], dtype=torch.int64, device="cuda")
    ids = torch.empty(B, K, L, dtype=torch.int64, device="cuda")
    sc = torch.empty(B, K, device="cuda")
    ln = torch.empty(B, K, dtype=torch.int32, device="cuda")
    ws = torch.empty(1 << 20, device="cuda")
    args = lambda: (_lib.ptr(f), _lib.ptr(dec.embed.weight), _lib.ptr_array(W_ih), _lib.ptr_array(W_hh),  # noqa: E731
                    _lib.ptr_array(b_ih), _lib.ptr_array(b_hh), _lib.ptr(dec.linear.weight), _lib.ptr(dec.linear.bias))

    def beam(c, k=K):
        return lib.gic_decode_beam_constrained(0, *args(), B, k, L, V, E, H, 1, 2, 0.0, C.byref(c), _lib.ptr(ids),
                                               _lib.ptr(sc), _lib.ptr(ln), None, _lib.ptr(ws), _lib.stream())

    def sample(c, k=0):
        return lib.gic_sample_captions_constrained(0, *args(), B, 1, L, V, E, H, 1, 2, 1.0, k, 1.0, C.byref(c),
                                                   _lib.ptr(ids), _lib.ptr(sc), _lib.ptr(ln), _lib.ptr(ws), _lib.stream())
    D = _lib.DecodeConstraints
    for c, k in ((D(-1, 0, None, 0), K), (D(L + 1, 0, None, 0), K), (D(0, -1, None, 0), K), (D(0, 0, _lib.ptr(bad), -1), K),
                 (D(1, 2, _lib.ptr(bad), V - 1 - (L - 1) - K + 1), K), (D(0, 0, _lib.ptr(bad), V - 16 + 1), 16)):
        assert beam(c, min(k, 16)) == 1
        assert sample(c, min(k, 16)) == 1
    assert beam(D(0, 0, None, 2)) == 2
    assert sample(D(0, 0, None, 2)) == 2
    assert beam(D(2, 2, _lib.ptr(bad), 2)) == 0
    torch.cuda.synchronize()
    h = torch.zeros(4, H, device="cuda")
    out = torch.empty(4, 4, device="cuda")
    tok = torch.empty(4, 4, dtype=torch.int64, device="cuda")
    assert lib.gic_vocab_topk_masked(1, _lib.ptr(h), _lib.ptr(dec.linear.weight), _lib.ptr(dec.linear.bias), 4, V, H, 4,
                                     _lib.ptr(out), _lib.ptr(tok), None, None, _lib.ptr(ws), _lib.stream()) == 2
    assert lib.gic_vocab_topk_masked(1, _lib.ptr(h), _lib.ptr(dec.linear.weight), _lib.ptr(dec.linear.bias), 4, V, H, 17,
                                     _lib.ptr(out), _lib.ptr(tok), None, _lib.ptr(ws), _lib.ptr(ws), _lib.stream()) == 1
    assert lib.gic_vocab_sample_masked(1, _lib.ptr(h), _lib.ptr(dec.linear.weight), _lib.ptr(dec.linear.bias), 4, V, H, 0,
                                       1.0, 0, 1.0, _lib.ptr(tok), _lib.ptr(out), None, _lib.ptr(ws), _lib.stream()) == 2
    assert lib.gic_vocab_sample_masked(1, _lib.ptr(h), _lib.ptr(dec.linear.weight), _lib.ptr(dec.linear.bias), 4, V, H, 0,
                                       0.0, 0, 1.0, _lib.ptr(tok), _lib.ptr(out), _lib.ptr(ws), _lib.ptr(ws),
                                       _lib.stream()) == 1
