"""CPU self-check of the constrained-generation oracle (oracle/ref_constrain.py: banned_tokens and the constrained
beam_search, sample_captions and step_check), against hand-worked cases, exhaustive search and the unconstrained oracles,
and the host-side constraint checks of Decoder / GANInstructor."""
import itertools

import pytest
import torch

from oracle import ref_beam as rx
from oracle import ref_constrain as rc
from oracle import ref_port as rp
from oracle import ref_sample as rs

from test_cpu_beam import _params, _seq_logprob


def test_banned_tokens_hand_worked():
    bt = rc.banned_tokens
    y = [5, 6, 5, 6, 5]
    # n = 1: every emitted token
    assert bt(y, 5, 10, 2, no_repeat_ngram_size=1) == {5, 6}
    assert bt(y, 0, 10, 2, no_repeat_ngram_size=1) == set()
    # n = 2: the last token 5 was followed by 6 before
    assert bt(y, 5, 10, 2, no_repeat_ngram_size=2) == {6}
    assert bt(y, 4, 10, 2, no_repeat_ngram_size=2) == {5}          # prefix 5 6 5 6: after 6 came 5
    # n = 3, overlapping repeats: tail (6, 5) occurred at s = 1 -> 6
    assert bt(y, 5, 10, 2, no_repeat_ngram_size=3) == {6}
    assert bt([7, 7, 7], 3, 10, 2, no_repeat_ngram_size=3) == {7}   # 7 7 7 overlaps itself
    assert bt([7, 7, 7], 3, 10, 2, no_repeat_ngram_size=2) == {7}
    # t < n - 1: nothing to match yet
    assert bt([4], 1, 10, 2, no_repeat_ngram_size=3) == set()
    assert bt([4, 4], 2, 10, 2, no_repeat_ngram_size=3) == set()
    # only the prefix y[0 .. t - 1] counts
    assert bt([4, 9, 4, 9, 9], 3, 10, 2, no_repeat_ngram_size=2) == {9}
    # min_length: EOS banned while t + 1 < min_length
    assert bt([], 0, 10, 2, min_length=0) == set()
    assert bt([], 0, 10, 2, min_length=1) == set()
    assert bt([], 0, 10, 2, min_length=2) == {2}
    L = 4
    assert [2 in bt([3] * t, t, 10, 2, min_length=L) for t in range(L)] == [True, True, True, False]
    # bad ids: duplicates and ids outside [0, V) are ignored
    assert bt([], 0, 10, 2, bad_ids=[0, 1, 1, 3, -1, 10, 99]) == {0, 1, 3}
    assert bt(y, 5, 10, 2, min_length=9, no_repeat_ngram_size=2, bad_ids=[0]) == {0, 2, 6}


def _admissible(seq, eos, V, min_length, n, bad):
    for t, w in enumerate(seq):
        if w in rc.banned_tokens(seq, t, V, eos, min_length, n, bad):
            return False
        if w == eos:
            return True
    return True


def test_constrained_beam_equals_exhaustive_search():
    cases = [dict(min_length=3), dict(no_repeat_ngram_size=1), dict(no_repeat_ngram_size=2, bad_ids=[0]),
             dict(bad_ids=[1, 3, 7], min_length=2)]
    for layers, (V, L), cons in itertools.product((1, 2), ((4, 3), (5, 3)), cases):
        K = V ** (L - 1)
        p = _params(V, 6, 8, layers, seed=31 + V + L + layers)
        feats = torch.randn(2, 6, generator=torch.Generator().manual_seed(5))
        out = rc.beam_search(p, feats, K, L, eos_id=2, **cons)
        args = (cons.get("min_length", 0), cons.get("no_repeat_ngram_size", 0), cons.get("bad_ids", ()))
        for b in range(2):
            best = {}
            for seq in itertools.product(range(V), repeat=L):
                if not _admissible(seq, 2, V, *args):
                    continue
                s, n = _seq_logprob(p, feats[b], seq, 2)
                best[tuple(seq[:n]) + (0,) * (L - n)] = (s, n)
            ranked = sorted(best.items(), key=lambda kv: -kv[1][0])
            want_ids, (want_s, want_n) = ranked[0]
            assert tuple(out["ids"][b, 0].tolist()) == want_ids, (layers, V, L, cons, b)
            assert abs(float(out["scores"][b, 0]) - want_s) < 1e-9
            assert int(out["lengths"][b, 0]) == want_n
            live = [r for r in out["ids"][b].tolist() if tuple(r) in best]
            assert set(tuple(r) for r in live) == set(k for k, _ in ranked[:len(live)])


CONS = dict(min_length=4, no_repeat_ngram_size=2, bad_ids=[0, 1, 3])


@pytest.mark.parametrize("layers", [1, 2])
def test_constrained_greedy_beam_is_constrained_top_k_1(layers):
    B, L, V, E, H = 5, 8, 12, 8, 12
    p = _params(V, E, H, layers, seed=3 + layers)
    p["decoder.linear.bias"][2] += 1.0
    feats = torch.randn(B, E, generator=torch.Generator().manual_seed(layers), dtype=torch.float64)
    U = torch.rand(L, B, V, generator=torch.Generator().manual_seed(9), dtype=torch.float64)
    got = rc.sample_captions(p, feats, 1, L, 0.7, 1, 1.0, 2, U, **CONS)
    ref = rc.beam_search(p, feats, 1, L, eos_id=2, **CONS)
    assert torch.equal(got["ids"], ref["ids"][:, 0])
    assert torch.equal(got["lengths"], ref["lengths"][:, 0])
    torch.testing.assert_close(got["caption_logp"], ref["scores"][:, 0], rtol=1e-12, atol=1e-12)


NONBINDING = dict(min_length=1, no_repeat_ngram_size=9, bad_ids=[-1, 40, 1000])      # L = 8, V = 12


@pytest.mark.parametrize("cons", [{}, NONBINDING])
def test_off_or_non_binding_constraints_reproduce_the_unconstrained_oracles(cons):
    B, L, V, E, H = 4, 8, 12, 8, 12
    p = _params(V, E, H, 2, seed=17)
    feats = torch.randn(B, E, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    U = torch.rand(L, B * 3, V, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    a, b = rx.beam_search(p, feats, 3, L, length_penalty=0.5), rc.beam_search(p, feats, 3, L, length_penalty=0.5, **cons)
    for k in ("ids", "scores", "lengths", "trace", "margin"):
        assert torch.equal(a[k], b[k]) if k != "margin" else a[k] == b[k], k
    for top_k, top_p in ((0, 1.0), (4, 0.8)):
        a = rs.sample_captions(p, feats, 3, L, 1.3, top_k, top_p, 2, U)
        b = rc.sample_captions(p, feats, 3, L, 1.3, top_k, top_p, 2, U, **cons)
        for k in a:
            assert torch.equal(a[k], b[k]), k
        ca = rs.step_check(p, feats, 3, a["ids"], 1.3, top_k, top_p, 2, U)
        cb = rc.step_check(p, feats, 3, a["ids"], 1.3, top_k, top_p, 2, U, **cons)
        for k in ca:
            assert torch.equal(ca[k], cb[k]), k


def _check_caption(ids, length, L, min_length, n, bad, eos=2):
    row = ids.tolist()
    live = row[:length]
    assert length >= min(min_length, L)
    assert not any(w in bad for w in live), row
    if n:
        grams = [tuple(live[s:s + n]) for s in range(len(live) - n + 1)]
        assert len(grams) == len(set(grams)), row
    assert all(w == 0 for w in row[length:])
    if length < L:
        assert live[-1] == eos


@pytest.mark.parametrize("cons", [CONS, dict(no_repeat_ngram_size=1), dict(min_length=8, bad_ids=[0, 1, 3, 5])])
def test_oracle_outputs_satisfy_constraints(cons):
    B, L, V, E, H = 6, 8, 12, 8, 12
    p = _params(V, E, H, 1, seed=23, scale=8.0)
    p["decoder.linear.bias"][2] += 2.0                # eager EOS, so min_length binds
    p["decoder.linear.bias"][0] += 2.0                # PAD would be likely without the ban
    feats = torch.randn(B, E, generator=torch.Generator().manual_seed(6), dtype=torch.float64)
    U = torch.rand(L, B * 2, V, generator=torch.Generator().manual_seed(7), dtype=torch.float64)
    args = (cons.get("min_length", 0), cons.get("no_repeat_ngram_size", 0), set(cons.get("bad_ids", ())))
    out = rc.beam_search(p, feats, 4, L, **cons)
    for b, k in itertools.product(range(B), range(4)):
        _check_caption(out["ids"][b, k], int(out["lengths"][b, k]), L, *args)
    for top_k, top_p in ((0, 1.0), (3, 0.9)):
        s = rc.sample_captions(p, feats, 2, L, 1.0, top_k, top_p, 2, U, **cons)
        for m in range(B * 2):
            _check_caption(s["ids"][m], int(s["lengths"][m]), L, *args)
        chk = rc.step_check(p, feats, 2, s["ids"], 1.0, top_k, top_p, 2, U, **cons)
        assert bool(torch.where(chk["live"], chk["win"] == s["ids"], torch.ones_like(chk["live"])).all())


# ---- host-side argument checks (V = 12, L = 2 unless given) ----
BAD = [dict(min_length=-1), dict(min_length=3), dict(no_repeat_ngram_size=-1), dict(bad_ids=[12]), dict(bad_ids=[-1]),
       dict(bad_ids=list(range(10)), min_length=1)]


def _no_gpu(monkeypatch):
    from gic_b200 import _lib

    def boom(*a, **k):
        raise AssertionError("GPU work started before the arguments were checked")
    monkeypatch.setattr(_lib, "require_cuda", boom)


def _decoder():
    from gic_b200.generator import Decoder
    return Decoder(rp.args_for(dict(B=1, L=2, V=12, E=8, H=8, layers=1, feat=0, filters=[4, 4, 4])))


@pytest.mark.parametrize("bad", BAD)
def test_decoder_rejects_bad_constraints(bad, monkeypatch):
    dec = _decoder()
    _no_gpu(monkeypatch)
    with pytest.raises(ValueError):
        dec.beam_search(torch.zeros(2, 8), beam_size=2, max_caption_len=2, **bad)
    with pytest.raises(ValueError):
        dec.sample_captions(torch.zeros(2, 8), max_caption_len=2, top_k=2, **bad)


def test_capacity_counts_width_and_ngram_budget(monkeypatch):
    dec = _decoder()
    _no_gpu(monkeypatch)
    # V 12 - 3 bad - 1 (min_length) - (L - 1) = 4 (n-gram) leaves 4: beam 5 / top_k 5 do not fit
    kw = dict(max_caption_len=5, min_length=2, no_repeat_ngram_size=2, bad_ids=[0, 1, 3])
    with pytest.raises(ValueError):
        dec.beam_search(torch.zeros(2, 8), beam_size=5, **kw)
    with pytest.raises(ValueError):
        dec.sample_captions(torch.zeros(2, 8), top_k=5, **kw)
    with pytest.raises(AssertionError):          # 4 fits: the checks pass and the GPU path starts
        dec.beam_search(torch.zeros(2, 8), beam_size=4, **kw)


@pytest.mark.parametrize("bad", BAD)
@pytest.mark.parametrize("cgan", [0, 1])
def test_instructor_rejects_bad_constraints(bad, cgan, monkeypatch):
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=12, gen_embed_dim=8, gen_hidden_dim=8, disc_num_filters=[4, 4, 4], conditional_gan=cgan,
                     feature_dim=6, device="cpu")
    inst = GANInstructor(a, device="cpu")
    _no_gpu(monkeypatch)
    kw = dict(pooled=torch.zeros(3, 6)) if cgan else dict(batch_size=3)
    with pytest.raises(ValueError):
        inst.generate(**kw, beam_size=2, max_caption_len=2, **bad)
    with pytest.raises(ValueError):
        inst.sample_captions(**kw, max_caption_len=2, top_k=2, **bad)
