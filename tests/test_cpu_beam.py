"""CPU self-check of the beam-search oracle (oracle/ref_beam.py beam_search): on tiny shapes with K >= V^(L-1) it must
return the exhaustive-search optimum, and K = 1 must be a plain greedy loop."""
import itertools

import torch
import torch.nn.functional as F

from oracle import ref_beam as rx
from oracle import ref_port as rp


def _params(V, E, H, layers, seed, scale=20.0):
    cfg = dict(B=2, L=4, V=V, E=E, H=H, layers=layers, feat=0, filters=[4, 4, 4])
    p = rp.make_params(rp.gen_param_shapes(rp.args_for(cfg)), seed)
    return {k: v * scale for k, v in p.items()}


def _seq_logprob(p, feat, seq, eos):
    """float64 log-probability of one caption (frozen after EOS: later tokens are PAD at probability 1)."""
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    layers = rx._decoder_layers(P)
    H = P["decoder.linear.weight"].shape[1]
    hs = [torch.zeros(1, H, dtype=torch.float64) for _ in range(layers)]
    cs = [torch.zeros(1, H, dtype=torch.float64) for _ in range(layers)]
    x = feat.double()[None]
    total, n = 0.0, len(seq)
    for t, w in enumerate(seq):
        top = rx._lstm_stack(P, x, hs, cs)
        total += float(F.log_softmax(F.linear(top, P["decoder.linear.weight"], P["decoder.linear.bias"]), -1)[0, w])
        if w == eos:
            n = t + 1
            break
        x = P["decoder.embed.weight"][w][None]
    return total, n


def test_beam_equals_exhaustive_search():
    for layers, (V, L), lp in itertools.product((1, 2), ((4, 3), (5, 3), (3, 4)), (0.0, 0.7)):
        K = V ** (L - 1)
        p = _params(V, 6, 8, layers, seed=11 + V + L + layers)
        feats = torch.randn(2, 6, generator=torch.Generator().manual_seed(3))
        out = rx.beam_search(p, feats, K, L, eos_id=2, length_penalty=lp)
        for b in range(2):
            best = {}
            for seq in itertools.product(range(V), repeat=L):
                s, n = _seq_logprob(p, feats[b], seq, 2)
                key = tuple(seq[:n]) + (0,) * (L - n)
                best[key] = (s, n)
            ranked = sorted(best.items(), key=lambda kv: -kv[1][0] / kv[1][1] ** lp)
            want_ids, (want_s, want_n) = ranked[0]
            assert tuple(out["ids"][b, 0].tolist()) == want_ids, (layers, V, L, lp, b)
            assert abs(float(out["scores"][b, 0]) - want_s) < 1e-9
            assert int(out["lengths"][b, 0]) == want_n
            if lp == 0.0:
                # beams are kept by raw score, so without a length penalty the K beams are the K best captions
                got = set(tuple(r) for r in out["ids"][b].tolist())
                assert got == set(k for k, _ in ranked[:K])


def test_k1_is_greedy():
    for layers in (1, 2):
        V, L = 7, 6
        p = _params(V, 6, 8, layers, seed=5 + layers, scale=10.0)
        feats = torch.randn(3, 6, generator=torch.Generator().manual_seed(4))
        out = rx.beam_search(p, feats, 1, L, eos_id=2)
        P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
        H = P["decoder.linear.weight"].shape[1]
        hs = [torch.zeros(3, H, dtype=torch.float64) for _ in range(layers)]
        cs = [torch.zeros(3, H, dtype=torch.float64) for _ in range(layers)]
        x = feats.double()
        done = torch.zeros(3, dtype=torch.bool)
        for t in range(L):
            top = rx._lstm_stack(P, x, hs, cs)
            tok = F.linear(top, P["decoder.linear.weight"], P["decoder.linear.bias"]).argmax(1)
            tok = torch.where(done, torch.zeros_like(tok), tok)
            assert torch.equal(out["ids"][:, 0, t], tok), (layers, t)
            done |= tok == 2
            x = P["decoder.embed.weight"][tok]


def test_output_invariants():
    p = _params(9, 6, 8, 2, seed=21, scale=15.0)
    feats = torch.randn(4, 6, generator=torch.Generator().manual_seed(8))
    out = rx.beam_search(p, feats, 4, 6, eos_id=2, length_penalty=0.5)
    ids, lens, sc = out["ids"], out["lengths"], out["scores"]
    for b in range(4):
        norm = sc[b] / lens[b].double() ** 0.5
        assert bool((norm[:-1] >= norm[1:]).all())
        rows = [tuple(r) for r in ids[b].tolist()]
        assert len(set(rows)) == len(rows)
        for k in range(4):
            n = int(lens[b, k])
            eos = (ids[b, k] == 2).nonzero()
            if len(eos):
                assert int(eos[0]) + 1 == n
                assert bool((ids[b, k, n:] == 0).all())
            else:
                assert n == ids.shape[2]
