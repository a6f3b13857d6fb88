"""CPU self-check of the sampled-caption oracle (oracle/ref_sample.py): top_k = 1 is greedy beam search (K = 1), n = 1 at
temperature 1 over the full vocabulary is Decoder.sample's Gumbel argmax with the same uniforms, nucleus filtering on
hand-made distributions, and the host-side argument checks of Decoder.sample_captions / GANInstructor.sample_captions."""
import pytest
import torch

from oracle import ref_beam as rx
from oracle import ref_port as rp
from oracle import ref_sample as rs


def _params(V, E, H, layers, seed, scale=20.0, eos_boost=0.0):
    cfg = dict(B=2, L=4, V=V, E=E, H=H, layers=layers, feat=0, filters=[4, 4, 4])
    p = {k: v * scale for k, v in rp.make_params(rp.gen_param_shapes(rp.args_for(cfg)), seed).items()}
    p["decoder.linear.bias"][2] += eos_boost
    return p


@pytest.mark.parametrize("layers", [1, 2])
def test_top_k_1_is_greedy_beam_search(layers):
    B, L, V, E, H = 5, 7, 30, 8, 12
    p = _params(V, E, H, layers, seed=3 + layers, eos_boost=1.0)
    feats = torch.randn(B, E, generator=torch.Generator().manual_seed(layers), dtype=torch.float64)
    U = torch.rand(L, B, V, generator=torch.Generator().manual_seed(9), dtype=torch.float64)
    for T in (0.5, 1.0, 2.0):                # top_k = 1: one candidate, temperature and noise are irrelevant
        got = rs.sample_captions(p, feats, 1, L, T, 1, 1.0, 2, U)
        ref = rx.beam_search(p, feats, 1, L, eos_id=2)
        assert torch.equal(got["ids"], ref["ids"][:, 0])
        assert torch.equal(got["lengths"], ref["lengths"][:, 0])
        torch.testing.assert_close(got["caption_logp"], ref["scores"][:, 0], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("layers", [1, 2])
def test_full_vocabulary_at_t1_is_decoder_sample(layers):
    B, L, V, E, H = 6, 8, 25, 8, 12
    p = _params(V, E, H, layers, seed=21 + layers, scale=5.0, eos_boost=1.5)
    feats = torch.randn(B, E, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    U = torch.rand(L, B, V, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    got = rs.sample_captions(p, feats, 1, L, 1.0, 0, 1.0, 2, U)
    P = {k: v.double() for k, v in p.items()}
    _, ids, _ = rp.decoder_sample(P, feats, U, 1.0, L, layers=layers)
    eos_rows = 0
    for b in range(B):
        eos = (ids[b] == 2).nonzero()
        n = int(eos[0]) + 1 if len(eos) else L
        eos_rows += n < L
        assert torch.equal(got["ids"][b, :n], ids[b, :n])
        assert int(got["lengths"][b]) == n
        assert bool((got["ids"][b, n:] == 0).all())
    assert eos_rows > 0


def test_nucleus_on_hand_made_distributions():
    z = torch.zeros(1, 4, dtype=torch.float64)              # q = 1/4 each: the cumulative masses are exact
    for top_p, kept in ((0.25, [0]), (0.2, [0]), (0.5, [0, 1]), (0.5000001, [0, 1, 2]), (0.75, [0, 1, 2]), (1.0, [0, 1, 2, 3])):
        S, _ = rs.candidate_mask(z, 1.0, 4, top_p)
        assert S[0].nonzero()[:, 0].tolist() == kept, top_p
    # probabilities 0.5, 0.3, 0.15, 0.05 in shuffled columns; temperature 1
    q = torch.tensor([[0.15, 0.5, 0.05, 0.3]], dtype=torch.float64)
    z = q.log()
    for top_p, kept in ((0.4, [1]), (0.7, [1, 3]), (0.9, [0, 1, 3]), (0.99, [0, 1, 2, 3])):
        S, _ = rs.candidate_mask(z, 1.0, 4, top_p)
        assert sorted(S[0].nonzero()[:, 0].tolist()) == kept, top_p
    # top_k cuts first, ties go to the lower token, and the nucleus is taken inside the top k
    z = torch.tensor([[1.0, 3.0, 3.0, 2.0, 0.0]], dtype=torch.float64)
    S, _ = rs.candidate_mask(z, 1.0, 2, 1.0)
    assert S[0].nonzero()[:, 0].tolist() == [1, 2]
    S, _ = rs.candidate_mask(z, 1.0, 3, 0.4)                # q over {1, 2, 3} = 0.42, 0.42, 0.16: equal heads, 1 first
    assert S[0].nonzero()[:, 0].tolist() == [1]
    S, _ = rs.candidate_mask(z, 1.0, 3, 0.5)
    assert S[0].nonzero()[:, 0].tolist() == [1, 2]
    # temperature sharpens / flattens the nucleus
    z = torch.tensor([[2.0, 1.0, 0.0]], dtype=torch.float64)
    assert int(rs.candidate_mask(z, 0.1, 3, 0.9)[0].sum()) == 1
    assert int(rs.candidate_mask(z, 10.0, 3, 0.9)[0].sum()) == 3
    # the draw never leaves S
    u = torch.rand(4000, 5, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    z = torch.tensor([[1.0, 3.0, 3.0, 2.0, 0.0]], dtype=torch.float64).expand(4000, 5)
    tok, _, S, _ = rs.draw(z, u, 1.3, 3, 0.8)
    assert bool(S.gather(1, tok[:, None]).all())


BAD = [dict(temperature=0.0), dict(temperature=-1.0), dict(temperature=float("inf")), dict(temperature=float("nan")),
       dict(top_p=0.0), dict(top_p=1.5), dict(top_k=-1), dict(top_k=17), dict(top_k=0, top_p=0.9),
       dict(top_k=13), dict(num_samples=0), dict(max_caption_len=0)]          # V = 12 below


def _no_gpu(monkeypatch):
    """Every GPU path of the package starts with _lib.require_cuda(): it must not be reached."""
    from gic_b200 import _lib

    def boom(*a, **k):
        raise AssertionError("GPU work started before the arguments were checked")
    monkeypatch.setattr(_lib, "require_cuda", boom)


@pytest.mark.parametrize("bad", BAD + [dict(eos_id=12), dict(eos_id=-1)])
def test_decoder_sample_captions_rejects_bad_arguments(bad, monkeypatch):
    from gic_b200.generator import Decoder
    dec = Decoder(rp.args_for(dict(B=1, L=2, V=12, E=8, H=8, layers=1, feat=0, filters=[4, 4, 4])))
    _no_gpu(monkeypatch)
    with pytest.raises(ValueError):
        dec.sample_captions(torch.zeros(2, 8), **bad)


@pytest.mark.parametrize("bad", BAD)
@pytest.mark.parametrize("cgan", [0, 1])
def test_instructor_sample_captions_rejects_bad_arguments(bad, cgan, monkeypatch):
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=12, gen_embed_dim=8, gen_hidden_dim=8, disc_num_filters=[4, 4, 4], conditional_gan=cgan,
                     feature_dim=6, device="cpu")
    inst = GANInstructor(a, device="cpu")
    _no_gpu(monkeypatch)
    kw = dict(pooled=torch.zeros(3, 6)) if cgan else dict(batch_size=3)
    with pytest.raises(ValueError):
        inst.sample_captions(**kw, **bad)
    with pytest.raises(ValueError):                         # no step-0 input
        inst.sample_captions()
