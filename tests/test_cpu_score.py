"""CPU self-check of the teacher-forced scoring oracle (oracle/ref_score.py teacher_forced_logp): it must equal a float64
torch.nn.LSTM (batch_first) + nn.Linear + log_softmax teacher-forced forward, and its totals must equal beam_rescore's."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import ref_beam as rx
from oracle import ref_score as rs
from oracle import ref_port as rp


def _params(V, E, H, layers, seed, scale=10.0):
    cfg = dict(B=2, L=4, V=V, E=E, H=H, layers=layers, feat=0, filters=[4, 4, 4])
    p = rp.make_params(rp.gen_param_shapes(rp.args_for(cfg)), seed)
    return {k: v * scale for k, v in p.items()}


def _torch_forward(p, feats, ids, layers):
    """The same teacher-forced forward with torch.nn modules: inputs [features, embed[ids[:, :-1]]]."""
    V, H = p["decoder.linear.weight"].shape
    E = p["decoder.embed.weight"].shape[1]
    lstm = nn.LSTM(E, H, layers, batch_first=True).double()
    lin = nn.Linear(H, V).double()
    with torch.no_grad():
        for l in range(layers):
            for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                getattr(lstm, "%s_l%d" % (n, l)).copy_(p["decoder.lstm.%s_l%d" % (n, l)].double())
        lin.weight.copy_(p["decoder.linear.weight"].double())
        lin.bias.copy_(p["decoder.linear.bias"].double())
        emb = p["decoder.embed.weight"].double()
        x = torch.cat([feats.double()[:, None], emb[ids[:, :-1]]], 1)
        out, _ = lstm(x)
        return F.log_softmax(lin(out), -1)


@pytest.mark.parametrize("layers", [1, 2])
def test_teacher_forced_logp_equals_nn_lstm(layers):
    V, E, H, N, L = 37, 12, 16, 6, 7
    p = _params(V, E, H, layers, seed=3 + layers)
    g = torch.Generator().manual_seed(layers)
    feats = torch.randn(N, E, generator=g)
    ids = torch.randint(0, V, (N, L), generator=g)
    lengths = torch.tensor([0, 1, 3, 7, 9, -2])
    r = rs.teacher_forced_logp(p, feats, ids, lengths)
    ref = _torch_forward(p, feats, ids, layers)
    want = ref.gather(2, ids[:, :, None])[:, :, 0]
    live = torch.arange(L)[None] < lengths.clamp(0, L)[:, None]
    torch.testing.assert_close(r["logp"], torch.where(live, want, torch.zeros_like(want)), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(r["total"], r["logp"].sum(1), rtol=0, atol=0)
    assert torch.equal(r["argmax"], ref.argmax(2))
    top2 = torch.topk(ref, 2, dim=2).values
    torch.testing.assert_close(r["gap"], top2[..., 0] - top2[..., 1], rtol=1e-9, atol=1e-9)
    assert bool((r["scale"] > 0).all())
    full = rs.teacher_forced_logp(p, feats, ids)
    torch.testing.assert_close(full["logp"], want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("layers", [1, 2])
def test_teacher_forced_totals_equal_beam_rescore(layers):
    V, E, H, B, K, L = 29, 10, 14, 3, 2, 6
    p = _params(V, E, H, layers, seed=20 + layers)
    g = torch.Generator().manual_seed(7)
    feats = torch.randn(B, E, generator=g)
    ids = torch.randint(0, V, (B, K, L), generator=g)
    lengths = torch.randint(1, L + 1, (B, K), generator=g, dtype=torch.int32)
    total, scale = rx.beam_rescore(p, feats, ids, lengths)
    r = rs.teacher_forced_logp(p, feats.repeat_interleave(K, 0), ids.reshape(B * K, L), lengths.reshape(-1))
    torch.testing.assert_close(r["total"].view(B, K), total, rtol=1e-12, atol=1e-12)
    live = torch.arange(L)[None] < lengths.reshape(-1, 1).long()
    torch.testing.assert_close(torch.where(live, r["scale"], torch.zeros_like(r["scale"])).sum(1).view(B, K), scale,
                               rtol=1e-12, atol=1e-12)
