"""CPU oracle for sampled caption generation (EXTENSION).  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED BY REFERENCE: kawshik8/GAN-Image-Captioning draws captions only through Decoder.sample's Gumbel-softmax
(src/generator.py:55-96), with no sampling temperature on the ids, no end of sentence and no top-k / top-p.  Sampling is
defined HERE, in float64, with the LSTM stack of ``oracle/ref_beam.py`` and the Gumbel noise of ``oracle/ref_port.py``; the
CUDA path (include/gic_b200.h gic_sample_captions, gic_vocab_sample) is tested against this file.  Only ``tests/`` may
import it.

Definition, for row m = b n + j at step t (mirrored in include/gic_b200.h):
  z = h_top W_out^T + b_out, lse = logsumexp(z) (temperature 1, no filter)
  S: top_k = 0 the whole vocabulary, else the top_k largest z (ties -> lower token); then, if top_p < 1, the shortest
     prefix of S in descending order whose cumulative softmax(z_S / temperature) is >= top_p (at least one token)
  token = argmax over S of z / temperature + gumbel_noise(U[t, m]) (ties -> lower token); logp = z_token - lse
  a row that emits eos_id is frozen: PAD (0) after, length = tokens up to and including EOS (L if none), caption_logp =
  sum of logp over its live steps; the next input is embed[token]
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import ref_port as rp
from .ref_beam import _decoder_layers, _lstm_stack


def candidate_order(z, top_k):
    """Columns of z[M,V] in descending order, ties -> lower column; the first top_k (all V when top_k = 0)."""
    order = torch.sort(z, dim=1, descending=True, stable=True).indices
    return order if top_k == 0 else order[:, :top_k]


def top_k_gap(z, top_k):
    """Per row of z[M,V]: the top_k-th largest z minus the next one (inf when top_k = 0 or top_k = V)."""
    if top_k == 0 or top_k >= z.shape[1]:
        return torch.full((z.shape[0],), float("inf"), dtype=torch.float64, device=z.device)
    v = torch.topk(z, top_k + 1, dim=1).values
    return v[:, top_k - 1] - v[:, top_k]


def candidate_mask(z, temperature, top_k, top_p):
    """Boolean S[M,V] of the definition, and per row the distance of the nucleus cut from top_p (inf when top_p = 1):
    min over the candidates of |exclusive cumulative mass - top_p|, the margin by which each one's membership is decided."""
    M, V = z.shape
    order = candidate_order(z, top_k)
    S = torch.zeros(M, V, dtype=torch.bool, device=z.device)
    cut = torch.full((M,), float("inf"), dtype=torch.float64, device=z.device)
    if top_p >= 1:
        S.scatter_(1, order, True)
        return S, cut
    q = F.softmax(z.gather(1, order) / temperature, dim=1)
    excl = torch.cumsum(q, 1) - q
    keep = excl < top_p
    keep[:, 0] = True
    S.scatter_(1, order, keep)
    cut = (excl[:, 1:] - top_p).abs().min(1).values if order.shape[1] > 1 else cut
    return S, cut


def draw(z, u, temperature, top_k, top_p):
    """The token of each row of z[M,V] with uniforms u[M,V]: returns (token[M], key[M,V] with -inf outside S, S, cut)."""
    S, cut = candidate_mask(z, temperature, top_k, top_p)
    key = torch.where(S, z / temperature + rp.gumbel_noise(u.double()), torch.full_like(z, -float("inf")))
    return key.argmax(1), key, S, cut          # argmax: first maximum, ties -> lower token


def sample_captions(p, features, n, L, temperature, top_k, top_p, eos_id, U):
    """float64 oracle: features[B,E], U[L, B n, V] -> dict(ids[B n, L], caption_logp[B n], lengths[B n] int32)."""
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    layers = _decoder_layers(P)
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    H = W_out.shape[1]
    dev = features.device
    x = features.double().repeat_interleave(n, 0)
    M = x.shape[0]
    hs = [torch.zeros(M, H, dtype=torch.float64, device=dev) for _ in range(layers)]
    cs = [torch.zeros(M, H, dtype=torch.float64, device=dev) for _ in range(layers)]
    ids = torch.zeros(M, L, dtype=torch.int64, device=dev)
    total = torch.zeros(M, dtype=torch.float64, device=dev)
    length = torch.full((M,), L, dtype=torch.int64, device=dev)
    fin = torch.zeros(M, dtype=torch.bool, device=dev)
    for t in range(L):
        top = _lstm_stack(P, x, hs, cs)
        z = F.linear(top, W_out, b_out)
        tok, _, _, _ = draw(z, U[t].to(dev), temperature, top_k, top_p)
        lp = z.gather(1, tok[:, None])[:, 0] - torch.logsumexp(z, 1)
        live = ~fin
        ids[:, t] = torch.where(live, tok, torch.zeros_like(tok))
        total += torch.where(live, lp, torch.zeros_like(lp))
        newly = live & (tok == eos_id)
        length = torch.where(newly, torch.full_like(length, t + 1), length)
        fin = fin | newly
        x = emb[tok]
    return dict(ids=ids, caption_logp=total, lengths=length.to(torch.int32))


def step_check(p, features, n, ids, temperature, top_k, top_p, eos_id, U):
    """Teacher-forced per-step checker: the oracle follows the GPU's own ids[B n, L] (so one flipped token does not make
    every later step diverge) and returns, per row and step, dict(win = the oracle's token, margin = its key minus the
    runner-up's among S, gpu_gap = its key minus the key of the GPU's token (inf when that token is outside S), in_S =
    whether the GPU's token is in S, kgap = z of the top_k-th candidate minus z of the next one (inf at top_k = 0: the
    margin by which the top-k set is decided), cut = the nucleus cut margin, scale = the logit scale max_w sum_j
    |h_j W[w,j]| (the operand-rounding bound is a multiple of it), live)."""
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    layers = _decoder_layers(P)
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    H = W_out.shape[1]
    dev = features.device
    ids = ids.to(dev)
    x = features.double().repeat_interleave(n, 0)
    M, L = ids.shape
    hs = [torch.zeros(M, H, dtype=torch.float64, device=dev) for _ in range(layers)]
    cs = [torch.zeros(M, H, dtype=torch.float64, device=dev) for _ in range(layers)]
    fin = torch.zeros(M, dtype=torch.bool, device=dev)
    out = {k: [] for k in ("win", "margin", "gpu_gap", "in_S", "kgap", "cut", "scale", "live")}
    for t in range(L):
        top = _lstm_stack(P, x, hs, cs)
        z = F.linear(top, W_out, b_out)
        tok, key, S, cut = draw(z, U[t].to(dev), temperature, top_k, top_p)
        two = torch.topk(key, 2, dim=1).values if key.shape[1] > 1 else torch.cat([key, key], 1)
        g = ids[:, t]
        kg = key.gather(1, g[:, None])[:, 0]
        out["win"].append(tok)
        out["margin"].append(two[:, 0] - two[:, 1])
        out["gpu_gap"].append(two[:, 0] - kg)
        out["in_S"].append(S.gather(1, g[:, None])[:, 0])
        out["kgap"].append(top_k_gap(z, top_k))
        out["cut"].append(cut)
        out["scale"].append((top.abs() @ W_out.abs().t()).max(1).values)
        out["live"].append(~fin)
        fin = fin | (g == eos_id)
        x = emb[g]
    return {k: torch.stack(v, 1) for k, v in out.items()}
