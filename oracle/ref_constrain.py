"""CPU oracle for constrained caption generation (EXTENSION).  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED BY REFERENCE: kawshik8/GAN-Image-Captioning has no beam search, no sampled captions and no decoding
constraints.  The constraints are defined HERE, in float64, on top of the beam search of ``oracle/ref_beam.py`` and the
sampling of ``oracle/ref_sample.py`` (whose functions are reused unchanged); the CUDA path (include/gic_b200.h
gic_decode_constraints_t, gic_decode_beam_constrained, gic_sample_captions_constrained, gic_vocab_topk_masked,
gic_vocab_sample_masked) is tested against this file.  Only ``tests/`` may import it.

Definition, for row m at step t with its generated prefix y[0..t-1] (sampling: ids[m, :t]; beam search: the tokens along
the beam's trace; the step-0 input is not part of it): Ban(m, t) = banned_tokens(y, t, ...), the union of
  bad_ids inside [0, V) (ids outside are ignored);
  {eos_id} while t + 1 < min_length (every returned length is then >= min(min_length, L));
  for n = no_repeat_ngram_size >= 1 and t >= n - 1: { y[s + n - 1] : 0 <= s <= t - n, y[s .. s + n - 2] ==
  y[t - n + 1 .. t - 1] } (no n-gram occurs twice in a caption; n = 1 bans every token already emitted).
Banned tokens are removed from the candidates and nothing else changes:
  beam search: a live beam k offers (k, w) only for w outside Ban, at score_k + log_softmax(z)[w] (the unfiltered model);
    frozen beams still offer (k, PAD);
  sampling: S is the top_k largest allowed z (every allowed column at top_k = 0), then the nucleus inside it; the keys
    z / T + g(u[t, m, w]) use the same uniforms; caption_logp stays unfiltered at temperature 1.
With every constraint off the functions here return what ref_beam.beam_search / ref_sample.sample_captions /
ref_sample.step_check return.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import ref_port as rp
from .ref_beam import PAD_ID, EOS_ID, _decoder_layers, _lstm_stack
from .ref_sample import candidate_mask, top_k_gap


def banned_tokens(prefix, t, V, eos_id, min_length=0, no_repeat_ngram_size=0, bad_ids=()):
    """The set Ban of the definition for a row whose generated tokens are prefix[0..t-1]."""
    y = [int(w) for w in prefix[:t]]
    ban = {int(w) for w in bad_ids if 0 <= int(w) < V}
    if t + 1 < min_length:
        ban.add(int(eos_id))
    n = int(no_repeat_ngram_size)
    if n >= 1 and t >= n - 1:
        tail = y[t - n + 1:t]
        for s in range(t - n + 1):
            if y[s:s + n - 1] == tail:
                ban.add(y[s + n - 1])
    return ban


def ban_mask(prefixes, t, V, eos_id, live, min_length=0, no_repeat_ngram_size=0, bad_ids=()):
    """Boolean [R, V]: row r's banned_tokens(prefixes[r], t, ...) where live[r], nothing where not."""
    mask = torch.zeros(prefixes.shape[0], V, dtype=torch.bool, device=prefixes.device)
    rows = prefixes[:, :t].tolist()
    for r, ok in enumerate(live.tolist()):
        if ok:
            for w in banned_tokens(rows[r], t, V, eos_id, min_length, no_repeat_ngram_size, bad_ids):
                mask[r, w] = True
    return mask


def draw(z, u, temperature, top_k, top_p, ban):
    """ref_sample.draw with the columns ban[M,V] removed before S is formed: (token[M], key[M,V], S, cut)."""
    S, cut = candidate_mask(z.masked_fill(ban, -float("inf")), temperature, top_k, top_p)
    S &= ~ban
    key = torch.where(S, z / temperature + rp.gumbel_noise(u.double()), torch.full_like(z, -float("inf")))
    return key.argmax(1), key, S, cut


def beam_search(p, features, K, L, eos_id=EOS_ID, length_penalty=0.0, min_length=0, no_repeat_ngram_size=0, bad_ids=()):
    """ref_beam.beam_search under the constraints: the same dict(ids, scores, lengths, trace, margin)."""
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    layers = _decoder_layers(P)
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    V, H = W_out.shape
    B = features.shape[0]
    hs = [features.new_zeros(B * K, H, dtype=torch.float64) for _ in range(layers)]
    cs = [features.new_zeros(B * K, H, dtype=torch.float64) for _ in range(layers)]
    x = features.double().repeat_interleave(K, 0)
    dev = features.device
    score = torch.full((B, K), -float("inf"), dtype=torch.float64, device=dev)
    score[:, 0] = 0.0
    fin = torch.zeros(B, K, dtype=torch.bool, device=dev)
    length = torch.full((B, K), L, dtype=torch.int64, device=dev)
    seq = torch.zeros(B, K, L, dtype=torch.int64, device=dev)
    trace = torch.zeros(L, B, K, 2, dtype=torch.int64, device=dev)
    margin = float("inf")
    for t in range(L):
        top = _lstm_stack(P, x, hs, cs)
        logp = F.log_softmax(F.linear(top, W_out, b_out), -1).view(B, K, V)
        cand = score[:, :, None] + logp
        ban = ban_mask(seq.view(B * K, L), t, V, eos_id, ~fin.view(-1), min_length, no_repeat_ngram_size, bad_ids)
        valid = ~fin[:, :, None].expand(B, K, V) & ~ban.view(B, K, V)
        valid[:, :, PAD_ID] |= fin
        cand = torch.where(fin[:, :, None], score[:, :, None].expand(B, K, V), cand)
        cand = torch.where(valid, cand, torch.full_like(cand, -float("inf")))
        flat = cand.view(B, K * V)
        order = torch.sort(flat, dim=1, descending=True, stable=True).indices
        vflat = valid.view(B, K * V)
        parent = torch.zeros(B, K, dtype=torch.int64, device=dev)
        tok = torch.zeros(B, K, dtype=torch.int64, device=dev)
        for b in range(B):
            vb, sel = vflat[b].tolist(), []
            for i in order[b].tolist():
                if vb[i]:
                    sel.append(i)
                    if len(sel) > K:
                        break
            fs = [float(flat[b, i]) for i in sel]
            for i in range(len(fs) - 1):
                if fs[i + 1] > -float("inf"):
                    margin = min(margin, fs[i] - fs[i + 1])
            sel = torch.tensor(sel[:K], device=dev)
            parent[b], tok[b] = sel // V, sel % V
        new_score = flat.gather(1, parent * V + tok)
        pf = fin.gather(1, parent)
        new_len = torch.where(pf, length.gather(1, parent), torch.where(tok == eos_id, torch.full_like(tok, t + 1),
                                                                       torch.full_like(tok, L)))
        seq = seq.gather(1, parent[:, :, None].expand(B, K, L)).clone()
        seq[:, :, t] = tok
        score, fin, length = new_score, pf | (tok == eos_id), new_len
        trace[t, :, :, 0], trace[t, :, :, 1] = parent, tok
        rows = (torch.arange(B, device=dev)[:, None] * K + parent).reshape(-1)
        hs = [h[rows] for h in hs]
        cs = [c[rows] for c in cs]
        x = emb[tok.reshape(-1)]
    norm = score / length.double() ** length_penalty
    order = torch.sort(norm, dim=1, descending=True, stable=True).indices
    if K > 1:
        sn = norm.gather(1, order)
        margin = min(margin, float((sn[:, :-1] - sn[:, 1:]).min()))
    return dict(ids=seq.gather(1, order[:, :, None].expand(B, K, L)), scores=score.gather(1, order),
                lengths=length.gather(1, order).to(torch.int32), trace=trace, margin=margin)


def sample_captions(p, features, n, L, temperature, top_k, top_p, eos_id, U, min_length=0, no_repeat_ngram_size=0,
                    bad_ids=()):
    """ref_sample.sample_captions under the constraints (the prefix of row m is its own ids[m, :t])."""
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    layers = _decoder_layers(P)
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    V, H = W_out.shape
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
        ban = ban_mask(ids, t, V, eos_id, ~fin, min_length, no_repeat_ngram_size, bad_ids)
        tok, _, _, _ = draw(z, U[t].to(dev), temperature, top_k, top_p, ban)
        lp = z.gather(1, tok[:, None])[:, 0] - torch.logsumexp(z, 1)
        live = ~fin
        ids[:, t] = torch.where(live, tok, torch.zeros_like(tok))
        total += torch.where(live, lp, torch.zeros_like(lp))
        newly = live & (tok == eos_id)
        length = torch.where(newly, torch.full_like(length, t + 1), length)
        fin = fin | newly
        x = emb[tok]
    return dict(ids=ids, caption_logp=total, lengths=length.to(torch.int32))


def step_check(p, features, n, ids, temperature, top_k, top_p, eos_id, U, min_length=0, no_repeat_ngram_size=0, bad_ids=()):
    """ref_sample.step_check under the constraints: the oracle follows the GPU's own ids[B n, L], its banned sets taken
    from that prefix; kgap is taken over the allowed columns.  Same dict of per-(row, step) tensors."""
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    layers = _decoder_layers(P)
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    V, H = W_out.shape
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
        ban = ban_mask(ids, t, V, eos_id, ~fin, min_length, no_repeat_ngram_size, bad_ids)
        tok, key, S, cut = draw(z, U[t].to(dev), temperature, top_k, top_p, ban)
        two = torch.topk(key, 2, dim=1).values if key.shape[1] > 1 else torch.cat([key, key], 1)
        g = ids[:, t]
        kg = key.gather(1, g[:, None])[:, 0]
        out["win"].append(tok)
        out["margin"].append(two[:, 0] - two[:, 1])
        out["gpu_gap"].append(two[:, 0] - kg)
        out["in_S"].append(S.gather(1, g[:, None])[:, 0])
        out["kgap"].append(top_k_gap(z.masked_fill(ban, -float("inf")), top_k))
        out["cut"].append(cut)
        out["scale"].append((top.abs() @ W_out.abs().t()).max(1).values)
        out["live"].append(~fin)
        fin = fin | (g == eos_id)
        x = emb[g]
    return {k: torch.stack(v, 1) for k, v in out.items()}
