"""CPU oracle for caption generation by beam search (EXTENSION).  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED BY REFERENCE: kawshik8/GAN-Image-Captioning has no beam search and no decoding other than
Decoder.sample (src/generator.py:55-81).  The search is defined HERE, in float64, composed from the reference-pinned
LSTM cell and vocab projection of ``oracle/ref_port.py``, and the CUDA path (include/gic_b200.h gic_decode_beam,
gic_vocab_topk) is tested against this file.  Only ``tests/`` may import it.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import ref_port as rp


# --------------------------------------------------------------------------------------------------------------
# Caption generation by beam search (EXTENSION, parity unpinned by reference: the reference has no beam search and
# no decoding other than Decoder.sample).  Definition, in float64 (mirrored in include/gic_b200.h gic_decode_beam):
#   start:     step 0's LSTM input is features[B,E] (as Decoder.sample), h = c = 0; beam 0 of each image at score 0,
#              beams 1..K-1 at -inf (step 0 expands one beam)
#   step:      logp = log_softmax(h_top W_out^T + b_out); live beam k offers (k, w) at score_k + logp[k, w]
#   frozen:    a beam that has emitted eos_id offers only (k, PAD = 0) at its own score (AllenNLP's BeamSearch); length fixed
#   selection: the image's K best candidates: higher score, then lower parent beam, then lower token; always L steps
#   output:    the K beams ordered by score / length ** length_penalty (ties -> lower slot); length = tokens up to and
#              including EOS, or L; ids[B,K,L] (PAD after EOS), scores[B,K] (raw sums), lengths[B,K]
# --------------------------------------------------------------------------------------------------------------
PAD_ID, EOS_ID = 0, 2


def _decoder_layers(p):
    n = 0
    while f"decoder.lstm.weight_ih_l{n}" in p:
        n += 1
    return n


def _lstm_stack(P, x, hs, cs):
    inp = x
    for l in range(len(hs)):
        hs[l], cs[l] = rp.lstm_cell(inp, hs[l], cs[l], P[f"decoder.lstm.weight_ih_l{l}"], P[f"decoder.lstm.weight_hh_l{l}"],
                                    P[f"decoder.lstm.bias_ih_l{l}"], P[f"decoder.lstm.bias_hh_l{l}"])
        inp = hs[l]
    return inp


def beam_search(p, features, K, L, eos_id=EOS_ID, length_penalty=0.0):
    """Returns dict(ids[B,K,L] int64, scores[B,K] float64, lengths[B,K] int32, trace[L,B,K,2] int64, margin): margin is the
    smallest gap that decided anything -- between neighbours among an image's K + 1 best candidates at any step (which
    slot a beam takes, and which beam is dropped), and between neighbours of the final ordering -- so a caller can tell
    whether a lower-precision implementation must agree exactly."""
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
        valid = ~fin[:, :, None].expand(B, K, V).clone()
        valid[:, :, PAD_ID] |= fin
        cand = torch.where(fin[:, :, None], score[:, :, None].expand(B, K, V), cand)
        cand = torch.where(valid, cand, torch.full_like(cand, -float("inf")))
        flat = cand.view(B, K * V)
        # stable descending sort over the (parent, token)-ordered flat index: equal scores keep the lower parent, then token
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


def beam_rescore(p, features, ids, lengths):
    """float64 sum of log-probabilities of given captions ids[B,K,L] (teacher-forced from features, as beam_search
    decodes them), over the first lengths[b,k] tokens; also returns the per-step logit scale max_w sum_j |h_j W[w,j]|."""
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    layers = _decoder_layers(P)
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    B, K, L = ids.shape
    H = W_out.shape[1]
    flat = ids.reshape(B * K, L)
    hs = [features.new_zeros(B * K, H, dtype=torch.float64) for _ in range(layers)]
    cs = [features.new_zeros(B * K, H, dtype=torch.float64) for _ in range(layers)]
    x = features.double().repeat_interleave(K, 0)
    total = features.new_zeros(B * K, dtype=torch.float64)
    scale = features.new_zeros(B * K, dtype=torch.float64)
    n = lengths.reshape(-1).long()
    for t in range(L):
        top = _lstm_stack(P, x, hs, cs)
        logp = F.log_softmax(F.linear(top, W_out, b_out), -1)
        live = t < n
        total += torch.where(live, logp.gather(1, flat[:, t:t + 1])[:, 0], torch.zeros_like(total))
        scale += torch.where(live, (top.abs() @ W_out.abs().t()).max(1).values, torch.zeros_like(scale))
        x = emb[flat[:, t]]
    return total.view(B, K), scale.view(B, K)
