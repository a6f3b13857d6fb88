"""CPU oracle for teacher-forced caption scoring (EXTENSION).  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED BY REFERENCE: kawshik8/GAN-Image-Captioning has no evaluation of the generator other than the GAN losses.
Scoring is defined HERE, in float64, with the LSTM stack and vocab projection that ``oracle/ref_beam.py`` composes from the
reference-pinned cell of ``oracle/ref_port.py``; the CUDA path (include/gic_b200.h gic_score_captions,
gic_vocab_target_logp) is tested against this file.  Only ``tests/`` may import it.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .ref_beam import _decoder_layers, _lstm_stack


def teacher_forced_logp(p, features, ids, lengths=None):
    """Teacher-forced scoring of captions ids[N,L] in float64 (mirrored in include/gic_b200.h gic_score_captions): step 0's
    input is features[N,E], h = c = 0; position t predicts ids[:, t], which is step t + 1's input.  Returns dict(
    logp[N,L] (log_softmax of the target, 0 for t >= lengths[n]; lengths None: all L), total[N] (sum of logp),
    argmax[N,L] (ties -> lower token), scale[N,L] (logit scale max_w sum_j |h_j W[w,j]|), gap[N,L] (top logit minus the
    second, for tie classification), lse[N,L])."""
    P = {k: v.double() for k, v in p.items() if k.startswith("decoder.")}
    layers = _decoder_layers(P)
    W_out, b_out, emb = P["decoder.linear.weight"], P["decoder.linear.bias"], P["decoder.embed.weight"]
    N, L = ids.shape
    H = W_out.shape[1]
    dev = features.device
    ids = ids.to(dev)
    n = (torch.full((N,), L, dtype=torch.int64, device=dev) if lengths is None
         else torch.as_tensor(lengths, device=dev).long().clamp(0, L))
    hs = [torch.zeros(N, H, dtype=torch.float64, device=dev) for _ in range(layers)]
    cs = [torch.zeros(N, H, dtype=torch.float64, device=dev) for _ in range(layers)]
    x = features.double()
    out = {k: [] for k in ("logp", "argmax", "scale", "gap", "lse")}
    for t in range(L):
        top = _lstm_stack(P, x, hs, cs)
        z = F.linear(top, W_out, b_out)
        lse = torch.logsumexp(z, 1)
        lp = z.gather(1, ids[:, t:t + 1])[:, 0] - lse
        out["logp"].append(torch.where(t < n, lp, torch.zeros_like(lp)))
        out["argmax"].append(z.argmax(1))          # first maximum: ties -> lower token
        two = torch.topk(z, 2, dim=1).values
        out["gap"].append(two[:, 0] - two[:, 1])
        out["scale"].append((top.abs() @ W_out.abs().t()).max(1).values)
        out["lse"].append(lse)
        x = emb[ids[:, t]]
    r = {k: torch.stack(v, 1) for k, v in out.items()}
    r["total"] = r["logp"].sum(1)
    return r
