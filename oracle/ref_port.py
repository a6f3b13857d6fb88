"""CPU oracle for the adversarial-captioning hot path.  TEST INFRASTRUCTURE ONLY.

This file is a CPU restatement (PyTorch fp32, explicit equations) of the reference's
algorithm for the hot path.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it; the product
package (``gan-image-captioning_b200/``) never does and fails loudly without its CUDA
library.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4), so this
oracle is pinned by *executing the reference's own modules*:
``oracle/make_golden.py`` imports ``<checkout>/src/{generator,discriminator,utils}.py``
unmodified, runs them on the seeded inputs produced by :func:`make_inputs`, and commits
the outputs under ``tests/golden/``.  ``tests/test_oracle_golden.py`` checks this
restatement against those fixtures.  Extensions the reference does not contain
(inverse-CDF sampler, rollouts, policy-gradient loss) are marked "parity unpinned by
reference" where they are defined.

Every random draw is an explicit input: Gumbel uniforms ``u[L,B,V]`` and dropout keep
masks ``[3][B*R,F]`` (SURVEY.md §0.1 Q7, §8b "Randomness").

All ``file:line`` citations are relative to the reference checkout.
"""
from __future__ import annotations

import math
from argparse import Namespace
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor
Params = Dict[str, Tensor]


# --------------------------------------------------------------------------------------
# configuration (src/args.py:12-193 defaults; get_args() itself is never called: it mkdirs)
# --------------------------------------------------------------------------------------
def default_args(**over) -> Namespace:
    a = Namespace(
        gen_hidden_dim=512, gen_embed_dim=32, gen_num_layers=1, gen_init="uniform",
        disc_embed_dim=64, disc_num_rep=64, disc_filter_sizes=[3, 4, 5],
        disc_num_filters=[300, 300, 300], disc_init="uniform", conditional_gan=0,
        vocab_size=-1, max_seq_len=34, padding_idx=0, temperature=100, temp_adpt="exp",
        clip_norm=5.0, adv_loss_type="standard", gen_lr=1e-4, disc_lr=1e-4,
        pretrain_lr=1e-2, adv_epochs=30, device="cpu", feature_dim=512,
    )
    for k, v in over.items():
        setattr(a, k, v)
    return a


# named hot-path configurations (BASELINE.json configs / SURVEY.md §8)
CONFIGS = {
    # tiny: every tensor is committed in full under tests/golden/
    "c0": dict(B=4, L=8, V=50, E=16, H=32, layers=1, feat=0, filters=[20, 24, 28]),
    "c0_l2": dict(B=3, L=7, V=37, E=12, H=20, layers=2, feat=24, filters=[8, 8, 8]),
    # BASELINE.json configs[0]: args.py defaults, 2048-d pooled features, vocab 1000, len 16
    "c1": dict(B=8, L=16, V=1000, E=32, H=512, layers=1, feat=2048, filters=[300, 300, 300]),
    # BASELINE.json configs[1] (Tier-A shape: pooled 7x7x2048 grid), the bench workload
    "c2": dict(B=256, L=20, V=10000, E=512, H=512, layers=1, feat=2048, filters=[300, 300, 300]),
}


def args_for(cfg: dict) -> Namespace:
    return default_args(vocab_size=cfg["V"], gen_embed_dim=cfg["E"], gen_hidden_dim=cfg["H"],
                        gen_num_layers=cfg["layers"], disc_num_filters=list(cfg["filters"]),
                        conditional_gan=1 if cfg["feat"] else 0, feature_dim=cfg["feat"] or 512)


# --------------------------------------------------------------------------------------
# synthetic weights / inputs (SURVEY.md §8d "Synthetic inputs")
# --------------------------------------------------------------------------------------
def gen_param_shapes(a: Namespace) -> List[Tuple[str, Tuple[int, ...]]]:
    """state_dict names/shapes of the reference Generator that the hot path touches
    (src/generator.py:15-16,31-33).  The ResNet trunk is out of scope (SURVEY.md §2 row 2)."""
    V, E, H = a.vocab_size, a.gen_embed_dim, a.gen_hidden_dim
    out = [("encoder.linear.weight", (E, a.feature_dim)), ("encoder.linear.bias", (E,)),
           ("encoder.bn.weight", (E,)), ("encoder.bn.bias", (E,)),
           ("decoder.embed.weight", (V, E))]
    for l in range(a.gen_num_layers):
        In = E if l == 0 else H
        out += [(f"decoder.lstm.weight_ih_l{l}", (4 * H, In)), (f"decoder.lstm.weight_hh_l{l}", (4 * H, H)),
                (f"decoder.lstm.bias_ih_l{l}", (4 * H,)), (f"decoder.lstm.bias_hh_l{l}", (4 * H,))]
    out += [("decoder.linear.weight", (V, H)), ("decoder.linear.bias", (V,))]
    return out


def disc_param_shapes(a: Namespace) -> List[Tuple[str, Tuple[int, ...]]]:
    """state_dict names/shapes of the reference Discriminator (src/discriminator.py:20-29)."""
    V, De = a.vocab_size, a.disc_embed_dim
    es = De // a.disc_num_rep
    Fd = sum(a.disc_num_filters)
    out = [("embeddings.weight", (De, V))]
    for i, (n, f) in enumerate(zip(a.disc_num_filters, a.disc_filter_sizes)):
        out += [(f"convs.{i}.weight", (n, 1, f, es)), (f"convs.{i}.bias", (n,))]
    out += [("highway.weight", (Fd, Fd)), ("highway.bias", (Fd,)),
            ("feature2out.weight", (100, Fd)), ("feature2out.bias", (100,)),
            ("out2logits.weight", (1, 100)), ("out2logits.bias", (1,))]
    return out


def make_params(shapes, seed: int) -> Params:
    """Every parameter ~ U(-0.05, 0.05) as init_params does (src/generator.py:116-123,
    src/discriminator.py:79-86; Q6), from a private generator so the draw order is ours."""
    g = torch.Generator().manual_seed(seed)
    return {k: (torch.rand(s, generator=g, dtype=torch.float32) * 0.1 - 0.05) for k, s in shapes}


def make_inputs(cfg: dict, seed: int = 1008, step: int = 0) -> dict:
    """All seeded inputs of one adversarial step (seed 1008: src/main.py:14-17)."""
    a = args_for(cfg)
    B, L, V = cfg["B"], cfg["L"], cfg["V"]
    R, Fd = a.disc_num_rep, sum(a.disc_num_filters)
    gp = make_params(gen_param_shapes(a), seed)
    dp = make_params(disc_param_shapes(a), seed + 1)
    g = torch.Generator().manual_seed(seed + 2 + step)
    pooled = torch.randn(B, a.feature_dim, generator=g) if cfg["feat"] else None
    u = torch.rand(L, B, V, generator=g, dtype=torch.float32)
    keep = (torch.rand(3, B * R, Fd, generator=g) >= 0.2).to(torch.float32)
    # collate contract (src/tasks.py:138-158): <S>=1, tokens, <E>=2, <PAD>=0 tail
    caps = torch.zeros(B, L, dtype=torch.int64)
    lens = torch.randint(max(1, L // 2 - 2), L - 1, (B,), generator=g)
    lens[0] = L - 2
    for b in range(B):
        n = int(lens[b])
        caps[b, 0] = 1
        caps[b, 1:1 + n] = torch.randint(4, V, (n,), generator=g)
        caps[b, 1 + n] = 2
    return dict(args=a, gen=gp, disc=dp, pooled=pooled, u=u, keep=keep, captions=caps)


# --------------------------------------------------------------------------------------
# generator: decode + Gumbel-softmax sampling
# --------------------------------------------------------------------------------------
def encoder_project(p: Params, pooled: Tensor, eps: float = 1e-5) -> Tensor:
    """Encoder.linear + Encoder.bn in train mode (src/generator.py:15-16,23-24): batch
    statistics, biased variance, eps 1e-5 (running stats are not on the hot path)."""
    y = F.linear(pooled, p["encoder.linear.weight"], p["encoder.linear.bias"])
    mu = y.mean(0, keepdim=True)
    var = ((y - mu) ** 2).mean(0, keepdim=True)
    return (y - mu) / torch.sqrt(var + eps) * p["encoder.bn.weight"] + p["encoder.bn.bias"]


def start_features(p: Params, B: int) -> Tensor:
    """Unconditional start input: embedding row 1 (<S>) for every caption
    (src/training.py:147)."""
    return p["decoder.embed.weight"][torch.ones(B, dtype=torch.int64)]


def lstm_cell(x: Tensor, h: Tensor, c: Tensor, W_ih, W_hh, b_ih, b_hh):
    """One nn.LSTM time step (src/generator.py:61): gates = x W_ih^T + b_ih + h W_hh^T + b_hh,
    chunk order i,f,g,o; c' = sig(f) c + sig(i) tanh(g); h' = sig(o) tanh(c')."""
    gates = F.linear(x, W_ih, b_ih) + F.linear(h, W_hh, b_hh)
    i, f, g, o = gates.chunk(4, dim=1)
    c2 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
    h2 = torch.sigmoid(o) * torch.tanh(c2)
    return h2, c2


def gumbel_noise(u: Tensor, eps: float = 1e-10) -> Tensor:
    """Decoder.add_gumbel with the uniform supplied (src/generator.py:84-96)."""
    return -torch.log(-torch.log(u + eps) + eps)


def decoder_sample(p: Params, features: Tensor, u: Optional[Tensor], temperature: float,
                   L: int, layers: int = 1, pretrain: bool = False,
                   forced_ids: Optional[Tensor] = None, return_hidden: bool = False):
    """Decoder.sample (src/generator.py:55-81).  Returns (outputs[B,L,V], ids[B,L], logits[B,L,V]).

    ``forced_ids`` (teacher forcing for parity runs, SURVEY.md §7 "hard parts"): the token fed
    back at step t is forced_ids[:, t] instead of this run's own argmax; the returned ids are
    still this run's own choices so mismatches can be classified."""
    B = features.shape[0]
    H = p["decoder.lstm.weight_hh_l0"].shape[1]
    h = [features.new_zeros(B, H) for _ in range(layers)]
    c = [features.new_zeros(B, H) for _ in range(layers)]
    x = features
    outs, ids, logit_list, hid = [], [], [], []
    for t in range(L):
        inp = x
        for l in range(layers):
            h[l], c[l] = lstm_cell(inp, h[l], c[l], p[f"decoder.lstm.weight_ih_l{l}"],
                                   p[f"decoder.lstm.weight_hh_l{l}"], p[f"decoder.lstm.bias_ih_l{l}"],
                                   p[f"decoder.lstm.bias_hh_l{l}"])
            inp = h[l]
        logits = F.linear(inp, p["decoder.linear.weight"], p["decoder.linear.bias"])   # :64,68
        logit_list.append(logits)
        hid.append(inp)
        if pretrain:
            outs.append(logits)                                                       # :65
            pred = F.softmax(logits, dim=-1)                                          # :66
        else:
            pred = F.softmax((logits + gumbel_noise(u[t])) * temperature, dim=-1)     # :69
            outs.append(pred)                                                         # :70
        tok = pred.max(1)[1]                                                          # :73 first max
        ids.append(tok)
        fed = tok if forced_ids is None else forced_ids[:, t]
        x = p["decoder.embed.weight"][fed.detach()]                                   # :75
    if return_hidden:      # top-layer hidden states [B,L,H]: the tests derive per-row rounding bounds on the logits from them
        return torch.stack(outs, 1), torch.stack(ids, 1), torch.stack(logit_list, 1), torch.stack(hid, 1)
    return torch.stack(outs, 1), torch.stack(ids, 1), torch.stack(logit_list, 1)


def sample_inverse_cdf(logits: Tensor, u_row: Tensor) -> Tensor:
    """EXTENSION, parity unpinned by reference (SURVEY.md §8a row B2): categorical draw by
    inverse CDF over softmax(logits) with a sequential fp32 cumulative sum; token = first
    index whose CDF exceeds u (clamped to V-1)."""
    pr = F.softmax(logits, dim=-1)
    cdf = torch.cumsum(pr, dim=-1)
    tok = (cdf <= u_row[:, None]).sum(-1)
    return tok.clamp(max=logits.shape[-1] - 1)


# --------------------------------------------------------------------------------------
# discriminator
# --------------------------------------------------------------------------------------
def disc_forward(p: Params, inp: Tensor, keep: Optional[Tensor], filter_sizes: Sequence[int],
                 drop_p: float = 0.2, return_parts: bool = False):
    """Discriminator.forward (src/discriminator.py:34-62) with the dropout keep-mask supplied
    (``keep`` None = eval mode).  inp [B,L,V] float -> logits [B*R]."""
    W_e = p["embeddings.weight"]                        # [De, V]
    B, L, _ = inp.shape
    R = W_e.shape[0]                                    # emb_dim_single == 1 (:17)
    emb = inp @ W_e.t()                                 # [B,L,R]           :40
    pools = []
    for i, f in enumerate(filter_sizes):
        w = p[f"convs.{i}.weight"][:, 0, :, 0]          # [n,f]
        win = emb.unfold(1, f, 1)                       # [B, L-f+1, R, f]
        conv = torch.einsum("btrk,nk->bntr", win, w) + p[f"convs.{i}.bias"][None, :, None, None]  # :42
        pools.append(F.relu(conv).max(dim=2)[0])        # [B,n,R]           :42,45
    x = torch.cat(pools, 1).permute(0, 2, 1).reshape(B * R, -1)     # :49-51, row = b*R + r
    hw = F.linear(x, p["highway.weight"], p["highway.bias"])        # :53
    sg = torch.sigmoid(hw)
    y = sg * F.relu(hw) + (1.0 - sg) * x                            # :55
    yd = y if keep is None else y * keep / (1.0 - drop_p)           # :58 nn.Dropout(0.2)
    z = F.linear(yd, p["feature2out.weight"], p["feature2out.bias"])  # :58
    logits = F.linear(z, p["out2logits.weight"], p["out2logits.bias"]).squeeze(1)  # :60
    if return_parts:
        return logits, dict(emb=emb, pooled=x, highway=y, hw=hw)
    return logits


def disc_forward_ids(p: Params, ids: Tensor, keep, filter_sizes, drop_p: float = 0.2):
    """Hard-token path: Linear of a one-hot == column pick of embeddings.weight
    (src/training.py:158 + src/discriminator.py:40; SURVEY.md §8a A8)."""
    V = p["embeddings.weight"].shape[1]
    return disc_forward(p, F.one_hot(ids, V).float(), keep, filter_sizes, drop_p)


# --------------------------------------------------------------------------------------
# losses (src/utils.py:10-53) and temperature schedule (src/utils.py:55-76)
# --------------------------------------------------------------------------------------
def bce_logits(x: Tensor, y: float) -> Tensor:
    """nn.BCEWithLogitsLoss(mean): mean(max(x,0) - x*y + log1p(exp(-|x|)))."""
    return (x.clamp(min=0) - x * y + torch.log1p(torch.exp(-x.abs()))).mean()


def get_losses(d_real: Tensor, d_fake: Tensor, g_out: Tensor, loss_type: str = "JS"):
    if loss_type in ("standard", "JS", "KL"):
        d_loss = bce_logits(d_real, 1.0) + bce_logits(d_fake, 0.0)
        if loss_type == "standard":
            g_loss = bce_logits(g_out, 1.0)
        elif loss_type == "JS":
            g_loss = -bce_logits(g_out, 0.0)
        else:
            g_loss = (-g_out).mean()
    elif loss_type == "hinge":      # Q4: reference calls nn.ReLU(x) (TypeError); F.relu intent
        d_loss = F.relu(1.0 - d_real).mean() + F.relu(1.0 + d_fake).mean()
        g_loss = -g_out.mean()
    elif loss_type == "tv":         # Q4: nn.Tanh(x) in the reference; torch.tanh intent
        d_loss = (torch.tanh(d_fake) - torch.tanh(d_real)).mean()
        g_loss = (-torch.tanh(g_out)).mean()
    elif loss_type == "rsgan":
        d_loss = bce_logits(d_real - d_fake, 1.0)
        g_loss = bce_logits(d_fake - d_real, 1.0)
    else:
        raise NotImplementedError("Divergence '%s' is not implemented" % loss_type)
    return g_loss, d_loss


def get_fixed_temperature(temper, i, N, adapt):
    if adapt == "no":
        return 1.0
    if adapt == "lin":
        return 1 + i / (N - 1) * (temper - 1)
    if adapt == "exp":
        return temper ** (i / N)
    if adapt == "log":
        return 1 + (temper - 1) / np.log(N) * np.log(i + 1)
    if adapt == "sigmoid":
        return (temper - 1) * 1 / (1 + np.exp((N / 2 - i) * 20 / N)) + 1
    if adapt == "quad":
        return (temper - 1) / (N - 1) ** 2 * i ** 2 + 1
    if adapt == "sqrt":
        return (temper - 1) / np.sqrt(N - 1) * np.sqrt(i) + 1
    raise Exception("Unknown adapt type!")


# --------------------------------------------------------------------------------------
# optimizer step (src/training.py:194-199, Adam ctor :24-26)
# --------------------------------------------------------------------------------------
def clip_coef(grads: Sequence[Tensor], max_norm: float) -> Tuple[float, float]:
    """clip_grad_norm_: global L2 norm over all grads; coef = max_norm/(norm+1e-6) clamped to 1."""
    total = math.sqrt(sum(float((g.double() ** 2).sum()) for g in grads if g is not None))
    return total, min(1.0, max_norm / (total + 1e-6))


def adam_update(p: Tensor, g: Tensor, m: Tensor, v: Tensor, step: int, lr: float,
                b1: float = 0.9, b2: float = 0.999, eps: float = 1e-8):
    """torch.optim.Adam single-tensor rule (weight_decay 0, amsgrad False)."""
    m.mul_(b1).add_(g, alpha=1 - b1)
    v.mul_(b2).addcmul_(g, g, value=1 - b2)
    bc1 = 1 - b1 ** step
    bc2 = 1 - b2 ** step
    denom = (v.sqrt() / math.sqrt(bc2)).add_(eps)
    p.addcdiv_(m, denom, value=-lr / bc1)


# --------------------------------------------------------------------------------------
# one adversarial step (src/training.py:136-169) with the Q1 ordering fix
# --------------------------------------------------------------------------------------
def adversarial_step(inp: dict, temperature: float, loss_type: str = "standard",
                     train: bool = True, adam_state: Optional[dict] = None, step: int = 1,
                     forced_ids: Optional[Tensor] = None, update: bool = True) -> dict:
    """Both gradients are taken on the same pre-update weights (SURVEY.md §0.1 Q1), then each
    set is clipped (clip_norm) and stepped with Adam.  Returns everything a parity test needs."""
    a = inp["args"]
    gp = {k: v.clone().requires_grad_(True) for k, v in inp["gen"].items()}
    dp = {k: v.clone().requires_grad_(True) for k, v in inp["disc"].items()}
    caps = inp["captions"]
    B, L = caps.shape
    fs = a.disc_filter_sizes
    feats = encoder_project(gp, inp["pooled"]) if a.conditional_gan else start_features(gp, B)   # :144-147
    probs, ids, logits, htop = decoder_sample(gp, feats, inp["u"], temperature, L, a.gen_num_layers,
                                              forced_ids=forced_ids, return_hidden=True)       # :150
    fake = probs.detach()                                                                       # :151
    real = F.one_hot(caps, a.vocab_size).float()                                                # :158
    keep = inp["keep"] if train else [None, None, None]
    d_real = disc_forward(dp, real, keep[0], fs)                                                # :162
    d_fake = disc_forward(dp, fake, keep[1], fs)                                                # :163
    g_out = disc_forward(dp, probs, keep[2], fs)                                                # :164
    g_loss, d_loss = get_losses(d_real, d_fake, g_out, loss_type)                               # :165
    out = dict(features=feats.detach(), probs=probs.detach(), ids=ids, logits=logits.detach(), htop=htop.detach(),
               d_real=d_real.detach(), d_fake=d_fake.detach(), g_out=g_out.detach(),
               g_loss=g_loss.detach(), d_loss=d_loss.detach())
    if not train:
        return out
    dnames, gnames = list(dp), list(gp)
    d_grads = torch.autograd.grad(d_loss, [dp[k] for k in dnames], retain_graph=True)
    if g_loss.requires_grad:
        g_grads = torch.autograd.grad(g_loss, [gp[k] for k in gnames], allow_unused=True)
    else:                                   # rsgan: g_loss has no path to G (A14)
        g_grads = [None] * len(gnames)
    out["d_grads"] = dict(zip(dnames, d_grads))
    out["g_grads"] = {k: g for k, g in zip(gnames, g_grads) if g is not None}
    dn, dc = clip_coef(d_grads, a.clip_norm)
    gn, gc = clip_coef([g for g in g_grads if g is not None], a.clip_norm)
    out.update(d_norm=dn, g_norm=gn, d_coef=dc, g_coef=gc)
    if update:
        st = adam_state if adam_state is not None else {}
        new_d, new_g = {}, {}
        for k in dnames:
            w = inp["disc"][k].clone()
            m, v = st.setdefault("d_m_" + k, torch.zeros_like(w)), st.setdefault("d_v_" + k, torch.zeros_like(w))
            adam_update(w, out["d_grads"][k] * dc, m, v, step, a.disc_lr)
            new_d[k] = w
        for k in gnames:
            w = inp["gen"][k].clone()
            if k in out["g_grads"]:
                m, v = st.setdefault("g_m_" + k, torch.zeros_like(w)), st.setdefault("g_v_" + k, torch.zeros_like(w))
                adam_update(w, out["g_grads"][k] * gc, m, v, step, a.gen_lr)
            new_g[k] = w
        out["new_disc"], out["new_gen"] = new_d, new_g
    return out


# ------------------------------------------------------------------------------------------------
# batch contract: collate_fn (src/tasks.py:138-158) -- the step immediately before the hot path (SURVEY.md 8f rank 2)
# ------------------------------------------------------------------------------------------------
def collate_captions(token_lists):
    """captions[B, max_len + 2] int64 = <S>=1, tokens, <E>=2, <PAD>=0 ...; lengths[B] int32 = len + 2; max_caption_len
    (src/tasks.py:143-156).  Plain loops, as the reference writes them."""
    max_caption_len = 0
    for toks in token_lists:                                    # :143-146
        max_caption_len = max(max_caption_len, len(toks))
    max_caption_len += 2
    captions = torch.zeros(len(token_lists), max_caption_len, dtype=torch.long)       # :149
    lengths = torch.zeros(len(token_lists), dtype=torch.int32)                        # :150
    for i, toks in enumerate(token_lists):                      # :152-155
        row = [1] + [int(t) for t in toks] + [2] + [0] * (max_caption_len - len(toks) - 2)
        captions[i] = torch.tensor(row, dtype=torch.long)
        lengths[i] = len(toks) + 2
    return captions, lengths, max_caption_len
