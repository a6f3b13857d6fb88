"""Generate tests/golden/*.npz by running the UNMODIFIED reference modules on CPU.

Needs a checkout of the original project (kawshik8/GAN-Image-Captioning):

    python oracle/make_golden.py <checkout>/src

It imports ``<checkout>/src/{generator,discriminator,utils}.py`` as they are, loads the
seeded synthetic weights from ``oracle.ref_port.make_inputs`` into the reference's own
``Decoder`` / ``Encoder`` / ``Discriminator`` modules via ``load_state_dict``, injects the
caller-supplied uniforms (by overriding ``Decoder.add_gumbel`` on the instance, keeping its
``eps`` arithmetic) and dropout keep-masks (by replacing the ``nn.Dropout`` instance), runs
one adversarial step exactly as ``src/training.py:144-169,194-199`` does except for the Q1
ordering fix (both grads on pre-update weights; SURVEY.md §0.1), and stores the results.
Nothing of the original project is copied; only numeric outputs are committed.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_port as rp  # noqa: E402


class SuppliedDropout(nn.Module):
    """nn.Dropout(0.2) with the Bernoulli keep-mask supplied by the caller (Q7)."""

    def __init__(self, p=0.2):
        super().__init__()
        self.p, self.keep = p, None

    def forward(self, x):
        if self.keep is None:
            return x
        return x * self.keep / (1.0 - self.p)


def load_reference(src):
    sys.path.insert(0, src)
    import generator as ref_gen       # noqa
    import discriminator as ref_disc  # noqa
    import utils as ref_utils         # noqa
    return ref_gen, ref_disc, ref_utils


def run_reference(src, cfg, temperature, loss_type, train=True):
    ref_gen, ref_disc, ref_utils = load_reference(src)
    inp = rp.make_inputs(cfg)
    a = inp["args"]
    B, L = inp["captions"].shape

    dec = ref_gen.Decoder(a)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in inp["gen"].items() if k.startswith("decoder.")})
    dec.temperature = temperature
    disc = ref_disc.Discriminator(a)
    disc.load_state_dict(inp["disc"])
    disc.dropout = SuppliedDropout(0.2)
    enc = None
    if a.conditional_gan:
        enc = ref_gen.Encoder(a)                      # builds the (out-of-scope) ResNet-18 trunk too
        enc.linear = nn.Linear(a.feature_dim, a.gen_embed_dim)   # same layer type, synthetic feature width
        enc.load_state_dict({k[len("encoder."):]: v for k, v in inp["gen"].items()
                             if k.startswith("encoder.")}, strict=False)
        enc.train()

    # uniforms: same arithmetic as Decoder.add_gumbel (src/generator.py:84-96), u supplied per step
    state = {"t": 0}

    def add_gumbel(self, o_t, eps=1e-10, gpu=0):
        u = inp["u"][state["t"]]
        state["t"] += 1
        g_t = -torch.log(-torch.log(u + eps) + eps)
        return o_t + g_t

    dec.add_gumbel = types.MethodType(add_gumbel, dec)
    if train:
        dec.train(); disc.train()
    else:
        dec.eval(); disc.eval()

    if a.conditional_gan:
        feats = enc.bn(enc.linear(inp["pooled"]))     # src/generator.py:23-24 without the trunk
    else:
        feats = dec.embed(torch.ones(B, 1, dtype=torch.long).squeeze(1))   # src/training.py:147
    gen_caps, gen_ids = dec.sample(feats, max_caption_len=L)               # :150
    fake = gen_caps.detach()
    real = F.one_hot(inp["captions"], a.vocab_size).float()                # :158
    outs = []
    for i, x in enumerate((real, fake, gen_caps)):                         # :162-164
        disc.dropout.keep = inp["keep"][i] if train else None
        outs.append(disc(x))
    d_real, d_fake, g_out = outs
    g_loss, d_loss = ref_utils.get_losses(d_real, d_fake, g_out, loss_type)   # :165
    res = dict(features=feats.detach(), probs=gen_caps.detach(), ids=gen_ids, d_real=d_real.detach(),
               d_fake=d_fake.detach(), g_out=g_out.detach(), g_loss=g_loss.detach(), d_loss=d_loss.detach())
    if not train:
        return inp, res
    gen_params = {("decoder." + k): p for k, p in dec.named_parameters()}
    if enc is not None:
        gen_params.update({("encoder." + k): p for k, p in enc.named_parameters() if not k.startswith("resnet")})
    disc_params = dict(disc.named_parameters())
    # Q1 fix: both gradients on the same pre-update weights
    dg = torch.autograd.grad(d_loss, list(disc_params.values()), retain_graph=True)
    if g_loss.requires_grad:
        gg = torch.autograd.grad(g_loss, list(gen_params.values()), allow_unused=True)
    else:
        gg = [None] * len(gen_params)
    for p, g in zip(disc_params.values(), dg):
        p.grad = g.clone()
    for p, g in zip(gen_params.values(), gg):
        p.grad = None if g is None else g.clone()
    res["d_grads"] = {k: p.grad.clone() for k, p in disc_params.items()}
    res["g_grads"] = {k: p.grad.clone() for k, p in gen_params.items() if p.grad is not None}
    # optimize(): clip_grad_norm_ then Adam.step (src/training.py:194-199, :24-26)
    d_opt = torch.optim.Adam(disc.parameters(), lr=a.disc_lr)
    res["d_norm"] = float(torch.nn.utils.clip_grad_norm_(disc.parameters(), a.clip_norm))
    d_opt.step()
    gps = [p for p in gen_params.values()]
    if any(p.grad is not None for p in gps):
        g_opt = torch.optim.Adam(gps, lr=a.gen_lr)
        res["g_norm"] = float(torch.nn.utils.clip_grad_norm_(gps, a.clip_norm))
        g_opt.step()
    else:
        res["g_norm"] = 0.0
    res["new_disc"] = {k: p.detach().clone() for k, p in disc_params.items()}
    res["new_gen"] = {k: p.detach().clone() for k, p in gen_params.items()}
    return inp, res


def sample_idx(n):
    """Deterministic sub-sample of a flat tensor: the first 256 entries + every 997th."""
    idx = np.unique(np.concatenate([np.arange(min(n, 256)), np.arange(0, n, 997)]))
    return idx


def pack(res, full):
    out = {}
    for k, v in res.items():
        if isinstance(v, dict):
            for kk, vv in v.items():
                flat = vv.detach().reshape(-1).numpy()
                out[f"{k}/{kk}/norm"] = np.float64(np.sqrt((flat.astype(np.float64) ** 2).sum()))
                out[f"{k}/{kk}"] = flat if full else flat[sample_idx(flat.size)]
        elif isinstance(v, torch.Tensor):
            arr = v.numpy()
            if not full and k == "probs":
                out["probs_max"] = arr.max(-1)
                out["probs_sumsq"] = (arr.astype(np.float64) ** 2).sum(-1)
                out["probs_head"] = arr[:, :, :32].copy()
            else:
                out[k] = arr
        else:
            out[k] = np.float64(v)
    return out


CASES = [
    # name, config, temperature, loss, train, store-everything
    ("c0_T1_standard", "c0", 1.0, "standard", True, True),
    ("c0_T100_JS", "c0", 100.0, "JS", True, True),
    ("c0_T3_rsgan", "c0", 3.0, "rsgan", True, True),
    ("c0_T1_eval", "c0", 1.0, "standard", False, True),
    ("c0l2_T5_KL", "c0_l2", 5.0, "KL", True, True),
    ("c1_T100_standard", "c1", 100.0, "standard", True, False),
    ("c1_T1_standard", "c1", 1.0, "standard", True, False),
]


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python oracle/make_golden.py <checkout of the original project>/src")
    torch.manual_seed(1008)
    torch.set_num_threads(4)
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    for name, cfg, T, loss, train, full in CASES:
        inp, res = run_reference(sys.argv[1], rp.CONFIGS[cfg], T, loss, train)
        blob = pack(res, full)
        blob["meta_temperature"] = np.float64(T)
        path = os.path.join(ROOT, "tests", "golden", name + ".npz")
        np.savez_compressed(path, **blob)
        print(name, "g_loss %.6f d_loss %.6f" % (float(res["g_loss"]), float(res["d_loss"])),
              "%.1f KB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
