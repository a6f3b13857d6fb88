"""get_losses / get_fixed_temperature with the reference's signatures (src/utils.py:10-76).
get_losses runs as one fused CUDA kernel that also produces the backward seeds."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib


def gan_loss_raw(loss_type, d_real, d_fake, g_out, losses, seeds, stream):
    """gic_gan_loss_fwd_bwd: losses[2] = (g_loss, d_loss) and the backward seeds[3, n] of d_real, d_fake and g_out."""
    P = _lib.ptr
    _lib.check(_lib.lib().gic_gan_loss_fwd_bwd(loss_type, P(d_real), P(d_fake), P(g_out), d_real.numel(), P(losses),
                                               P(seeds[0]), P(seeds[1]), P(seeds[2]), stream), "gic_gan_loss_fwd_bwd")


class _GanLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, d_real, d_fake, g_out, loss_type):
        _lib.require_cuda()
        d_real, d_fake, g_out = (t.detach().contiguous().float() for t in (d_real, d_fake, g_out))
        n = d_real.numel()
        if d_fake.numel() != n or g_out.numel() != n:
            raise ValueError("get_losses: d_out_real, d_out_fake and g_out must have the same number of logits")
        dev = d_real.device
        losses = torch.empty(2, device=dev)
        seeds = torch.empty(3, n, device=dev)
        gan_loss_raw(loss_type, d_real, d_fake, g_out, losses, seeds, _lib.stream())
        ctx.save_for_backward(seeds)
        ctx.shapes = (d_real.shape, d_fake.shape, g_out.shape)
        ctx.rsgan = (loss_type == _lib.LOSS_TYPES["rsgan"])
        return losses[0], losses[1]

    @staticmethod
    def backward(ctx, dg_loss, dd_loss):
        (seeds,) = ctx.saved_tensors
        s0, s1, s2 = ctx.shapes
        g_real, g_fake = seeds[0] * dd_loss, seeds[1] * dd_loss
        if ctx.rsgan:
            # g_loss = BCE(d_fake - d_real, 1) also depends on the D outputs (src/utils.py:48); with
            # x = d_real - d_fake and seeds[0] = (sig(x) - 1)/n:  d g_loss / d d_real = sig(x)/n = seeds[0] + 1/n
            n = seeds.shape[1]
            g_real = g_real + (seeds[0] + 1.0 / n) * dg_loss
            g_fake = g_fake - (seeds[0] + 1.0 / n) * dg_loss
        return (g_real.view(s0), g_fake.view(s1), (seeds[2] * dg_loss).view(s2), None)


def get_losses(d_out_real, d_out_fake, g_out, loss_type="JS"):
    """Get different adversarial losses according to given loss_type -> (g_loss, d_loss)."""
    if loss_type not in _lib.LOSS_TYPES:
        raise NotImplementedError("Divergence '%s' is not implemented" % loss_type)
    return _GanLoss.apply(d_out_real, d_out_fake, g_out, _lib.LOSS_TYPES[loss_type])


def get_fixed_temperature(temper, i, N, adapt):
    """A function to set up different temperature control policies (host-side scalar)."""
    if adapt == "no":
        temper_var_np = 1.0
    elif adapt == "lin":
        temper_var_np = 1 + i / (N - 1) * (temper - 1)
    elif adapt == "exp":
        temper_var_np = temper ** (i / N)
    elif adapt == "log":
        temper_var_np = 1 + (temper - 1) / np.log(N) * np.log(i + 1)
    elif adapt == "sigmoid":
        temper_var_np = (temper - 1) * 1 / (1 + np.exp((N / 2 - i) * 20 / N)) + 1
    elif adapt == "quad":
        temper_var_np = (temper - 1) / (N - 1) ** 2 * i ** 2 + 1
    elif adapt == "sqrt":
        temper_var_np = (temper - 1) / np.sqrt(N - 1) * np.sqrt(i) + 1
    else:
        raise Exception("Unknown adapt type!")
    return temper_var_np
