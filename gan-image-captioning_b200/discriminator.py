"""RelGAN-style multi-representation CNN discriminator with the reference's interface
(src/discriminator.py:9-86): same constructor, parameter names/shapes and ``forward(inp[B,L,V]) ->
logits[B*num_rep]``.  Compute runs in libgic_b200.so (gic_disc_fwd / gic_disc_bwd)."""
from __future__ import annotations

import math

import torch
import torch.nn as nn

import gic_b200
from . import _lib


def _f32c(t):
    return t.detach().contiguous().float()


def disc_weights(disc):
    """The discriminator's tensors in the order disc_fwd_raw / disc_bwd_raw take them: (W_e, conv weights, conv biases,
    W_h, b_h, W_f, b_f, W_o, b_o), the conv tensors as per-filter-group lists."""
    return (disc.embeddings.weight, [c.weight for c in disc.convs], [c.bias for c in disc.convs], disc.highway.weight,
            disc.highway.bias, disc.feature2out.weight, disc.feature2out.bias, disc.out2logits.weight,
            disc.out2logits.bias)


def disc_fwd_raw(lib, mode, inp_soft, ids, N, L, V, De, R, fsz, nfl, W_e, cw, cb, W_h, b_h, W_f, b_f, W_o, b_o, keeps,
                 drop_p, dev):
    """Thin call of gic_disc_fwd: returns (list of logits per head, saved)."""
    Fd = sum(nfl)
    logits = [torch.empty(N * R, device=dev) for _ in keeps]
    saved = torch.empty(lib.gic_disc_saved_floats(N, L, De, R, Fd), device=dev)
    ws = torch.empty(lib.gic_disc_fwd_workspace_floats(Fd), device=dev)
    _lib.check(lib.gic_disc_fwd(mode, _lib.ptr(inp_soft), _lib.ptr(ids), N, L, V, De, R, len(fsz),
                                _lib.int_array(fsz), _lib.int_array(nfl), _lib.ptr(W_e), _lib.ptr_array(cw),
                                _lib.ptr_array(cb), _lib.ptr(W_h), _lib.ptr(b_h), _lib.ptr(W_f), _lib.ptr(b_f),
                                W_f.shape[0], _lib.ptr(W_o), _lib.ptr(b_o), len(keeps), _lib.ptr_array(keeps),
                                float(drop_p), _lib.ptr_array(logits), _lib.ptr(saved), _lib.ptr(ws), _lib.stream()),
               "gic_disc_fwd")
    return logits, saved


def disc_bwd_raw(mode, dlogits, keep, drop_p, inp_soft, ids, N, L, V, De, R, fsz, nfl, W, saved, ws, dW, dinp, want_param,
                 accumulate, stream):
    """gic_disc_bwd of one head.  W: disc_weights() order; dW: gradient outputs in the same structure (written when
    want_param, added to when accumulate); dinp: d loss / d inp_soft or None."""
    W_e, cw, cb, W_h, _, W_f, b_f, W_o, b_o = W
    dW_e, dcw, dcb, dW_h, db_h, dW_f, db_f, dW_o, db_o = dW
    P, PA = _lib.ptr, _lib.ptr_array
    _lib.check(_lib.lib().gic_disc_bwd(mode, P(dlogits), P(keep), drop_p, P(inp_soft), P(ids), N, L, V, De, R, len(fsz),
                                       _lib.int_array(fsz), _lib.int_array(nfl), P(W_e), PA(cw), PA(cb), P(W_h), P(W_f),
                                       P(b_f), W_f.shape[0], P(W_o), P(b_o), P(saved), P(ws), P(dW_e), PA(dcw), PA(dcb),
                                       P(dW_h), P(db_h), P(dW_f), P(db_f), P(dW_o), P(db_o), P(dinp), want_param,
                                       accumulate, stream), "gic_disc_bwd")


class _DiscForward(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inp, ids, keep, drop_p, mode, fsz, nfl, R, W_e, W_h, b_h, W_f, b_f, W_o, b_o, *convs):
        _lib.require_cuda()
        lib = _lib.lib()
        ng = len(fsz)
        W_e, W_h, b_h, W_f, b_f, W_o, b_o = map(_f32c, (W_e, W_h, b_h, W_f, b_f, W_o, b_o))
        cw = [_f32c(c) for c in convs[:ng]]
        cb = [_f32c(c) for c in convs[ng:]]
        De, V = W_e.shape
        if inp is not None:
            inp = _f32c(inp)
            N, L, Vin = inp.shape
            if Vin != V:
                raise ValueError("discriminator input has vocab %d, expected %d" % (Vin, V))
            dev = inp.device
        else:
            ids = ids.detach().contiguous().long()
            N, L = ids.shape
            dev = ids.device
        if keep is not None:
            keep = keep.detach().to(torch.uint8).contiguous()
        logits, saved = disc_fwd_raw(lib, mode, inp, ids, N, L, V, De, R, fsz, nfl, W_e, cw, cb, W_h, b_h, W_f, b_f,
                                     W_o, b_o, [keep], drop_p, dev)
        ctx.save_for_backward(saved, inp, ids, keep, W_e, W_h, b_h, W_f, b_f, W_o, b_o, *cw, *cb)
        ctx.meta = (N, L, V, De, R, list(fsz), list(nfl), float(drop_p), mode)
        return logits[0]

    @staticmethod
    def backward(ctx, dlogits):
        N, L, V, De, R, fsz, nfl, drop_p, mode = ctx.meta
        ng = len(fsz)
        saved, inp, ids, keep, W_e, *rest = ctx.saved_tensors
        head, cw, cb = rest[:6], rest[6:6 + ng], rest[6 + ng:]
        ws = torch.empty(_lib.lib().gic_disc_bwd_workspace_floats(N, L, De, R, sum(nfl)), device=saved.device)
        want_inp = inp is not None and ctx.needs_input_grad[0]
        want_param = any(ctx.needs_input_grad[8:])
        dW = (torch.empty_like(W_e), [torch.empty_like(c) for c in cw], [torch.empty_like(c) for c in cb],
              *(torch.empty_like(t) for t in head))
        dinp = torch.empty(N, L, V, device=saved.device) if want_inp else None
        disc_bwd_raw(mode, _f32c(dlogits), keep, drop_p, inp, ids, N, L, V, De, R, fsz, nfl, (W_e, cw, cb, *head), saved,
                     ws, dW, dinp, int(want_param), 0, _lib.stream())
        if not want_param:
            return (dinp,) + (None,) * (14 + 2 * ng)
        return (dinp, None, None, None, None, None, None, None, dW[0], *dW[3:], *dW[1], *dW[2])


class Discriminator(nn.Module):
    def __init__(self, args, gpu=False, dropout=0.2):
        super().__init__()
        self.vocab_size = args.vocab_size
        self.embed_dim = args.disc_embed_dim
        self.padding_idx = args.padding_idx
        self.feature_dim = sum(args.disc_num_filters)
        self.emb_dim_single = int(args.disc_embed_dim / args.disc_num_rep)
        self.num_rep = args.disc_num_rep
        self.filter_sizes = list(args.disc_filter_sizes)
        self.num_filters = list(args.disc_num_filters)
        self.gpu = gpu
        self.embeddings = nn.Linear(self.vocab_size, self.embed_dim, bias=False)
        self.convs = nn.ModuleList([
            nn.Conv2d(1, n, (f, self.emb_dim_single), stride=(1, self.emb_dim_single))
            for (n, f) in zip(self.num_filters, self.filter_sizes)])
        self.highway = nn.Linear(self.feature_dim, self.feature_dim)
        self.feature2out = nn.Linear(self.feature_dim, 100)
        self.out2logits = nn.Linear(100, 1)
        self.dropout = nn.Dropout(dropout)
        self.args = args
        self.init_params()

    def _run(self, inp, ids, keep):
        N = (inp if inp is not None else ids).shape[0]
        if keep is None and self.training and self.dropout.p > 0:
            # same behaviour as nn.Dropout in train mode: a fresh Bernoulli(1-p) keep mask per call
            dev = (inp if inp is not None else ids).device
            keep = torch.rand(N * self.num_rep, self.feature_dim, device=dev) >= self.dropout.p
        W_e, cw, cb, *head = disc_weights(self)
        return _DiscForward.apply(inp, ids, keep, self.dropout.p, gic_b200.get_gemm_mode(), self.filter_sizes,
                                  self.num_filters, self.num_rep, W_e, *head, *cw, *cb)

    def forward(self, inp, keep=None):
        """Get logits of discriminator.  inp: batch_size * seq_len * vocab_size (soft or one-hot) ->
        logits [batch_size * num_rep].  ``keep`` optionally supplies the dropout keep-mask [B*R, F]."""
        return self._run(inp, None, keep)

    def forward_ids(self, ids, keep=None):
        """Hard-token path: equals forward(F.one_hot(ids, V).float()) without materialising the one-hot
        (src/training.py:158)."""
        return self._run(None, ids, keep)

    def get_feature(self, inp):
        raise NotImplementedError("Discriminator.get_feature is never called by the reference and is shape-invalid "
                                  "for num_rep > 1 (SURVEY.md section 2 row 4)")

    def init_params(self):
        for param in self.parameters():
            if param.requires_grad and len(param.shape) > 0:
                stddev = 1 / math.sqrt(param.shape[0])
                if self.args.disc_init == "uniform":
                    torch.nn.init.uniform_(param, a=-0.05, b=0.05)
                elif self.args.disc_init == "normal":
                    torch.nn.init.normal_(param, std=stddev)
