"""Caption generator with the reference's interface (src/generator.py): ``Encoder``, ``Decoder`` and
``Generator`` keep their constructor signatures, attribute names and ``state_dict`` keys, so
``optim.Adam(gen.parameters())`` and checkpoints written by the reference keep working.  The compute
of ``Decoder.sample`` (the live entry point, src/training.py:71,150) runs in libgic_b200.so.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

import gic_b200
from . import _lib


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().contiguous().float()


class _EncoderProject(torch.autograd.Function):
    """Encoder.linear + Encoder.bn, train mode (src/generator.py:23-24)."""

    @staticmethod
    def forward(ctx, pooled, W, b, gamma, beta, eps, mode, running=None):
        _lib.require_cuda()
        pooled, W, b, gamma, beta = map(_f32c, (pooled, W, b, gamma, beta))
        B, Fin = pooled.shape
        E = W.shape[0]
        lin = torch.empty(B, E, device=pooled.device)
        mean = torch.empty(E, device=pooled.device)
        rstd = torch.empty(E, device=pooled.device)
        feats = torch.empty(B, E, device=pooled.device)
        _lib.check(_lib.lib().gic_encoder_fwd(mode, _lib.ptr(pooled), B, Fin, E, _lib.ptr(W), _lib.ptr(b),
                                              _lib.ptr(gamma), _lib.ptr(beta), eps, _lib.ptr(lin), _lib.ptr(mean),
                                              _lib.ptr(rstd), _lib.ptr(feats), _lib.stream()), "gic_encoder_fwd")
        if running is not None:
            bn_running_update(running, mean, rstd, eps, B)
        ctx.save_for_backward(pooled, W, gamma, lin, mean, rstd)
        ctx.mode = mode
        return feats

    @staticmethod
    def backward(ctx, dfeats):
        pooled, W, gamma, lin, mean, rstd = ctx.saved_tensors
        B, Fin = pooled.shape
        E = W.shape[0]
        dfeats = _f32c(dfeats)
        ws = torch.empty(B, E, device=pooled.device)
        dW, db = torch.empty_like(W), torch.empty(E, device=W.device)
        dgamma, dbeta = torch.empty_like(db), torch.empty_like(db)
        _lib.check(_lib.lib().gic_encoder_bwd(ctx.mode, _lib.ptr(dfeats), _lib.ptr(pooled), _lib.ptr(lin),
                                              _lib.ptr(mean), _lib.ptr(rstd), _lib.ptr(W), _lib.ptr(gamma), B, Fin, E,
                                              _lib.ptr(ws), _lib.ptr(dW), _lib.ptr(db), _lib.ptr(dgamma),
                                              _lib.ptr(dbeta), 0, _lib.stream()), "gic_encoder_bwd")
        return None, dW, db, dgamma, dbeta, None, None, None


def bn_running_update(bn, mean, rstd, eps, count):
    """nn.BatchNorm1d's training-mode bookkeeping (momentum 0.01, src/generator.py:16) from the batch statistics the
    projection kernel saved: running_mean / running_var (unbiased) / num_batches_tracked, so that checkpoints and the
    eval-mode forward see what the reference's would."""
    if bn.running_mean is None or not bn.track_running_stats:
        return
    mom = 0.1 if bn.momentum is None else float(bn.momentum)
    _lib.check(_lib.lib().gic_encoder_bn_running_update(_lib.ptr(mean), _lib.ptr(rstd), mean.numel(), float(eps), float(count),
                                                        mom, _lib.ptr(bn.running_mean), _lib.ptr(bn.running_var),
                                                        _lib.ptr(bn.num_batches_tracked), _lib.stream()),
               "gic_encoder_bn_running_update")


def encoder_eval(enc, pooled, mode):
    """Encoder.linear + Encoder.bn with the running statistics (gen.eval(), src/training.py:213-214); forward only."""
    _lib.require_cuda()
    pooled = _f32c(pooled)
    B, Fin = pooled.shape
    E = enc.linear.weight.shape[0]
    lin = torch.empty(B, E, device=pooled.device)
    feats = torch.empty(B, E, device=pooled.device)
    bn = enc.bn
    _lib.check(_lib.lib().gic_encoder_fwd_eval(mode, _lib.ptr(pooled), B, Fin, E, _lib.ptr(_f32c(enc.linear.weight)),
                                               _lib.ptr(_f32c(enc.linear.bias)), _lib.ptr(_f32c(bn.weight)),
                                               _lib.ptr(_f32c(bn.bias)), bn.eps, _lib.ptr(bn.running_mean),
                                               _lib.ptr(bn.running_var), _lib.ptr(lin), _lib.ptr(feats), _lib.stream()),
               "gic_encoder_fwd_eval")
    return feats


class Encoder(nn.Module):
    """Feature projection of the reference's Encoder (src/generator.py:8-25).

    The frozen ResNet trunk (``self.resnet``, run under ``no_grad``) is out of the hot path's scope
    (SURVEY.md section 2 row 2): this Encoder consumes the pooled CNN feature ``[B, feature_dim]``
    that trunk would produce and applies ``linear`` + ``bn`` exactly as lines 23-24 do."""

    def __init__(self, args):
        super().__init__()
        self.feature_dim = getattr(args, "feature_dim", 512)     # resnet18.fc.in_features
        self.linear = nn.Linear(self.feature_dim, args.gen_embed_dim)
        self.bn = nn.BatchNorm1d(args.gen_embed_dim, momentum=0.01)
        self.args = args

    def forward(self, pooled):
        if pooled.dim() != 2 or pooled.shape[1] != self.feature_dim:
            raise ValueError("Encoder expects pooled CNN features [B, %d]" % self.feature_dim)
        if not self.training:
            # eval mode (the reference validates with gen.eval(), src/training.py:213): running statistics, no autograd
            with torch.no_grad():
                return encoder_eval(self, pooled, gic_b200.get_gemm_mode())
        return _EncoderProject.apply(pooled, self.linear.weight, self.linear.bias, self.bn.weight, self.bn.bias,
                                     self.bn.eps, gic_b200.get_gemm_mode(), self.bn)


class _DecodeSample(torch.autograd.Function):
    """Decoder.sample forward/backward through gic_decode_sample_{fwd,bwd}."""

    @staticmethod
    def forward(ctx, features, u, temperature, pretrain, L, forced_ids, mode, layers, W_emb, W_out, b_out, *lstm):
        _lib.require_cuda()
        lib = _lib.lib()
        dev = features.device
        features = _f32c(features)
        W_emb, W_out, b_out = map(_f32c, (W_emb, W_out, b_out))
        lstm = [_f32c(w) for w in lstm]
        W_ih, W_hh, b_ih, b_hh = (lstm[i::4] for i in range(4))
        B, E = features.shape
        V, H = W_out.shape
        if u is not None:
            u = _f32c(u)
            if tuple(u.shape) != (L, B, V):
                raise ValueError("uniforms must have shape [L, B, V] = %r" % ((L, B, V),))
        if forced_ids is not None:
            forced_ids = forced_ids.detach().contiguous().long()
        out = torch.empty(B, L, V, device=dev)
        ids = torch.empty(B, L, dtype=torch.int64, device=dev)
        saved = torch.empty(lib.gic_decode_saved_floats(B, L, E, H, layers), device=dev)
        ws = torch.empty(lib.gic_decode_fwd_workspace_floats(B, V, H), device=dev)
        _lib.check(lib.gic_decode_sample_fwd(
            mode, _lib.ptr(features), _lib.ptr(W_emb), _lib.ptr_array(W_ih), _lib.ptr_array(W_hh),
            _lib.ptr_array(b_ih), _lib.ptr_array(b_hh), _lib.ptr(W_out), _lib.ptr(b_out), _lib.ptr(u),
            float(temperature), int(bool(pretrain)), _lib.ptr(forced_ids), B, L, V, E, H, layers, _lib.ptr(out),
            _lib.ptr(ids), _lib.ptr(saved), _lib.ptr(ws), _lib.stream()), "gic_decode_sample_fwd")
        fed = ids if forced_ids is None else forced_ids
        ctx.save_for_backward(out, fed, saved, W_emb, W_out, *W_ih, *W_hh)
        ctx.dims = (B, L, V, E, H, layers, float(temperature), bool(pretrain), mode)
        ctx.mark_non_differentiable(ids)
        return out, ids

    @staticmethod
    def backward(ctx, dout, _dids):
        lib = _lib.lib()
        B, L, V, E, H, layers, T, pretrain, mode = ctx.dims
        out, fed, saved, W_emb, W_out = ctx.saved_tensors[:5]
        W_ih = ctx.saved_tensors[5:5 + layers]
        W_hh = ctx.saved_tensors[5 + layers:5 + 2 * layers]
        dev = out.device
        dout = _f32c(dout)
        ws = torch.empty(lib.gic_decode_bwd_workspace_floats(B, L, V, E, H, layers), device=dev)
        dW_emb, dW_out = torch.empty_like(W_emb), torch.empty_like(W_out)
        db_out = torch.empty(V, device=dev)
        dW_ih = [torch.empty_like(w) for w in W_ih]
        dW_hh = [torch.empty_like(w) for w in W_hh]
        db_ih = [torch.empty(4 * H, device=dev) for _ in range(layers)]
        db_hh = [torch.empty(4 * H, device=dev) for _ in range(layers)]
        dfeat = torch.empty(B, E, device=dev)
        _lib.check(lib.gic_decode_sample_bwd(
            mode, _lib.ptr(dout), _lib.ptr(out), _lib.ptr(fed), _lib.ptr(W_emb), _lib.ptr_array(W_ih),
            _lib.ptr_array(W_hh), _lib.ptr(W_out), T, int(pretrain), B, L, V, E, H, layers, _lib.ptr(saved),
            _lib.ptr(ws), _lib.ptr(dW_emb), _lib.ptr_array(dW_ih), _lib.ptr_array(dW_hh), _lib.ptr_array(db_ih),
            _lib.ptr_array(db_hh), _lib.ptr(dW_out), _lib.ptr(db_out), _lib.ptr(dfeat), 0, _lib.stream()),
            "gic_decode_sample_bwd")
        lstm_grads = []
        for l in range(layers):
            lstm_grads += [dW_ih[l], dW_hh[l], db_ih[l], db_hh[l]]
        return (dfeat, None, None, None, None, None, None, None, dW_emb, dW_out, db_out, *lstm_grads)


class _DecodeSampleAttn(torch.autograd.Function):
    """Decoder.sample with the attention cell (EXTENSION, SURVEY.md 8a row B1) through gic_decode_sample_{fwd,bwd}_attn."""

    @staticmethod
    def forward(ctx, features, grid, u, temperature, L, forced_ids, mode, W_k, W_v, W_q, w_e, W_emb, W_out, b_out, W_ih,
                W_hh, b_ih, b_hh):
        _lib.require_cuda()
        lib = _lib.lib()
        dev = features.device
        features, grid, u = _f32c(features), _f32c(grid), _f32c(u)
        W_k, W_v, W_q, w_e, W_emb, W_out, b_out, W_ih, W_hh, b_ih, b_hh = map(
            _f32c, (W_k, W_v, W_q, w_e, W_emb, W_out, b_out, W_ih, W_hh, b_ih, b_hh))
        B, E = features.shape
        V, H = W_out.shape
        Pn, Da = grid.shape[1], W_k.shape[0]
        if forced_ids is not None:
            forced_ids = forced_ids.detach().contiguous().long()
        out = torch.empty(B, L, V, device=dev)
        ids = torch.empty(B, L, dtype=torch.int64, device=dev)
        saved = torch.empty(lib.gic_decode_saved_floats(B, L, E, H, 1), device=dev)
        asaved = torch.empty(lib.gic_attn_saved_floats(B, L, Pn, Da, E), device=dev)
        ws = torch.empty(lib.gic_decode_fwd_workspace_floats(B, V, H), device=dev)
        blk = _lib.attn_block(grid, W_k, W_v, W_q, w_e.reshape(-1), asaved)
        import ctypes as C
        _lib.check(lib.gic_decode_sample_fwd_attn(
            C.byref(blk), mode, _lib.ptr(features), _lib.ptr(W_emb), _lib.ptr_array([W_ih]), _lib.ptr_array([W_hh]),
            _lib.ptr_array([b_ih]), _lib.ptr_array([b_hh]), _lib.ptr(W_out), _lib.ptr(b_out), _lib.ptr(u),
            float(temperature), 0, _lib.ptr(forced_ids), B, L, V, E, H, 1, _lib.ptr(out), _lib.ptr(ids), _lib.ptr(saved),
            _lib.ptr(ws), _lib.stream()), "gic_decode_sample_fwd_attn")
        fed = ids if forced_ids is None else forced_ids
        ctx.save_for_backward(out, fed, saved, asaved, grid, W_k, W_v, W_q, w_e, W_emb, W_out, W_ih, W_hh)
        ctx.dims = (B, L, V, E, H, Pn, Da, float(temperature), mode)
        ctx.mark_non_differentiable(ids)
        return out, ids

    @staticmethod
    def backward(ctx, dout, _dids):
        import ctypes as C
        lib = _lib.lib()
        B, L, V, E, H, Pn, Da, T, mode = ctx.dims
        out, fed, saved, asaved, grid, W_k, W_v, W_q, w_e, W_emb, W_out, W_ih, W_hh = ctx.saved_tensors
        dev = out.device
        dout = _f32c(dout)
        ws = torch.empty(lib.gic_decode_bwd_workspace_floats(B, L, V, E, H, 1), device=dev)
        aws = torch.empty(lib.gic_attn_bwd_workspace_floats(B, L, Pn, Da, E), device=dev)
        dW_k, dW_v, dW_q, dw_e = (torch.empty_like(t) for t in (W_k, W_v, W_q, w_e))
        dW_emb, dW_out = torch.empty_like(W_emb), torch.empty_like(W_out)
        db_out = torch.empty(V, device=dev)
        dW_ih, dW_hh = torch.empty_like(W_ih), torch.empty_like(W_hh)
        db_ih, db_hh = torch.empty(4 * H, device=dev), torch.empty(4 * H, device=dev)
        dfeat = torch.empty(B, E, device=dev)
        blk = _lib.attn_block(grid, W_k, W_v, W_q, w_e.reshape(-1), asaved, aws, dW_k, dW_v, dW_q, dw_e)
        _lib.check(lib.gic_decode_sample_bwd_attn(
            C.byref(blk), mode, _lib.ptr(dout), None, None, None, 0, _lib.ptr(out), _lib.ptr(fed), _lib.ptr(W_emb),
            _lib.ptr_array([W_ih]), _lib.ptr_array([W_hh]), _lib.ptr(W_out), T, 0, B, L, V, E, H, 1, _lib.ptr(saved),
            _lib.ptr(ws), _lib.ptr(dW_emb), _lib.ptr_array([dW_ih]), _lib.ptr_array([dW_hh]), _lib.ptr_array([db_ih]),
            _lib.ptr_array([db_hh]), _lib.ptr(dW_out), _lib.ptr(db_out), _lib.ptr(dfeat), _lib.stream()),
            "gic_decode_sample_bwd_attn")
        return (dfeat, None, None, None, None, None, None, dW_k, dW_v, dW_q, dw_e, dW_emb, dW_out, db_out, dW_ih, dW_hh,
                db_ih, db_hh)


def decode_beam(dec, features, beam_size, max_caption_len, length_penalty=0.0, eos_id=2, mode=None, trace=None):
    """gic_decode_beam over the decoder's weights -> (ids[B,K,L] int64, scores[B,K], lengths[B,K] int32).  trace[L,B,K,2]
    (int32, optional) receives the (parent slot, token) chosen at every step."""
    _lib.require_cuda()
    lib = _lib.lib()
    mode = gic_b200.get_gemm_mode() if mode is None else mode
    features = _f32c(features)
    B, E = features.shape
    K, L = int(beam_size), int(max_caption_len)
    V, H = dec.linear.weight.shape
    layers = dec.lstm.num_layers
    dev = features.device
    lp = [_f32c(w) for w in dec.lstm_params()]
    W_ih, W_hh, b_ih, b_hh = lp[0::4], lp[1::4], lp[2::4], lp[3::4]
    W_emb, W_out, b_out = _f32c(dec.embed.weight), _f32c(dec.linear.weight), _f32c(dec.linear.bias)
    ids = torch.empty(B, K, L, dtype=torch.int64, device=dev)
    scores = torch.empty(B, K, device=dev)
    lengths = torch.empty(B, K, dtype=torch.int32, device=dev)
    ws = torch.empty(lib.gic_decode_beam_workspace_floats(B, K, L, V, E, H, layers), device=dev)
    _lib.check(lib.gic_decode_beam(mode, _lib.ptr(features), _lib.ptr(W_emb), _lib.ptr_array(W_ih), _lib.ptr_array(W_hh),
                                   _lib.ptr_array(b_ih), _lib.ptr_array(b_hh), _lib.ptr(W_out), _lib.ptr(b_out), B, K, L, V,
                                   E, H, layers, int(eos_id), float(length_penalty), _lib.ptr(ids), _lib.ptr(scores),
                                   _lib.ptr(lengths), _lib.ptr(trace), _lib.ptr(ws), _lib.stream()), "gic_decode_beam")
    return ids, scores, lengths


class Decoder(nn.Module):
    """LSTM caption decoder (src/generator.py:27-96).  ``embed``/``lstm``/``linear`` are parameter
    containers with the reference's state_dict keys; ``sample`` runs on the B200 kernels."""

    def __init__(self, args):
        super().__init__()
        self.embed = nn.Embedding(args.vocab_size, args.gen_embed_dim)
        self.lstm = nn.LSTM(args.gen_embed_dim, args.gen_hidden_dim, args.gen_num_layers, batch_first=True)
        self.linear = nn.Linear(args.gen_hidden_dim, args.vocab_size)
        self.max_seq_length = args.max_seq_len
        self.temperature = args.temperature
        self.args = args
        # EXTENSION (SURVEY.md 8a row B1): additive attention over the CNN feature grid; off by default so that the
        # reference's state_dict is unchanged
        self.attention = bool(getattr(args, "gen_attention", 0))
        if self.attention:
            Cf, Da = args.feature_channels, args.attn_dim
            self.attn_k = nn.Linear(Cf, Da, bias=False)
            self.attn_v = nn.Linear(Cf, args.gen_embed_dim, bias=False)
            self.attn_q = nn.Linear(args.gen_hidden_dim, Da, bias=False)
            self.attn_e = nn.Linear(Da, 1, bias=False)

    def lstm_params(self):
        ps = []
        for l in range(self.lstm.num_layers):
            ps += [getattr(self.lstm, f"weight_ih_l{l}"), getattr(self.lstm, f"weight_hh_l{l}"),
                   getattr(self.lstm, f"bias_ih_l{l}"), getattr(self.lstm, f"bias_hh_l{l}")]
        return ps

    def attn_params(self):
        return [self.attn_k.weight, self.attn_v.weight, self.attn_q.weight, self.attn_e.weight]

    def sample(self, features, states=None, pretrain=False, max_caption_len=34, u=None, forced_ids=None, grid=None):
        """Generate captions (src/generator.py:55-81) -> (outputs[B,L,V], sampled_ids[B,L]).

        Extensions over the reference signature (keyword-only in spirit): ``u[L,B,V]`` supplies the
        uniforms ``add_gumbel`` would draw (default: drawn on-device, src/generator.py:90);
        ``forced_ids[B,L]`` teacher-forces the fed-back token for parity runs."""
        if states is not None:
            raise NotImplementedError("sample(states=...) is never used by the reference's training loops")
        L = int(max_caption_len)
        if u is None and not pretrain:
            u = torch.rand(L, features.shape[0], self.linear.out_features, device=features.device)
        if grid is not None:
            if not self.attention:
                raise ValueError("a feature grid was given but the decoder was built without --gen-attention 1")
            if pretrain or self.lstm.num_layers != 1:
                raise NotImplementedError("the attention cell is implemented for single-layer adversarial decoding")
            return _DecodeSampleAttn.apply(features, grid, u, float(self.temperature), L, forced_ids,
                                           gic_b200.get_gemm_mode(), *self.attn_params(), self.embed.weight,
                                           self.linear.weight, self.linear.bias, *self.lstm_params())
        return _DecodeSample.apply(features, u, float(self.temperature), bool(pretrain), L, forced_ids,
                                   gic_b200.get_gemm_mode(), self.lstm.num_layers, self.embed.weight,
                                   self.linear.weight, self.linear.bias, *self.lstm_params())

    @torch.no_grad()
    def beam_search(self, features, beam_size=3, max_caption_len=34, length_penalty=0.0, eos_id=2):
        """The most likely captions of features[B,E] (the step-0 input, as in sample) by beam search (EXTENSION; the
        reference has none, oracle/ref_beam.py defines it) -> (ids[B,K,L], scores[B,K], lengths[B,K]), the K beams of each
        image best first by score / length ** length_penalty.  ids hold PAD (0) after <E> (eos_id); scores are sums of
        log-probabilities; lengths count tokens up to and including <E>.  beam_size = 1 is greedy decoding."""
        if self.attention:
            raise NotImplementedError("beam search is implemented for the plain LSTM decoder, not the attention cell")
        return decode_beam(self, features, beam_size, max_caption_len, length_penalty, eos_id)

    def add_gumbel(self, o_t, eps=1e-10, gpu=0):
        """Kept for interface parity (src/generator.py:84-96); the hot path fuses this into the sampler."""
        u = torch.rand_like(o_t)
        return o_t - torch.log(-torch.log(u + eps) + eps)

    def forward(self, features, caps, lengths, pretrain=False):
        raise NotImplementedError("Decoder.forward (teacher-forced packed path, src/generator.py:39-53) is never "
                                  "called by the reference's training loops; use sample()")


class Generator(nn.Module):
    """Owns encoder + decoder and the U(-0.05, 0.05) re-initialisation (src/generator.py:98-123)."""

    def __init__(self, args):
        super().__init__()
        self.encoder = Encoder(args)
        self.decoder = Decoder(args)
        self.args = args
        self.init_params()

    def forward(self, images, caps, lengths, pretrain=False):
        raise NotImplementedError("Generator.forward is broken in the reference (reads args.cgan, SURVEY Q3) and "
                                  "never called; use encoder(...) / decoder.sample(...)")

    def init_params(self):
        for param in self.parameters():
            if param.requires_grad and len(param.shape) > 0:
                stddev = 1 / math.sqrt(param.shape[0])
                if self.args.gen_init == "uniform":
                    torch.nn.init.uniform_(param, a=-0.05, b=0.05)
                elif self.args.gen_init == "normal":
                    torch.nn.init.normal_(param, std=stddev)
