"""Caption generator with the reference's interface (src/generator.py): ``Encoder``, ``Decoder`` and
``Generator`` keep their constructor signatures, attribute names and ``state_dict`` keys, so
``optim.Adam(gen.parameters())`` and checkpoints written by the reference keep working.  The compute
of ``Decoder.sample`` (the live entry point, src/training.py:71,150) runs in libgic_b200.so.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.nn as nn

import gic_b200
from . import _lib


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().contiguous().float()


def lstm_split(lstm):
    """Per-layer lists (W_ih, W_hh, b_ih, b_hh) of a flat list in Decoder.lstm_params() order."""
    return lstm[0::4], lstm[1::4], lstm[2::4], lstm[3::4]


# ---- one binding per compute entry point: each owns its ctypes argument list, allocates nothing, never synchronises ----
def encoder_fwd_raw(mode, pooled, W, b, gamma, beta, eps, lin, mean, rstd, feats, stream):
    """gic_encoder_fwd: Encoder.linear + Encoder.bn with the batch statistics; lin / mean / rstd are saved for the backward."""
    B, Fin = pooled.shape
    P = _lib.ptr
    _lib.check(_lib.lib().gic_encoder_fwd(mode, P(pooled), B, Fin, W.shape[0], P(W), P(b), P(gamma), P(beta), eps, P(lin),
                                          P(mean), P(rstd), P(feats), stream), "gic_encoder_fwd")


def encoder_fwd_eval_raw(mode, pooled, W, b, gamma, beta, eps, running_mean, running_var, lin, feats, stream):
    """gic_encoder_fwd_eval: the same projection with the running statistics; lin is workspace."""
    B, Fin = pooled.shape
    P = _lib.ptr
    _lib.check(_lib.lib().gic_encoder_fwd_eval(mode, P(pooled), B, Fin, W.shape[0], P(W), P(b), P(gamma), P(beta), eps,
                                               P(running_mean), P(running_var), P(lin), P(feats), stream),
               "gic_encoder_fwd_eval")


def encoder_bwd_raw(mode, dfeats, pooled, lin, mean, rstd, W, gamma, dlin, dW, db, dgamma, dbeta, stream):
    """gic_encoder_bwd of encoder_fwd_raw: dW / db / dgamma / dbeta overwritten, dlin is workspace."""
    B, Fin = pooled.shape
    P = _lib.ptr
    _lib.check(_lib.lib().gic_encoder_bwd(mode, P(dfeats), P(pooled), P(lin), P(mean), P(rstd), P(W), P(gamma), B, Fin,
                                          W.shape[0], P(dlin), P(dW), P(db), P(dgamma), P(dbeta), 0, stream),
               "gic_encoder_bwd")


def decode_fwd_raw(mode, features, W_emb, lstm, W_out, b_out, u, temperature, pretrain, forced_ids, out, ids, saved, ws,
                   stream, attn=None):
    """gic_decode_sample_fwd (Decoder.sample into out[B,L,V] / ids[B,L]), or gic_decode_sample_fwd_attn when attn is the
    gic_attn_t of the attention cell (_lib.attn_block).  lstm: Decoder.lstm_params() order."""
    W_ih, W_hh, b_ih, b_hh = lstm_split(lstm)
    B, L = ids.shape
    V, H = W_out.shape
    P, PA = _lib.ptr, _lib.ptr_array
    args = (mode, P(features), P(W_emb), PA(W_ih), PA(W_hh), PA(b_ih), PA(b_hh), P(W_out), P(b_out), P(u),
            float(temperature), int(pretrain), P(forced_ids), B, L, V, W_emb.shape[1], H, len(W_ih), P(out), P(ids),
            P(saved), P(ws), stream)
    if attn is None:
        _lib.check(_lib.lib().gic_decode_sample_fwd(*args), "gic_decode_sample_fwd")
    else:
        _lib.check(_lib.lib().gic_decode_sample_fwd_attn(C.byref(attn), *args), "gic_decode_sample_fwd_attn")


def decode_bwd_raw(mode, dout, out, fed, W_emb, lstm, W_out, temperature, pretrain, saved, ws, dW_emb, dlstm, dW_out,
                   db_out, dfeat, stream, factored=None, attn=None):
    """Backward of decode_fwd_raw; the gradients (dlstm in Decoder.lstm_params() order) are overwritten.  The incoming
    gradient is dout[B,L,V] (gic_decode_sample_bwd), or factored = (demb, emb, W_e, De) with dout = None
    (gic_decode_sample_bwd_factored).  attn: the forward's gic_attn_t with its backward workspace and gradients
    (gic_decode_sample_bwd_attn, either form of the incoming gradient)."""
    W_ih, W_hh = lstm[0::4], lstm[1::4]
    dW_ih, dW_hh, db_ih, db_hh = lstm_split(dlstm)
    B, L = fed.shape
    V, H = W_out.shape
    E, layers = W_emb.shape[1], len(W_ih)
    P, PA = _lib.ptr, _lib.ptr_array
    grads = (P(saved), P(ws), P(dW_emb), PA(dW_ih), PA(dW_hh), PA(db_ih), PA(db_hh), P(dW_out), P(db_out), P(dfeat))
    if attn is not None:
        demb, emb, W_e, De = factored or (None, None, None, 0)
        _lib.check(_lib.lib().gic_decode_sample_bwd_attn(
            C.byref(attn), mode, P(dout), P(demb), P(emb), P(W_e), De, P(out), P(fed), P(W_emb), PA(W_ih), PA(W_hh),
            P(W_out), temperature, int(pretrain), B, L, V, E, H, layers, *grads, stream), "gic_decode_sample_bwd_attn")
    elif factored is not None:
        demb, emb, W_e, De = factored
        _lib.check(_lib.lib().gic_decode_sample_bwd_factored(
            mode, P(demb), P(emb), P(W_e), De, P(out), P(fed), P(W_emb), PA(W_ih), PA(W_hh), P(W_out), temperature, B, L,
            V, E, H, layers, *grads, 0, stream), "gic_decode_sample_bwd_factored")
    else:
        _lib.check(_lib.lib().gic_decode_sample_bwd(
            mode, P(dout), P(out), P(fed), P(W_emb), PA(W_ih), PA(W_hh), P(W_out), temperature, int(pretrain), B, L, V, E,
            H, layers, *grads, 0, stream), "gic_decode_sample_bwd")


class _EncoderProject(torch.autograd.Function):
    """Encoder.linear + Encoder.bn, train mode (src/generator.py:23-24)."""

    @staticmethod
    def forward(ctx, pooled, W, b, gamma, beta, eps, mode, running=None):
        _lib.require_cuda()
        pooled, W, b, gamma, beta = map(_f32c, (pooled, W, b, gamma, beta))
        B = pooled.shape[0]
        E = W.shape[0]
        lin = torch.empty(B, E, device=pooled.device)
        mean = torch.empty(E, device=pooled.device)
        rstd = torch.empty(E, device=pooled.device)
        feats = torch.empty(B, E, device=pooled.device)
        encoder_fwd_raw(mode, pooled, W, b, gamma, beta, eps, lin, mean, rstd, feats, _lib.stream())
        if running is not None:
            bn_running_update(running, mean, rstd, eps, B)
        ctx.save_for_backward(pooled, W, gamma, lin, mean, rstd)
        ctx.mode = mode
        return feats

    @staticmethod
    def backward(ctx, dfeats):
        pooled, W, gamma, lin, mean, rstd = ctx.saved_tensors
        dfeats = _f32c(dfeats)
        ws = torch.empty_like(lin)
        dW, db = torch.empty_like(W), torch.empty_like(mean)
        dgamma, dbeta = torch.empty_like(db), torch.empty_like(db)
        encoder_bwd_raw(ctx.mode, dfeats, pooled, lin, mean, rstd, W, gamma, ws, dW, db, dgamma, dbeta, _lib.stream())
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
    B = pooled.shape[0]
    E = enc.linear.weight.shape[0]
    lin = torch.empty(B, E, device=pooled.device)
    feats = torch.empty(B, E, device=pooled.device)
    bn = enc.bn
    encoder_fwd_eval_raw(mode, pooled, _f32c(enc.linear.weight), _f32c(enc.linear.bias), _f32c(bn.weight), _f32c(bn.bias),
                         bn.eps, bn.running_mean, bn.running_var, lin, feats, _lib.stream())
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
    """Decoder.sample forward/backward through decode_fwd_raw / decode_bwd_raw."""

    @staticmethod
    def forward(ctx, features, u, temperature, pretrain, L, forced_ids, mode, W_emb, W_out, b_out, *lstm):
        _lib.require_cuda()
        lib = _lib.lib()
        dev = features.device
        features = _f32c(features)
        W_emb, W_out, b_out = map(_f32c, (W_emb, W_out, b_out))
        lstm = [_f32c(w) for w in lstm]
        layers = len(lstm) // 4
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
        decode_fwd_raw(mode, features, W_emb, lstm, W_out, b_out, u, temperature, pretrain, forced_ids, out, ids, saved, ws,
                       _lib.stream())
        fed = ids if forced_ids is None else forced_ids
        ctx.save_for_backward(out, fed, saved, W_emb, W_out, *lstm)
        ctx.meta = (float(temperature), bool(pretrain), mode)
        ctx.mark_non_differentiable(ids)
        return out, ids

    @staticmethod
    def backward(ctx, dout, _dids):
        T, pretrain, mode = ctx.meta
        out, fed, saved, W_emb, W_out, *lstm = ctx.saved_tensors
        B, L, V = out.shape
        E, H = W_emb.shape[1], W_out.shape[1]
        dev = out.device
        ws = torch.empty(_lib.lib().gic_decode_bwd_workspace_floats(B, L, V, E, H, len(lstm) // 4), device=dev)
        dW_emb, dW_out = torch.empty_like(W_emb), torch.empty_like(W_out)
        db_out = torch.empty(V, device=dev)
        dlstm = [torch.empty_like(w) for w in lstm]
        dfeat = torch.empty(B, E, device=dev)
        decode_bwd_raw(mode, _f32c(dout), out, fed, W_emb, lstm, W_out, T, pretrain, saved, ws, dW_emb, dlstm, dW_out,
                       db_out, dfeat, _lib.stream())
        return (dfeat, None, None, None, None, None, None, dW_emb, dW_out, db_out, *dlstm)


class _DecodeSampleAttn(torch.autograd.Function):
    """Decoder.sample with the attention cell (EXTENSION, SURVEY.md 8a row B1) through decode_fwd_raw / decode_bwd_raw."""

    @staticmethod
    def forward(ctx, features, grid, u, temperature, L, forced_ids, mode, W_k, W_v, W_q, w_e, W_emb, W_out, b_out, *lstm):
        _lib.require_cuda()
        lib = _lib.lib()
        dev = features.device
        features, grid, u = _f32c(features), _f32c(grid), _f32c(u)
        W_k, W_v, W_q, w_e, W_emb, W_out, b_out = map(_f32c, (W_k, W_v, W_q, w_e, W_emb, W_out, b_out))
        lstm = [_f32c(w) for w in lstm]
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
        decode_fwd_raw(mode, features, W_emb, lstm, W_out, b_out, u, temperature, 0, forced_ids, out, ids, saved, ws,
                       _lib.stream(), attn=blk)
        fed = ids if forced_ids is None else forced_ids
        ctx.save_for_backward(out, fed, saved, asaved, grid, W_k, W_v, W_q, w_e, W_emb, W_out, *lstm)
        ctx.meta = (float(temperature), mode)
        ctx.mark_non_differentiable(ids)
        return out, ids

    @staticmethod
    def backward(ctx, dout, _dids):
        T, mode = ctx.meta
        out, fed, saved, asaved, grid, W_k, W_v, W_q, w_e, W_emb, W_out, *lstm = ctx.saved_tensors
        B, L, V = out.shape
        E, H = W_emb.shape[1], W_out.shape[1]
        Pn, Da = grid.shape[1], W_k.shape[0]
        dev = out.device
        lib = _lib.lib()
        ws = torch.empty(lib.gic_decode_bwd_workspace_floats(B, L, V, E, H, 1), device=dev)
        aws = torch.empty(lib.gic_attn_bwd_workspace_floats(B, L, Pn, Da, E), device=dev)
        dW_k, dW_v, dW_q, dw_e = (torch.empty_like(t) for t in (W_k, W_v, W_q, w_e))
        dW_emb, dW_out = torch.empty_like(W_emb), torch.empty_like(W_out)
        db_out = torch.empty(V, device=dev)
        dlstm = [torch.empty_like(w) for w in lstm]
        dfeat = torch.empty(B, E, device=dev)
        blk = _lib.attn_block(grid, W_k, W_v, W_q, w_e.reshape(-1), asaved, aws, dW_k, dW_v, dW_q, dw_e)
        decode_bwd_raw(mode, _f32c(dout), out, fed, W_emb, lstm, W_out, T, 0, saved, ws, dW_emb, dlstm, dW_out, db_out,
                       dfeat, _lib.stream(), attn=blk)
        return (dfeat, None, None, None, None, None, None, dW_k, dW_v, dW_q, dw_e, dW_emb, dW_out, db_out, *dlstm)


def check_constraints(min_length, no_repeat_ngram_size, bad_ids, max_caption_len, V, width):
    """ValueError for constraints gic_decode_beam_constrained / gic_sample_captions_constrained reject, and bad ids outside
    [0, V) (checked on the host, before any GPU work); width = beam_size, or top_k for sampling."""
    L = int(max_caption_len)
    if not 0 <= int(min_length) <= L:
        raise ValueError("min_length must lie in [0, max_caption_len] = [0, %d]" % L)
    if int(no_repeat_ngram_size) < 0:
        raise ValueError("no_repeat_ngram_size must be >= 0")
    bad = [int(w) for w in (bad_ids if bad_ids is not None else ())]
    if any(not 0 <= w < V for w in bad):
        raise ValueError("bad_ids must lie in [0, %d)" % V)
    allowed = V - len(bad) - (int(min_length) > 0) - (L - 1 if int(no_repeat_ngram_size) > 0 else 0)
    if max(int(width), 1) > allowed:
        raise ValueError("the constraints may leave %d allowed tokens per step, fewer than %d" % (allowed, max(int(width), 1)))


def _constraints(min_length, no_repeat_ngram_size, bad_ids, dev):
    """(gic_decode_constraints_t or None, the device bad ids it points at).  bad_ids is a host sequence, copied here, or
    an int64 tensor already on the device (no copy: the call stays capturable into a CUDA graph)."""
    if torch.is_tensor(bad_ids) and bad_ids.is_cuda:
        ids = bad_ids.to(torch.int64).contiguous()
    else:
        bad = [int(w) for w in (bad_ids if bad_ids is not None else ())]
        ids = torch.tensor(bad, dtype=torch.int64, device=dev) if bad else None
    n_bad = 0 if ids is None else ids.numel()
    if int(min_length) == 0 and int(no_repeat_ngram_size) == 0 and n_bad == 0:
        return None, None
    return _lib.DecodeConstraints(int(min_length), int(no_repeat_ngram_size), _lib.ptr(ids), n_bad), ids


def decode_beam(dec, features, beam_size, max_caption_len, length_penalty=0.0, eos_id=2, mode=None, trace=None,
                min_length=0, no_repeat_ngram_size=0, bad_ids=None):
    """gic_decode_beam_constrained over the decoder's weights -> (ids[B,K,L] int64, scores[B,K], lengths[B,K] int32).
    trace[L,B,K,2] (int32, optional) receives the (parent slot, token) chosen at every step.  min_length /
    no_repeat_ngram_size / bad_ids: the constraints of include/gic_b200.h gic_decode_constraints_t (none by default)."""
    _lib.require_cuda()
    lib = _lib.lib()
    mode = gic_b200.get_gemm_mode() if mode is None else mode
    features = _f32c(features)
    B, E = features.shape
    K, L = int(beam_size), int(max_caption_len)
    V, H = dec.linear.weight.shape
    layers = dec.lstm.num_layers
    dev = features.device
    W_ih, W_hh, b_ih, b_hh = lstm_split([_f32c(w) for w in dec.lstm_params()])
    W_emb, W_out, b_out = _f32c(dec.embed.weight), _f32c(dec.linear.weight), _f32c(dec.linear.bias)
    ids = torch.empty(B, K, L, dtype=torch.int64, device=dev)
    scores = torch.empty(B, K, device=dev)
    lengths = torch.empty(B, K, dtype=torch.int32, device=dev)
    c, _bad = _constraints(min_length, no_repeat_ngram_size, bad_ids, dev)
    cp = None if c is None else C.byref(c)
    ws = torch.empty(lib.gic_decode_beam_constrained_workspace_floats(B, K, L, V, E, H, layers, cp), device=dev)
    _lib.check(lib.gic_decode_beam_constrained(mode, _lib.ptr(features), _lib.ptr(W_emb), _lib.ptr_array(W_ih),
                                               _lib.ptr_array(W_hh), _lib.ptr_array(b_ih), _lib.ptr_array(b_hh),
                                               _lib.ptr(W_out), _lib.ptr(b_out), B, K, L, V, E, H, layers, int(eos_id),
                                               float(length_penalty), cp, _lib.ptr(ids), _lib.ptr(scores),
                                               _lib.ptr(lengths), _lib.ptr(trace), _lib.ptr(ws), _lib.stream()),
               "gic_decode_beam_constrained")
    return ids, scores, lengths


def score_captions(dec, features, captions, lengths=None, mode=None):
    """gic_score_captions over the decoder's weights -> (logp[B,L], caption_logp[B], correct[B,L] uint8).  No
    host sync: ids outside [0, V) are not checked here (they give NaN, see Decoder.score)."""
    _lib.require_cuda()
    lib = _lib.lib()
    mode = gic_b200.get_gemm_mode() if mode is None else mode
    features = _f32c(features)
    captions = captions.detach().to(features.device).contiguous().long()
    B, E = features.shape
    if captions.dim() != 2 or captions.shape[0] != B:
        raise ValueError("captions must have shape [B, L] with B = %d" % B)
    L = captions.shape[1]
    if lengths is not None:
        lengths = torch.as_tensor(lengths, device=features.device).to(torch.int32).contiguous()
        if tuple(lengths.shape) != (B,):
            raise ValueError("lengths must have shape [B] = [%d]" % B)
    V, H = dec.linear.weight.shape
    layers = dec.lstm.num_layers
    dev = features.device
    W_ih, W_hh, b_ih, b_hh = lstm_split([_f32c(w) for w in dec.lstm_params()])
    W_emb, W_out, b_out = _f32c(dec.embed.weight), _f32c(dec.linear.weight), _f32c(dec.linear.bias)
    logp = torch.empty(B, L, device=dev)
    total = torch.empty(B, device=dev)
    corr = torch.empty(B, L, dtype=torch.uint8, device=dev)
    ws = torch.empty(lib.gic_score_captions_workspace_floats(B, L, V, E, H, layers), device=dev)
    _lib.check(lib.gic_score_captions(mode, _lib.ptr(features), _lib.ptr(captions), _lib.ptr(lengths), _lib.ptr(W_emb),
                                      _lib.ptr_array(W_ih), _lib.ptr_array(W_hh), _lib.ptr_array(b_ih), _lib.ptr_array(b_hh),
                                      _lib.ptr(W_out), _lib.ptr(b_out), B, L, V, E, H, layers, _lib.ptr(logp),
                                      _lib.ptr(total), _lib.ptr(corr), _lib.ptr(ws), _lib.stream()), "gic_score_captions")
    return logp, total, corr


def check_sample_args(num_samples, max_caption_len, temperature, top_k, top_p, eos_id, V):
    """ValueError for sampling arguments gic_sample_captions rejects (checked on the host, before any GPU work)."""
    if int(num_samples) < 1:
        raise ValueError("num_samples must be >= 1")
    if int(max_caption_len) < 1:
        raise ValueError("max_caption_len must be >= 1")
    if not (math.isfinite(float(temperature)) and float(temperature) > 0):
        raise ValueError("temperature must be finite and > 0")
    if not 0 <= int(top_k) <= min(16, V):
        raise ValueError("top_k must lie in [0, min(16, V)] = [0, %d]" % min(16, V))
    if not 0 < float(top_p) <= 1:
        raise ValueError("top_p must lie in (0, 1]")
    if float(top_p) < 1 and int(top_k) == 0:
        raise ValueError("top_p < 1 needs 1 <= top_k <= 16: nucleus sampling works inside the top 16 tokens")
    if not 0 <= int(eos_id) < V:
        raise ValueError("eos_id must lie in [0, %d)" % V)


def sample_captions(dec, features, num_samples=1, max_caption_len=34, temperature=1.0, top_k=0, top_p=1.0, eos_id=2,
                    mode=None, min_length=0, no_repeat_ngram_size=0, bad_ids=None):
    """gic_sample_captions_constrained over the decoder's weights -> (ids[B,n,L] int64, caption_logp[B,n], lengths[B,n]
    int32).  The draws read the library's Philox state (gic_set_rng) of the current context.  min_length /
    no_repeat_ngram_size / bad_ids: the constraints of include/gic_b200.h gic_decode_constraints_t (none by default)."""
    _lib.require_cuda()
    lib = _lib.lib()
    mode = gic_b200.get_gemm_mode() if mode is None else mode
    features = _f32c(features)
    B, E = features.shape
    n, L = int(num_samples), int(max_caption_len)
    V, H = dec.linear.weight.shape
    layers = dec.lstm.num_layers
    dev = features.device
    W_ih, W_hh, b_ih, b_hh = lstm_split([_f32c(w) for w in dec.lstm_params()])
    W_emb, W_out, b_out = _f32c(dec.embed.weight), _f32c(dec.linear.weight), _f32c(dec.linear.bias)
    ids = torch.empty(B, n, L, dtype=torch.int64, device=dev)
    logp = torch.empty(B, n, device=dev)
    lengths = torch.empty(B, n, dtype=torch.int32, device=dev)
    c, _bad = _constraints(min_length, no_repeat_ngram_size, bad_ids, dev)
    cp = None if c is None else C.byref(c)
    ws = torch.empty(lib.gic_sample_captions_constrained_workspace_floats(B, n, L, V, E, H, layers, int(top_k), cp),
                     device=dev)
    _lib.check(lib.gic_sample_captions_constrained(mode, _lib.ptr(features), _lib.ptr(W_emb), _lib.ptr_array(W_ih),
                                                   _lib.ptr_array(W_hh), _lib.ptr_array(b_ih), _lib.ptr_array(b_hh),
                                                   _lib.ptr(W_out), _lib.ptr(b_out), B, n, L, V, E, H, layers, int(eos_id),
                                                   float(temperature), int(top_k), float(top_p), cp, _lib.ptr(ids),
                                                   _lib.ptr(logp), _lib.ptr(lengths), _lib.ptr(ws), _lib.stream()),
               "gic_sample_captions_constrained")
    return ids, logp, lengths


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
                                   gic_b200.get_gemm_mode(), self.embed.weight, self.linear.weight, self.linear.bias,
                                   *self.lstm_params())

    @torch.no_grad()
    def beam_search(self, features, beam_size=3, max_caption_len=34, length_penalty=0.0, eos_id=2, min_length=0,
                    no_repeat_ngram_size=0, bad_ids=None):
        """The most likely captions of features[B,E] (the step-0 input, as in sample) by beam search (EXTENSION; the
        reference has none, oracle/ref_beam.py defines it) -> (ids[B,K,L], scores[B,K], lengths[B,K]), the K beams of each
        image best first by score / length ** length_penalty.  ids hold PAD (0) after <E> (eos_id); scores are sums of
        log-probabilities; lengths count tokens up to and including <E>.  beam_size = 1 is greedy decoding.

        Optional constraints (oracle/ref_constrain.py banned_tokens), none by default: ``min_length`` bans <E> until the
        caption has that many tokens; ``no_repeat_ngram_size`` = n bans every token that would repeat an n-gram of the
        caption; ``bad_ids`` (a host sequence of ids) are never emitted -- ``bad_ids=(0, 1, 3)`` keeps PAD, <S> and <UNK>
        out of captions.  Scores stay log-probabilities of the unconstrained model.  Raises ValueError on an invalid
        constraint before any GPU work."""
        if self.attention:
            raise NotImplementedError("beam search is implemented for the plain LSTM decoder, not the attention cell")
        check_constraints(min_length, no_repeat_ngram_size, bad_ids, max_caption_len, self.linear.out_features, beam_size)
        return decode_beam(self, features, beam_size, max_caption_len, length_penalty, eos_id, min_length=min_length,
                           no_repeat_ngram_size=no_repeat_ngram_size, bad_ids=bad_ids)

    @torch.no_grad()
    def score(self, features, captions, lengths=None):
        """Teacher-forced log-likelihood of given captions (EXTENSION; oracle/ref_score.py teacher_forced_logp defines it)
        -> (logp[B,L], caption_logp[B], correct[B,L] bool).  Step 0's input is features[B,E], as in sample; position t
        predicts captions[:, t], which is fed to step t + 1.  logp[b, t] = log_softmax(h W_out^T + b_out)[captions[b, t]]
        for t < lengths[b] (clamped to [0, L]; None: all L positions) and 0 after; caption_logp[b] is their sum; correct
        marks the positions whose target is the argmax (ties -> lower token, as sample(pretrain=True) picks).  Raises
        ValueError when an id lies outside [0, V); that check is one host read."""
        if self.attention:
            raise NotImplementedError("caption scoring is implemented for the plain LSTM decoder, not the attention cell")
        V = self.linear.out_features
        if captions.numel() and bool(((captions < 0) | (captions >= V)).any()):
            raise ValueError("caption ids must lie in [0, %d)" % V)
        logp, total, corr = score_captions(self, features, captions, lengths)
        return logp, total, corr.bool()

    @torch.no_grad()
    def sample_captions(self, features, num_samples=1, max_caption_len=34, temperature=1.0, top_k=0, top_p=1.0, eos_id=2,
                        min_length=0, no_repeat_ngram_size=0, bad_ids=None):
        """Draw num_samples captions per row of features[B,E] (EXTENSION; oracle/ref_sample.py sample_captions defines it)
        -> (ids[B,n,L], caption_logp[B,n], lengths[B,n]).  Each step draws from softmax(logits / temperature) restricted
        to the top_k tokens (0: the whole vocabulary), then to the smallest prefix of them holding top_p of the mass
        (top_p < 1 needs top_k >= 1).  ``temperature`` divides the logits; it is not ``Decoder.temperature``, which scales
        the Gumbel-softmax output of ``sample``.  A caption stops at <E> (eos_id): PAD (0) follows, lengths count tokens up
        to and including <E>, and caption_logp is the caption's log-likelihood under the unfiltered model at temperature 1.
        Draws come from the library's Philox stream (gic_set_rng); GANInstructor.sample_captions seeds it.  The optional
        constraints ``min_length``, ``no_repeat_ngram_size`` and ``bad_ids`` are those of beam_search (e.g.
        ``bad_ids=(0, 1, 3)`` for PAD, <S> and <UNK>): banned tokens leave the candidate set before top_k / top_p are
        applied.  Raises ValueError on an invalid argument before any GPU work."""
        if self.attention:
            raise NotImplementedError("caption sampling is implemented for the plain LSTM decoder, not the attention cell")
        V = self.linear.out_features
        check_sample_args(num_samples, max_caption_len, temperature, top_k, top_p, eos_id, V)
        check_constraints(min_length, no_repeat_ngram_size, bad_ids, max_caption_len, V, top_k)
        return sample_captions(self, features, num_samples, max_caption_len, temperature, top_k, top_p, eos_id,
                               min_length=min_length, no_repeat_ngram_size=no_repeat_ngram_size, bad_ids=bad_ids)

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
