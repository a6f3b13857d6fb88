"""Adversarial training driver with the reference's ``GANInstructor`` surface (src/training.py:15-235)
for the hot path: ``adv_loop`` body (:136-183), ``optimize`` (:194-199), ``update_temperature`` (:190-191).

``adv_step`` is the fused B200 path: it calls the C ABI directly (no autograd graph), shares the
discriminator trunk between ``disc(fake)`` and ``disc(gen_captions)`` (same values, different dropout
masks, src/training.py:163-164), never materialises ``F.one_hot(real)`` (:158), writes gradients
straight into flat buffers, and finishes with fused clip + Adam.  Ordering follows the Q1 fix
(SURVEY.md section 0.1): both gradients are taken on the pre-update weights, then D and G step.

Data parallel: one process per GPU, each rank owns B/world rows; the only exchange is an all-reduce
(sum) of the flat G and D gradient buffers before the clip (SURVEY.md section 8e)."""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.nn as nn

import gic_b200
from . import _lib, parallel
from .discriminator import Discriminator, disc_fwd_raw
from .generator import Generator, bn_running_update, encoder_eval
from .utils import get_fixed_temperature, get_losses


def _in_ctx(fn):
    """Runs a GANInstructor method with the instructor's library context current (include/gic_b200.h "contexts"): the
    temperature pointer, prepared discriminator weights, Philox state and event hooks it installs are its own."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        with self._ctx:
            return fn(self, *args, **kwargs)
    return wrapped


class FlatParams:
    """Re-homes a list of parameters into one contiguous fp32 buffer (params become views), with matching
    flat grad / Adam-moment buffers.  state_dict keys and nn.Parameter identities are unchanged."""

    def __init__(self, params, device, grad_alloc=None):
        self.params = [p for p in params]
        self.sizes = [p.numel() for p in self.params]
        self.offsets = []
        off = 0
        for n in self.sizes:
            self.offsets.append(off)
            off += (n + 3) & ~3          # keep every tensor 16-byte aligned inside the flat buffer
        self.n = off
        self.flat = torch.zeros(self.n, device=device)
        # data parallel: the gradient buffer lives in the peer communicator's symmetric allocation (gic_allreduce reduces it
        # in place over NVLink peer memory); otherwise a plain tensor
        self.grad = grad_alloc(self.n) if grad_alloc is not None else torch.zeros(self.n, device=device)
        self.m = torch.zeros(self.n, device=device)
        self.v = torch.zeros(self.n, device=device)
        self.step = 0
        for p, o, n in zip(self.params, self.offsets, self.sizes):
            view = self.flat[o:o + n].view(p.shape)
            view.copy_(p.data)
            p.data = view
        self._index = {id(p): i for i, p in enumerate(self.params)}

    def g(self, p):
        i = self._index[id(p)]
        return self.grad[self.offsets[i]:self.offsets[i] + self.sizes[i]].view(p.shape)

    def homed(self):
        return all(p.data_ptr() == self.flat.data_ptr() + 4 * o for p, o in zip(self.params, self.offsets))


class GANInstructor:
    def __init__(self, args, train_dataset=None, dev_dataset=None, device=None):
        _lib.lib()        # fail loudly at construction if the CUDA library is missing
        self._ctx = _lib.Context()
        self.args = args
        self.device = torch.device(device if device is not None else args.device)
        self.gen = Generator(args).to(self.device)
        self.disc = Discriminator(args).to(self.device)
        self.train_dataset, self.dev_dataset = train_dataset, dev_dataset
        self.cgan = (args.conditional_gan == 1)
        self.adv_epoch = -1
        self.pretrain_steps = self.gen_steps = self.disc_steps = 0
        self._flat_g: Optional[FlatParams] = None
        self._flat_d: Optional[FlatParams] = None
        self._cache = {}
        self._retired = []
        self._graphs = {}
        self._dyn = None          # device scalars of the captured step: [T, D lr/bc1, D 1/sqrt(bc2), G lr/bc1, G 1/sqrt(bc2)]
        self._dyn_host = None
        self._in_graph = False
        self._side = None
        self._comm = None
        self.timeline = None         # list of (name, timing event) when a profiling script asks for markers
        # Philox key of the library-side draws (u / dropout masks not supplied by the caller): torch's seed at construction
        self._rng_seed = int(torch.initial_seed()) & ((1 << 63) - 1)
        self._rng_offset = 0
        self._rng_dyn = None
        self._vocab_ev = None
        self._embed_ev = None
        self.bucketed = os.environ.get("GIC_NO_BUCKET", "0") != "1"
        # data parallel: Encoder.bn over the GLOBAL batch (two [2, E] all-reduces per step) instead of per shard;
        # opt-in (args.sync_bn / GIC_SYNC_BN=1): the reference is single-GPU, per-shard statistics are the documented default
        self.sync_bn = bool(getattr(args, "sync_bn", 0)) or os.environ.get("GIC_SYNC_BN", "0") == "1"
        self.overlap = os.environ.get("GIC_NO_OVERLAP", "0") != "1"
        self.d_priority = os.environ.get("GIC_D_PRIORITY", "0") == "1"
        self._hp = None
        self.world, self.rank = 1, 0
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            self.world = torch.distributed.get_world_size()
            self.rank = torch.distributed.get_rank()
        self._peer = None            # parallel.PeerComm: symmetric gradient buffers + one-kernel all-reduce over peer memory
        self._peer_failed = False
        self.skip_allreduce = False  # measurement only (bench.py comm_ms_exposed): run the step without the gradient exchange
        self._passthrough = {}       # encoder.resnet.* tensors of a reference-written checkpoint (re-emitted on save)

    # ---- library-side random draws: one Philox stream per (seed, rank, step) -------------------------------------
    RANK_SHIFT = 40

    def _next_rng_offset(self):
        """Philox offset of the next step's library-side draws.  The rank sits in the high bits (it reaches the counter
        word that also carries the stream tag, philox.cuh): data-parallel ranks seeded identically -- main.py seeds 1008
        everywhere so that the weights agree -- still draw DIFFERENT Gumbel noise and dropout masks for their rows."""
        if self._rng_seed is None:
            self._rng_seed = int(torch.initial_seed()) & ((1 << 63) - 1)
        self._rng_offset += 1
        assert self._rng_offset < (1 << self.RANK_SHIFT)
        return (int(self.rank) << self.RANK_SHIFT) | self._rng_offset

    # ---- reference-compatible pieces -------------------------------------------------------------
    def update_temperature(self, i, N):
        self.gen.decoder.temperature = get_fixed_temperature(self.args.temperature, i, N, self.args.temp_adpt)

    def optimize(self, opt, loss, model=None, retain_graph=False):
        """Autograd-driven variant kept for drop-in use with torch optimizers (src/training.py:194-199)."""
        opt.zero_grad()
        loss.backward(retain_graph=retain_graph)
        if model is not None:
            torch.nn.utils.clip_grad_norm_(model.parameters(), self.args.clip_norm)
        opt.step()

    def _mark(self, name):
        """Timeline marker (profiles/step_timeline.py): a timing event on the current stream, also inside graph capture."""
        if self.timeline is None:
            return
        # external=True: captured as an event-record NODE, so the event can be timed after every replay
        ev = torch.cuda.Event(enable_timing=True, external=True)
        ev.record(torch.cuda.current_stream())
        self.timeline.append((name, ev))

    def _side_stream(self):
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        return self._side

    def _comm_stream(self):
        if self._comm is None:
            self._comm = torch.cuda.Stream(device=self.device)
        return self._comm

    def _gen_backward_early_bucket(self, run_backward):
        """Data parallel, phase 1: generator backward with the C library's hook event registered; the
        [linear.weight | linear.bias] bucket (final before the BPTT tail) is all-reduced on a third stream as soon as
        the event fires.  Returns True when phase 2 (_gen_allreduce_rest) must follow."""
        fg = self._flat_g
        if self.world <= 1 or not self.bucketed or fg.n_early <= 0 or fg.n_early >= fg.n:
            run_backward()
            return False
        lib = _lib.lib()
        cur = torch.cuda.current_stream()
        if self._vocab_ev is None:
            self._vocab_ev, self._embed_ev = torch.cuda.Event(), torch.cuda.Event()
            self._vocab_ev.record(cur)                  # materialises the cudaEvent_t handles
            self._embed_ev.record(cur)
        ev, ev2 = self._vocab_ev, self._embed_ev
        two = fg.n_early < fg.n_mid < fg.n              # second bucket: embed.weight, final before the weight-gradient GEMMs
        lib.gic_set_vocab_grads_event(ev.cuda_event)
        if two:
            lib.gic_set_embed_grads_event(ev2.cuda_event)
        try:
            run_backward()
        finally:
            lib.gic_set_vocab_grads_event(None)
            lib.gic_set_embed_grads_event(None)
        comm = self._comm_stream()
        comm.wait_event(ev)
        with torch.cuda.stream(comm):
            self._mark("comm: early bucket (linear.weight) ready")
            self._allreduce(fg.grad[:fg.n_early], 1, self._sq_g[0:1])
            self._mark("comm: early bucket all-reduced")
            if two:
                comm.wait_event(ev2)
                self._mark("comm: embed bucket ready")
                self._allreduce(fg.grad[fg.n_early:fg.n_mid], 3, self._sq_g[1:2])
                self._mark("comm: embed bucket all-reduced")
        return 2 if two else 1

    def _gen_allreduce_rest(self, bucketed):
        """Phase 2 (issued after the discriminator's all-reduce so that NCCL's queue order is early bucket, D, rest)."""
        fg = self._flat_g
        if self.world <= 1:
            return
        if bucketed:
            lo = fg.n_mid if bucketed == 2 else fg.n_early
            self._allreduce(fg.grad[lo:], 2, self._sq_g[2:3])
            torch.cuda.current_stream().wait_stream(self._comm_stream())
        else:
            self._allreduce(fg.grad, 2, self._sq_g[2:3])

    # ---- gradient exchange -------------------------------------------------------------------------------------------
    def _allreduce(self, t, channel, sq=None):
        """Sum of a flat gradient slice over the ranks, in place, on the current stream.  Peer transport: ONE kernel that
        also adds the square norm of the reduced slice to `sq` (a device scalar; returns True then).  NCCL fallback:
        torch.distributed, the norm is left to gic_grad_sqnorm (returns False)."""
        if self.world <= 1 or self.skip_allreduce:
            return False
        if self._peer is not None and self._peer.owns(t):
            self._peer.allreduce_(t, channel, sq)
            return sq is not None
        parallel.allreduce_sum_(t)
        return False

    def _peer_alloc(self, n_total_floats):
        """Creates the peer communicator on first use (data parallel only); None -> plain gradient tensors + NCCL."""
        if self.world <= 1 or self._peer_failed or not parallel.peer_transport_enabled() or self.device.type != "cuda":
            return None
        if self._peer is None:
            try:
                self._peer = parallel.PeerComm(int(n_total_floats) * 4 + 4096, self.device)
            except Exception as exc:             # peers cannot be mapped (no IPC / no P2P): documented fallback
                self._peer_failed = True
                import warnings
                warnings.warn("gic_b200: peer-memory all-reduce unavailable (%s); using torch.distributed" % (exc,))
                return None
        return self._peer.alloc

    # ---- Encoder.linear + Encoder.bn (src/generator.py:15-16,23-24), per-shard or synchronised statistics ------------
    def _sync_bn_on(self):
        return self.sync_bn and self.world > 1

    def _encoder_fwd(self, mode, pooled, B, Fin, E, lin, mean, rstd, feats, stream):
        lib, P, enc = _lib.lib(), _lib.ptr, self.gen.encoder
        if not enc.training:
            # gen.eval() (the reference's validation loops, src/training.py:213-215): running statistics, row-local
            _lib.check(lib.gic_encoder_fwd_eval(mode, P(pooled), B, Fin, E, P(enc.linear.weight), P(enc.linear.bias),
                                                P(enc.bn.weight), P(enc.bn.bias), enc.bn.eps, P(enc.bn.running_mean),
                                                P(enc.bn.running_var), P(lin), P(feats), stream), "gic_encoder_fwd_eval")
            return
        if not self._sync_bn_on():
            _lib.check(lib.gic_encoder_fwd(mode, P(pooled), B, Fin, E, P(enc.linear.weight), P(enc.linear.bias),
                                           P(enc.bn.weight), P(enc.bn.bias), enc.bn.eps, P(lin), P(mean), P(rstd),
                                           P(feats), stream), "gic_encoder_fwd")
            bn_running_update(enc.bn, mean, rstd, enc.bn.eps, B)
            return
        # SyncBN: local sums -> all-reduce of [2, E] -> normalise with the global-batch statistics (SURVEY.md 8e)
        stats = self._buf("enc_stats", 2 * E)
        _lib.check(lib.gic_encoder_fwd_stats(mode, P(pooled), B, Fin, E, P(enc.linear.weight), P(enc.linear.bias), P(lin),
                                             P(stats), stream), "gic_encoder_fwd_stats")
        parallel.allreduce_sum_(stats)
        _lib.check(lib.gic_encoder_fwd_apply(P(lin), B, E, P(enc.bn.weight), P(enc.bn.bias), enc.bn.eps, P(stats),
                                             float(B * self.world), P(mean), P(rstd), P(feats), stream), "gic_encoder_fwd_apply")
        bn_running_update(enc.bn, mean, rstd, enc.bn.eps, B * self.world)

    def _encoder_bwd(self, mode, dfeat, pooled, lin, mean, rstd, B, E, stream):
        lib, P, enc = _lib.lib(), _lib.ptr, self.gen.encoder
        if not enc.training:
            raise NotImplementedError("training step with the encoder in eval mode: call gen.train() (the reference trains "
                                      "with gen.train(), src/training.py:215)")
        gg = self._flat_g.g
        dlin = self._buf("enc_dlin", B * E)
        if not self._sync_bn_on():
            _lib.check(lib.gic_encoder_bwd(mode, P(dfeat), P(pooled), P(lin), P(mean), P(rstd), P(enc.linear.weight),
                                           P(enc.bn.weight), B, pooled.shape[1], E, P(dlin), P(gg(enc.linear.weight)),
                                           P(gg(enc.linear.bias)), P(gg(enc.bn.weight)), P(gg(enc.bn.bias)), 0, stream),
                       "gic_encoder_bwd")
            return
        stats = self._buf("enc_bstats", 2 * E)
        _lib.check(lib.gic_encoder_bwd_stats(P(dfeat), P(lin), P(mean), P(rstd), B, E, P(stats), stream), "gic_encoder_bwd_stats")
        parallel.allreduce_sum_(stats)
        _lib.check(lib.gic_encoder_bwd_apply(mode, P(dfeat), P(pooled), P(lin), P(mean), P(rstd), P(enc.bn.weight), B,
                                             pooled.shape[1], E, P(stats), float(B * self.world), 1.0 / self.world, P(dlin),
                                             P(gg(enc.linear.weight)), P(gg(enc.linear.bias)), P(gg(enc.bn.weight)),
                                             P(gg(enc.bn.bias)), stream), "gic_encoder_bwd_apply")

    # ---- flat buffers ---------------------------------------------------------------------------
    def _gen_params(self):
        dec = self.gen.decoder
        # the vocab projection comes first: its gradients are final before the BPTT tail, so data-parallel runs all-reduce
        # that contiguous bucket early (n_early) underneath the rest of the backward
        ps = [dec.linear.weight, dec.linear.bias, dec.embed.weight, *dec.lstm_params()]
        if dec.attention:
            ps += dec.attn_params()
        if self.cgan:
            enc = self.gen.encoder
            ps += [enc.linear.weight, enc.linear.bias, enc.bn.weight, enc.bn.bias]
        return ps

    def _disc_params(self):
        d = self.disc
        ps = [d.embeddings.weight]
        for c in d.convs:
            ps += [c.weight, c.bias]
        ps += [d.highway.weight, d.highway.bias, d.feature2out.weight, d.feature2out.bias, d.out2logits.weight,
               d.out2logits.bias]
        return ps

    def _rehome(self, old, params, grad_alloc=None):
        """(Re)builds the flat buffers.  When a parameter was moved out of them (gen.to(), .float(),
        load_state_dict(assign=True)) the Adam moments and step counts of every parameter that kept its shape carry
        over, and the captured graphs -- which address the OLD buffers -- are dropped."""
        try:
            new = FlatParams(params, self.device, grad_alloc)
        except MemoryError:                      # the symmetric buffer was sized for the first layout: plain tensor + NCCL
            new = FlatParams(params, self.device)
        if old is not None:
            new.step = old.step
            if hasattr(old, "m_pre"):
                new.m_pre, new.v_pre, new.step_pre = torch.zeros_like(new.m), torch.zeros_like(new.v), old.step_pre
            old_at = {id(p): (o, n) for p, o, n in zip(old.params, old.offsets, old.sizes)}
            for p, o, n in zip(new.params, new.offsets, new.sizes):
                if old_at.get(id(p), (0, -1))[1] == n:
                    oo = old_at[id(p)][0]
                    new.m[o:o + n].copy_(old.m[oo:oo + n]); new.v[o:o + n].copy_(old.v[oo:oo + n])
                    if hasattr(old, "m_pre"):
                        new.m_pre[o:o + n].copy_(old.m_pre[oo:oo + n]); new.v_pre[o:o + n].copy_(old.v_pre[oo:oo + n])
            self._graphs.clear()
        return new

    def _ensure_flat(self):
        need_g = self._flat_g is None or not self._flat_g.homed()
        need_d = self._flat_d is None or not self._flat_d.homed()
        if not (need_g or need_d):
            return
        gp, dp = self._gen_params(), self._disc_params()
        total = sum((p.numel() + 3) & ~3 for p in gp) + sum((p.numel() + 3) & ~3 for p in dp) + 256
        alloc = self._peer_alloc(total)
        if need_g:
            self._flat_g = self._rehome(self._flat_g, gp, alloc)
            self._flat_g.n_early = self._flat_g.offsets[2]          # [linear.weight | linear.bias]
            self._flat_g.n_mid = self._flat_g.offsets[3]            # ... | embed.weight]
        if need_d:
            self._flat_d = self._rehome(self._flat_d, dp, alloc)

    def _zero_unwritten_attn_grads(self):
        """A step that does not run the attention cell (no grid; the policy-gradient step) writes no attn_* gradients:
        clear those slots so that Adam does not re-apply the gradients of an earlier attention step."""
        dec = self.gen.decoder
        if dec.attention:
            for p_ in dec.attn_params():
                self._flat_g.g(p_).zero_()

    def _buf(self, key, numel, dtype=torch.float32):
        t = self._cache.get(key)
        if t is None or t.numel() < numel or t.dtype != dtype:
            if t is not None and self._graphs:
                self._retired.append(t)      # a captured graph may still replay on the old buffer: keep it alive
            t = torch.empty(int(numel), dtype=dtype, device=self.device)
            self._cache[key] = t
        return t[:int(numel)]            # a smaller batch after a larger one reuses the front of the cached buffer

    # ---- the fused adversarial step ---------------------------------------------------------------
    @_in_ctx
    @torch.no_grad()
    def adv_step(self, captions, pooled=None, u=None, keep=None, train=True, forced_ids=None, loss_type=None,
                 update=True, graph=False, grid=None):
        """One adversarial step on a batch (src/training.py:136-169).

        captions [B,L] int64 (collate contract); pooled [B,feature_dim] CNN features when conditional;
        u [L,B,V] uniforms and keep [3,B*R,F] dropout keep-masks are drawn on-device when omitted.
        Returns a dict with g_loss/d_loss (device scalars), ids, probs and the D logits.

        graph=True replays the whole step as one CUDA graph (captured on first use per batch shape): inputs are
        copied into static buffers, the temperature and Adam's bias corrections are read from device memory
        (gic_set_temperature_device / gic_clip_adam_dyn), so one replay call enqueues all ~150 kernels.  The tensors
        in the dict a replay returns (losses, probs, ids, D logits) are the graph's STATIC buffers: the next replay
        overwrites them -- clone what must outlive the step."""
        if graph:
            if grid is not None and graph != "static":
                raise NotImplementedError("graph replay with the attention grid: pass graph='static' (resident inputs) or graph=False")
            return self._adv_step_graph(captions, pooled, u, keep, loss_type, static=(graph == "static"), grid=grid)
        _lib.require_cuda()
        lib = _lib.lib()
        a, dev = self.args, self.device
        mode = gic_b200.get_gemm_mode()
        loss_type = loss_type or a.adv_loss_type
        if loss_type not in _lib.LOSS_TYPES:
            raise NotImplementedError("Divergence '%s' is not implemented" % loss_type)
        self._ensure_flat()
        fg, fd = self._flat_g, self._flat_d
        dec, disc = self.gen.decoder, self.disc
        captions = captions.to(dev).long().contiguous()
        B, L = captions.shape
        V, E, H, layers = a.vocab_size, a.gen_embed_dim, a.gen_hidden_dim, a.gen_num_layers
        De, R, Fd = a.disc_embed_dim, a.disc_num_rep, sum(a.disc_num_filters)
        fsz, nfl = list(a.disc_filter_sizes), list(a.disc_num_filters)
        T = float(dec.temperature)
        stream = _lib.stream()
        P = _lib.ptr
        if self._in_graph:
            lib.gic_set_temperature_device(P(self._dyn[0:1]))
        # derived D weights (collapsed head, bf16 highway.weight) once per step: all six D calls below see the same
        # pre-update weights (Q1)
        prep = self._buf("disc_prep", lib.gic_disc_prepared_floats(Fd))
        _lib.check(lib.gic_disc_prepare(mode, P(disc.highway.weight), P(disc.feature2out.weight), P(disc.feature2out.bias),
                                        disc.feature2out.weight.shape[0], P(disc.out2logits.weight),
                                        P(disc.out2logits.bias), Fd, P(prep), stream), "gic_disc_prepare")
        lib.gic_disc_set_prepared(P(prep))
        try:
            return self._adv_step_body(captions, pooled, u, keep, train, forced_ids, loss_type, update, grid, prep)
        finally:
            lib.gic_disc_set_prepared(None)
            lib.gic_set_rng(0, 0, None)
            if self._in_graph:
                lib.gic_set_temperature_device(None)

    def _adv_step_body(self, captions, pooled, u, keep, train, forced_ids, loss_type, update, grid, prep):
        lib = _lib.lib()
        a, dev = self.args, self.device
        mode = gic_b200.get_gemm_mode()
        fg, fd = self._flat_g, self._flat_d
        dec, disc = self.gen.decoder, self.disc
        B, L = captions.shape
        V, E, H, layers = a.vocab_size, a.gen_embed_dim, a.gen_hidden_dim, a.gen_num_layers
        De, R, Fd = a.disc_embed_dim, a.disc_num_rep, sum(a.disc_num_filters)
        fsz, nfl = list(a.disc_filter_sizes), list(a.disc_num_filters)
        T = float(dec.temperature)
        stream = _lib.stream()
        P = _lib.ptr
        # -- discriminator on the real captions (hard tokens, :158,162): independent of the decode, so it runs on a
        #    side stream underneath the latency-bound autoregressive loop
        if u is None or (train and keep is None):
            # draws not supplied: Philox inside the library (the Gumbel uniforms are generated in the fused decode kernel
            # itself; the reference draws with uniform_ / nn.Dropout, src/generator.py:86-90, src/discriminator.py:30)
            if self._in_graph:
                lib.gic_set_rng(0, 0, P(self._rng_dyn))
            else:
                off = self._next_rng_offset()
                lib.gic_set_rng(self._rng_seed, off, None)
        if train:
            if keep is None:
                keep = self._buf("keep_u8", 3 * B * R * Fd, dtype=torch.uint8).view(3, B * R, Fd)
                _lib.check(lib.gic_philox_keep_mask(_lib.RNG_TAG_DROPOUT, keep.numel(), float(disc.dropout.p), P(keep),
                                                    stream), "gic_philox_keep_mask")
            keep = keep.to(dev).to(torch.uint8).contiguous()
            k0, k1, k2 = keep[0], keep[1], keep[2]
        else:
            k0 = k1 = k2 = None
        cw = [c.weight for c in disc.convs]
        cb = [c.bias for c in disc.convs]
        dW = (disc.embeddings.weight, cw, cb, disc.highway.weight, disc.highway.bias, disc.feature2out.weight,
              disc.feature2out.bias, disc.out2logits.weight, disc.out2logits.bias)
        drop_p = disc.dropout.p
        main = torch.cuda.current_stream()
        side = self._side_stream() if (train and self.overlap) else None
        self._mark("start (masks drawn)")
        # -- backward helper: D parameter gradients from (real, fake); generator gradients through D(gen) (:168-169, Q1)
        bws = self._buf("disc_bws", lib.gic_disc_bwd_workspace_floats(B, L, De, R, Fd))
        g = fd.g
        dcw, dcb = [g(c.weight) for c in disc.convs], [g(c.bias) for c in disc.convs]

        def disc_bwd(seed, kp, inp, idz, saved, want_param, acc, dinp, bws, stream):
            _lib.check(lib.gic_disc_bwd(mode, P(seed), P(kp), drop_p, P(inp), P(idz), B, L, V, De, R, len(fsz),
                                        _lib.int_array(fsz), _lib.int_array(nfl), P(disc.embeddings.weight),
                                        _lib.ptr_array(cw), _lib.ptr_array(cb), P(disc.highway.weight),
                                        P(disc.feature2out.weight), P(disc.feature2out.bias),
                                        disc.feature2out.weight.shape[0], P(disc.out2logits.weight),
                                        P(disc.out2logits.bias), P(saved), P(bws), P(g(disc.embeddings.weight)),
                                        _lib.ptr_array(dcw), _lib.ptr_array(dcb), P(g(disc.highway.weight)),
                                        P(g(disc.highway.bias)), P(g(disc.feature2out.weight)),
                                        P(g(disc.feature2out.bias)), P(g(disc.out2logits.weight)),
                                        P(g(disc.out2logits.bias)), P(dinp), want_param, acc, stream), "gic_disc_bwd")

        # The seed of d_loss w.r.t. D(real) does not depend on D(fake) (every divergence except rsgan), and neither does
        # anything else in backward(real), so it CAN run on the side stream right behind forward(real), underneath the
        # decode loop.  Measured (profiles/step_timeline.py): the decode kernels need nearly every SM (126-128 CTAs of
        # ~200 KB shared memory), so whatever runs beside them stalls them almost one for one: decode 989 -> 1232 us, the
        # phase after the losses 1346 -> 1150 us, step 2.62 -> 2.67 ms.  Opt-in only (GIC_EARLY_REAL=1).
        early_real = train and self.overlap and loss_type != "rsgan" and os.environ.get("GIC_EARLY_REAL", "0") == "1"
        real_bwd_done = None
        if side is not None:
            side.wait_stream(main)
            with torch.cuda.stream(side):
                (d_real,), saved_r = disc_fwd_raw(lib, mode, None, captions, B, L, V, De, R, fsz, nfl, *dW, [k0], drop_p,
                                                  dev)
                self._mark("side: D(real) forward done")
                if early_real:
                    nR = B * R
                    seed_real = self._buf("seed_real", nR)
                    _lib.check(lib.gic_gan_loss_fwd_bwd(_lib.LOSS_TYPES[loss_type], P(d_real), P(d_real), P(d_real), nR,
                                                        P(self._buf("loss_scratch", 2)), P(seed_real), None, None,
                                                        side.cuda_stream), "gic_gan_loss_fwd_bwd")
                    disc_bwd(seed_real, k0, None, captions, saved_r, 1, 0, None, bws, side.cuda_stream)
                    real_bwd_done = torch.cuda.Event()
                    real_bwd_done.record(side)
                    self._mark("side: D backward(real) done")
        else:
            (d_real,), saved_r = disc_fwd_raw(lib, mode, None, captions, B, L, V, De, R, fsz, nfl, *dW, [k0], drop_p, dev)
        # -- step-0 input (:144-147)
        attn = grid is not None
        if attn:
            import ctypes as C
            if not dec.attention or layers != 1:
                raise ValueError("grid given: build the generator with gen_attention=1 and one LSTM layer")
            grid = grid.to(dev).float().contiguous()
            if pooled is None and self.cgan:
                pooled = grid.mean(1)                       # the reference's pooled feature = mean over the locations
            Pn, Da = grid.shape[1], a.attn_dim
            asaved = self._buf("attn_saved", lib.gic_attn_saved_floats(B, L, Pn, Da, E))
            we = dec.attn_e.weight.view(-1)
        if self.cgan:
            enc = self.gen.encoder
            pooled = pooled.to(dev).float().contiguous()
            Fin = pooled.shape[1]
            lin, mean, rstd = self._buf("enc_lin", B * E).view(B, E), self._buf("enc_mean", E), self._buf("enc_rstd", E)
            feats = self._buf("feats", B * E).view(B, E)
            self._encoder_fwd(mode, pooled, B, Fin, E, lin, mean, rstd, feats, stream)
        else:
            feats = dec.embed.weight[1].expand(B, E).contiguous()
        # -- Decoder.sample (:150)
        if u is not None:
            u = u.to(dev).float().contiguous()
        probs = self._buf("probs", B * L * V).view(B, L, V)
        ids = torch.empty(B, L, dtype=torch.int64, device=dev)
        dsaved = self._buf("dec_saved", lib.gic_decode_saved_floats(B, L, E, H, layers))
        dws = self._buf("dec_ws", lib.gic_decode_fwd_workspace_floats(B, V, H))
        lp = dec.lstm_params()
        W_ih, W_hh, b_ih, b_hh = lp[0::4], lp[1::4], lp[2::4], lp[3::4]
        if forced_ids is not None:
            forced_ids = forced_ids.to(dev).long().contiguous()
        if attn:
            blk = _lib.attn_block(grid, dec.attn_k.weight, dec.attn_v.weight, dec.attn_q.weight, we, asaved)
            _lib.check(lib.gic_decode_sample_fwd_attn(C.byref(blk), mode, P(feats), P(dec.embed.weight),
                                                      _lib.ptr_array(W_ih), _lib.ptr_array(W_hh), _lib.ptr_array(b_ih),
                                                      _lib.ptr_array(b_hh), P(dec.linear.weight), P(dec.linear.bias),
                                                      P(u), T, 0, P(forced_ids), B, L, V, E, H, layers, P(probs), P(ids),
                                                      P(dsaved), P(dws), stream), "gic_decode_sample_fwd_attn")
        else:
            _lib.check(lib.gic_decode_sample_fwd(mode, P(feats), P(dec.embed.weight), _lib.ptr_array(W_ih),
                                                 _lib.ptr_array(W_hh), _lib.ptr_array(b_ih), _lib.ptr_array(b_hh),
                                                 P(dec.linear.weight), P(dec.linear.bias), P(u), T, 0, P(forced_ids), B,
                                                 L, V, E, H, layers, P(probs), P(ids), P(dsaved), P(dws), stream),
                       "gic_decode_sample_fwd")
        self._mark("main: decode done")
        # -- discriminator on the generated captions: fake / gen share one trunk, two dropout masks (:163-164)
        (d_fake, g_out), saved_f = disc_fwd_raw(lib, mode, probs, None, B, L, V, De, R, fsz, nfl, *dW, [k1, k2],
                                                drop_p, dev)
        self._mark("main: D(fake/gen) forward done")
        if side is not None:
            main.wait_stream(side)
        # -- losses + seeds (:165)
        n = B * R
        losses = torch.empty(2, device=dev)
        seeds = self._buf("seeds", 3 * n).view(3, n)
        _lib.check(lib.gic_gan_loss_fwd_bwd(_lib.LOSS_TYPES[loss_type], P(d_real), P(d_fake), P(g_out), n, P(losses),
                                            P(seeds[0]), P(seeds[1]), P(seeds[2]), stream), "gic_gan_loss_fwd_bwd")
        self._mark("main: losses done")
        out = dict(g_loss=losses[0], d_loss=losses[1], ids=ids, probs=probs, d_real=d_real, d_fake=d_fake,
                   g_out=g_out, features=feats)
        if not train:
            return out

        g_has_grad = loss_type != "rsgan"          # A14: rsgan's g_loss only sees detached D outputs

        def gen_chain(ws_d, st):
            # D's input gradient stays factored (demb x W_e): the dense d(probs)[B,L,V] is never written; the
            # decoder backward fuses demb W_e with the tempered-softmax backward (gic_decode_sample_bwd_factored)
            disc_bwd(seeds[2], k2, probs, None, saved_f, 0, 0, None, ws_d, st)
            self._mark("G chain: D input gradient (demb) done")
            off = lib.gic_disc_bwd_demb_offset_floats(B, L, De, R, Fd)
            demb = ws_d[off:off + B * L * De]
            emb = saved_f[:B * L * De]
            gg = fg.g
            gws = self._buf("dec_bws", lib.gic_decode_bwd_workspace_floats(B, L, V, E, H, layers))
            dfeat = self._buf("dfeat", B * E).view(B, E)
            fed = ids if forced_ids is None else forced_ids
            if attn:
                aws = self._buf("attn_ws", lib.gic_attn_bwd_workspace_floats(B, L, Pn, Da, E))
                blk = _lib.attn_block(grid, dec.attn_k.weight, dec.attn_v.weight, dec.attn_q.weight, we, asaved, aws,
                                      gg(dec.attn_k.weight), gg(dec.attn_v.weight), gg(dec.attn_q.weight),
                                      gg(dec.attn_e.weight).view(-1))
                _lib.check(lib.gic_decode_sample_bwd_attn(
                    C.byref(blk), mode, None, P(demb), P(emb), P(disc.embeddings.weight), De, P(probs), P(fed),
                    P(dec.embed.weight), _lib.ptr_array(W_ih), _lib.ptr_array(W_hh), P(dec.linear.weight), T, 0, B, L, V,
                    E, H, layers, P(dsaved), P(gws), P(gg(dec.embed.weight)), _lib.ptr_array([gg(w) for w in W_ih]),
                    _lib.ptr_array([gg(w) for w in W_hh]), _lib.ptr_array([gg(w) for w in b_ih]),
                    _lib.ptr_array([gg(w) for w in b_hh]), P(gg(dec.linear.weight)), P(gg(dec.linear.bias)), P(dfeat),
                    st), "gic_decode_sample_bwd_attn")
            else:
                self._zero_unwritten_attn_grads()
                _lib.check(lib.gic_decode_sample_bwd_factored(
                    mode, P(demb), P(emb), P(disc.embeddings.weight), De, P(probs), P(fed), P(dec.embed.weight),
                    _lib.ptr_array(W_ih), _lib.ptr_array(W_hh), P(dec.linear.weight), T, B, L, V, E, H, layers,
                    P(dsaved), P(gws), P(gg(dec.embed.weight)), _lib.ptr_array([gg(w) for w in W_ih]),
                    _lib.ptr_array([gg(w) for w in W_hh]), _lib.ptr_array([gg(w) for w in b_ih]),
                    _lib.ptr_array([gg(w) for w in b_hh]), P(gg(dec.linear.weight)), P(gg(dec.linear.bias)), P(dfeat), 0,
                    st), "gic_decode_sample_bwd_factored")
            self._mark("G chain: decoder backward done")
            if self.cgan:
                self._encoder_bwd(mode, dfeat, pooled, lin, mean, rstd, B, E, st)
            else:
                gg(dec.embed.weight)[1] += dfeat.sum(0)      # features = embed(<S>) for every row (:147)

        # Two independent chains after the loss: D parameter gradients (real, then fake accumulated) and the generator
        # chain (D input gradient -> decoder BPTT).  The generator chain is latency-bound (L serial BPTT steps), so it
        # runs on a side stream under the D chain.  Q1: both read the PRE-update weights, so D's Adam waits for the
        # generator chain's last read of D weights.
        # square norms of the reduced gradients (the peer all-reduce accumulates them); one slot per generator bucket: two
        # buckets may finish in either order, and a float sum must not depend on that (the replicas have to stay identical)
        self._sq_g = torch.zeros(4, device=dev)
        self._sq_d = torch.zeros(1, device=dev)
        if side is not None and g_has_grad:
            bws2 = self._buf("disc_bws2", lib.gic_disc_bwd_workspace_floats(B, L, De, R, Fd))
            side.wait_stream(main)
            with torch.cuda.stream(side):
                gen_done = torch.cuda.Event()

                def _bwd():
                    gen_chain(bws2, side.cuda_stream)
                    gen_done.record(side)
                g_bucketed = self._gen_backward_early_bucket(_bwd)
            # GIC_D_PRIORITY=1 (experiment): the D chain on a high-priority stream, so that it finishes ahead of the
            # generator chain and its gradient all-reduce runs under the generator chain's tail
            dst = main
            if self.d_priority:
                if self._hp is None:
                    self._hp = torch.cuda.Stream(device=self.device, priority=-1)
                dst = self._hp
                dst.wait_stream(main)
            with torch.cuda.stream(dst):
                ds = dst.cuda_stream
                if real_bwd_done is None:
                    disc_bwd(seeds[0], k0, None, captions, saved_r, 1, 0, None, bws, ds)
                    self._mark("D chain: backward(real) done")
                else:
                    dst.wait_event(real_bwd_done)         # fake accumulates onto real's parameter gradients
                disc_bwd(seeds[1], k1, probs, None, saved_f, 1, 1, None, bws, ds)
                self._mark("D chain: backward(fake) done")
                d_sq = self._allreduce(fd.grad, 0, self._sq_d)
                self._mark("D chain: gradients all-reduced")
            with torch.cuda.stream(side):
                self._mark("G chain: backward done")
                self._gen_allreduce_rest(g_bucketed)
                self._mark("G chain: gradients all-reduced")
                g_sq = self._peer is not None and self.world > 1 and not self.skip_allreduce and self._peer.owns(fg.grad)
                out["g_sqnorm"] = self._clip_adam(fg, a.gen_lr, update, 3, self._sq_g.sum().reshape(1) if g_sq else None)
                self._mark("G chain: clip + Adam done")
            with torch.cuda.stream(dst):
                dst.wait_event(gen_done)
                out["d_sqnorm"] = self._clip_adam(fd, a.disc_lr, update, 1, self._sq_d if d_sq else None)
                self._mark("D chain: clip + Adam done")
            if dst is not main:
                main.wait_stream(dst)
            main.wait_stream(side)
            self._mark("end")
        else:
            disc_bwd(seeds[0], k0, None, captions, saved_r, 1, 0, None, bws, stream)
            disc_bwd(seeds[1], k1, probs, None, saved_f, 1, 1, None, bws, stream)
            if g_has_grad:
                gen_chain(bws, stream)
            # -- data-parallel exchange: summed gradients, averaged inside the optimizer kernel
            d_sq = self._allreduce(fd.grad, 0, self._sq_d)
            g_sq = self._allreduce(fg.grad, 2, self._sq_g[2:3]) if g_has_grad else False
            out["d_sqnorm"] = self._clip_adam(fd, a.disc_lr, update, 1, self._sq_d if d_sq else None)
            if g_has_grad:
                out["g_sqnorm"] = self._clip_adam(fg, a.gen_lr, update, 3, self._sq_g.sum().reshape(1) if g_sq else None)
        out["g_has_grad"] = g_has_grad
        return out

    def _clip_adam(self, fp: FlatParams, lr: float, update: bool, dyn_slot: int = 1, sq=None):
        """sq: square norm of fp.grad already on the device (the peer all-reduce computes it in the same pass)."""
        lib = _lib.lib()
        stream = _lib.stream()
        if sq is None:
            sq = torch.zeros(1, device=self.device)
            _lib.check(lib.gic_grad_sqnorm(_lib.ptr(fp.grad), fp.n, _lib.ptr(sq), stream), "gic_grad_sqnorm")
        if update and self._in_graph:
            _lib.check(lib.gic_clip_adam_dyn(_lib.ptr(fp.flat), _lib.ptr(fp.grad), _lib.ptr(fp.m), _lib.ptr(fp.v), fp.n,
                                             _lib.ptr(sq), float(self.args.clip_norm), 1.0 / self.world,
                                             _lib.ptr(self._dyn[dyn_slot:dyn_slot + 2]), 0.9, 0.999, 1e-8, stream),
                       "gic_clip_adam_dyn")
        elif update:
            fp.step += 1
            _lib.check(lib.gic_clip_adam(_lib.ptr(fp.flat), _lib.ptr(fp.grad), _lib.ptr(fp.m), _lib.ptr(fp.v), fp.n,
                                         _lib.ptr(sq), float(self.args.clip_norm), 1.0 / self.world, fp.step,
                                         float(lr), 0.9, 0.999, 1e-8, stream), "gic_clip_adam")
        return sq

    # ---- CUDA-graph replay of the fused step -------------------------------------------------------
    def _adv_step_graph(self, captions, pooled, u, keep, loss_type, static=False, grid=None):
        """static=True: the given device tensors themselves are the graph's inputs (no copies; one graph per distinct
        set of buffers) -- for callers that keep their batches resident."""
        a, dev = self.args, self.device
        loss_type = loss_type or a.adv_loss_type
        B, L = captions.shape
        key = (B, L, loss_type, pooled is not None, u is not None, keep is not None, bool(self.gen.encoder.training),
               gic_b200.get_gemm_mode())
        if static:
            key = key + tuple(None if t is None else t.data_ptr() for t in (captions, pooled, u, keep, grid))
        st = self._graphs.get(key)
        if self._dyn is None:
            self._dyn = torch.zeros(8, device=dev)
            # ring of pinned staging slots: the host may run ahead of the GPU, so a slot is rewritten only after the
            # copy that read it has executed (event per slot)
            self._dyn_host = [torch.zeros(8).pin_memory() for _ in range(16)]
            self._dyn_ev = [None] * 16
            self._dyn_i = 0
            self._rng_dyn = torch.zeros(2, dtype=torch.int64, device=dev)
            self._rng_host = [torch.zeros(2, dtype=torch.int64).pin_memory() for _ in range(16)]
        if st is None and static:
            st = dict(captions=captions, pooled=pooled, u=u, keep=keep, grid=grid)
            self._graphs[key] = st
        if st is None:
            st = dict(captions=torch.empty(B, L, dtype=torch.int64, device=dev),
                      pooled=None if pooled is None else torch.empty(pooled.shape, device=dev),
                      u=None if u is None else torch.empty(u.shape, device=dev),
                      keep=None if keep is None else torch.empty(keep.shape, dtype=torch.uint8, device=dev))
            self._graphs[key] = st

        def load_inputs():
            if static:
                return
            st["captions"].copy_(captions, non_blocking=True)
            if pooled is not None:
                st["pooled"].copy_(pooled, non_blocking=True)
            if u is not None:
                st["u"].copy_(u, non_blocking=True)
            if keep is not None:
                st["keep"].copy_(keep, non_blocking=True)

        def load_scalars():
            self._ensure_flat()
            i = self._dyn_i = (self._dyn_i + 1) % 16
            if self._dyn_ev[i] is not None:
                self._dyn_ev[i].synchronize()
            h = self._dyn_host[i]
            h[0] = float(self.gen.decoder.temperature)
            for slot, fp, lr in ((1, self._flat_d, a.disc_lr), (3, self._flat_g, a.gen_lr)):
                t = fp.step + 1
                h[slot] = lr / (1.0 - 0.9 ** t)
                h[slot + 1] = 1.0 / (1.0 - 0.999 ** t) ** 0.5
            self._dyn.copy_(h, non_blocking=True)
            off = self._next_rng_offset()
            hr = self._rng_host[i]
            hr[0] = self._rng_seed
            hr[1] = off
            self._rng_dyn.copy_(hr, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            self._dyn_ev[i] = ev

        load_inputs()
        if "graph" not in st:
            # one eager step allocates every cached buffer and compiles nothing new during capture; it is a real
            # training step (same semantics), so the captured replay starts at step 2
            out = self.adv_step(st["captions"], pooled=st["pooled"], u=st["u"], keep=st["keep"], loss_type=loss_type,
                                grid=st.get("grid"))
            torch.cuda.synchronize(dev)
            load_scalars()
            g = torch.cuda.CUDAGraph()
            n0 = _lib.lib().gic_launch_count()
            self._in_graph = True
            try:
                with torch.cuda.graph(g):
                    st["out"] = self.adv_step(st["captions"], pooled=st["pooled"], u=st["u"], keep=st["keep"],
                                              loss_type=loss_type, grid=st.get("grid"))
            finally:
                self._in_graph = False
                _lib.lib().gic_set_temperature_device(None)
            st["graph"] = g
            st["g_has_grad"] = st["out"]["g_has_grad"]
            self.graph_launches_per_step = int(_lib.lib().gic_launch_count() - n0)   # kernels of ours in one replay
            return out          # the eager step's results (capture itself does not execute the kernels)
        load_scalars()
        st["graph"].replay()
        self._flat_d.step += 1
        if st["g_has_grad"]:
            self._flat_g.step += 1
        return st["out"]

    # ---- EXTENSION: caption generation by beam search (the reference has none) -------------------------------------
    @_in_ctx
    @torch.no_grad()
    def generate(self, pooled=None, batch_size=None, beam_size=3, max_caption_len=34, length_penalty=0.0):
        """Captions of a trained generator -> (ids[B,K,L], scores[B,K], lengths[B,K]) (Decoder.beam_search).  Conditional
        mode: the pooled CNN features [B, feature_dim] go through the encoder projection in eval mode (running statistics,
        as gen.eval() would); unconditional mode: every caption starts from embed.weight[1] (<S>), batch_size of them.
        Inference only: parameters, gradients, optimizer state, step counters, temperature and the library's random stream
        are left as they were."""
        _lib.require_cuda()
        dev = self.device
        dec = self.gen.decoder
        if self.cgan:
            if pooled is None:
                raise ValueError("conditional generation needs the pooled image features")
            feats = encoder_eval(self.gen.encoder, pooled.to(dev).float(), gic_b200.get_gemm_mode())
        else:
            if batch_size is None:
                if pooled is None:
                    raise ValueError("unconditional generation needs batch_size")
                batch_size = pooled.shape[0]
            feats = dec.embed.weight[1].expand(int(batch_size), dec.embed.weight.shape[1]).contiguous()
        return dec.beam_search(feats, beam_size=beam_size, max_caption_len=max_caption_len, length_penalty=length_penalty)

    # ---- generator pre-training step (src/training.py:53-95; SURVEY.md 8f rank 1) -------------------------------
    @_in_ctx
    @torch.no_grad()
    def pretrain_step(self, captions, pooled=None, update=True):
        """Free-running greedy decode (sample(pretrain=True), :71) -> CrossEntropyLoss over all positions incl. PAD
        (:81-83) -> optimize(pretrain_opt, loss, gen) (:86): clip 5.0 + Adam(lr = pretrain_lr) with its own moments."""
        _lib.require_cuda()
        lib = _lib.lib()
        a, dev = self.args, self.device
        mode = gic_b200.get_gemm_mode()
        self._ensure_flat()
        fg = self._flat_g
        dec = self.gen.decoder
        captions = captions.to(dev).long().contiguous()
        B, L = captions.shape
        V, E, H, layers = a.vocab_size, a.gen_embed_dim, a.gen_hidden_dim, a.gen_num_layers
        stream = _lib.stream()
        P = _lib.ptr
        if self.cgan:
            enc = self.gen.encoder
            pooled = pooled.to(dev).float().contiguous()
            Fin = pooled.shape[1]
            lin, mean, rstd = self._buf("enc_lin", B * E).view(B, E), self._buf("enc_mean", E), self._buf("enc_rstd", E)
            feats = self._buf("feats", B * E).view(B, E)
            self._encoder_fwd(mode, pooled, B, Fin, E, lin, mean, rstd, feats, stream)
        else:
            feats = dec.embed.weight[1].expand(B, E).contiguous()
        logits = self._buf("pg_logits", B * L * V).view(B, L, V)
        ids = torch.empty(B, L, dtype=torch.int64, device=dev)
        dsaved = self._buf("dec_saved", lib.gic_decode_saved_floats(B, L, E, H, layers))
        dws = self._buf("dec_ws", lib.gic_decode_fwd_workspace_floats(B, V, H))
        lp = dec.lstm_params()
        W_ih, W_hh, b_ih, b_hh = lp[0::4], lp[1::4], lp[2::4], lp[3::4]
        _lib.check(lib.gic_decode_sample_fwd(mode, P(feats), P(dec.embed.weight), _lib.ptr_array(W_ih),
                                             _lib.ptr_array(W_hh), _lib.ptr_array(b_ih), _lib.ptr_array(b_hh),
                                             P(dec.linear.weight), P(dec.linear.bias), None, 1.0, 1, None, B, L, V, E, H,
                                             layers, P(logits), P(ids), P(dsaved), P(dws), stream), "gic_decode_sample_fwd")
        loss = torch.empty(1, device=dev)
        dlogits = self._buf("pg_dlogits", B * L * V).view(B, L, V)
        _lib.check(lib.gic_ce_loss_fwd_bwd(P(logits), P(captions), B, L, V, P(loss), P(dlogits), stream), "gic_ce_loss_fwd_bwd")
        gg = fg.g
        fg.grad.zero_()
        gws = self._buf("dec_bws", lib.gic_decode_bwd_workspace_floats(B, L, V, E, H, layers))
        dfeat = self._buf("dfeat", B * E).view(B, E)
        _lib.check(lib.gic_decode_sample_bwd(
            mode, P(dlogits), None, P(ids), P(dec.embed.weight), _lib.ptr_array(W_ih), _lib.ptr_array(W_hh),
            P(dec.linear.weight), 1.0, 1, B, L, V, E, H, layers, P(dsaved), P(gws), P(gg(dec.embed.weight)),
            _lib.ptr_array([gg(w) for w in W_ih]), _lib.ptr_array([gg(w) for w in W_hh]),
            _lib.ptr_array([gg(w) for w in b_ih]), _lib.ptr_array([gg(w) for w in b_hh]), P(gg(dec.linear.weight)),
            P(gg(dec.linear.bias)), P(dfeat), 0, stream), "gic_decode_sample_bwd")
        if self.cgan:
            enc = self.gen.encoder
            _lib.check(lib.gic_encoder_bwd(mode, P(dfeat), P(pooled), P(lin), P(mean), P(rstd), P(enc.linear.weight),
                                           P(enc.bn.weight), B, pooled.shape[1], E, P(self._buf("enc_dlin", B * E)),
                                           P(gg(enc.linear.weight)), P(gg(enc.linear.bias)), P(gg(enc.bn.weight)),
                                           P(gg(enc.bn.bias)), 0, stream), "gic_encoder_bwd")
        else:
            gg(dec.embed.weight)[1] += dfeat.sum(0)
        self._allreduce(fg.grad, 2)
        # pretrain_opt is its own Adam instance in the reference (:24-26): separate moments and step count
        if not hasattr(fg, "m_pre"):
            fg.m_pre, fg.v_pre, fg.step_pre = torch.zeros_like(fg.m), torch.zeros_like(fg.v), 0
        sq = torch.zeros(1, device=dev)
        _lib.check(lib.gic_grad_sqnorm(P(fg.grad), fg.n, P(sq), stream), "gic_grad_sqnorm")
        if update:
            fg.step_pre += 1
            _lib.check(lib.gic_clip_adam(P(fg.flat), P(fg.grad), P(fg.m_pre), P(fg.v_pre), fg.n, P(sq),
                                         float(a.clip_norm), 1.0 / self.world, fg.step_pre, float(a.pretrain_lr), 0.9,
                                         0.999, 1e-8, stream), "gic_clip_adam")
        self.pretrain_steps += 1
        return dict(loss=loss[0], ids=ids, logits=logits, sqnorm=sq)

    # ---- discriminator step on hard captions (real vs generated ids): D pre-training sweep (BASELINE configs[4]) and
    #      the D half of the policy-gradient step.  F.one_hot is never materialised (column gather, src/training.py:158).
    @_in_ctx
    @torch.no_grad()
    def disc_step(self, real_ids, fake_ids, keep=None, update=True):
        _lib.require_cuda()
        lib = _lib.lib()
        a, dev = self.args, self.device
        mode = gic_b200.get_gemm_mode()
        self._ensure_flat()
        fd, disc = self._flat_d, self.disc
        real_ids = real_ids.to(dev).long().contiguous()
        fake_ids = fake_ids.to(dev).long().contiguous()
        B, L = real_ids.shape
        V, De, R, Fd = a.vocab_size, a.disc_embed_dim, a.disc_num_rep, sum(a.disc_num_filters)
        fsz, nfl = list(a.disc_filter_sizes), list(a.disc_num_filters)
        stream = _lib.stream()
        P = _lib.ptr
        cw = [c.weight for c in disc.convs]
        cb = [c.bias for c in disc.convs]
        dW = (disc.embeddings.weight, cw, cb, disc.highway.weight, disc.highway.bias, disc.feature2out.weight,
              disc.feature2out.bias, disc.out2logits.weight, disc.out2logits.bias)
        drop_p = disc.dropout.p
        if keep is None:
            keep = torch.rand(2, B * R, Fd, device=dev) >= drop_p
        keep = keep.to(dev).to(torch.uint8).contiguous()
        (d_real,), saved_r = disc_fwd_raw(lib, mode, None, real_ids, B, L, V, De, R, fsz, nfl, *dW, [keep[0]], drop_p, dev)
        (d_fake,), saved_f = disc_fwd_raw(lib, mode, None, fake_ids, B, L, V, De, R, fsz, nfl, *dW, [keep[1]], drop_p, dev)
        nn_ = B * R
        losses = torch.empty(2, device=dev)
        seeds = self._buf("seeds", 3 * nn_).view(3, nn_)
        _lib.check(lib.gic_gan_loss_fwd_bwd(_lib.LOSS_TYPES["standard"], P(d_real), P(d_fake), P(d_fake), nn_, P(losses),
                                            P(seeds[0]), P(seeds[1]), P(seeds[2]), stream), "gic_gan_loss_fwd_bwd")
        bws = self._buf("disc_bws", lib.gic_disc_bwd_workspace_floats(B, L, De, R, Fd))
        g = fd.g
        dcw, dcb = [g(c.weight) for c in disc.convs], [g(c.bias) for c in disc.convs]
        for seed, kp, idz, saved, acc in ((seeds[0], keep[0], real_ids, saved_r, 0), (seeds[1], keep[1], fake_ids, saved_f, 1)):
            _lib.check(lib.gic_disc_bwd(mode, P(seed), P(kp), drop_p, None, P(idz), B, L, V, De, R, len(fsz),
                                        _lib.int_array(fsz), _lib.int_array(nfl), P(disc.embeddings.weight),
                                        _lib.ptr_array(cw), _lib.ptr_array(cb), P(disc.highway.weight),
                                        P(disc.feature2out.weight), P(disc.feature2out.bias),
                                        disc.feature2out.weight.shape[0], P(disc.out2logits.weight),
                                        P(disc.out2logits.bias), P(saved), P(bws), P(g(disc.embeddings.weight)),
                                        _lib.ptr_array(dcw), _lib.ptr_array(dcb), P(g(disc.highway.weight)),
                                        P(g(disc.highway.bias)), P(g(disc.feature2out.weight)),
                                        P(g(disc.feature2out.bias)), P(g(disc.out2logits.weight)),
                                        P(g(disc.out2logits.bias)), None, 1, acc, stream), "gic_disc_bwd")
        self._allreduce(fd.grad, 0)
        return dict(d_loss=losses[1], d_real=d_real, d_fake=d_fake, d_sqnorm=self._clip_adam(fd, a.disc_lr, update, 1))

    # ---- EXTENSION: SeqGAN-style policy-gradient step (north-star stages 2-4; not in the reference) -------------
    @_in_ctx
    @torch.no_grad()
    def pg_step(self, captions, pooled=None, u=None, u_roll=None, keep=None, n_roll=16, baseline_mode=1, update=True,
                d_update=True, score_chunk=2048):
        """Generator update by REINFORCE with Monte-Carlo rollouts, discriminator update on hard captions.

        1. captions are sampled by inverse CDF (u[L,B]); 2. for every prefix n_roll continuations are rolled out
        (u_roll[L, (L-1)*B*n_roll]) -- one batched LSTM step + vocab projection over all live rollouts per position;
        3. the discriminator scores all rollouts (hard-token gather path, eval mode) -> Q[B,L]; 4. fused
        reward/baseline/log-prob-weighted loss + backward through the decoder; clip + Adam.  5. (d_update) D step on
        real vs sampled captions with the 'standard' BCE loss.  Returns ids, roll_ids, Q, pg_loss, logp, d_loss."""
        _lib.require_cuda()
        lib = _lib.lib()
        a, dev = self.args, self.device
        mode = gic_b200.get_gemm_mode()
        self._ensure_flat()
        fg, fd = self._flat_g, self._flat_d
        dec, disc = self.gen.decoder, self.disc
        captions = captions.to(dev).long().contiguous()
        B, L = captions.shape
        V, E, H, layers = a.vocab_size, a.gen_embed_dim, a.gen_hidden_dim, a.gen_num_layers
        if layers != 1:
            raise NotImplementedError("rollouts support a single-layer decoder")
        De, R, Fd = a.disc_embed_dim, a.disc_num_rep, sum(a.disc_num_filters)
        fsz, nfl = list(a.disc_filter_sizes), list(a.disc_num_filters)
        stream = _lib.stream()
        P = _lib.ptr
        n = int(n_roll)
        Mmax = (L - 1) * B * n
        if self.cgan:
            feats = self.gen.encoder(pooled.to(dev).float()).detach().contiguous()
        else:
            feats = dec.embed.weight[1].expand(B, E).contiguous()
        if u is None:
            u = torch.rand(L, B, device=dev)
        if u_roll is None:
            u_roll = torch.rand(L, Mmax, device=dev)
        u, u_roll = u.to(dev).float().contiguous(), u_roll.to(dev).float().contiguous()
        logits = self._buf("pg_logits", B * L * V).view(B, L, V)
        ids = torch.empty(B, L, dtype=torch.int64, device=dev)
        logp = torch.empty(B, L, device=dev)
        dsaved = self._buf("dec_saved", lib.gic_decode_saved_floats(B, L, E, H, layers))
        dws = self._buf("dec_ws", lib.gic_decode_fwd_workspace_floats(B, V, H))
        lp = dec.lstm_params()
        W_ih, W_hh, b_ih, b_hh = lp[0::4], lp[1::4], lp[2::4], lp[3::4]
        _lib.check(lib.gic_decode_sample_cdf_fwd(mode, P(feats), P(dec.embed.weight), _lib.ptr_array(W_ih),
                                                 _lib.ptr_array(W_hh), _lib.ptr_array(b_ih), _lib.ptr_array(b_hh),
                                                 P(dec.linear.weight), P(dec.linear.bias), P(u), None, B, L, V, E, H,
                                                 layers, P(logits), P(ids), P(logp), P(dsaved), P(dws), stream),
                   "gic_decode_sample_cdf_fwd")
        roll_ids = torch.empty(Mmax, L, dtype=torch.int64, device=dev)
        rws = self._buf("roll_ws", lib.gic_decode_rollouts_workspace_floats(B, L, V, E, H, n))
        _lib.check(lib.gic_decode_rollouts(mode, P(dsaved), P(ids), P(dec.embed.weight), P(W_ih[0]), P(W_hh[0]),
                                           P(b_ih[0]), P(b_hh[0]), P(dec.linear.weight), P(dec.linear.bias), P(u_roll),
                                           B, L, V, E, H, n, P(roll_ids), P(rws), stream), "gic_decode_rollouts")
        # -- D scores of every rollout and of the captions themselves (eval mode, hard-token gather path)
        cw = [c.weight for c in disc.convs]
        cb = [c.bias for c in disc.convs]
        dW = (disc.embeddings.weight, cw, cb, disc.highway.weight, disc.highway.bias, disc.feature2out.weight,
              disc.feature2out.bias, disc.out2logits.weight, disc.out2logits.bias)
        drop_p = disc.dropout.p
        roll_logits = torch.empty(Mmax * R, device=dev)
        for m0 in range(0, Mmax, score_chunk):
            mc = min(score_chunk, Mmax - m0)
            (lg,), _ = disc_fwd_raw(lib, mode, None, roll_ids[m0:m0 + mc], mc, L, V, De, R, fsz, nfl, *dW, [None], drop_p, dev)
            roll_logits[m0 * R:(m0 + mc) * R] = lg
        (main_logits,), _ = disc_fwd_raw(lib, mode, None, ids, B, L, V, De, R, fsz, nfl, *dW, [None], drop_p, dev)
        Q = torch.empty(B, L, device=dev)
        _lib.check(lib.gic_rollout_rewards(P(roll_logits), P(main_logits), B, L, n, R, P(Q), stream), "gic_rollout_rewards")
        # -- fused reward/baseline/log-prob-weighted loss and its backward; decoder backward w.r.t. the logits
        loss = torch.empty(1, device=dev)
        dlogits = self._buf("pg_dlogits", B * L * V).view(B, L, V)
        _lib.check(lib.gic_pg_loss_fwd_bwd(P(logits), P(ids), P(Q), int(baseline_mode), B, L, V, P(loss), P(dlogits), None,
                                           stream), "gic_pg_loss_fwd_bwd")
        gg = fg.g
        self._zero_unwritten_attn_grads()
        gws = self._buf("dec_bws", lib.gic_decode_bwd_workspace_floats(B, L, V, E, H, layers))
        dfeat = self._buf("dfeat", B * E).view(B, E)
        _lib.check(lib.gic_decode_sample_bwd(
            mode, P(dlogits), None, P(ids), P(dec.embed.weight), _lib.ptr_array(W_ih), _lib.ptr_array(W_hh),
            P(dec.linear.weight), 1.0, 1, B, L, V, E, H, layers, P(dsaved), P(gws), P(gg(dec.embed.weight)),
            _lib.ptr_array([gg(w) for w in W_ih]), _lib.ptr_array([gg(w) for w in W_hh]),
            _lib.ptr_array([gg(w) for w in b_ih]), _lib.ptr_array([gg(w) for w in b_hh]), P(gg(dec.linear.weight)),
            P(gg(dec.linear.bias)), P(dfeat), 0, stream), "gic_decode_sample_bwd")
        if self.cgan:
            enc = self.gen.encoder
            for p_ in (enc.linear.weight, enc.linear.bias, enc.bn.weight, enc.bn.bias):
                gg(p_).zero_()                       # the encoder projection is not trained by the PG step here
        else:
            gg(dec.embed.weight)[1] += dfeat.sum(0)
        out = dict(ids=ids, roll_ids=roll_ids, Q=Q, pg_loss=loss[0], logp=logp, logits=logits, roll_logits=roll_logits,
                   main_logits=main_logits)
        self._allreduce(fg.grad, 2)
        out["g_sqnorm"] = self._clip_adam(fg, a.gen_lr, update, 3)
        if d_update:
            d = self.disc_step(captions, ids, keep=keep, update=update)
            out["d_loss"], out["d_sqnorm"] = d["d_loss"], d["d_sqnorm"]
        return out

    # ---- checkpoints (src/training.py:116-119 pretrained_model.ckpt, :223-227 adv_model.ckpt; SURVEY.md 8f rank 4) -----
    # The reference only ever SAVES (plain state_dict dumps) and has no load / resume.  The files written here keep its
    # formats -- a reference-side torch.load(...)["generator"] keeps working -- and add one extra key with what a
    # resumed run needs: Adam moments and step counts (per parameter NAME, so the flat layout may change), temperature,
    # epoch / step counters.
    def _named_flat(self, fp, module):
        names = {id(p): n for n, p in module.named_parameters()}
        return [(names[id(p)], o, n) for p, o, n in zip(fp.params, fp.offsets, fp.sizes)]

    def _optim_state(self):
        self._ensure_flat()
        out = {}
        for tag, fp, mod in (("gen", self._flat_g, self.gen), ("disc", self._flat_d, self.disc)):
            st = {"step": int(fp.step), "m": {}, "v": {}}
            for name, o, n in self._named_flat(fp, mod):
                st["m"][name] = fp.m[o:o + n].detach().cpu().clone()
                st["v"][name] = fp.v[o:o + n].detach().cpu().clone()
            if hasattr(fp, "m_pre"):
                st["step_pre"] = int(fp.step_pre)
                st["m_pre"] = {name: fp.m_pre[o:o + n].detach().cpu().clone() for name, o, n in self._named_flat(fp, mod)}
                st["v_pre"] = {name: fp.v_pre[o:o + n].detach().cpu().clone() for name, o, n in self._named_flat(fp, mod)}
            out[tag] = st
        return out

    def save_pretrained(self, path):
        """pretrained_model.ckpt: the generator's state_dict, exactly as src/training.py:118."""
        torch.save(self._gen_state(), path)

    def save_checkpoint(self, path, resume_state=True):
        """adv_model.ckpt: {"generator": ..., "discriminator": ...} as src/training.py:225-226 (+ "gic_resume")."""
        blob = {"generator": self._gen_state(), "discriminator": self.disc.state_dict()}
        if resume_state:
            blob["gic_resume"] = {"optim": self._optim_state(), "temperature": float(self.gen.decoder.temperature),
                                  "adv_epoch": int(self.adv_epoch), "pretrain_steps": int(self.pretrain_steps),
                                  "gen_steps": int(self.gen_steps), "disc_steps": int(self.disc_steps), "format": 1}
        torch.save(blob, path)

    RESNET_PREFIX = "encoder.resnet."

    def _load_gen_state(self, sd, strict):
        """The reference's Generator.state_dict() always carries the frozen ResNet trunk (encoder.resnet.*,
        src/generator.py:12-14), which is outside this path (SURVEY.md section 2 row 2): those tensors are set aside --
        and written back by save_checkpoint / save_pretrained, so a file that came from the reference can go back to it --
        and everything else is loaded with the requested strictness."""
        self._passthrough = {k: v for k, v in sd.items() if k.startswith(self.RESNET_PREFIX)}
        self.gen.load_state_dict({k: v for k, v in sd.items() if not k.startswith(self.RESNET_PREFIX)}, strict=strict)

    def _gen_state(self):
        sd = self.gen.state_dict()
        sd.update(self._passthrough)
        return sd

    def load_checkpoint(self, path, strict=True, unsafe_pickle=False):
        """Loads either file format (a bare generator state_dict, or the generator/discriminator dict) and, when the
        file carries it, the resume state.  Parameters stay views of the flat buffers (load_state_dict copies in place),
        captured CUDA graphs stay valid.  Returns True when optimizer / schedule state was restored.
        Files are read with torch.load(weights_only=True) -- both formats hold only tensors and plain containers;
        unsafe_pickle=True opts into full unpickling for files from a trusted source that hold anything else."""
        blob = torch.load(path, map_location="cpu", weights_only=not unsafe_pickle)
        if not isinstance(blob, dict):
            raise ValueError("%s: not a checkpoint written by this code or the reference" % path)
        if "generator" in blob or "discriminator" in blob:
            if "generator" in blob:
                self._load_gen_state(blob["generator"], strict)
            if "discriminator" in blob:
                self.disc.load_state_dict(blob["discriminator"], strict=strict)
        else:
            self._load_gen_state(blob, strict)              # pretrained_model.ckpt
        rs = blob.get("gic_resume") if isinstance(blob.get("gic_resume", None), dict) else None
        if rs is None:
            return False
        self._ensure_flat()
        for tag, fp, mod in (("gen", self._flat_g, self.gen), ("disc", self._flat_d, self.disc)):
            st = rs["optim"][tag]
            fp.step = int(st["step"])
            for name, o, n in self._named_flat(fp, mod):
                if name not in st["m"]:
                    if strict:
                        raise KeyError("checkpoint has no Adam state for %s.%s" % (tag, name))
                    continue
                fp.m[o:o + n].copy_(st["m"][name].reshape(-1))
                fp.v[o:o + n].copy_(st["v"][name].reshape(-1))
            if "m_pre" in st:
                fp.m_pre, fp.v_pre, fp.step_pre = torch.zeros_like(fp.m), torch.zeros_like(fp.v), int(st["step_pre"])
                for name, o, n in self._named_flat(fp, mod):
                    fp.m_pre[o:o + n].copy_(st["m_pre"][name].reshape(-1))
                    fp.v_pre[o:o + n].copy_(st["v_pre"][name].reshape(-1))
        self.gen.decoder.temperature = rs["temperature"]
        self.adv_epoch, self.pretrain_steps = rs["adv_epoch"], rs["pretrain_steps"]
        self.gen_steps, self.disc_steps = rs["gen_steps"], rs["disc_steps"]
        return True

    def adv_loop(self, what, batches, total_batches=None, graph=False):
        """Body of the reference's adv_loop over an iterable of (pooled_or_None, captions) batches."""
        gen_loss, disc_loss = [], []
        nb = total_batches or (len(batches) if hasattr(batches, "__len__") else 1)
        for i, (pooled, captions) in enumerate(batches, start=1):
            r = self.adv_step(captions, pooled=pooled, train=(what == "train"), graph=(graph and what == "train"))
            # graph replay returns views of the graph's static loss buffer (overwritten by the next replay): keep copies,
            # so that the mean is over the per-batch values as the reference's np.mean(gen_loss) is (src/training.py:185)
            gen_loss.append(r["g_loss"].clone())
            disc_loss.append(r["d_loss"].clone())
            self.gen_steps += 1
            self.disc_steps += 1
            self.update_temperature(self.adv_epoch + i / nb, self.args.adv_epochs)      # :183
        g = torch.stack(gen_loss).mean().item() if gen_loss else float("nan")
        d = torch.stack(disc_loss).mean().item() if disc_loss else float("nan")
        return g, d
