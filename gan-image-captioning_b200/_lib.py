"""ctypes binding of libgic_b200.so (C ABI in include/gic_b200.h).  No torch types cross this boundary:
tensors are passed as raw device pointers + sizes, the stream as a cudaStream_t handle.

There is deliberately no CPU fallback: if the library is missing, or a compute entry point is called
without an sm_100 device, this raises."""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgic_b200.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "gic_b200.h")

GEMM_FP32, GEMM_TF32, GEMM_BF16 = 0, 1, 3
LOSS_TYPES = {"standard": 0, "JS": 1, "KL": 2, "hinge": 3, "tv": 4, "rsgan": 5}

_lib = None


class AttnBlock(C.Structure):
    """gic_attn_t of include/gic_b200.h."""
    _fields_ = [("grid", C.c_void_p), ("P", C.c_int), ("Cf", C.c_int), ("Da", C.c_int), ("W_k", C.c_void_p),
                ("W_v", C.c_void_p), ("W_q", C.c_void_p), ("w_e", C.c_void_p), ("saved", C.c_void_p), ("ws", C.c_void_p),
                ("dW_k", C.c_void_p), ("dW_v", C.c_void_p), ("dW_q", C.c_void_p), ("dw_e", C.c_void_p)]


def attn_block(grid, W_k, W_v, W_q, w_e, saved, ws=None, dW_k=None, dW_v=None, dW_q=None, dw_e=None):
    B, Pn, Cf = grid.shape
    return AttnBlock(ptr(grid), Pn, Cf, W_k.shape[0], ptr(W_k), ptr(W_v), ptr(W_q), ptr(w_e), ptr(saved), ptr(ws),
                     ptr(dW_k), ptr(dW_v), ptr(dW_q), ptr(dw_e))


class DecodeConstraints(C.Structure):
    """gic_decode_constraints_t (include/gic_b200.h): constrained beam search / sampling."""
    _fields_ = [("min_length", C.c_int), ("no_repeat_ngram_size", C.c_int), ("bad_ids", C.c_void_p), ("n_bad", C.c_int)]


class GicError(RuntimeError):
    pass


def header_symbols():
    """Names of all functions include/gic_b200.h declares."""
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gic_[a-z0-9_]+)\s*\(", src)))


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GicError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the hot path is CUDA-only; there is no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


P = C.c_void_p
I = C.c_int
F = C.c_float
Z = C.c_size_t


RNG_TAG_GUMBEL, RNG_TAG_DROPOUT, RNG_TAG_SAMPLE = 0x47, 0x44, 0x53


def _declare(L):
    L.gic_version.restype = I
    L.gic_last_error.restype = C.c_char_p
    L.gic_check_device.restype = I
    L.gic_launch_count.restype = C.c_ulonglong
    L.gic_kernel_launches.restype = C.c_ulonglong
    L.gic_kernel_launches.argtypes = [C.c_char_p]
    L.gic_kernel_names.argtypes = [C.c_char_p, I]
    L.gic_prof_begin.restype = None
    L.gic_prof_end.restype = None
    L.gic_prof_end.argtypes = [P, P, P]
    L.gic_gemm.argtypes = [I, I, I, I, I, I, F, P, I, P, I, F, P, I, P, P]
    L.gic_gemm_bf16.argtypes = [I, I, I, I, I, F, P, I, P, I, F, P, I, P, P]
    L.gic_encoder_fwd.argtypes = [I, P, I, I, I, P, P, P, P, F, P, P, P, P, P]
    L.gic_encoder_bwd.argtypes = [I, P, P, P, P, P, P, P, I, I, I, P, P, P, P, P, I, P]
    L.gic_encoder_bn_running_update.argtypes = [P, P, I, F, F, F, P, P, P, P]
    L.gic_encoder_fwd_eval.argtypes = [I, P, I, I, I, P, P, P, P, F, P, P, P, P, P]
    L.gic_sample_step.argtypes = [I, P, P, F, I, I, I, I, P, P, P, P, I, P, P]
    for f in (L.gic_decode_saved_floats, L.gic_decode_fwd_workspace_floats, L.gic_decode_bwd_workspace_floats,
              L.gic_disc_saved_floats, L.gic_disc_fwd_workspace_floats, L.gic_disc_bwd_workspace_floats,
              L.gic_disc_bwd_demb_offset_floats):
        f.restype = Z
    L.gic_decode_saved_floats.argtypes = [I] * 5
    L.gic_decode_fwd_workspace_floats.argtypes = [I] * 3
    L.gic_decode_bwd_workspace_floats.argtypes = [I] * 6
    L.gic_disc_saved_floats.argtypes = [I] * 5
    L.gic_disc_fwd_workspace_floats.argtypes = [I]
    L.gic_disc_bwd_workspace_floats.argtypes = [I] * 5
    L.gic_disc_bwd_demb_offset_floats.argtypes = [I] * 5
    L.gic_decode_sample_bwd_factored.argtypes = [I, P, P, P, I, P, P, P, P, P, P, F, I, I, I, I, I, I, P, P, P, P, P, P,
                                                 P, P, P, P, I, P]
    L.gic_decode_sample_fwd.argtypes = [I, P, P, P, P, P, P, P, P, P, F, I, P, I, I, I, I, I, I, P, P, P, P, P]
    L.gic_decode_sample_bwd.argtypes = [I, P, P, P, P, P, P, P, F, I, I, I, I, I, I, I, P, P, P, P, P, P, P, P, P, P,
                                        I, P]
    L.gic_disc_fwd.argtypes = [I, P, P, I, I, I, I, I, I, P, P, P, P, P, P, P, P, P, I, P, P, I, P, F, P, P, P, P]
    L.gic_disc_bwd.argtypes = [I, P, P, F, P, P, I, I, I, I, I, I, P, P, P, P, P, P, P, P, I, P, P, P, P, P, P, P, P,
                               P, P, P, P, P, P, I, I, P]
    L.gic_gan_loss_fwd_bwd.argtypes = [I, P, P, P, I, P, P, P, P, P]
    L.gic_grad_sqnorm.argtypes = [P, Z, P, P]
    L.gic_clip_adam.argtypes = [P, P, P, P, Z, P, F, F, I, F, F, F, F, P]
    L.gic_clip_adam_dyn.argtypes = [P, P, P, P, Z, P, F, F, P, F, F, F, P]
    L.gic_decode_sample_cdf_fwd.argtypes = [I, P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, P, P, P, P, P, P]
    L.gic_attn_saved_floats.restype = Z
    L.gic_attn_saved_floats.argtypes = [I] * 5
    L.gic_attn_bwd_workspace_floats.restype = Z
    L.gic_attn_bwd_workspace_floats.argtypes = [I] * 5
    L.gic_decode_sample_fwd_attn.argtypes = [P] + [I, P, P, P, P, P, P, P, P, P, F, I, P, I, I, I, I, I, I, P, P, P, P, P]
    L.gic_decode_sample_bwd_attn.argtypes = [P, I, P, P, P, P, I, P, P, P, P, P, P, F, I, I, I, I, I, I, I, P, P, P, P, P,
                                             P, P, P, P, P, P]
    L.gic_sample_cdf_step.argtypes = [P, P, I, I, I, I, P, P, P, P, P, I, P, P]
    L.gic_decode_rollouts_workspace_floats.restype = Z
    L.gic_decode_rollouts_workspace_floats.argtypes = [I] * 6
    L.gic_decode_rollouts.argtypes = [I, P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, P, P, P]
    L.gic_rollout_rewards.argtypes = [P, P, I, I, I, I, P, P]
    L.gic_ce_loss_fwd_bwd.argtypes = [P, P, I, I, I, P, P, P]
    L.gic_pg_loss_fwd_bwd.argtypes = [P, P, P, I, I, I, I, P, P, P, P]
    L.gic_set_temperature_device.restype = None
    L.gic_set_temperature_device.argtypes = [P]
    L.gic_disc_prepared_floats.restype = Z
    L.gic_disc_prepared_floats.argtypes = [I]
    L.gic_disc_prepare.argtypes = [I, P, P, P, I, P, P, I, P, P]
    L.gic_pack_captions.argtypes = [P, P, I, I, P, P, P]
    L.gic_set_rng.restype = None
    L.gic_set_rng.argtypes = [C.c_ulonglong, C.c_ulonglong, P]
    L.gic_philox_uniform.argtypes = [C.c_uint, Z, P, P]
    L.gic_philox_keep_mask.argtypes = [C.c_uint, Z, F, P, P]
    L.gic_encoder_fwd_stats.argtypes = [I, P, I, I, I, P, P, P, P, P]
    L.gic_encoder_fwd_apply.argtypes = [P, I, I, P, P, F, P, F, P, P, P, P]
    L.gic_encoder_bwd_stats.argtypes = [P, P, P, P, I, I, P, P]
    L.gic_encoder_bwd_apply.argtypes = [I, P, P, P, P, P, P, I, I, I, P, F, F, P, P, P, P, P, P]
    L.gic_set_vocab_grads_event.restype = None
    L.gic_set_vocab_grads_event.argtypes = [P]
    L.gic_set_embed_grads_event.restype = None
    L.gic_set_embed_grads_event.argtypes = [P]
    L.gic_disc_set_prepared.restype = None
    L.gic_disc_set_prepared.argtypes = [P]
    L.gic_comm_create.restype = P
    L.gic_comm_create.argtypes = [I, I, Z]
    L.gic_comm_handle_bytes.restype = Z
    L.gic_comm_ipc_handle.argtypes = [P, P]
    L.gic_comm_open.argtypes = [P, P]
    L.gic_comm_buffer.restype = P
    L.gic_comm_buffer.argtypes = [P]
    L.gic_comm_buffer_bytes.restype = Z
    L.gic_comm_buffer_bytes.argtypes = [P]
    L.gic_comm_error.argtypes = [P]
    L.gic_comm_destroy.restype = None
    L.gic_comm_destroy.argtypes = [P]
    L.gic_allreduce.argtypes = [P, Z, P, I, P, P]
    L.gic_comm_local_group.argtypes = [P, I]
    L.gic_allreduce_local_group.argtypes = [P, P, P, Z, I, I, P]
    L.gic_ctx_create.restype = P
    L.gic_ctx_set_current.restype = P
    L.gic_ctx_set_current.argtypes = [P]
    L.gic_ctx_destroy.restype = None
    L.gic_ctx_destroy.argtypes = [P]
    L.gic_trap_info.restype = None
    L.gic_trap_info.argtypes = [C.POINTER(C.c_ulonglong)]
    L.gic_trap_notes.argtypes = [C.POINTER(C.c_ulonglong), I]
    L.gic_ctx_set_option.argtypes = [C.c_char_p, I]
    L.gic_ctx_clear_option.restype = None
    L.gic_ctx_clear_option.argtypes = [C.c_char_p]
    L.gic_ctx_get_option.argtypes = [C.c_char_p, I]
    L.gic_vocab_topk_workspace_floats.restype = Z
    L.gic_vocab_topk_workspace_floats.argtypes = [I] * 3
    L.gic_vocab_topk.argtypes = [I, P, P, P, I, I, I, I, P, P, P, P, P]
    L.gic_decode_beam_workspace_floats.restype = Z
    L.gic_decode_beam_workspace_floats.argtypes = [I] * 7
    L.gic_decode_beam.argtypes = [I, P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, C.c_int64, F, P, P, P, P, P, P]
    L.gic_vocab_target_logp_workspace_floats.restype = Z
    L.gic_vocab_target_logp_workspace_floats.argtypes = [I] * 2
    L.gic_vocab_target_logp.argtypes = [I, P, P, P, P, I, I, I, P, P, P, P, P]
    L.gic_score_captions_workspace_floats.restype = Z
    L.gic_score_captions_workspace_floats.argtypes = [I] * 6
    L.gic_score_captions.argtypes = [I, P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, P, P, P, P, P]
    L.gic_vocab_sample_workspace_floats.restype = Z
    L.gic_vocab_sample_workspace_floats.argtypes = [I] * 3
    L.gic_vocab_sample.argtypes = [I, P, P, P, I, I, I, I, F, I, F, P, P, P, P]
    L.gic_sample_captions_workspace_floats.restype = Z
    L.gic_sample_captions_workspace_floats.argtypes = [I] * 7
    L.gic_sample_captions.argtypes = [I, P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, C.c_int64, F, I, F, P, P, P, P, P]
    CP = C.POINTER(DecodeConstraints)
    L.gic_vocab_topk_masked.argtypes = [I, P, P, P, I, I, I, I, P, P, P, P, P, P]
    L.gic_vocab_sample_masked.argtypes = [I, P, P, P, I, I, I, I, F, I, F, P, P, P, P, P]
    L.gic_decode_beam_constrained_workspace_floats.restype = Z
    L.gic_decode_beam_constrained_workspace_floats.argtypes = [I] * 7 + [CP]
    L.gic_decode_beam_constrained.argtypes = [I, P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, C.c_int64, F, CP, P, P, P, P,
                                              P, P]
    L.gic_sample_captions_constrained_workspace_floats.restype = Z
    L.gic_sample_captions_constrained_workspace_floats.argtypes = [I] * 8 + [CP]
    L.gic_sample_captions_constrained.argtypes = [I, P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, C.c_int64, F, I, F, CP, P,
                                                  P, P, P, P]
    for name in header_symbols():      # every declared entry point must be exported
        getattr(L, name)


def kernel_launches(name=None) -> int:
    """Launches so far of the kernel `name` (e.g. "vocab_sample_kernel"); None = every kernel of the library."""
    return int(lib().gic_kernel_launches(None if name is None else name.encode()))


def kernel_counts() -> dict:
    """{kernel name: launches so far} for every kernel this process has launched."""
    buf = C.create_string_buffer(8192)
    lib().gic_kernel_names(buf, 8192)
    return {n: kernel_launches(n) for n in buf.value.decode().split("\n") if n}


class expect_kernels:
    """Context manager for tests: every kernel named must be launched at least once inside the block -- a fused path
    that silently declines (handled = false) fails the test instead of comparing the fallback with itself."""

    def __init__(self, *names, absent=()):
        self.names, self.absent = names, tuple(absent)

    def __enter__(self):
        self.before = {n: kernel_launches(n) for n in self.names + self.absent}
        return self

    def __exit__(self, et, ev, tb):
        if et is not None:
            return False
        self.delta = {n: kernel_launches(n) - self.before[n] for n in self.names + self.absent}
        missing = [n for n in self.names if self.delta[n] <= 0]
        extra = [n for n in self.absent if self.delta[n] > 0]
        if missing or extra:
            raise AssertionError("kernels expected but not launched: %s; launched but expected absent: %s" % (missing, extra))
        return False


class Context:
    """A library context (include/gic_b200.h "contexts"): the temperature pointer, prepared discriminator weights, Philox
    state and vocab-gradient event that the setters install are per context, not per process.  ``with ctx:`` makes it the
    calling thread's current context for the block (re-entrant)."""

    def __init__(self):
        self.handle = lib().gic_ctx_create()
        if not self.handle:
            raise MemoryError("gic_ctx_create")
        self._prev = []

    def __enter__(self):
        self._prev.append(lib().gic_ctx_set_current(self.handle))
        return self

    def __exit__(self, *exc):
        lib().gic_ctx_set_current(self._prev.pop())
        return False

    def set_option(self, name: str, value: int):
        with self:
            set_option(name, value)

    def clear_option(self, name: str):
        with self:
            clear_option(name)

    def get_option(self, name: str, default: int = 0) -> int:
        with self:
            return get_option(name, default)

    def __del__(self):
        try:
            if getattr(self, "handle", None) and _lib is not None:
                _lib.gic_ctx_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def trap_info():
    """(site, word, blockIdx.x, threadIdx.x, globaltimer) of the bounded device-side wait that gave up, or None
    (include/gic_b200.h, gic_trap_info); readable after the CUDA context has died."""
    out = (C.c_ulonglong * 4)()
    lib().gic_trap_info(out)
    if out[0] == 0:
        return None
    notes = (C.c_ulonglong * 128)()
    n = lib().gic_trap_notes(notes, 32)
    waits = [dict(site=int(notes[4 * i]), word=hex(int(notes[4 * i + 1])), block=int(notes[4 * i + 2] >> 32),
                  thread=int(notes[4 * i + 2] & 0xffffffff)) for i in range(n)]
    return dict(site=int(out[0]), word=hex(int(out[1])), block=int(out[2] >> 32), thread=int(out[2] & 0xffffffff), globaltimer=int(out[3]),
                waits=waits)


def set_option(name: str, value: int):
    """Set a kernel-variant / tuning switch of the calling thread's CURRENT context (gic_ctx_set_option)."""
    check(lib().gic_ctx_set_option(name.encode(), int(value)), "gic_ctx_set_option")


def clear_option(name: str):
    lib().gic_ctx_clear_option(name.encode())


def get_option(name: str, default: int = 0) -> int:
    return int(lib().gic_ctx_get_option(name.encode(), int(default)))


class options:
    """``with _lib.options(GIC_DECODE_STEP=0, ...):`` -- switches of the current context for the block, cleared afterwards
    (back to environment / built-in default)."""

    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        for k, v in self.kw.items():
            set_option(k, v)
        return self

    def __exit__(self, *exc):
        for k in self.kw:
            clear_option(k)
        return False


def check(rc: int, what: str = ""):
    if rc == 0:
        return
    msg = lib().gic_last_error().decode(errors="replace")
    if rc == 6:
        raise NotImplementedError(msg)
    raise GicError(f"{what}: {msg} (status {rc})")


def ptr(t):
    """Device pointer of a contiguous torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), "libgic_b200 takes dense row-major tensors"
    return t.data_ptr()


def ptr_array(ts):
    """C array of device pointers (for per-layer / per-filter-group weights)."""
    arr = (C.c_void_p * len(ts))()
    for i, t in enumerate(ts):
        arr[i] = None if t is None else ptr(t)
    return arr


def int_array(xs):
    return (C.c_int * len(xs))(*[int(x) for x in xs])


def stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda():
    """Fail loudly when the CUDA path cannot run (no silent fallback)."""
    import torch
    if not torch.cuda.is_available():
        raise GicError("no CUDA device: the gic_b200 hot path is CUDA-only (sm_100a) and has no CPU fallback")
    check(lib().gic_check_device(), "gic_check_device")
