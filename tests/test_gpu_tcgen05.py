"""tcgen05 / TMA GEMM (kind::tf32, fp32 accumulate in TMEM) against an fp64 product of the same operands.

TF32 keeps 10 mantissa bits: per-product relative error <= 2^-11 with round-to-nearest staging, so a
K-term dot product of O(1) operands is expected within ~1e-3 * sqrt(K) absolute; the bound used here is
rtol 2e-3 against max |C| (the fp32-exact path is tested in test_gpu_parity.py)."""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
REPORT = {}


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "tcgen05_report.json"), "w") as f:
        json.dump(REPORT, f, indent=1, sort_keys=True)


def run_gemm(mode, tA, tB, M, N, K, alpha=1.0, beta=0.0, use_bias=False, seed=0):
    import gic_b200
    from gic_b200 import _lib as L
    L.require_cuda()
    g = torch.Generator().manual_seed(seed + M * 7 + N * 3 + K + tA * 2 + tB)
    A = torch.randn((K, M) if tA else (M, K), generator=g)
    B = torch.randn((N, K) if tB else (K, N), generator=g)
    C0 = torch.randn(M, N, generator=g)
    bias = torch.randn(N, generator=g) if use_bias else None
    Ad, Bd, Cd = A.to(dev()), B.to(dev()), C0.clone().to(dev())
    bd = bias.to(dev()) if use_bias else None
    want = alpha * ((Ad.t() if tA else Ad).double() @ (Bd.t() if tB else Bd).double()) + beta * Cd.double()
    if use_bias:
        want = want + bd.double()
    L.check(L.lib().gic_gemm(mode, tA, tB, M, N, K, alpha, L.ptr(Ad), A.shape[1], L.ptr(Bd), B.shape[1], beta,
                             L.ptr(Cd), N, L.ptr(bd), L.stream()), "gic_gemm")
    torch.cuda.synchronize()
    scale = float(want.abs().max())
    err = float((Cd.double() - want).abs().max())
    return err, scale


SHAPES = [(128, 128, 32), (128, 128, 64), (256, 2048, 1024), (256, 10000, 512), (300, 900, 900), (16384, 900, 900),
          (5120, 64, 10000), (900, 900, 2048), (130, 100, 36), (5120, 512, 10000)]


@pytest.mark.parametrize("tA,tB", [(0, 1), (0, 0), (1, 0), (1, 1)])
@pytest.mark.parametrize("M,N,K", SHAPES)
def test_gemm_tf32_vs_fp64(tA, tB, M, N, K):
    err, scale = run_gemm(1, tA, tB, M, N, K, seed=1)
    REPORT[f"tf32/{M}x{N}x{K}/tA{tA}tB{tB}"] = dict(err=err, scale=scale, rel=err / scale)
    assert err <= 2e-3 * scale, f"rel err {err / scale:.3e}"


def test_gemm_tf32_alpha_beta_bias():
    err, scale = run_gemm(1, 0, 1, 384, 900, 900, alpha=0.75, beta=0.5, use_bias=True, seed=2)
    REPORT["tf32/alpha_beta_bias"] = dict(err=err, scale=scale, rel=err / scale)
    assert err <= 2e-3 * scale


def test_gemm_tf32_unaligned_falls_back_to_exact_kernel():
    # lda = 37 is not TMA-addressable: the dispatcher must use the exact-fp32 kernel (still CUDA, still ours)
    err, scale = run_gemm(1, 0, 1, 70, 90, 37, seed=3)
    assert err <= 1e-5 * scale


# ---- bf16 operands (tcgen05 kind::f16, fp32 accumulate): GIC_GEMM_BF16 mode's contraction ----------------------
def run_gemm_bf16(tA, tB, M, N, K, alpha=1.0, beta=0.0, use_bias=False, seed=0, pad=0):
    """Operands are rounded to bf16 first, so the fp64 product of the rounded operands is the exact target and the
    only error left is the fp32 accumulation order."""
    from gic_b200 import _lib as L
    L.require_cuda()
    g = torch.Generator().manual_seed(seed + M * 7 + N * 3 + K + tA * 2 + tB)
    ra, ca = ((K, M) if tA else (M, K))
    rb, cb = ((N, K) if tB else (K, N))
    lda, ldb = ((ca + 7) // 8) * 8 + pad, ((cb + 7) // 8) * 8 + pad
    A = torch.zeros(ra, lda, dtype=torch.bfloat16); A[:, :ca] = torch.randn(ra, ca, generator=g).to(torch.bfloat16)
    B = torch.zeros(rb, ldb, dtype=torch.bfloat16); B[:, :cb] = torch.randn(rb, cb, generator=g).to(torch.bfloat16)
    C0 = torch.randn(M, N, generator=g)
    bias = torch.randn(N, generator=g) if use_bias else None
    Ad, Bd, Cd = A.to(dev()), B.to(dev()), C0.clone().to(dev())
    bd = bias.to(dev()) if use_bias else None
    Aop = (A[:, :ca].double().t() if tA else A[:, :ca].double())
    Bop = (B[:, :cb].double().t() if tB else B[:, :cb].double())
    want = alpha * (Aop @ Bop) + beta * C0.double()
    if use_bias:
        want = want + bias.double()
    L.check(L.lib().gic_gemm_bf16(tA, tB, M, N, K, alpha, L.ptr(Ad), lda, L.ptr(Bd), ldb, beta, L.ptr(Cd), N, L.ptr(bd),
                                  L.stream()), "gic_gemm_bf16")
    torch.cuda.synchronize()
    scale = float(want.abs().max())
    err = float((Cd.double().cpu() - want).abs().max())
    return err, scale


@pytest.mark.parametrize("tA,tB", [(0, 1), (0, 0), (1, 0), (1, 1)])
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 256, 128), (300, 900, 900), (16384, 900, 900), (900, 900, 4096),
                                   (130, 100, 72), (2048, 512, 5120)])
def test_gemm_bf16_vs_fp64(tA, tB, M, N, K):
    err, scale = run_gemm_bf16(tA, tB, M, N, K, seed=4)
    REPORT[f"bf16/{M}x{N}x{K}/tA{tA}tB{tB}"] = dict(err=err, scale=scale, rel=err / scale)
    assert err <= 2e-5 * scale, f"rel err {err / scale:.3e}"          # exact bf16 products, fp32 accumulation


@pytest.mark.parametrize("tB,M,N,K", [(1, 16384 + 130, 900, 900), (0, 8192 + 256 + 8, 900, 900), (1, 8192, 256, 512),
                                      (0, 19200, 1024, 192), (1, 18944, 200, 72), (0, 18944, 328, 1000)])
def test_gemm_bf16_cta_pair_kernel_bias_ragged_rows(tB, M, N, K):
    """Shapes that take the cta_group::2 kernel (gemm_pair_tcgen05.cu): rows that are not a multiple of the 256-row pair
    tile, bias, alpha, padded pitches; and the same call with GIC_GEMM_2CTA=0 (one CTA per tile)."""
    from gic_b200 import _lib
    # the pair kernel takes a shape when its 256 x 256 tiles give every SM pair (74 on a B200) at least one tile
    pair = ((M + 255) // 256) * ((N + 255) // 256) >= 74
    with _lib.expect_kernels(*(["gemm_pair_kernel"] if pair else ["gemm_p_kernel"]),
                             absent=() if pair else ("gemm_pair_kernel",)):   # a declined dispatch must fail, not pass silently
        err, scale = run_gemm_bf16(0, tB, M, N, K, alpha=0.5, use_bias=True, seed=9, pad=8)
    REPORT[f"bf16_pair/{M}x{N}x{K}/tB{tB}"] = dict(err=err, scale=scale, rel=err / scale)
    assert err <= 2e-5 * scale, f"rel err {err / scale:.3e}"
    with _lib.options(GIC_GEMM_2CTA=0), _lib.expect_kernels("gemm_p_kernel", absent=("gemm_pair_kernel",)):
        err0, _ = run_gemm_bf16(0, tB, M, N, K, alpha=0.5, use_bias=True, seed=9, pad=8)
    assert err0 <= 2e-5 * scale


def test_gemm_bf16_alpha_beta_bias_padded_pitch():
    err, scale = run_gemm_bf16(0, 1, 384, 900, 900, alpha=0.75, beta=1.0, use_bias=True, seed=5, pad=56)
    assert err <= 2e-5 * scale


# ---- decode-step kernels (vocab_sample_tcgen05.cu): three ways to run Decoder.sample in TF32 mode ----------------------
#   "step"   one kernel per step: projection + sample of step t, recurrent contraction and LSTM cell of step t + 1 (default)
#   "two"    GIC_DECODE_STEP=0: fused LSTM-step kernel + fused projection / sample kernel (round-1 path; attention and
#            multi-layer decoders still take it)
#   "three"  GIC_FUSED_SAMPLE=0: fused LSTM-step kernel, projection GEMM, sampler kernel
# Every variant asserts, through the library's launch counters, that ITS kernels ran.
_DECODE_ENV = {"step": {}, "two": {"GIC_DECODE_STEP": "0"}, "three": {"GIC_FUSED_SAMPLE": "0"}}
_DECODE_KERNELS = {"step": (("decode_step_kernel", "lstm_step_tf32_kernel"), ()),
                   "two": (("vocab_sample_kernel", "lstm_step_tf32_kernel"), ("decode_step_kernel",)),
                   "three": (("sample_step_reg_kernel", "lstm_step_tf32_kernel"), ("decode_step_kernel", "vocab_sample_kernel"))}


def _decode_variants(B, L, V, E, H, T, forced=False, seed=0, variants=("step", "two", "three")):
    import gic_b200
    import gic_b200.generator as G
    from gic_b200 import _lib
    from gic_b200.args import default_args
    a = default_args(vocab_size=V, gen_embed_dim=E, gen_hidden_dim=H, gen_num_layers=1, conditional_gan=0, device="cuda")
    torch.manual_seed(seed)
    gen = G.Generator(a).to("cuda:0")
    gen.train()
    gen.decoder.temperature = T
    g = torch.Generator(device="cuda:0").manual_seed(seed + 1)
    u = torch.rand(L, B, V, generator=g, device="cuda:0")
    feats = torch.randn(B, E, generator=g, device="cuda:0") * 0.05
    fz = torch.randint(0, V, (B, L), generator=g, device="cuda:0") if forced else None
    old = gic_b200.get_gemm_mode()
    gic_b200.set_gemm_mode(gic_b200.GEMM_TF32)
    res = {}
    try:
        for v in variants:
            want, absent = _DECODE_KERNELS[v]
            with _lib.options(**_DECODE_ENV[v]), _lib.expect_kernels(*want, absent=absent) as ek:
                with torch.no_grad():
                    p, ids = gen.decoder.sample(feats, max_caption_len=L, u=u, forced_ids=fz)
                torch.cuda.synchronize()
            if v == "step":      # step 0's LSTM kernel, L - 1 fused steps, and the last step (nothing follows it) as the plain kernel
                assert ek.delta["decode_step_kernel"] == L - 1 and ek.delta["lstm_step_tf32_kernel"] == 1, ek.delta
            res[v] = (p.clone(), ids.clone())
    finally:
        gic_b200.set_gemm_mode(old)
    return res


@pytest.mark.parametrize("B,L,V,E,H,T,forced", [
    (8, 6, 1000, 32, 512, 1.0, False),        # c1-like: one row block, 8 column tiles, rows padded to 128
    (8, 6, 1000, 32, 512, 100.0, True),       # saturated softmax (first-max tie rule), teacher forcing
    (256, 4, 10000, 512, 512, 1.0, False),    # c2 shape: 2 x 63 tiles of 128 x 160
    (200, 3, 10000, 64, 256, 5.0, False),     # ragged last row block
    (130, 3, 4004, 64, 128, 1.0, True),       # V not a multiple of the tile width
])
def test_fused_vocab_sample_matches_unfused(B, L, V, E, H, T, forced):
    """"two" vs "three": both read the same TF32 accumulators, so the sampled ids must be IDENTICAL and the probabilities
    equal up to the different summation order of the softmax normaliser."""
    res = _decode_variants(B, L, V, E, H, T, forced, variants=("two", "three"))
    (p1, i1), (p0, i0) = res["two"], res["three"]
    nm = f"vocab_sample/B{B}V{V}T{T}"
    mism = int((i1 != i0).sum())
    REPORT[nm + "/id_mismatches"] = dict(err=float(mism), scale=float(i0.numel()), rel=mism / i0.numel())
    assert mism == 0, f"{mism} of {i0.numel()} sampled ids differ between the fused and the separate kernels"
    err = float((p1 - p0).abs().max())
    REPORT[nm + "/probs"] = dict(err=err, scale=float(p0.max()), rel=err / float(p0.max()))
    assert err <= 1e-5 * float(p0.max()) + 1e-12
    rs = p1.sum(-1)
    assert float((rs - 1).abs().max()) < 1e-4


@pytest.mark.parametrize("B,L,V,E,H,T", [
    (8, 6, 1000, 32, 512, 1.0),               # c1-like: 8 projection tiles, 128 narrow rec tiles
    (8, 16, 1000, 32, 512, 100.0),            # saturated softmax
    (256, 20, 10000, 512, 512, 1.0),          # c2: 126 projection tiles + 22 rec tiles of 192 columns
    (200, 5, 10000, 64, 256, 5.0),            # ragged last row block
    (130, 4, 4004, 64, 128, 1.0),             # V not a multiple of the tile width
    (128, 3, 30000, 512, 1024, 1.0),          # c4 per-GPU shape: 118 projection tiles of 256, 30 rec tiles
])
def test_fused_decode_step_matches_two_kernel_path(B, L, V, E, H, T):
    """"step" vs "two", teacher-forced (the same tokens are fed back, so one flipped near-tie cannot cascade).  The fused
    step sums the LSTM pre-activation as (embed[tok] W_ih^T) + (h W_hh^T) -- two TF32 accumulators added in fp32 -- where the
    LSTM-step kernel runs one accumulator over K = E + H: same products, different association, so h agrees to fp32
    round-off, the logits to ~1e-6, and a sampled id may differ only where the top two perturbed logits are that close."""
    res = _decode_variants(B, L, V, E, H, T, forced=True, seed=7, variants=("step", "two"))
    (p1, i1), (p0, i0) = res["step"], res["two"]
    mism = (i1 != i0)
    nm = f"decode_step/B{B}V{V}H{H}T{T}"
    n_mism = int(mism.sum())
    same = ~mism
    err = float(((p1 - p0).abs().amax(-1))[same].max())
    REPORT[nm] = dict(err=err, scale=float(p0.max()), rel=err / float(p0.max()), id_mismatches=n_mism)
    assert n_mism <= max(1, i0.numel() // 2000), f"{n_mism} of {i0.numel()} sampled ids differ"
    # d p <= p (1 - p) T d z with d z ~ 1e-6: rows that agree on the token agree on p to 1e-5 T of the largest p
    assert err <= 1e-5 * max(T, 1.0) * float(p0.max()) + 1e-12, err
    assert float((p1.sum(-1) - 1).abs().max()) < 1e-4


# ---- fused dz kernel (dz_fused_tcgen05.cu): D-embedding input gradient + tempered-softmax backward + db_out ------------
def _adv_grads(fused_dz, B, L, V, E, H, T=1.0, expect=(), absent=(), options=None):
    import gic_b200
    from gic_b200 import _lib
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=V, gen_embed_dim=E, gen_hidden_dim=H, gen_num_layers=1, conditional_gan=0, device="cuda")
    torch.manual_seed(3)
    inst = GANInstructor(a, device="cuda:0")
    inst.gen.train(); inst.disc.train(); inst.gen.decoder.temperature = T
    g = torch.Generator(device="cuda:0").manual_seed(11)
    caps = torch.randint(4, V, (B, L), generator=g, device="cuda:0")
    u = torch.rand(L, B, V, generator=g, device="cuda:0")
    keep = (torch.rand(3, B * 64, 900, generator=g, device="cuda:0") >= 0.2).to(torch.uint8)
    inst._ctx.set_option("GIC_FUSED_DZ_BF16", 1 if fused_dz else 0)       # switches are per context: the instructor's own
    for k, v in (options or {}).items():
        inst._ctx.set_option(k, v)
    with _lib.expect_kernels(*expect, absent=absent):
        inst.adv_step(caps, u=u, keep=keep, update=False)
        torch.cuda.synchronize()
    return {k: inst._flat_g.g(p).clone() for k, p in inst.gen.named_parameters() if id(p) in inst._flat_g._index}


@pytest.mark.parametrize("B,L,V,E,H,T", [(24, 10, 1000, 64, 64, 1.0), (64, 12, 4000, 128, 256, 3.0)])
def test_fused_dz_matches_separate_kernels(B, L, V, E, H, T):
    """GIC_GEMM_BF16: the streaming dz kernel against GEMM + softmax-backward + column-sum kernels.  Both round the same
    fp32 dz to bf16, so every generator gradient agrees to summation order; db_out is summed from the fp32 values in the
    fused kernel (from the bf16 copy in the separate one) and agrees to bf16 rounding."""
    import gic_b200
    old = gic_b200.get_gemm_mode()
    gic_b200.set_gemm_mode(gic_b200.GEMM_BF16)
    try:
        g1 = _adv_grads(True, B, L, V, E, H, T, expect=("dz_fused_kernel",))
        g0 = _adv_grads(False, B, L, V, E, H, T, expect=("softmax_bwd_dot_bf16_kernel",), absent=("dz_fused_kernel",))
    finally:
        gic_b200.set_gemm_mode(old)
    for k in g0:
        scale = float(g0[k].abs().max())
        err = float((g1[k] - g0[k]).abs().max())
        REPORT[f"dz_fused/B{B}V{V}/{k}"] = dict(err=err, scale=scale, rel=err / max(scale, 1e-30))
        tol = 2e-2 if k.endswith("linear.bias") else 5e-3     # bf16 rounding flips of dz where dp - dot cancels
        assert err <= tol * scale + 1e-12, f"{k}: err {err:.3e} scale {scale:.3e}"


# ---- fused BPTT step (bptt_tcgen05.cu): recurrent contraction over a 4-CTA cluster + cell backward in one kernel ------
@pytest.mark.parametrize("B,L,V,E,H", [(256, 6, 1000, 512, 512), (200, 5, 1000, 64, 64), (130, 5, 1000, 128, 1024), (256, 20, 1000, 512, 512),
                                       (8, 5, 1000, 32, 512), (40, 5, 1000, 64, 128)])
def test_fused_bptt_step_matches_gemm_plus_cell_kernel(B, L, V, E, H):
    """TF32 mode with GIC_BPTT_FUSED=1 (split-K over a cluster, DSMEM reduction in rank order, cell backward in the
    epilogue) and =0 (stream-K GEMM + lstm_cell_bwd_kernel): same TF32 products, different association of the K sum, so
    every generator gradient agrees to fp32 round-off accumulated over the L steps."""
    import gic_b200
    old = gic_b200.get_gemm_mode()
    gic_b200.set_gemm_mode(gic_b200.GEMM_TF32)
    res = []
    try:
        # (persistent launch over all steps, per-step fused kernel) -> persistent / per-step fused / GEMM + cell kernel
        pers_ok = H <= 512                   # the persistent recurrence keeps a W_hh slice resident: H <= 512
        for pers, fused, want, gone in (
                ("1", "1", ("bptt_persistent_kernel",) if pers_ok else ("bptt_step_kernel",), ()),
                ("0", "1", ("bptt_step_kernel",), ("bptt_persistent_kernel",)),
                ("0", "0", ("lstm_cell_bwd_kernel",), ("bptt_persistent_kernel", "bptt_step_kernel"))):
            res.append(_adv_grads(True, B, L, V, E, H, 1.0, expect=want, absent=gone,
                                  options=dict(GIC_BPTT_PERSISTENT=int(pers), GIC_BPTT_FUSED=int(fused))))
    finally:
        gic_b200.set_gemm_mode(old)
    gp, g1, g0 = res
    for nm, gx in (("persistent", gp), ("step", g1)):
        for k in g0:
            scale = float(g0[k].abs().max())
            err = float((gx[k] - g0[k]).abs().max())
            REPORT[f"bptt_{nm}/B{B}H{H}/{k}"] = dict(err=err, scale=scale, rel=err / max(scale, 1e-30))
            assert err <= 2e-4 * scale + 1e-12, f"{nm} {k}: err {err:.3e} scale {scale:.3e}"


# ---- mma.sync conv + ReLU + max-pool forward (disc.cu, tensor-core modes) vs the CUDA-core kernel --------------------
def _a4(n):
    return (n + 3) & ~3


def _conv_pool_pair(N, L, V, fsz, nfl, seed=0, R=64):
    """gic_disc_fwd on hard token ids (the embedding gather is exact in every mode) in TF32 mode, once with the mma.sync
    conv kernel (bf16 hi/lo split) and once with GIC_CONV_MMA=0 (CUDA-core FFMA kernel): (pooled, arg, logits) of both."""
    import gic_b200
    from gic_b200 import _lib
    from gic_b200.discriminator import disc_fwd_raw
    d = dev()
    lib = _lib.lib()
    g = torch.Generator(device=d).manual_seed(seed)
    De, Fd, Hd = R, sum(nfl), 100
    u = lambda *s: (torch.rand(*s, generator=g, device=d) - 0.5) * 0.1
    W_e = u(De, V) * 10          # embedding values of order 0.5: conv outputs of order 0.1
    cw = [u(n, 1, f, 1).contiguous() for n, f in zip(nfl, fsz)]
    cb = [u(n) for n in nfl]
    W_h, b_h, W_f, b_f, W_o, b_o = u(Fd, Fd), u(Fd), u(Hd, Fd), u(Hd), u(1, Hd), u(1)
    ids = torch.randint(0, V, (N, L), generator=g, device=d)
    res = []
    for flag in ("1", "0"):
        want, gone = ("conv_pool_fwd_mma_kernel", "conv_pool_fwd_kernel") if flag == "1" else ("conv_pool_fwd_kernel", "conv_pool_fwd_mma_kernel")
        with _lib.options(GIC_CONV_MMA=int(flag)), _lib.expect_kernels(want, absent=(gone,)):
            logits, saved = disc_fwd_raw(lib, gic_b200.GEMM_TF32, None, ids, N, L, V, De, R, fsz, nfl, W_e, cw, cb, W_h, b_h,
                                         W_f, b_f, W_o, b_o, [None], 0.0, d)
            torch.cuda.synchronize()
        rows = N * R
        o = _a4(N * L * De)
        pooled = saved[o:o + rows * Fd].view(rows, Fd).clone()
        o2 = o + 2 * _a4(rows * Fd)
        arg = saved[o2:o2 + _a4((rows * Fd + 3) // 4)].view(torch.uint8)[:rows * Fd].view(rows, Fd).clone()
        res.append((pooled, arg, logits[0].clone()))
    return res


@pytest.mark.parametrize("N,L,V,fsz,nfl", [
    (8, 16, 1000, [3, 4, 5], [300, 300, 300]),      # c1 discriminator
    (64, 20, 2000, [3, 4, 5], [300, 300, 300]),     # c2 caption length, several captions per SM
    (5, 32, 500, [2, 3, 4, 5], [100, 52, 300, 20]), # c5 length; groups that are not multiples of 16 channels
    (3, 6, 200, [3, 5], [24, 40]),                  # short captions: T = 2 for the widest filter
    (2, 8, 300, [5, 1], [16, 36]),                  # f = 5 (all taps of a part) and f = 1
    (3, 34, 300, [3, 4, 5], [20, 16, 12]),          # T = 32 for the narrowest filter: the largest step the 5-bit tag holds
])
def test_conv_pool_mma_matches_cuda_core_kernel(N, L, V, fsz, nfl):
    (p1, a1, l1), (p0, a0, l0) = _conv_pool_pair(N, L, V, fsz, nfl)
    scale = float(p0.max())
    err = float((p1 - p0).abs().max())
    mism = int((a1 != a0).sum())
    nm = f"conv_pool_mma/N{N}L{L}F{sum(nfl)}"
    REPORT[nm] = dict(err=err, scale=scale, rel=err / scale, arg_mismatches=mism, n=int(a0.numel()))
    # bf16 hi/lo split of both operands: ~2^-16 relative per operand (the TF32 contractions of these modes carry 2^-11)
    assert err <= 5e-5 * scale + 1e-7, f"pooled differs by {err:.3e} (scale {scale:.3e})"
    # the arg-max (routing of the gradient) may differ only where two time steps tie at that level
    assert mism <= max(2, int(1e-3 * a0.numel())), f"{mism} of {a0.numel()} arg-max indices differ"
    assert bool(((a1 == 255) == (a0 == 255)).all() or mism > 0)
    lerr = float((l1 - l0).abs().max())
    assert lerr <= 2e-4 * float(l0.abs().max()) + 1e-6
