"""CPU-side checks: the C-ABI library loads and exports every declared symbol, host logic (flat buffers,
argument surface, temperature schedule) works, and the product path fails loudly without CUDA."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge
    ge.build()
    import gic_b200
    return gic_b200


def test_library_exports_every_header_symbol(built):
    from gic_b200 import _lib
    L = _lib.lib()
    syms = _lib.header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), s
    assert L.gic_version() >= 100
    # size helpers are pure host functions
    assert L.gic_decode_saved_floats(4, 8, 16, 32, 1) > 0
    assert L.gic_disc_saved_floats(4, 8, 64, 64, 72) > 0


def test_sass_is_sm100a_only(built):
    from gic_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out


def test_no_cpu_fallback(built):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from gic_b200 import _lib
    from gic_b200.utils import get_losses
    x = torch.zeros(4)
    with pytest.raises(_lib.GicError):
        get_losses(x, x, x, "standard")
    import gic_b200.discriminator as D
    from gic_b200.args import default_args
    disc = D.Discriminator(default_args(vocab_size=20, disc_num_filters=[4, 4, 4]))
    with pytest.raises(_lib.GicError):
        disc(torch.rand(2, 8, 20))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "gan-image-captioning_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            src = open(os.path.join(pkg, f)).read()
            assert "oracle" not in src.replace("oracle/", ""), f


def test_each_compute_entry_point_has_one_call_site():
    """Every C ABI call that takes a stream is spelled out once in the package: the autograd modules and the fused steps
    share one binding per entry point instead of repeating its ctypes argument list."""
    import re
    header = open(os.path.join(ROOT, "include", "gic_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    names = [m.group(1) for m in re.finditer(r"\b(gic_[a-z0-9_]+)\s*\(([^;{]*)\)\s*;", header)
             if "gic_stream_t" in m.group(2)]
    assert len(names) >= 30
    pkg = os.path.join(ROOT, "gan-image-captioning_b200")
    lines = [line for f in sorted(os.listdir(pkg)) if f.endswith(".py")
             for line in open(os.path.join(pkg, f)).read().splitlines()]
    many = {n: c for n in names if (c := sum(("." + n + "(") in line for line in lines)) > 1}
    assert not many, many


def test_args_surface_matches_reference_defaults(built):
    from gic_b200.args import default_args, get_args
    a = get_args([])
    assert (a.gen_hidden_dim, a.gen_embed_dim, a.gen_num_layers) == (512, 32, 1)
    assert (a.disc_embed_dim, a.disc_num_rep) == (64, 64)
    assert a.disc_filter_sizes == [3, 4, 5] and a.disc_num_filters == [300, 300, 300]
    assert a.temperature == 100 and a.temp_adpt == "exp" and a.clip_norm == 5.0
    assert a.adv_loss_type == "standard" and a.gen_lr == 1e-4 and a.disc_lr == 1e-4
    b = get_args(["--gen-embed-dim", "512", "--gen-num-layers", "2", "--disc-filter-sizes", "2,3,4"])
    assert b.gen_embed_dim == 512 and b.gen_num_layers == 2 and b.disc_filter_sizes == [2, 3, 4]
    with pytest.raises(AttributeError):
        default_args(nope=1)


def test_state_dict_keys_match_reference(built):
    import gic_b200.discriminator as D
    import gic_b200.generator as G
    from gic_b200.args import default_args
    from oracle import ref_port as rp
    a = default_args(vocab_size=40, gen_num_layers=2, disc_num_filters=[5, 6, 7], conditional_gan=1)
    gen, disc = G.Generator(a), D.Discriminator(a)
    gk = set(gen.state_dict())
    for k, shape in rp.gen_param_shapes(a):
        assert k in gk and tuple(gen.state_dict()[k].shape) == shape, k
    assert {k for k, _ in rp.disc_param_shapes(a)} == set(disc.state_dict())
    for p in list(gen.parameters()) + list(disc.parameters()):
        if p.dim() > 0:
            assert float(p.detach().min()) >= -0.05 - 1e-7 and float(p.detach().max()) <= 0.05 + 1e-7   # init_params, Q6 (fp32(0.05) rounds outward)


def test_temperature_schedule_matches_oracle(built):
    from gic_b200.utils import get_fixed_temperature
    from oracle import ref_port as rp
    for adapt in ("no", "lin", "exp", "log", "sigmoid", "quad", "sqrt"):
        for i in (0, 1, 7.5, 29):
            assert get_fixed_temperature(100, i, 30, adapt) == rp.get_fixed_temperature(100, i, 30, adapt)
    with pytest.raises(Exception):
        get_fixed_temperature(100, 1, 30, "bogus")


def test_flat_params_views(built):
    from gic_b200.training import FlatParams
    ps = [torch.nn.Parameter(torch.randn(3, 5)), torch.nn.Parameter(torch.randn(7)), torch.nn.Parameter(torch.randn(2, 2))]
    vals = [p.detach().clone() for p in ps]
    fp = FlatParams(ps, "cpu")
    assert fp.homed() and fp.n % 4 == 0
    for p, v in zip(ps, vals):
        assert torch.equal(p.detach(), v)
    fp.flat.mul_(2.0)
    for p, v in zip(ps, vals):
        assert torch.equal(p.detach(), 2 * v)          # params are views of the flat buffer
    fp.g(ps[1]).fill_(1.0)
    assert float(fp.grad.sum()) == 7.0


def test_checkpoint_formats_and_resume_state_roundtrip(tmp_path):
    """src/training.py:118 (pretrained_model.ckpt = generator state_dict) and :225-226 (adv_model.ckpt =
    {"generator", "discriminator"}) keep their formats; the extra "gic_resume" key restores Adam moments per parameter
    name, step counts, temperature and counters.  Host logic only (no kernels run)."""
    import torch
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=50, gen_embed_dim=8, gen_hidden_dim=16, disc_num_filters=[4, 4, 4], conditional_gan=1,
                     feature_dim=12, device="cpu")
    torch.manual_seed(0)
    inst = GANInstructor(a, device="cpu")
    inst._ensure_flat()
    for fp in (inst._flat_g, inst._flat_d):
        fp.m.uniform_(-1, 1); fp.v.uniform_(0, 1); fp.step = 7
    inst._flat_g.m_pre, inst._flat_g.v_pre, inst._flat_g.step_pre = torch.rand_like(inst._flat_g.m), torch.rand_like(inst._flat_g.v), 3
    inst.gen.decoder.temperature, inst.adv_epoch, inst.gen_steps, inst.disc_steps, inst.pretrain_steps = 12.5, 4, 40, 41, 2
    adv, pre = str(tmp_path / "adv_model.ckpt"), str(tmp_path / "pretrained_model.ckpt")
    inst.save_checkpoint(adv); inst.save_pretrained(pre)
    # reference-side readers: plain dicts of tensors with the reference's keys
    blob = torch.load(adv, map_location="cpu", weights_only=False)
    assert set(blob) == {"generator", "discriminator", "gic_resume"}
    assert "decoder.lstm.weight_ih_l0" in blob["generator"] and "highway.weight" in blob["discriminator"]
    assert "decoder.embed.weight" in torch.load(pre, map_location="cpu", weights_only=False)
    torch.manual_seed(1)
    other = GANInstructor(a, device="cpu")
    assert other.load_checkpoint(adv) is True
    for k, v in inst.gen.state_dict().items():
        assert torch.equal(other.gen.state_dict()[k], v), k
    for k, v in inst.disc.state_dict().items():
        assert torch.equal(other.disc.state_dict()[k], v), k
    assert other._flat_g.homed() and other._flat_d.homed()            # parameters are still views of the flat buffers
    for f0, f1 in ((inst._flat_g, other._flat_g), (inst._flat_d, other._flat_d)):
        assert f0.step == f1.step == 7
        for o, n in zip(f0.offsets, f0.sizes):                         # (the 16-byte alignment gaps between tensors carry no state)
            assert torch.equal(f0.m[o:o + n], f1.m[o:o + n]) and torch.equal(f0.v[o:o + n], f1.v[o:o + n])
            assert torch.equal(f0.flat[o:o + n], f1.flat[o:o + n])
    for o, n in zip(inst._flat_g.offsets, inst._flat_g.sizes):
        assert torch.equal(inst._flat_g.m_pre[o:o + n], other._flat_g.m_pre[o:o + n])
    assert other._flat_g.step_pre == 3
    assert other.gen.decoder.temperature == 12.5 and (other.adv_epoch, other.gen_steps, other.disc_steps, other.pretrain_steps) == (4, 40, 41, 2)
    third = GANInstructor(a, device="cpu")
    assert third.load_checkpoint(pre) is False                       # weights only: no optimizer state in that format
    assert torch.equal(third.gen.state_dict()["decoder.linear.weight"], inst.gen.state_dict()["decoder.linear.weight"])


def test_reference_written_checkpoint_round_trip(tmp_path):
    """A file written by the REFERENCE (Generator.state_dict() always carries the frozen ResNet trunk as
    encoder.resnet.*, src/generator.py:12-14, and BatchNorm's running statistics) loads with strict=True: the trunk's
    tensors are set aside, everything else lands in our modules; saving writes them back, so the file can return to the
    reference.  weights_only loading is the default."""
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=30, gen_embed_dim=8, gen_hidden_dim=16, disc_num_filters=[4, 4, 4], conditional_gan=1,
                     feature_dim=12, device="cpu")
    torch.manual_seed(3)
    src = GANInstructor(a, device="cpu")
    ref_sd = {k: v.clone() for k, v in src.gen.state_dict().items()}
    ref_sd["encoder.bn.running_mean"] = torch.full_like(ref_sd["encoder.bn.running_mean"], 0.25)
    ref_sd["encoder.bn.num_batches_tracked"] = torch.tensor(11)
    trunk = {"encoder.resnet.0.weight": torch.randn(4, 3, 3, 3), "encoder.resnet.1.running_var": torch.rand(4)}
    ref_sd.update(trunk)
    path = str(tmp_path / "ref_adv_model.ckpt")
    torch.save({"generator": ref_sd, "discriminator": src.disc.state_dict()}, path)       # src/training.py:225-226
    inst = GANInstructor(a, device="cpu")
    assert inst.load_checkpoint(path, strict=True) is False
    assert float(inst.gen.encoder.bn.running_mean[0]) == 0.25 and int(inst.gen.encoder.bn.num_batches_tracked) == 11
    out = str(tmp_path / "ours.ckpt")
    inst.save_checkpoint(out)
    back = torch.load(out, map_location="cpu", weights_only=True)["generator"]
    assert set(back) == set(ref_sd)
    for k, v in trunk.items():
        assert torch.equal(back[k], v)
    inst.save_pretrained(str(tmp_path / "pre.ckpt"))
    assert set(torch.load(str(tmp_path / "pre.ckpt"), map_location="cpu", weights_only=True)) == set(ref_sd)


def test_rehoming_parameters_keeps_adam_state_and_drops_graphs():
    """gen.to() / .float() / load_state_dict(assign=True) move parameters out of the flat buffers: the rebuilt flat
    buffers must carry the Adam moments and step counts over, and captured graphs (which address the old buffers) go."""
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=30, gen_embed_dim=8, gen_hidden_dim=16, disc_num_filters=[4, 4, 4], device="cpu")
    inst = GANInstructor(a, device="cpu")
    inst._ensure_flat()
    fg = inst._flat_g
    fg.m.uniform_(-1, 1); fg.v.uniform_(0, 1); fg.step = 5
    fg.m_pre, fg.v_pre, fg.step_pre = torch.rand_like(fg.m), torch.rand_like(fg.v), 2
    w = inst.gen.decoder.linear.weight
    o, n = fg.offsets[fg._index[id(w)]], w.numel()
    m_w, mp_w = fg.m[o:o + n].clone(), fg.m_pre[o:o + n].clone()
    inst._graphs["stale"] = object()
    w.data = w.data.clone()                      # re-homed: no longer a view of the flat buffer
    assert not fg.homed()
    inst._ensure_flat()
    f2 = inst._flat_g
    assert f2 is not fg and f2.homed() and f2.step == 5 and f2.step_pre == 2 and not inst._graphs
    o2 = f2.offsets[f2._index[id(w)]]
    assert torch.equal(f2.m[o2:o2 + n], m_w) and torch.equal(f2.m_pre[o2:o2 + n], mp_w)
    assert f2.n_early == f2.offsets[2]


def test_library_side_rng_offsets_differ_per_rank():
    """Data-parallel ranks are seeded identically (main.py seeds 1008 everywhere so the weights agree); the Philox offset
    of the library-side draws carries the rank, so two ranks never share a (seed, offset) pair."""
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=30, gen_embed_dim=8, gen_hidden_dim=16, disc_num_filters=[4, 4, 4], device="cpu")
    torch.manual_seed(1008)
    r0, r1 = GANInstructor(a, device="cpu"), GANInstructor(a, device="cpu")
    r1.rank = 1
    offs0 = [r0._next_rng_offset() for _ in range(4)]
    offs1 = [r1._next_rng_offset() for _ in range(4)]
    assert r0._rng_seed == r1._rng_seed
    assert not set(offs0) & set(offs1)
    assert [o & ((1 << 40) - 1) for o in offs1] == [1, 2, 3, 4] and all(o >> 40 == 1 for o in offs1)


def test_kernel_launch_counters_are_exported(built):
    from gic_b200 import _lib
    assert _lib.kernel_launches("vocab_sample_kernel") == 0      # nothing can launch without a GPU
    assert _lib.kernel_counts() == {} or all(v >= 0 for v in _lib.kernel_counts().values())
    with pytest.raises(AssertionError):
        with _lib.expect_kernels("vocab_sample_kernel"):
            pass


def test_contexts_isolate_the_setters(built):
    """The temperature pointer / prepared weights / Philox state / event hook live in a context; a thread's current context
    is its own.  (Host-side bookkeeping only: nothing is launched.)"""
    import threading
    from gic_b200 import _lib
    L = _lib.lib()
    a, b = _lib.Context(), _lib.Context()
    assert a.handle and b.handle and a.handle != b.handle
    with a:
        L.gic_set_rng(11, 22, None)
        with b:                                       # nested: b is current, a's state untouched
            L.gic_set_rng(33, 44, None)
        prev = L.gic_ctx_set_current(a.handle)        # already current: returns a
        assert prev == a.handle
    assert L.gic_ctx_set_current(None) in (None, 0)   # outside every `with`: the thread's default was current
    seen = {}

    def other():
        seen["prev"] = L.gic_ctx_set_current(b.handle)    # a fresh thread starts on ITS default, whatever the main thread did
        L.gic_ctx_set_current(None)
    with a:
        t = threading.Thread(target=other); t.start(); t.join()
    assert seen["prev"] in (None, 0)
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    args = default_args(vocab_size=30, gen_embed_dim=8, gen_hidden_dim=16, disc_num_filters=[4, 4, 4], device="cpu")
    i1, i2 = GANInstructor(args, device="cpu"), GANInstructor(args, device="cpu")
    assert i1._ctx.handle != i2._ctx.handle


def test_context_options_are_per_context_and_read_environment_once(monkeypatch):
    """Kernel-variant switches live in the library context (include/gic_b200.h gic_ctx_set_option): set > environment (read
    once per context) > built-in default; another context does not see them."""
    from gic_b200 import _lib
    monkeypatch.setenv("GIC_TEST_OPT_A", "7")
    a, b = _lib.Context(), _lib.Context()
    assert a.get_option("GIC_TEST_OPT_A", 1) == 7              # from the environment, first lookup
    monkeypatch.setenv("GIC_TEST_OPT_A", "9")
    assert a.get_option("GIC_TEST_OPT_A", 1) == 7              # remembered: a later setenv does not re-route context a
    assert b.get_option("GIC_TEST_OPT_A", 1) == 9              # context b looks for the first time now
    a.set_option("GIC_TEST_OPT_A", 3)
    assert a.get_option("GIC_TEST_OPT_A", 1) == 3 and b.get_option("GIC_TEST_OPT_A", 1) == 9
    a.clear_option("GIC_TEST_OPT_A")
    assert a.get_option("GIC_TEST_OPT_A", 1) == 9              # cleared: the environment again
    monkeypatch.delenv("GIC_TEST_OPT_A")
    assert _lib.Context().get_option("GIC_TEST_OPT_A", 5) == 5   # neither set nor in the environment: the default
    with a, _lib.options(GIC_TEST_OPT_B=0):
        assert _lib.get_option("GIC_TEST_OPT_B", 1) == 0
    assert a.get_option("GIC_TEST_OPT_B", 1) == 1
    with pytest.raises(_lib.GicError):
        _lib.set_option("X" * 40, 1)


def test_trap_info_is_empty_when_nothing_trapped():
    from gic_b200 import _lib
    assert _lib.trap_info() is None


def test_generator_gradient_buckets_follow_the_order_the_backward_finishes_them():
    """Data parallel (DESIGN.md section 6): the flat generator gradient leaves in three contiguous buckets -- [linear.weight |
    linear.bias] (final before the BPTT tail), [embed.weight] (formed before the weight-gradient GEMMs), the rest -- so the
    flat layout has to start with exactly those tensors, each bucket 16-byte aligned."""
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    a = default_args(vocab_size=30, gen_embed_dim=8, gen_hidden_dim=16, disc_num_filters=[4, 4, 4], device="cpu", conditional_gan=1,
                     feature_dim=12)
    inst = GANInstructor(a, device="cpu")
    inst._ensure_flat()
    fg, dec = inst._flat_g, inst.gen.decoder
    assert fg.params[0] is dec.linear.weight and fg.params[1] is dec.linear.bias and fg.params[2] is dec.embed.weight
    assert fg.n_early == fg.offsets[2] and fg.n_mid == fg.offsets[3]
    assert 0 < fg.n_early < fg.n_mid < fg.n
    assert fg.n_early % 4 == 0 and fg.n_mid % 4 == 0 and fg.n % 4 == 0
    assert fg.n_mid - fg.n_early >= dec.embed.weight.numel()
    # the views the backward writes into are the slices the buckets cover
    assert fg.g(dec.embed.weight).data_ptr() == fg.grad.data_ptr() + 4 * fg.n_early
    assert fg.g(dec.lstm_params()[0]).data_ptr() == fg.grad.data_ptr() + 4 * fg.n_mid
