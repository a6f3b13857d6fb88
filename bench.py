#!/usr/bin/env python
"""Benchmark of the adversarial-captioning hot path (BASELINE.json: adversarial train steps/s and sampled
caption tokens/s at 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores

A "step" is one full adversarial train step (src/training.py:136-169) on the COCO-shaped workload
(BASELINE.json configs[1], Tier-A shape): per GPU batch 256, caption length 20, vocab 10 000, E = H = 512,
2048-d pooled CNN features through Encoder.linear+bn, discriminator with 64 representations and 3x300
filters, loss 'standard', clip 5.0, Adam.  Data parallel = weak scaling: every rank owns 256 rows and the
flat G/D gradients are all-reduced before the clip.

Prints ONE JSON line (rank 0).  `value` = steps/s with every input already resident in HBM (two input sets
of 250 MB alternate, each larger than L2); `e2e` = the same step through GANInstructor.adv_step with the
user-facing inputs (captions, pooled features) copied from pinned host memory every step, the uniforms and
dropout masks drawn on-device as the reference does (src/generator.py:90, nn.Dropout), and the two losses
read back to the host.  Beside them, in the same line:
  modes       the same step in the other precision modes (tf32, exact fp32) -- the fp32 mode is the one that meets the
              fp32 parity bar on the reference's golden vectors; the headline mode is held to the bar stated for it
  sustained   the headline step replayed for >= 1 s (hundreds of steps): the long-run regime, with its own clock record
  roofline    the FLOP-dominant kernel class (discriminator GEMMs) and `time_dominant`, the fused decode step
  workloads   BASELINE.json's other configs: c2a (attention over the 7x7x2048 grid), c3 (Monte-Carlo rollouts),
              c4 (hidden 1024, vocab 30k: one GPU's 128 rows), c5 (discriminator-only, 4096 + 4096 captions of length 32)
  comm        (N > 1) exposed milliseconds of the gradient exchange, its transport, and whether the replicas are bit-identical

--dump-outputs DIR writes what the last timed step computed (see dump_outputs) so that two builds can be compared output for
output: the inputs and the weights are seeded, so the same arguments give the same inputs on every run.  The step itself
is not bit-reproducible (two runs of one build differ in the last bits, and the Adam updates carry that over the steps
before the dumped one), so compare with a tolerance.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True                   # the benchmark leaves the tree it runs from as it found it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1] (Tier-A: mean-pooled 7x7x2048 grid -> 2048-d feature)
    "c2": dict(B=256, L=20, V=10000, E=512, H=512, layers=1, feat=2048, filters=[300, 300, 300]),
    # the same with additive attention over the [B, 49, 2048] grid in every decode step (north-star extension B1)
    "c2a": dict(B=256, L=20, V=10000, E=512, H=512, layers=1, feat=2048, filters=[300, 300, 300]),
    # BASELINE.json configs[0] (args.py defaults; CPU-runnable)
    "c1": dict(B=8, L=16, V=1000, E=32, H=512, layers=1, feat=2048, filters=[300, 300, 300]),
    # BASELINE.json configs[2]: SeqGAN-style reward, 128 captions x 16 rollouts per prefix (secondary line: --workload c3)
    "c3": dict(B=128, L=20, V=10000, E=512, H=512, layers=1, feat=0, filters=[300, 300, 300], n_roll=16),
    # BASELINE.json configs[3]: scaled decoder (hidden 1024, vocab 30k, global batch 1024 over 8 GPUs = 128 rows per GPU; --workload c4)
    "c4": dict(B=128, L=20, V=30000, E=512, H=1024, layers=1, feat=2048, filters=[300, 300, 300]),
    # BASELINE.json configs[4]: discriminator-only step, 4096 real + 4096 fake captions of length 32 (--workload c5)
    "c5": dict(B=4096, L=32, V=10000, E=512, H=512, layers=1, feat=0, filters=[300, 300, 300]),
}
MODES = {"fp32": 0, "tf32": 1, "bf16": 3}
DTYPE_NAME = {"fp32": "f32", "tf32": "tf32 (fp32 accumulate)", 
              "bf16": "bf16 operands on the discriminator's highway/dx/dW_h contractions, tf32 on the others (fp32 accumulate)"}


def load_peaks():
    """tf_burst: dense bf16 for a kernel timed ALONE (short, boost clocks); tf: the sustained figure for a kernel timed
    inside a long step (the profiling recipe's distinction)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d.get("hbm_gbs", 6650.0), tf=d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)),
                    tf_burst=d.get("bf16_tflops", 1590.0), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf=1400.0, tf_burst=1590.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


DUMP_BYTES = 64 << 20


def dump_outputs(path, out, modules):
    """--dump-outputs: one step's results as <path>/<name>.npy -- every tensor of the dict the step returned, under its key,
    and the state of each model after the step (the updated weights and buffers) as <tag>.<state_dict key>.  Floating
    tensors are written in float32 (float64 stays float64), integer ones in float64, which holds them exactly.  When the
    whole set would exceed DUMP_BYTES, every array of more than `cap` entries is replaced by `cap` of its flattened
    entries, drawn with a fixed seed: the same entries on every run, so that two builds compare entry for entry."""
    import numpy as np
    import torch
    arrays = {k: v.detach() for k, v in out.items() if isinstance(v, torch.Tensor)}
    for tag, m in modules.items():
        arrays.update({f"{tag}.{k}": v.detach() for k, v in m.state_dict().items()})
    wide = {k for k, v in arrays.items() if v.dtype == torch.float64 or not v.is_floating_point()}
    cap = 1 << 24
    while sum(min(v.numel(), cap) * (8 if k in wide else 4) for k, v in arrays.items()) > DUMP_BYTES:
        cap //= 2
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        if v.numel() > cap:
            idx = np.sort(np.random.default_rng(1008).choice(v.numel(), cap, replace=False))
            v = v.reshape(-1)[torch.from_numpy(idx).to(v.device)]
        np.save(os.path.join(path, k + ".npy"), (v.double() if k in wide else v.float()).cpu().numpy())
    print("bench: %d arrays of the last timed step written to %s (arrays of more than %d entries sampled)" % (len(arrays), path, cap),
          file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation (oracle port with the same torch library ops)
# ------------------------------------------------------------------------------------------------------
def cpu_reference_step_time(cfg, sample_B, steps, warmup, threads):
    """Seconds per step of the library-op CPU port (oracle/ref_modules.py: nn.LSTM / nn.Conv2d / autograd / optim.Adam, the
    ops the reference itself reaches on a CPU) on `sample_B` rows of the workload: the WHOLE step of src/training.py:144-169
    -- Encoder.linear + bn on the pooled features, Decoder.sample with its own uniform draws, F.one_hot, three discriminator
    passes with their own dropout masks, losses, both gradients, clip, both Adam steps."""
    import torch
    from oracle import ref_modules as rm
    from oracle import ref_port as rp
    torch.set_num_threads(threads)
    inp = rp.make_inputs(dict(cfg, B=sample_B))
    a = inp["args"]
    a.temperature = 1.0
    if cfg["feat"]:
        enc, dec, disc = rm.load_port(a, inp["gen"], inp["disc"], with_encoder=True)
        g_params = list(dec.parameters()) + list(enc.parameters())
    else:
        (dec, disc), enc = rm.load_port(a, inp["gen"], inp["disc"]), None
        g_params = list(dec.parameters())
    g_opt = torch.optim.Adam(g_params, lr=a.gen_lr)
    d_opt = torch.optim.Adam(disc.parameters(), lr=a.disc_lr)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        feats = None if enc is not None else dec.embed(torch.ones(sample_B, dtype=torch.long))
        rm.port_adv_step(a, dec, disc, g_opt, d_opt, inp["captions"], feats, enc=enc, pooled=inp["pooled"])   # draws u / dropout itself
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return statistics.median(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    sample_B = min(cfg["B"], args.cpu_sample_rows or cfg["B"])
    steps, warmup = args.steps, args.warmup
    t = cpu_reference_step_time(cfg, sample_B, steps, warmup, threads)
    scale = cfg["B"] / sample_B
    step_s = t * scale
    val = 1.0 / step_s
    sample = (f"the whole step (encoder projection, decode, 3 discriminator passes, both gradients, clip, 2 x Adam) on {sample_B} of "
              f"{cfg['B']} rows" + (f", time scaled x{scale:g}" if scale != 1 else "") + f"; {steps} timed + {warmup} warm-up steps, median; "
              f"{threads} host threads (oracle/ref_modules.py: torch library-op port of the reference path)")
    conf = workload_config(args, cfg, 1)          # the WORKLOAD is the GPU arm's (same keys, same values); how this arm runs it:
    impl_conf = {"arithmetic": "fp32 (torch CPU: MKL / oneDNN)", "memory": "host", "launch": "eager PyTorch on the host cores",
                 "rows_per_step": sample_B, "encoder_projection": bool(cfg["feat"]),
                 "parallelism": "1 CPU process, %d threads; the config's gemm_mode / cache / launch keys describe the GPU arm only, and "
                                "this arm does not scale with --gpus" % threads}
    line = {
        "impl": "reference", "metric": "adversarial_train_steps_per_sec", "value": val, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": conf, "impl_config": impl_conf,
        "tokens_per_sec": None,
        "cpu_baseline": {"value": val, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, cfg, world):
    return {"workload": f"{args.workload}: COCO-shaped adversarial step, per-GPU batch {cfg['B']}, len {cfg['L']}, "
                        f"vocab {cfg['V']}, E {cfg['E']}, H {cfg['H']}, feat {cfg['feat']} (pooled 7x7x2048 grid), "
                        f"D 64 reps x {sum(cfg['filters'])} filters, loss standard",
            "global_batch": cfg["B"] * world, "seq_len": cfg["L"], "vocab": cfg["V"], "parallelism": f"dp{world}",
            "gemm_mode": args.mode, "cache": "two 250 MB input sets alternate (each > 126 MB L2)",
            "launch": "eager" if args.no_graph else "one CUDA graph per step",
            "setup": "graph capture + %d settling replays (untimed) before the warm-up steps" % getattr(args, "settle", 0)}


# ------------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import gic_b200
    from gic_b200 import _lib
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    _lib.require_cuda()
    lib = _lib.lib()
    gic_b200.set_gemm_mode(MODES[args.mode])

    cfg = WORKLOADS[args.workload]
    B, L, V = cfg["B"], cfg["L"], cfg["V"]
    a = default_args(vocab_size=V, gen_embed_dim=cfg["E"], gen_hidden_dim=cfg["H"], gen_num_layers=cfg["layers"],
                     disc_num_filters=list(cfg["filters"]), conditional_gan=1, feature_dim=cfg["feat"], device="cuda")
    torch.manual_seed(1008)                      # identical weights on every rank (src/main.py:14-17)
    inst = GANInstructor(a, device=dev)
    inst.gen.train(); inst.disc.train()
    inst.gen.decoder.temperature = 1.0           # exp schedule start (reported config); T is a kernel argument
    R, Fd = a.disc_num_rep, sum(a.disc_num_filters)

    # synthetic inputs, sharded by batch row: rank r owns rows [r*B, (r+1)*B) of the global batch
    def make_set(seed):
        g = torch.Generator(device=dev).manual_seed(seed * 1000 + rank)
        caps = torch.randint(4, V, (B, L), generator=g, device=dev)
        caps[:, 0] = 1; caps[:, L - 1] = 2
        return dict(caps=caps, pooled=torch.randn(B, cfg["feat"], generator=g, device=dev),
                    u=torch.rand(L, B, V, generator=g, device=dev),
                    keep=(torch.rand(3, B * R, Fd, generator=g, device=dev) >= 0.2).to(torch.uint8))
    sets = [make_set(1008 + i) for i in range(2)]
    h_caps = [s["caps"].cpu().pin_memory() for s in sets]
    h_pool = [s["pooled"].cpu().pin_memory() for s in sets]

    use_graph = not args.no_graph
    last = {}

    def step_resident(i):
        s = sets[i % 2]
        last["out"] = inst.adv_step(s["caps"], pooled=s["pooled"], u=s["u"], keep=s["keep"], graph="static" if use_graph else False)
        return last["out"]

    # end to end: host buffers in, losses out.  Every step's two losses are copied to pinned host memory and READ on the host;
    # the read of step i happens while step i + 1 runs (one step of pipelining: the host never idles the GPU to fetch a number
    # it only logs -- the reference's own loop blocks on .item() four times per step, src/training.py:177-181)
    host_loss = [torch.zeros(2).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    loss_log = []
    pending = [None]

    def drain():
        if pending[0] is not None:
            loss_ev[pending[0]].synchronize()
            loss_log.append((float(host_loss[pending[0]][0]), float(host_loss[pending[0]][1])))
            pending[0] = None

    def step_e2e(i):
        # with the graph the H2D copies land in the graph's static input buffers
        if use_graph:
            r = inst.adv_step(h_caps[i % 2], pooled=h_pool[i % 2], graph=True)
        else:
            caps = h_caps[i % 2].to(dev, non_blocking=True)
            pooled = h_pool[i % 2].to(dev, non_blocking=True)
            r = inst.adv_step(caps, pooled=pooled)                     # uniforms / masks drawn on-device
        k = i % 2
        host_loss[k].copy_(torch.stack([r["g_loss"], r["d_loss"]]), non_blocking=True)      # D2H of the step's result
        loss_ev[k].record()
        drain()                                                      # the PREVIOUS step's losses, read on the host now
        pending[0] = k

    def timed(fn, steps, warmup, sample_clocks=False, finalize=None):
        for i in range(warmup):
            fn(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()
        n0 = lib.gic_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        if finalize is not None:
            finalize()                       # e.g. the host read of the last step's result: inside the timed region
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        launches = lib.gic_launch_count() - n0
        if use_graph and launches == 0:
            launches = steps * getattr(inst, "graph_launches_per_step", 0)     # kernels replayed from the captured step
        clocks = sampler.stop() if sampler else None
        if world > 1:
            dist.barrier()
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, clocks

    # set-up (untimed, before the W warm-up steps): the first call per input set runs one eager step and captures the graph;
    # a few replays then let the uploaded graphs, the caches and the clocks settle (20 steps are 45 ms of GPU time in all)
    for i in range(2 + args.settle):
        step_resident(i)
    torch.cuda.synchronize()
    ms, launches, clocks = timed(step_resident, args.steps, args.warmup, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["out"], {"gen": inst.gen, "disc": inst.disc})
    ms_step = ms / args.steps
    value = world / (ms_step * 1e-3)             # global steps/s: every rank completes one 256-row step per iteration

    # sampled-caption tokens/s: decode only (Decoder.sample), device resident
    dec = inst.gen.decoder

    def decode_only(i):
        s = sets[i % 2]
        feats = inst.gen.encoder(s["pooled"])
        with torch.no_grad():
            return dec.sample(feats, max_caption_len=L, u=s["u"])
    # Decoder.sample replayed as a CUDA graph per input set (the public call is dec.sample; the graph removes the host's
    # ~60 launches per caption batch from the critical path exactly as the step graph does)
    dec_graphs = []
    with torch.no_grad():
        for i in range(2):
            decode_only(i); torch.cuda.synchronize()
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph):
                decode_only(i)
            dec_graphs.append(gph)
        if args.no_graph:
            dms, _, _ = timed(decode_only, args.steps, args.warmup)
        else:
            dms, _, _ = timed(lambda i: dec_graphs[i % 2].replay(), args.steps, args.warmup)
    tokens_per_sec = world * B * L / (dms / args.steps * 1e-3)

    for i in range(2 + args.settle):
        step_e2e(i)
    drain()
    torch.cuda.synchronize()
    e2e_ms, _, _ = timed(step_e2e, args.steps, args.warmup, finalize=drain)     # the last step's losses are read inside the timed region too
    e2e_val = world / (e2e_ms / args.steps * 1e-3)
    e2e_losses_read = len(loss_log)
    h2d = h_caps[0].numel() * 8 + h_pool[0].numel() * 4

    # ---- the long-run regime: the same resident step for >= ~1 s (the K timed steps above last ~50 ms: boost clocks)
    sustained = None
    if not args.no_sustained:
        n_long = int(min(2000, max(200, 1.0 / (ms_step * 1e-3))))
        # chunks of 50 steps with an event between them and the host's enqueue time beside them: tells a GPU that slows down
        # from a host that cannot enqueue a replay per step time
        sampler = ClockSampler(local) if rank == 0 else None
        for i in range(3):
            step_resident(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        if sampler:
            sampler.start()
        evs = [torch.cuda.Event(enable_timing=True)]
        evs[0].record()
        h0 = time.perf_counter()
        for i in range(n_long):
            step_resident(3 + i)
            if (i + 1) % 50 == 0 or i + 1 == n_long:
                e = torch.cuda.Event(enable_timing=True); e.record(); evs.append(e)
        host_ms = (time.perf_counter() - h0) * 1e3
        torch.cuda.synchronize()
        lclocks = sampler.stop() if sampler else None
        lms = evs[0].elapsed_time(evs[-1])
        if world > 1:
            t = torch.tensor([lms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); lms = float(t.item())
        chunks = [evs[j].elapsed_time(evs[j + 1]) / min(50, n_long - 50 * j) for j in range(len(evs) - 1)]
        sustained = {"steps": n_long, "ms_per_step": lms / n_long, "value": world / (lms / n_long * 1e-3), "unit": "steps/s",
                     "ms_per_step_first_50": chunks[0], "ms_per_step_last_50": chunks[-1],
                     "host_enqueue_ms_per_step": host_ms / n_long, "clocks": lclocks}

    # ---- exposed cost of the gradient exchange (N > 1): the same step with the all-reduce left out
    comm = None
    if world > 1:
        # after identical updates from identical reduced gradients the replicas must be bit-identical (checked BEFORE the
        # no-exchange run below, which lets every rank follow its own shard's gradient)
        flat = torch.cat([inst._flat_g.flat, inst._flat_d.flat])
        ref0 = flat.clone(); dist.broadcast(ref0, 0)
        same = torch.tensor([1.0 if torch.equal(ref0, flat) else 0.0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        inst.skip_allreduce = True
        inst._graphs.clear()
        nms, _, _ = timed(step_resident, args.steps, args.warmup)
        inst.skip_allreduce = False
        inst._graphs.clear()
        for fp in (inst._flat_g, inst._flat_d):          # back to identical replicas: rank 0's parameters and Adam moments
            for t in (fp.flat, fp.m, fp.v):
                dist.broadcast(t, 0)
        for i in range(3):
            step_resident(i)                 # re-capture the real step (the later measurements replay it)
        torch.cuda.synchronize()
        nbytes = 4 * (inst._flat_g.n + inst._flat_d.n)
        peer = inst._peer is not None
        comm = {"comm_ms_exposed": ms_step - nms / args.steps, "ms_per_step_without_exchange": nms / args.steps,
                "allreduce_bytes_per_step": nbytes,
                "transport": ("gic_allreduce: one kernel over NVLink peer memory (reduce-scatter + all-gather in rank order, fused square norm)"
                              if peer else "torch.distributed all_reduce (NCCL)"),
                "replicas_bit_identical": bool(same.item() > 0.5),
                "peer_wait_expired": bool(inst._peer.error()) if peer else None}

    # ---- the other precision modes on the same workload (device-resident value and e2e)
    modes = {args.mode: {"value": value, "ms_per_step": ms_step, "e2e": e2e_val, "dtype": DTYPE_NAME[args.mode]}}
    if not args.no_modes:
        for m in ("bf16", "tf32", "fp32"):
            if m in modes:
                continue
            gic_b200.set_gemm_mode(MODES[m])
            k = max(3, min(args.steps, 10 if m != "fp32" else 5))
            mms, _, _ = timed(step_resident, k, 3)
            ems, _, _ = timed(step_e2e, k, 3, finalize=drain)
            modes[m] = {"value": world / (mms / k * 1e-3), "ms_per_step": mms / k, "e2e": world / (ems / k * 1e-3), "steps": k,
                        "dtype": DTYPE_NAME[m]}
        gic_b200.set_gemm_mode(MODES[args.mode])
        modes["parity"] = ("fp32: ids bit-exact, rtol 1e-3 vs the reference's golden vectors (tests/test_gpu_parity.py); tf32 / bf16: "
                           "stated separately, oracle-checked at MID / c2 / c4 / c5 shapes with classified token mismatches "
                           "(tests/test_gpu_parity_modes.py)")

    # roofline of the dominant kernel class: instrumented steps (events around every launch of the class)
    peaks = load_peaks()
    NK = 9
    K = C.c_double * NK
    ms_k, work_k, calls_k = K(), K(), (C.c_ulonglong * NK)()
    use_graph = False          # events around individual launches need the eager path
    psteps = min(args.steps, 3)
    names = ["gemm_other", "sample_step", "conv_pool_fwd", "softmax_bwd", "clip_adam", "head_fwd", "gemm_disc", "gemm_decode",
             "vocab_sample_fused"]

    def instrumented(overlap):
        """psteps eager steps with CUDA events around every launch of each kernel class (on the launching stream).
        overlap=True: the step's two streams run side by side as in the timed region, so a kernel's events also cover
        the time it shares the SMs with the other chain's kernels.  overlap=False: one stream, every kernel alone on the
        machine -- the duration that belongs to the kernel (and the one ncu's serialised launch list can be compared with)."""
        prev = inst.overlap
        inst.overlap = overlap
        try:
            step_resident(0); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            lib.gic_prof_begin()
            e0.record()
            for i in range(psteps):
                step_resident(i)
            e1.record()
            torch.cuda.synchronize()
            lib.gic_prof_end(ms_k, work_k, calls_k)
        finally:
            inst.overlap = prev
        out = {}
        for k, nm in enumerate(names):
            if calls_k[k]:
                out[nm] = dict(ms_per_step=ms_k[k] / psteps, calls_per_step=calls_k[k] / psteps, work_per_step=work_k[k] / psteps)
        return out, e0.elapsed_time(e1) / psteps

    classes_2s, _ = instrumented(True)
    classes, ms_serial = instrumented(False)
    # FLOP-dominant kernel class: the discriminator's [B*R, F] x [F, F] contractions (highway forward, dx, dW_h): 7 launches of
    # 2*B*R*F*F flop each (SURVEY.md 8d: 2*R*F^2 per caption).  `achieved` / `frac`: every launch timed ALONE on the machine
    # (eager, one stream) against the BURST bf16 peak -- that is what the measured-peaks file calls the figure for a kernel
    # timed alone; `in_step`: the same launches with the step's two streams side by side, against the SUSTAINED peak.
    g = classes.get("gemm_disc")
    roofline = None
    if g:
        traffic = None
        for tp in (os.path.join(ROOT, "profiles", "r2", "traffic.json"), os.path.join(ROOT, "profiles", "r1", "traffic.json")):
            if args.workload == "c2" and os.path.exists(tp):
                tj = json.load(open(tp)).get(args.mode)
                if tj:
                    traffic = tj["dram_bytes_read_per_launch"] + tj["dram_bytes_write_per_launch"]
                    break
        flops_launch = g["work_per_step"] / g["calls_per_step"]
        us_launch = g["ms_per_step"] * 1e3 / g["calls_per_step"]
        ach = flops_launch / (us_launch * 1e-6) / 1e12
        g2 = classes_2s.get("gemm_disc", g)
        us_launch_2s = g2["ms_per_step"] * 1e3 / g2["calls_per_step"]
        ach_2s = flops_launch / (us_launch_2s * 1e-6) / 1e12
        kname = ("gemm_pair_kernel (tcgen05 cta_group::2, M = 256: highway forward, dx) + gemm_p_kernel (persistent, stream-K: dW_h), "
                 "kind::f16 bf16 operands" if args.mode == "bf16" else "gemm_p_kernel (tcgen05 kind::tf32, persistent)")
        tf32_note = "" if args.mode == "bf16" else " (TF32 runs at half the bf16 rate)"
        roofline = {"kernel": (f"{kname}: discriminator highway / dx / dW_h, {B * R}x{Fd}x{Fd}") if args.mode != "fp32" else "sgemm_kernel (fp32 FFMA)",
                    "bound": "tensor", "achieved": ach, "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": ach / peaks["tf_burst"],
                    "traffic": traffic,
                    "peak_source": peaks["src"] + ": dense bf16 BURST (kernel timed alone)" + tf32_note,
                    "measured": "CUDA events around every launch of the class (on its own stream), eager steps on ONE stream: each kernel alone "
                                "on the machine, warm L2",
                    "share_of_step": g["ms_per_step"] / ms_serial, "serialised_step_ms": ms_serial,
                    "launches_per_step": g["calls_per_step"],
                    "algorithmic_flops_per_launch": flops_launch, "us_per_launch": us_launch,
                    "in_step": {"achieved": ach_2s, "peak": peaks["tf"], "frac": ach_2s / peaks["tf"], "us_per_launch": us_launch_2s,
                                "share_of_timed_step": g2["ms_per_step"] / ms_step,
                                "note": "the step's two streams side by side, as in the timed region; SUSTAINED bf16 peak"}}
        # time-dominant kernel: the fused decode step (one launch per sampled position).  It is a serial, latency-bound chain
        # (L launches that each wait for the previous token), so both of its rooflines are reported: HBM (8 B V bytes per launch:
        # read u, write p) and tensor (2 B V H + 2 B 4H H flop per launch).
        c = classes.get("vocab_sample_fused")
        if c:
            us_eager = c["ms_per_step"] * 1e3 / c["calls_per_step"]
            # per decode step inside the replayed graph (decode_ms covers L steps + the one-off EW GEMM and step-0 LSTM kernel):
            # the eager, event-bracketed figure also contains the host's tensor-map encoding between the two event records
            us = dms / args.steps * 1e3 / L
            by = 8.0 * B * V
            fl = 2.0 * B * V * cfg["H"] + 2.0 * B * 4 * cfg["H"] * cfg["H"]
            roofline["time_dominant"] = {
                "kernel": "vocab_sample_kernel in its fused-decode-step role (decode_step_kernel): projection + Gumbel-softmax + sample of "
                          "step t, recurrent contraction and LSTM cell of step t + 1; tcgen05 kind::tf32",
                "bound": "latency (serial chain); HBM and tensor figures for reference",
                "launches_per_step": c["calls_per_step"], "us_per_launch": us, "us_per_launch_eager_events": us_eager,
                "share_of_step": (dms / args.steps) / ms_step,
                "hbm": {"achieved": by / (us * 1e-6) / 1e9, "peak": peaks["hbm"], "unit": "GB/s", "frac": by / (us * 1e-6) / 1e9 / peaks["hbm"],
                        "algorithmic_bytes_per_launch": by},
                "tensor": {"achieved": fl / (us * 1e-6) / 1e12, "peak": peaks["tf_burst"] / 2, "unit": "TFLOP/s (TF32 = half the bf16 peak)",
                           "frac": fl / (us * 1e-6) / 1e12 / (peaks["tf_burst"] / 2), "algorithmic_flops_per_launch": fl},
                "decode_ms_graph_replay": dms / args.steps}
    tensor_classes = {}
    for nm in ("gemm_disc", "gemm_decode", "gemm_other"):
        c = classes.get(nm)
        if c:
            tf = c["work_per_step"] / (c["ms_per_step"] * 1e-3) / 1e12
            tensor_classes[nm] = {"achieved_TFLOPs": tf, "frac_of_bf16_burst_peak": tf / peaks["tf_burst"], "ms_per_step": c["ms_per_step"],
                                  "launches_per_step": c["calls_per_step"]}
    hbm = {}
    for nm in ("sample_step", "vocab_sample_fused", "conv_pool_fwd", "softmax_bwd", "clip_adam", "head_fwd"):
        c = classes.get(nm)
        if c:
            gbs = c["work_per_step"] / (c["ms_per_step"] * 1e-3) / 1e9
            hbm[nm] = {"achieved_GBps": gbs, "frac_of_hbm_peak": gbs / peaks["hbm"], "ms_per_step": c["ms_per_step"],
                       "launches_per_step": c["calls_per_step"]}

    # ---- BASELINE.json's other configs, each a short run on its own models (rank 0's GPU; N = 1 only)
    workloads = None
    if world == 1 and not args.no_workloads and args.workload == "c2":
        del sets, dec_graphs
        inst._graphs.clear()
        torch.cuda.empty_cache()
        workloads = {}
        for w in ("c2a", "c3", "c4", "c5"):
            try:
                workloads[w] = run_workload(w, args.mode, dev, peaks)
            except Exception as exc:            # a secondary workload must not take the headline line down
                workloads[w] = {"error": "%s: %s" % (type(exc).__name__, exc)}
            torch.cuda.empty_cache()

    def shutdown():
        """Release the captured graphs before tearing NCCL down; a watchdog ends the process if the teardown of a
        communicator that was captured into CUDA graphs does not return (observed with NCCL 2.28 + torch 2.11)."""
        if world <= 1:
            return
        inst._graphs.clear()
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        t = threading.Timer(15.0, lambda: os._exit(0))
        t.daemon = True
        t.start()
        dist.destroy_process_group()
        t.cancel()

    if rank != 0:
        shutdown()
        return

    # CPU baseline beside it (rank 0, N = 1 only): bounded sample of the same workload on the host cores
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        sb = min(B, args.cpu_sample_rows or B)
        t = cpu_reference_step_time(cfg, sb, 3, 1, threads)
        cpu = {"value": 1.0 / (t * B / sb), "unit": "steps/s", "cores": threads, "kind": "port",
               "sample": f"the whole step (encoder projection included) on {sb} of {B} rows" + (f", time scaled x{B / sb:g}" if sb != B else "") +
                         "; 3 timed + 1 warm-up steps, median (oracle/ref_modules.py: nn.LSTM / nn.Conv2d / autograd / optim.Adam port of the reference path)"}

    line = {
        "metric": "adversarial_train_steps_per_sec", "value": value, "unit": "steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": DTYPE_NAME[args.mode], "data": "synthetic",
        "config": workload_config(args, cfg, world),
        "value_definition": ("%d-row adversarial steps per second, summed over the %d ranks (weak scaling: every rank completes one "
                             "%d-row shard of a %d-row global step per iteration; global steps/s = value / n_gpus)"
                             % (B, world, B, B * world)) if world > 1 else "%d-row adversarial steps per second" % B,
        "tokens_per_sec": tokens_per_sec, "decode_ms": dms / args.steps,
        "e2e": {"value": e2e_val, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                "ms_per_step": e2e_ms / args.steps,
                "d2h": "both losses of every step copied to pinned memory and read on the host, one step behind the GPU "
                       "(%d reads for %d warm-up + timed steps)" % (e2e_losses_read, args.warmup + args.steps)},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "tensor_kernels": tensor_classes,
        "hbm_kernels": hbm, "modes": modes, "sustained": sustained, "comm": comm, "workloads": workloads,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)
    shutdown()


def run_workload(w, mode, dev, peaks, steps=None, world=1, rank=0, dump=None):
    """One of BASELINE.json's other configs on its own models: a dict for the `workloads` block of the headline line (or a
    line of its own with --workload).  Device-resident synthetic inputs, two input sets alternating, CUDA events.
    dump: directory for dump_outputs of the last timed step (rank 0)."""
    import torch
    import torch.distributed as dist
    import gic_b200
    from gic_b200.args import default_args
    from gic_b200.training import GANInstructor
    gic_b200.set_gemm_mode(MODES[mode])
    cfg = WORKLOADS[w]
    B, L, V, E, H = cfg["B"], cfg["L"], cfg["V"], cfg["E"], cfg["H"]
    R, Fd = 64, sum(cfg["filters"])
    cond = 1 if cfg["feat"] else 0
    a = default_args(vocab_size=V, gen_embed_dim=E, gen_hidden_dim=H, gen_num_layers=cfg["layers"], disc_num_filters=list(cfg["filters"]),
                     conditional_gan=cond, feature_dim=cfg["feat"] or 512, device="cuda", gen_attention=1 if w == "c2a" else 0)
    torch.manual_seed(1008)
    inst = GANInstructor(a, device=dev)
    inst.gen.train(); inst.disc.train(); inst.gen.decoder.temperature = 1.0
    g = torch.Generator(device=dev).manual_seed(1008 + rank)

    def caps_():
        c = torch.randint(4, V, (B, L), generator=g, device=dev); c[:, 0] = 1; c[:, L - 1] = 2
        return c
    out = {"config": {"workload": WORKLOAD_NOTES[w], **{k: v for k, v in cfg.items()}}, "dtype": DTYPE_NAME[mode], "data": "synthetic"}
    if w in ("c2a", "c4"):
        sets = []
        for i in range(2):
            d = dict(caps=caps_(), u=torch.rand(L, B, V, generator=g, device=dev),
                     keep=(torch.rand(3, B * R, Fd, generator=g, device=dev) >= 0.2).to(torch.uint8))
            if w == "c2a":
                d["grid"] = torch.randn(B, 49, 2048, generator=g, device=dev)
                d["pooled"] = d["grid"].mean(1)
            else:
                d["pooled"] = torch.randn(B, cfg["feat"], generator=g, device=dev)
            sets.append(d)
        fn = lambda i: inst.adv_step(sets[i % 2]["caps"], pooled=sets[i % 2]["pooled"], u=sets[i % 2]["u"], keep=sets[i % 2]["keep"],
                                     grid=sets[i % 2].get("grid"), graph="static")
        units, metric, unit = 1, "adversarial_train_steps_per_sec", "steps/s"
        k = steps or 10
        # decode contractions (gates 8 H (E + H) + vocab 2 H V flop per row-step, SURVEY.md 8d) forward; backward ~ 2x
        flops = None
    elif w == "c3":
        n = cfg["n_roll"]
        Mmax = (L - 1) * B * n
        caps = caps_()
        sets = [dict(u=torch.rand(L, B, generator=g, device=dev), ur=torch.rand(L, Mmax, generator=g, device=dev)) for _ in range(2)]
        units = B * L + B * n * (L * (L - 1) // 2)               # sampled row-steps per step (SURVEY.md 8a row B2)
        fn = lambda i: inst.pg_step(caps, u=sets[i % 2]["u"], u_roll=sets[i % 2]["ur"], n_roll=n)
        metric, unit = "sampled_caption_tokens_per_sec", "tokens/s"
        k = steps or 3
        flops = units * (8.0 * H * (E + H) + 2.0 * H * V)        # forward decode contractions of every sampled row-step
    else:
        caps = caps_()
        fake = torch.randint(4, V, (B, L), generator=g, device=dev)
        keeps = [(torch.rand(2, B * R, Fd, generator=g, device=dev) >= 0.2).to(torch.uint8) for _ in range(2)]
        units = 1
        fn = lambda i: inst.disc_step(caps, fake, keep=keeps[i % 2])
        metric, unit = "discriminator_steps_per_sec", "steps/s"
        k = steps or 5
        # highway forward + dx + dW_h for both trunks: 3 x 2 x (2 B R F^2); plus head 2 B R F 100 x 3
        flops = 2.0 * (3 * 2.0 * B * R * Fd * Fd + 3 * 2.0 * B * R * Fd * 100)
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(k):
        r = fn(i)
    e1.record(); torch.cuda.synchronize()
    if dump and rank == 0:
        dump_outputs(dump, r, {"gen": inst.gen, "disc": inst.disc})
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    out.update({"metric": metric, "value": world * units * k / (ms * 1e-3), "unit": unit, "ms_per_step": ms / k, "steps": k, "warmup": 3})
    if flops:
        tf = flops / (ms / k * 1e-3) / 1e12
        out["tensor"] = {"algorithmic_flops_per_step": flops, "achieved_TFLOPs": tf, "frac_of_bf16_burst_peak": tf / peaks["tf_burst"],
                         "note": ("forward decode contractions of all sampled row-steps over the WHOLE step time (sampling, discriminator "
                                  "scoring of 39 040 captions and the policy-gradient backward included)") if w == "c3" else
                                 "highway / dx / dW_h / head contractions of both trunks over the WHOLE step time (gather, conv + pool, loss, Adam included)"}
    if w == "c2a":
        out["note"] = ("additive attention over the [256, 49, 2048] grid inside every decode step (EXTENSION: the reference has no "
                       "attention; oracle/ref_ext.py defines it, parity unpinned by reference); per-step q projection + attention kernel + "
                       "LSTM step + fused projection / sample")
    inst._graphs.clear()
    del inst
    return out


WORKLOAD_NOTES = {
    "c2": "BASELINE.json configs[1], Tier-A shape (mean-pooled grid)",
    "c2a": "BASELINE.json configs[1] WITH attention over the 7x7x2048 grid (north-star extension B1)",
    "c3": "BASELINE.json configs[2]: SeqGAN-style policy-gradient step, 128 captions x 16 Monte-Carlo rollouts per prefix",
    "c4": "BASELINE.json configs[3]: hidden 1024, vocab 30k; one GPU's 128 rows of the 1024-row global batch",
    "c5": "BASELINE.json configs[4]: discriminator-only step on 4096 real + 4096 fake captions of length 32",
}


def run_secondary(args):
    """--workload c2a / c3 / c4 / c5 as a line of its own (under torchrun: weak scaling over the ranks)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    r = run_workload(args.workload, args.mode, dev, load_peaks(), steps=args.steps, world=world, rank=rank, dump=args.dump_outputs)
    if rank == 0:
        r.update({"n_gpus": world, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "secondary": True})
        print(json.dumps(r), flush=True)
    if world > 1:
        torch.cuda.synchronize(); dist.barrier()
        t = threading.Timer(15.0, lambda: os._exit(0)); t.daemon = True; t.start()
        dist.destroy_process_group(); t.cancel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default=os.environ.get("GIC_GEMM_MODE", "bf16"), choices=sorted(MODES))
    ap.add_argument("--cpu-sample-rows", type=int, default=0, help="rows of the CPU arm's step (0 = the whole per-GPU batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--settle", type=int, default=20, help="untimed set-up replays after graph capture, before the warm-up steps")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 1 s long-run measurement")
    ap.add_argument("--no-modes", action="store_true", help="skip the tf32 / fp32 measurements of the same step")
    ap.add_argument("--no-workloads", action="store_true", help="skip the c2a / c3 / c4 / c5 block")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every kernel from the host instead of replaying the captured step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                                                          "(float32 / float64, at most 64 MB: larger arrays as a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
        return
    try:
        if args.workload in ("c2a", "c3", "c4", "c5"):
            run_secondary(args)
        else:
            run_ours(args)
    except Exception:
        # a bounded device-side wait that gave up says which one (host-mapped memory outlives the CUDA context)
        try:
            from gic_b200 import _lib
            info = _lib.trap_info()
            if info:
                print("gic_b200: device-side wait expired: %r (sites: include/gic_b200.h, gic_trap_info)" % (info,), file=sys.stderr, flush=True)
        except Exception:
            pass
        raise


if __name__ == "__main__":
    main()
