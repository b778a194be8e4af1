#!/usr/bin/env python
"""bench.py -- bar-VAE generator training throughput (bars/s) on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (libbarvae.so)
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's loss (.npy)

A "step" is one pass of the hot path over one batch of synthetic piano-roll bars: zero_grad, generator forward
(phrase encoder, encoder x2, decoder), BCE loss, backward, (NCCL gradient all-reduce), Adam -- the pre-training
branch of the reference's agent/barGen.py:249-252,302-335.  Workload = BASELINE.json configs[1]: batch 512 bars per
GPU, bf16 tensor-core arithmetic with fp32 accumulation/statistics/parameters.  Weak scaling: 512 bars per GPU at
every N (N = 8 is configs[2]'s global batch 4096).

One JSON line on stdout (rank 0).  `value` = whole-job bars/s with inputs resident in HBM; `e2e` = the same step
driven through the public nn.Module API from pinned HOST tensors (H2D copy of the batch and D2H read of the loss
inside the timed region).  `roofline` = the contraction kernels (tcgen05 implicit GEMMs) timed live with CUDA events.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "musicgeneration_vae-torch_b200"

# algorithmic work per bar (SURVEY.md section 8d): forward 9.8314 GFLOP, forward+backward 29.494 GFLOP
GFLOP_PER_BAR_TRAIN = 29.494
N_PARAMS = 89537290


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1383.1), d.get("hbm_gbs", 6547.8), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def synthetic_batch(B, seed, device, pin=False):
    """SURVEY.md section 8(d): binary piano-roll bars at ~5 % density (agent/barGen.py:134-141 shapes)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    note = (torch.rand(B, 1, 96, 60, generator=g) < 0.05).float()
    pre_note = (torch.rand(B, 1, 96, 60, generator=g) < 0.05).float()
    phrase = (torch.rand(B, 1, 384, 60, generator=g) < 0.05).float()
    position = torch.randint(0, 332, (B,), generator=g)
    ts = (note, pre_note, phrase, position)
    if device is not None:
        return tuple(t.to(device) for t in ts)
    return tuple(t.pin_memory() for t in ts) if pin else ts


def dump_outputs(out_dir, loss):
    """--dump-outputs: what the last timed training step returns to its caller -- its loss -- as DIR/loss.npy (float32).
    The gradients and updated parameters it leaves in the model are not written: with the reference's N(-1,1)
    initialisation the step is so ill-conditioned that the order of the fp32 atomic additions in the InstanceNorm
    statistics and the norm-block backward decides them (measured on one B200, 10 timed steps after 3 warm-up steps: two
    runs' sampled gradients differ by 112 % rel-Frobenius, and the loss itself by 0.4-1.9 %), so they cannot be compared
    between builds; the loss is the only value of the step a caller receives."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().reshape(1).cpu().numpy())


def cpu_reference_arm(batch, steps, warmup, target_s=0.0):
    """The reference algorithm (CPU oracle port of graph/*.py + bar_loss.py + torch.optim.Adam semantics) on all host
    cores; returns bars/s.  Bounded sample: `batch` bars per step."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import barvae_oracle as O
    from collections import OrderedDict
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = O.make_state_dict(O.generator_spec(), 0, "reference")
    b = O.make_inputs(batch, 1234)
    m = OrderedDict((k, torch.zeros_like(v)) for k, v in sd.items())
    v = OrderedDict((k, torch.zeros_like(t)) for k, t in sd.items())
    times = []
    i = 0
    while i < warmup + steps:
        t0 = time.perf_counter()
        O.train_step(sd, b, m, v, i + 1, 0.002, None, True)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
            if target_s and len(times) == 1:        # size the bounded sample to ~target_s seconds of CPU work
                steps = max(steps, min(40, int(target_s / max(times[0], 1e-3) + 0.999)))
        i += 1
    dt = sum(times) / len(times)
    return batch / dt, dt, cores, torch.get_num_threads(), len(times)


GFLOP_PER_BAR_DECODE_CACHED = 5.3223     # SURVEY.md section 8d: phrase feature computed once per 4 bars
NB_ALGO_BYTES_PER_BAR = 4.26e6 * (4 + 6)   # SURVEY.md section 8d: 4.26 M InstanceNorm-site elements/bar, 4 B fwd + 6 B bwd


def decode_measure(pkg, Model, dev, rank, world, songs, phrases, model=None, refine=False):
    """BASELINE configs[4]: the maker_bar.py:32-44 sampling loop, `songs` songs in lock-step per GPU (songs are
    independent, so ranks need no collective).  One step = one 4-bar phrase: phrase encoder once, then 4 x (encoder +
    decoder).  Returns a dict (max over ranks of the CUDA-event time)."""
    import torch
    import torch.distributed as dist
    maker = importlib.import_module(PKG + ".maker_bar")
    if model is None:
        model = Model().to(dev)
    model.eval()
    g = torch.Generator(device=dev).manual_seed(99 + rank)

    def run(n):
        lat = torch.randn(n * 4, songs, 1152, device=dev, generator=g)
        return maker.sample_songs(model, lat, n)

    run(1)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    n0 = pkg.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    roll = run(phrases)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    bars = songs * 4 * phrases * world
    tf_peak, _, how = measured_peaks()
    val = bars / (ms * 1e-3)
    tfl = GFLOP_PER_BAR_DECODE_CACHED * 1e9 * val / world / 1e12          # per GPU
    return {"metric": "decode_bars_per_sec", "value": val, "unit": "bars/s", "n_gpus": world, "phrases": phrases,
            "songs_per_gpu": songs, "ms_per_phrase": ms / phrases, "gpu_launches": pkg.launch_count() - n0,
            "tflops_per_gpu": tfl, "frac_of_tensor_peak": tfl / tf_peak,
            "ceiling_bars_per_sec_per_gpu": tf_peak * 1e12 / (GFLOP_PER_BAR_DECODE_CACHED * 1e9),
            "peak_source": how, "notes_on": float(roll.float().mean()),
            "what": "maker_bar sampling loop, %d songs/GPU in lock-step, 4 bars per phrase, phrase feature computed once "
                    "per phrase, threshold 0.3 on the device; dp%d, independent songs, no collective" % (songs, world)}


def decode_bench(args, pkg, Model, dev, rank, world):
    import torch.distributed as dist
    d = decode_measure(pkg, Model, dev, rank, world, args.songs, max(1, args.steps))
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    emit({"metric": d["metric"], "value": d["value"], "unit": "bars/s", "n_gpus": world, "steps": d["phrases"], "warmup": 1,
          "ms_per_step": d["ms_per_phrase"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
          "dtype": "bf16", "data": "synthetic",
          "config": {"workload": d["what"], "songs_per_gpu": args.songs, "parallelism": "dp%d" % world},
          "gpu_launches": d["gpu_launches"], "tflops_end_to_end": d["tflops_per_gpu"] * world,
          "frac_of_tensor_peak": d["frac_of_tensor_peak"], "peak_source": d["peak_source"], "notes_on": d["notes_on"]})


def torch_eager_gpu(dev, bars, steps=3):
    """SURVEY.md section 8(d) 'library comparator': the reference algorithm (oracle port: stock torch.nn.functional ops ->
    cuDNN / cuBLAS / ATen kernels) run by PyTorch eager on the SAME B200, fp32 and bf16-autocast, forward + backward +
    torch.optim.Adam.  `bars` per step is bounded (eager autograd keeps ~10x the activations this repo's path saves)."""
    import torch
    from collections import OrderedDict
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import barvae_oracle as O
    out = {"bars_per_step": bars, "steps": steps,
           "what": "oracle port of the reference modules on cuda through PyTorch eager (cuDNN/cuBLAS/ATen), fwd+bwd+"
                   "torch.optim.Adam; fp32 row = fp32 storage with TF32 tensor-core convolutions and matmuls allowed "
                   "(the faster setting), bf16 row = torch.autocast(bfloat16)"}
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True          # as the reference sets it (agent/barGen.py:26)
    sd = O.make_state_dict(O.generator_spec(), 0, "reference")
    batch = tuple(t.to(dev) for t in O.make_inputs(bars, 1234))
    for name, autocast in (("fp32", False), ("bf16_autocast", True)):
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        try:
            leaves = OrderedDict((k, v.to(dev).clone().requires_grad_(True)) for k, v in sd.items())
            opt = torch.optim.Adam(list(leaves.values()), lr=0.002)

            def step():
                opt.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    gen = O.model_forward(*batch, leaves, True, None)[0]
                loss = O.loss_forward(gen.float(), batch[0], True)
                loss.backward()
                opt.step()

            step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"bars_per_sec": bars / (ms * 1e-3), "ms_per_step": ms,
                         "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 2 ** 30}
            del leaves, opt
        except Exception as exc:            # an auxiliary comparator must not take the headline measurement down
            out[name] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
    return out


def ncu_traffic_table():
    """per-launch DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) from `ncu --set full` captures, kept under
    profiles/ (this round's file first); keyed by kernel instance"""
    for name in ("traffic_r3.json", "traffic_r2.json", "traffic_r1.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            try:
                return json.load(open(p)), name
            except ValueError:
                pass
    return {}, None


def gan_bench(args, pkg, dev, rank, world):
    """BASELINE configs[3]: the adversarial step of agent/barGen_with_gan.py on N GPUs -- per iteration a discriminator
    step (generator frozen: forward only, incl. the re-encode of the thresholded bar) + a generator step, for both phases:
    train_wae (z discriminators; generator step = BCE + 3 adversarial terms) and train_gan (conv BarDiscriminator + feature
    discriminator; generator step from noise).  Whole-job bars/s = bars per iteration / time per iteration."""
    import torch
    import torch.distributed as dist
    Config = importlib.import_module(PKG + ".config").Config
    G = importlib.import_module(PKG + ".agent.barGen_with_gan")
    SyntheticBars = importlib.import_module(PKG + ".data.bar_dataset").SyntheticBars
    import tempfile

    class Cfg(Config):
        root_path = tempfile.mkdtemp(prefix="bvae_gan_bench_")
        batch_size = 1
        pretraining_step_size = 0

    agent = G.BarGen(Cfg(), dataset=SyntheticBars(world, 1, 1))
    B = args.batch
    batch = synthetic_batch(B, 1234 + rank, dev)
    valid, fake = torch.ones(B, device=dev), torch.zeros(B, device=dev)
    sink = lambda loss: None
    agent.epoch = 1

    def it_wae():
        agent.train_wae(*batch, sink, sink, sink, fake, valid, 0)       # (epoch + curr_it) % 2 == 1: discriminator step too

    def it_gan():
        agent.train_gan(*batch, sink, sink, sink, fake, valid, 0)

    def it_horovod():                                   # agent/barGen_horovod.py:312-324, GAN phase
        agent.train_discriminator(*batch, sink, sink, sink, sink, fake, valid)
        agent.train_add_gan(*batch, sink, valid)

    out = {}
    for name, fn in (("wae", it_wae), ("gan", it_gan), ("horovod_gan", it_horovod)):
        for _ in range(max(3, args.warmup)):          # (the allocator still grows in the second iteration of a phase)
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        n0 = pkg.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        out[name] = {"ms_per_iteration": ms, "bars_per_sec": B * world / (ms * 1e-3),
                     "gpu_launches_per_iteration": (pkg.launch_count() - n0) / args.steps}
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    emit({"metric": "gan_step_bars_per_sec", "value": out["gan"]["bars_per_sec"], "unit": "bars/s", "n_gpus": world,
          "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": out["gan"]["ms_per_iteration"],
          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
          "config": {"workload": "barGen_with_gan adversarial iteration (discriminator step + generator step), %d bars/GPU, "
                                 "reference-init weights; value = train_gan phase, extra.wae = train_wae phase, extra.horovod_gan = "
                                 "the barGen_horovod.py iteration (train_discriminator + train_add_gan)" % B,
                     "bars_per_gpu": B, "parallelism": "dp%d" % world},
          "gpu_launches": int(out["gan"]["gpu_launches_per_iteration"] * args.steps), "extra": out})


_JSON_OUT = None


def _protect_stdout():
    """Keep stdout to the ONE JSON line the driver parses.  Libraries write to file descriptor 1 behind Python's back
    (NCCL printf()s its version banner there at NCCL_DEBUG=VERSION and above -- measured on the 2-GPU run): point fd 1
    at stderr for the whole run and write the JSON line to a saved duplicate of the original descriptor.  A
    VERSION-only NCCL_DEBUG (set on some boxes) is dropped as well; an explicit WARN / INFO / TRACE request is left alone
    and simply lands on stderr."""
    global _JSON_OUT
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        del os.environ["NCCL_DEBUG"]
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="barvae", choices=["barvae", "reference"])
    ap.add_argument("--batch", type=int, default=512, help="bars per GPU")
    ap.add_argument("--cpu-batch", type=int, default=16, help="bars per step of the CPU arm (BASELINE configs[0])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--micro-bars", type=int, default=0,
                    help="train: run the step as gradient-accumulated chunks of this many bars (BASELINE configs[2]: "
                         "--gpus 2 --batch 2048 --micro-bars 512 is global batch 4096)")
    ap.add_argument("--mode", default="train", choices=["train", "decode", "gan"],
                    help="train = BASELINE configs[1] (the driver's default); decode = configs[4], maker_bar sampling")
    ap.add_argument("--songs", type=int, default=8192, help="decode: songs generated in lock-step per GPU")
    ap.add_argument("--no-decode", action="store_true", help="train mode: skip the extra.decode measurement")
    ap.add_argument("--no-eager", action="store_true", help="train mode: skip extra.torch_eager_gpu")
    ap.add_argument("--eager-bars", type=int, default=256, help="bars per step of the PyTorch-eager comparator")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="train mode: after the timed steps, write the loss the last timed step returned as DIR/loss.npy "
                         "(see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.mode != "train" or args.impl != "barvae"):
        ap.error("--dump-outputs applies to the training step of this repo's CUDA path (--mode train --impl barvae)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = {"workload": "barGen bar-VAE generator training step (fwd+bwd+Adam), %d bars/GPU, synthetic 5%%-density "
                       "piano-roll bars [B,1,96,60] + phrases [B,1,384,60], reference-init weights" % args.batch,
           "bars_per_gpu": args.batch, "global_batch": args.batch * world, "parallelism": "dp%d" % world,
           "l2": "per-step working set (~25 MB/bar of saved activations) is >> 126 MB L2; no flush needed"}

    if args.impl == "reference":
        # The reference's own CPU implementation of the path (oracle port of graph/*.py + bar_loss.py + Adam; the
        # reference is a script tree without setup.py, /root/reference does not exist on the GPU box) on all host cores.
        # Same metric / unit / config as this repo's arm; --steps and --warmup are honoured as given; each step is a
        # BOUNDED SAMPLE of the workload: --cpu-batch bars (BASELINE configs[0]) instead of the 512 of one GPU step.
        if rank != 0:
            return
        steps, warm = max(1, args.steps), max(0, args.warmup)
        bars_s, dt, cores, threads, nst = cpu_reference_arm(args.cpu_batch, steps, warm)
        line = {"impl": "reference", "metric": "train_bars_per_sec", "value": bars_s, "unit": "bars/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": cfg,
                "cpu_baseline": {"value": bars_s, "unit": "bars/s", "cores": threads, "kind": "port",
                                 "sample": "%d timed steps (after %d warm-up) of %d bars each (fwd+bwd+Adam) -- a bounded "
                                           "sample of the %d-bar step; oracle port of the reference modules on %d host "
                                           "threads" % (nst, warm, args.cpu_batch, args.batch, threads)},
                "e2e": {"value": bars_s, "unit": "bars/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch
    import torch.distributed as dist
    pkg = importlib.import_module(PKG)
    par = importlib.import_module(PKG + ".parallel")
    Model = importlib.import_module(PKG + ".graph.model").Model
    Trainer = importlib.import_module(PKG + ".trainer").GeneratorTrainer
    eng = pkg.engine
    rank, world, local = par.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B = args.batch

    torch.manual_seed(0)
    if args.mode == "decode":
        return decode_bench(args, pkg, Model, dev, rank, world)
    if args.mode == "gan":
        return gan_bench(args, pkg, dev, rank, world)
    model = Model().to(dev).train()          # reference initialisation (graph/weights_initializer.py semantics)
    flat = model.flatten_parameters()
    reducer = None
    if world > 1:
        reducer = par.GradReducer.for_model(model, flat)
        reducer.broadcast_parameters(0)
    # Graph replay: the trainer's default is on for one process and opt-in under torch.distributed (trainer.py: a process
    # that still holds a graph with captured NCCL kernels when the process group is destroyed hangs in NCCL teardown).
    # This script releases the graphs before it destroys the group -- also on an exception, see the finally below -- so it
    # opts in at every N (measured on one 8xB200 node: 95.8 k vs 94.7 k bars/s, e2e 95.0 k vs 92.7 k; BVAE_GRAPH=0 disables).
    use_graph = None if world == 1 else (os.environ.get("BVAE_GRAPH", "1") != "0")
    trainer = Trainer(model, lr=0.002, reducer=reducer, micro_bars=args.micro_bars, use_graph=use_graph)
    try:
        return _train_bench(args, pkg, eng, par, Model, trainer, model, flat, reducer, cfg, dev, rank, world, local, B)
    finally:
        trainer.release_graphs()


def _train_bench(args, pkg, eng, par, Model, trainer, model, flat, reducer, cfg, dev, rank, world, local, B):
    import torch
    import torch.distributed as dist
    if args.micro_bars:
        cfg["micro_bars"] = args.micro_bars
        cfg["workload"] += " (gradient-accumulated in chunks of %d bars)" % args.micro_bars

    dbatch = synthetic_batch(B, 1234 + rank, dev)
    hbatch = synthetic_batch(B, 4321 + rank, None, pin=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    last_loss = [None]

    def step_resident():
        last_loss[0] = trainer.step(*dbatch)

    def step_e2e():
        loss = trainer.step_from_host(*hbatch)      # pinned host tensors -> H2D copies -> step, strictly in sequence
        return loss.item()               # D2H read of the step's result, as agent/barGen.py:335 does

    def loop_e2e(batch, k):
        """the loop BarGen.train_epoch runs (public API): k host batches through trainer.prefetch -- batch i+1's H2D
        copy is issued on a copy stream before step i -- one optimisation step and one loss read-back per batch.  The
        iterator is created here, so all k copies (the first one exposed) are inside the timed region."""
        for db in trainer.prefetch(batch for _ in range(k)):
            trainer.step_batch(db).item()

    # untimed warm-up: W (>= 3) steps; with CUDA-graph replay on (the default) the last two of them are the step that captures
    # the graph and one replay, so that the timed region below contains replays only
    n_warm = max(3, args.warmup)
    if trainer.use_graph:
        trainer.graph_after = n_warm - 2          # eager steps, then the capturing step, then one replay: W untimed steps
    for _ in range(n_warm):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    pkg.reset_launch_count()
    ms = timed(step_resident, args.steps)
    launches = pkg.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    value = B * world * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:          # before the e2e loops below train the model further
        dump_outputs(args.dump_outputs, last_loss[0])

    loop_e2e(hbatch, 2)
    ms_e2e = timed(lambda: loop_e2e(hbatch, args.steps), 1)
    e2e = B * world * args.steps / (ms_e2e * 1e-3)
    h2d = sum(t.numel() * t.element_size() for t in hbatch)
    step_e2e()
    ms_seq = timed(step_e2e, args.steps)
    e2e_seq = {"value": B * world * args.steps / (ms_seq * 1e-3), "unit": "bars/s", "ms_per_step": ms_seq / args.steps,
               "what": "trainer.step_from_host + .item(): copy, step and read-back strictly in sequence (the reference "
                       "loop's order, agent/barGen.py:302-335); no copy/compute overlap"}

    # the same loop fed from BIT-PACKED pinned host batches (data/packed.py, SURVEY.md section 8f N3): one 2.2 MB H2D
    # copy + bvae_unpack_bits per step instead of 70.8 MB of fp32.  Reported beside `e2e` (which stays on the
    # reference-format fp32 host tensors), never instead of it.
    e2e_packed = None
    try:
        Packed = importlib.import_module(PKG + ".data.packed").PackedBatch
        pbatch = Packed.from_arrays(*hbatch, pin=True)
        loop_e2e(pbatch, 2 + (trainer.graph_after + 1 if trainer.use_graph else 0))   # (its own input signature / graph)
        ms_p = timed(lambda: loop_e2e(pbatch, args.steps), 1)
        e2e_packed = {"value": B * world * args.steps / (ms_p * 1e-3), "unit": "bars/s",
                      "h2d_bytes_per_step": pbatch.nbytes, "d2h_bytes_per_step": 4, "ms_per_step": ms_p / args.steps}
    except Exception as exc:      # an auxiliary number must not take the headline measurement down with it
        e2e_packed = {"error": "%s: %s" % (type(exc).__name__, exc)}

    # live roofline of the contraction kernels: CUDA events around every bvae_conv_gemm / bvae_wgrad_gemm launch
    roofline = None
    roofline_hbm = None
    extra = {}
    if not args.no_profile:
        prof_steps = 2
        # per-kernel CUDA-event timing needs the launches serialised on one stream: switch the branch / weight-gradient
        # stream overlap off for these (untimed) profiling steps only
        saved_env = {k: os.environ.get(k) for k in ("BVAE_STREAMS", "BVAE_WGRAD_STREAM")}
        os.environ["BVAE_STREAMS"] = "0"
        os.environ["BVAE_WGRAD_STREAM"] = "0"
        step_resident()
        torch.cuda.synchronize()
        eng.profile_begin()
        for _ in range(prof_steps):
            step_resident()
        torch.cuda.synchronize()
        prof = eng.profile_end()
        for k, v in saved_env.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        detail = prof.pop("detail", {})
        classes = prof.pop("classes", {})
        if os.environ.get("BVAE_PROFILE_DETAIL") and rank == 0:
            for k, (t, n) in sorted(detail.items(), key=lambda kv: -kv[1][0]):
                print("%9.3f ms %4d  %s" % (t / prof_steps, n // prof_steps, k), file=sys.stderr)
        tf_peak, hbm_peak, how = measured_peaks()
        gemm_ms = (prof.get("conv_gemm", 0.0) + prof.get("wgrad_gemm", 0.0)) / prof_steps
        nb_ms = (prof.get("nb_forward", 0.0) + prof.get("nb_backward", 0.0)) / prof_steps
        flops = GFLOP_PER_BAR_TRAIN * 1e9 * B
        ach = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        how_timed = ("CUDA events around every launch on its launching stream, in a profiling pass with the branch / "
                     "weight-gradient stream overlap switched off (the timed steps run with it on)")
        aggregate = {"achieved": ach, "frac": ach / tf_peak, "kernel_ms_per_step": gemm_ms,
                     "launches_per_step": prof.get("n_gemm", 0) / prof_steps,
                     "kernels": "every contraction launch of one step (conv_tc2 / wgrad_tc / wgrad_halo / stem kernels)"}
        # per kernel INSTANCE (template arguments as launched, bvae_last_kernel): the dominant one is the roofline headline
        kernels = prof.pop("kernels", {})
        by_kernel, dom = {}, None
        for name, kk in kernels.items():
            tf = kk["flops"] / (kk["ms"] * 1e-3) / 1e12 if kk["ms"] > 0 else 0.0
            by_kernel[name] = {"ms_per_step": kk["ms"] / prof_steps, "tflops": tf, "frac": tf / tf_peak,
                               "launches_per_step": kk["launches"] / prof_steps}
            if kk["flops"] > 0 and (dom is None or kk["ms"] > kernels[dom]["ms"]):
                dom = name
        traffic_tab, traffic_src = ncu_traffic_table()
        if dom is not None:
            kk = kernels[dom]
            top_layer, (lms, lfl, ln) = max(kk["layers"].items(), key=lambda kv: kv[1][0])
            tr = traffic_tab.get(dom)
            roofline = {"bound": "tensor", "kernel": dom, "achieved": by_kernel[dom]["tflops"], "peak": tf_peak,
                        "unit": "TFLOP/s", "frac": by_kernel[dom]["frac"],
                        "traffic": tr.get("dram_bytes_per_launch") if isinstance(tr, dict) else None,
                        "traffic_note": (dict(tr, source="profiles/" + traffic_src) if isinstance(tr, dict) else
                                         "no ncu --set full capture of this kernel instance under profiles/"),
                        "peak_source": how + " (sustained cuBLAS bf16)", "how": how_timed,
                        "algorithmic_flops_per_launch": kk["flops"] / kk["launches"],
                        "avg_launch_ms": kk["ms"] / kk["launches"], "launches_per_step": kk["launches"] / prof_steps,
                        "ms_per_step": kk["ms"] / prof_steps,
                        "share_of_step": kk["ms"] / max(prof.get("total_ms", 0.0), 1e-9),
                        "top_layer": {"layer": top_layer, "ms_per_launch": lms / ln,
                                      "tflops": lfl / (lms * 1e-3) / 1e12 if lms > 0 else 0.0},
                        "all_contractions": aggregate, "by_kernel": by_kernel}
        else:
            roofline = dict(aggregate, bound="tensor", peak=tf_peak, unit="TFLOP/s", traffic=None,
                            peak_source=how + " (sustained cuBLAS bf16)", how=how_timed)
        # the same launches split by their narrower channel count: FLOPs accounted per launch by engine.GemmLayer
        # (SURVEY.md section 8 convention), time = CUDA events around that launch
        try:
            by_class = {}
            for name, (cms, cfl, cn) in sorted(classes.items()):
                tf = cfl / (cms * 1e-3) / 1e12 if cms > 0 else 0.0
                by_class[name] = {"ms_per_step": cms / prof_steps, "tflops": tf, "frac": tf / tf_peak,
                                  "launches_per_step": cn / prof_steps,
                                  "share_of_flops": cfl / prof_steps / flops if flops else None}
            roofline["by_class"] = by_class
            roofline["flops_accounted_frac"] = sum(c[1] for c in classes.values()) / prof_steps / flops
        except Exception as exc:
            roofline["by_class"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        # the HBM-bound half of the step: all norm-block launches against their ALGORITHMIC bytes (SURVEY.md 8d)
        nb_bytes = NB_ALGO_BYTES_PER_BAR * B
        nb_gbs = nb_bytes / (nb_ms * 1e-3) / 1e9 if nb_ms > 0 else 0.0
        roofline_hbm = {"bound": "hbm", "kernel": "norm-block sweeps (all bvae_nb_forward / bvae_nb_backward launches)",
                        "achieved": nb_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": nb_gbs / hbm_peak,
                        "algorithmic_bytes_per_step": nb_bytes, "ms_per_step": nb_ms,
                        "launches_per_step": (prof.get("n_nb_forward", 0) + prof.get("n_nb_backward", 0)) / prof_steps,
                        "traffic": (traffic_tab.get("norm_blocks") or {}).get("dram_bytes_per_step"),
                        "peak_source": how + " (copy bandwidth)", "how": how_timed}
        extra = {"normblock_ms_per_step": nb_ms, "step_ms_under_event_profiling": prof.get("total_ms", 0.0) / prof_steps,
                 "adam_gbs": None}
        # fused Adam alone: 28 B/param
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(5):
            eng.adam_step(flat, 0.0, 100 + i, repack=False)
        e1.record()
        torch.cuda.synchronize()
        extra["adam_gbs"] = flat.numel * 28 / (e0.elapsed_time(e1) / 5 * 1e-3) / 1e9
        extra["adam_frac_of_hbm_peak"] = extra["adam_gbs"] / hbm_peak
        # the one-launch refresh of all bf16 contraction operands that follows Adam (4 B read + 2 B written per packed value)
        e0.record()
        for i in range(5):
            eng.repack_weights(flat)
        e1.record()
        torch.cuda.synchronize()
        extra["repack_ms"] = e0.elapsed_time(e1) / 5

    # a 64-bar/GPU point (VERDICT r1 item 5): with the step replayed as one CUDA graph the host is out of the picture, what
    # remains is the device-side latency of ~520 small launches
    if not args.no_profile and not args.micro_bars:
        try:
            sb = synthetic_batch(64, 99 + rank, dev)
            for _ in range(trainer.graph_after + 3 if trainer.use_graph else 4):
                trainer.step(*sb)
            ms64 = timed(lambda: trainer.step(*sb), 10) / 10
            extra["small_batch"] = {"bars_per_gpu": 64, "ms_per_step": ms64, "bars_per_sec": 64 * world / (ms64 * 1e-3),
                                    "per_bar_rate_vs_%d_bars" % B: (64 * world / (ms64 * 1e-3)) / value,
                                    "graph_replay": bool(trainer.use_graph)}
            del sb
        except Exception as exc:
            extra["small_batch"] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
    # BASELINE configs[4] in the same record, at every N: maker_bar sampling, 8192 songs per GPU, 2 phrases (8 bars/song)
    if not args.no_decode:
        try:
            del dbatch
            torch.cuda.empty_cache()
            extra["decode"] = decode_measure(pkg, Model, dev, rank, world, args.songs, 2, model=model)
            model.train()
        except Exception as exc:
            extra["decode"] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
    trainer_used_graph = bool(trainer._graphs)
    trainer.release_graphs()            # graphs that captured NCCL kernels must go before the process group does
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if world == 1 and not args.no_eager:
        del trainer, model, flat
        torch.cuda.empty_cache()
        extra["torch_eager_gpu"] = torch_eager_gpu(dev, args.eager_bars)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        bars_s, dt, cores, threads, nst = cpu_reference_arm(args.cpu_batch, 3, 1, target_s=12.0)
        cpu = {"value": bars_s, "unit": "bars/s", "cores": threads, "kind": "port",
               "sample": "%d steps of %d bars (fwd+bwd+Adam) of the oracle port, %.1f s/step" % (nst, args.cpu_batch, dt)}
    line = {"metric": "train_bars_per_sec", "value": value, "unit": "bars/s", "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfg,
            "e2e": {"value": e2e, "unit": "bars/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps,
                    "what": "the BarGen.train_epoch loop: for batch in trainer.prefetch(pinned fp32 host batches): "
                            "trainer.step_batch(batch).item() -- every step's H2D copy and loss read-back inside the "
                            "timed region, batch i+1's copy overlapping step i on a copy stream"},
            "e2e_sequential": e2e_seq,
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_hbm": roofline_hbm,
            "cpu_baseline": cpu,
            "tflops_end_to_end": GFLOP_PER_BAR_TRAIN * 1e9 * value / 1e12, "e2e_packed": e2e_packed,
            "graph_replay": bool(trainer_used_graph), "extra": extra}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
