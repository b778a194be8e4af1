"""Cost of the Bernoulli sampler (csrc/sample.cu) on its own and inside the sampling loop.

  1. bvae_bernoulli_sample at --bars bars (8192 by default: 47 M cells, 0.38 GB moved, three times the L2, so every
     launch streams from HBM): CUDA events around --iters back-to-back launches after a warm-up; achieved GB/s against
     the algorithmic 8 B per cell (4 B logit read, 4 B cell written).
  2. maker_bar.sample_songs at --songs songs x --phrases phrases with sampler="threshold" and sampler="bernoulli",
     alternating the two --rounds times in this process (CUDA events, one warm-up run of each first); bars/s per run.

Prints one JSON object (also written to --out) with the card's name and power limit read in the same run.

    python tools/bench_sampling.py --out profiles/sampling_bench.json
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "musicgeneration_vae-torch_b200"
sys.path.insert(0, ROOT)
CELLS = 96 * 60


def card():
    """name, power limit and max SM clock of the current device (read-only nvidia-smi query)"""
    info = {"name": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                            "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:                               # the figure then says it is unknown
        info["power_limit"] = "unknown (%s)" % type(e).__name__
    return info


def time_kernel(packed, bars, iters):
    g = torch.Generator(device="cuda").manual_seed(0)
    logits = torch.randn(bars, 1, 96, 60, device="cuda", generator=g)
    out = torch.empty_like(logits)
    for _ in range(5):
        packed.bernoulli_sample(logits, 1.0, 1, 0, 0, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        packed.bernoulli_sample(logits, 1.0, 1, 0, i, out=out)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    nbytes = 8 * bars * CELLS
    return {"bars": bars, "cells": bars * CELLS, "iters": iters, "us_per_launch": us, "algorithmic_bytes": nbytes,
            "achieved_GBps": nbytes / (us * 1e-6) / 1e9, "notes_on": float(out.mean())}


def time_decode(maker, model, songs, phrases, rounds):
    g = torch.Generator(device="cuda").manual_seed(99)
    lat = torch.randn(phrases * 4, songs, 1152, device="cuda", generator=g)
    modes = ("threshold", "bernoulli")
    for m in modes:                                           # warm-up: every shape of the timed runs
        maker.sample_songs(model, lat[:4], 1, sampler=m, seed=1)
    torch.cuda.synchronize()
    runs = {m: [] for m in modes}
    for _ in range(rounds):
        for m in modes:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            roll = maker.sample_songs(model, lat, phrases, sampler=m, seed=1)
            e1.record()
            torch.cuda.synchronize()
            runs[m].append(songs * 4 * phrases / (e0.elapsed_time(e1) * 1e-3))
            runs[m + "_notes_on"] = float(roll.mean())
    res = {"songs": songs, "phrases": phrases, "rounds": rounds}
    for m in modes:
        res[m] = {"bars_per_sec_runs": runs[m], "bars_per_sec_median": statistics.median(runs[m]),
                  "notes_on": runs[m + "_notes_on"]}
    res["bernoulli_over_threshold"] = res["bernoulli"]["bars_per_sec_median"] / res["threshold"]["bars_per_sec_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bars", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--songs", type=int, default=8192)
    ap.add_argument("--phrases", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sampling: needs a CUDA device; nothing is measured without one")
    packed = importlib.import_module(PKG + ".data.packed")
    maker = importlib.import_module(PKG + ".maker_bar")
    Model = importlib.import_module(PKG + ".graph.model").Model
    res = {"card": card(), "kernel": time_kernel(packed, args.bars, args.iters)}
    model = Model().cuda().eval()          # the reference's initialisation, as bench.py --mode decode
    res["decode"] = time_decode(maker, model, args.songs, args.phrases, args.rounds)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
