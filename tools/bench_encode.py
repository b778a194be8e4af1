"""Cost of the per-bar score (csrc/sample.cu) and of the song-level encode / teacher-forced passes (maker_bar).

  1. bvae_bar_score at --bars bars (8192 by default: 47 M cells, 0.38 GB read, three times the L2, so every launch
     streams from HBM): CUDA events around --iters back-to-back launches after a warm-up; achieved TB/s against the
     algorithmic 8 B per cell (4 B logit and 4 B target read; the outputs are 16 B per bar).
  2. maker_bar.encode_songs over --bars bars (--bars / 4 one-phrase songs, one pass): bars/s, median of --rounds.
  3. maker_bar.reconstruct_songs against maker_bar.sample_songs (threshold), alternated --rounds times in this process,
     medians reported:
       - throughput at --songs songs x --phrases phrases: bars/s from CUDA events;
       - latency of one song of --latency-phrases phrases: host wall time of the call ending in a device synchronise.
     sample_songs has to run bar after bar (each bar needs the previous generated bar); the teacher-forced pass knows
     every bar's inputs in advance and runs all bars of all songs as batched passes.

The model has the reference's initialisation (as bench.py --mode decode); the songs are seeded random 5 %-density
rolls.  Prints one JSON object (also written to --out) with the card's name and power limit read in the same run.

    python tools/bench_encode.py --out profiles/encode/bench_encode.json
"""
import argparse
import importlib
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "musicgeneration_vae-torch_b200"
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_sampling import card  # noqa: E402

CELLS = 96 * 60


def songs(S, L, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.rand(S, L * 384, 60, device="cuda", generator=g) < 0.05).float()


def events_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def time_kernel(packed, bars, iters):
    g = torch.Generator(device="cuda").manual_seed(0)
    logits = torch.randn(bars, 1, 96, 60, device="cuda", generator=g) * 3
    target = (torch.rand(bars, 1, 96, 60, device="cuda", generator=g) < 0.05).float()
    for _ in range(5):
        packed.score_bars(logits, target)
    torch.cuda.synchronize()
    ms, _ = events_ms(lambda: [packed.score_bars(logits, target) for _ in range(iters)])
    us = ms * 1e3 / iters
    nbytes = 8 * bars * CELLS
    nll, counts = packed.score_bars(logits, target)
    return {"bars": bars, "cells": bars * CELLS, "iters": iters, "us_per_launch": us, "algorithmic_bytes": nbytes,
            "achieved_TBps": nbytes / (us * 1e-6) / 1e12, "nll_per_bar_mean": float(nll.double().mean()),
            "counts_sum": [int(v) for v in counts.sum(0, dtype=torch.int64).tolist()]}


def time_encode(maker, model, bars, rounds):
    roll = songs(bars // 4, 1, 1)
    maker.encode_songs(model, roll)                        # warm-up of the timed shape
    runs = [bars / (events_ms(lambda: maker.encode_songs(model, roll))[0] * 1e-3) for _ in range(rounds)]
    return {"bars": bars, "bars_per_sec_runs": runs, "bars_per_sec_median": statistics.median(runs)}


def compare(maker, model, S, L, rounds, wall):
    """reconstruct_songs against sample_songs on the same songs' latents, alternated; bars/s (events) or wall ms"""
    roll = songs(S, L, 2)
    lat = maker.encode_songs(model, roll)
    calls = {"reconstruct_songs": lambda: maker.reconstruct_songs(model, roll),
             "sample_songs": lambda: maker.sample_songs(model, lat, L)}
    for fn in calls.values():                             # warm-up: every shape of the timed runs
        fn()
    torch.cuda.synchronize()
    runs = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            if wall:
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                runs[k].append((time.perf_counter() - t0) * 1e3)
            else:
                runs[k].append(S * 4 * L / (events_ms(fn)[0] * 1e-3))
    unit = "wall_ms" if wall else "bars_per_sec"
    res = {"songs": S, "phrases": L, "bars": S * 4 * L, "rounds": rounds}
    for k in calls:
        res[k] = {unit + "_runs": runs[k], unit + "_median": statistics.median(runs[k])}
    a, b = res["reconstruct_songs"][unit + "_median"], res["sample_songs"][unit + "_median"]
    res["speedup_of_reconstruct"] = b / a if wall else a / b
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bars", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--songs", type=int, default=2048)
    ap.add_argument("--phrases", type=int, default=4)
    ap.add_argument("--latency-phrases", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_encode: needs a CUDA device; nothing is measured without one")
    packed = importlib.import_module(PKG + ".data.packed")
    maker = importlib.import_module(PKG + ".maker_bar")
    Model = importlib.import_module(PKG + ".graph.model").Model
    res = {"card": card(), "score_kernel": time_kernel(packed, args.bars, args.iters)}
    model = Model().cuda().eval()
    res["encode_songs"] = time_encode(maker, model, args.bars, args.rounds)
    res["throughput"] = compare(maker, model, args.songs, args.phrases, args.rounds, wall=False)
    res["latency_one_song"] = compare(maker, model, 1, args.latency_phrases, args.rounds, wall=True)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
