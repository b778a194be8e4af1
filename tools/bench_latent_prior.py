"""Cost of the latent prior (csrc/prior.cu, prior.py).

  1. bvae_latent_moments on one --chunk-latent chunk (8192 x 1152 fp32, 38 MB: L2 resident): CUDA events around --iters
     back-to-back launches after a warm-up; fp64 TFLOP/s against the algorithmic 2 * n * d(d+1)/2 (one DFMA per row and
     upper-triangle element).
  2. Its share of one Encoder.encode pass over the same number of bars (bf16 input, CUDA events, median of --rounds).
  3. fit_latent_prior from a packed-array directory of --fit-bars seeded 5 %-density bars against encode_songs alone on
     the same bars: bars/s from host wall time of calls that end in a device synchronise (the fit ends in the host
     finalisation), median of --rounds.
  4. LatentPrior.sample at --draw-songs songs x --draw-bars bars (CUDA events, median of --rounds).
  5. For illustration only: the norm of held-out encoded bars against N(0, I) draws and draws from the fitted prior.

The model has the reference's initialisation (as bench.py --mode decode).  Prints one JSON object (also written to
--out) with the card's name and power limit read in the same run.

    python tools/bench_latent_prior.py --out profiles/prior/bench_latent_prior.json
"""
import argparse
import importlib
import json
import os
import statistics
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "musicgeneration_vae-torch_b200"
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_encode import events_ms, songs  # noqa: E402
from bench_sampling import card  # noqa: E402

D = 1152


def time_kernel(P, n, iters):
    g = torch.Generator(device="cuda").manual_seed(0)
    z = 500.0 + 30.0 * torch.randn(n, D, device="cuda", generator=g)
    s = torch.zeros(D, dtype=torch.float64, device="cuda")
    gram = torch.zeros(D, D, dtype=torch.float64, device="cuda")
    for _ in range(5):
        P.latent_moments(z, s, gram)
    torch.cuda.synchronize()
    ms, _ = events_ms(lambda: [P.latent_moments(z, s, gram) for _ in range(iters)])
    per = ms / iters
    flop = 2.0 * n * D * (D + 1) / 2
    return {"latents": n, "d": D, "iters": iters, "ms_per_launch": per, "algorithmic_fp64_flop": flop,
            "achieved_fp64_TFLOPs": flop / (per * 1e-3) / 1e12}


def time_encode_pass(model, n, rounds):
    x = songs(n // 4, 1, 3).view(n, 1, 96, 60).to(torch.bfloat16)
    with torch.no_grad():
        model.encoder.encode(x)
        runs = [events_ms(lambda: model.encoder.encode(x))[0] for _ in range(rounds)]
    return {"bars": n, "ms_runs": runs, "ms_median": statistics.median(runs)}


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def time_fit(P, maker, packed, model, bars, rounds):
    roll = songs(bars // 4, 1, 4)
    bits = packed.pack_cells(roll.cpu()).reshape(bars, packed.BAR_BYTES)
    with tempfile.TemporaryDirectory() as tmp:
        np.save(os.path.join(tmp, "note_bits.npy"), bits)
        calls = {"fit_latent_prior_packed": lambda: P.fit_latent_prior(model, P.bars_of_packed(tmp)),
                 "encode_songs": lambda: maker.encode_songs(model, roll)}
        for fn in calls.values():
            fn()
        runs = {k: [] for k in calls}
        prior = None
        for _ in range(rounds):
            for k, fn in calls.items():
                t, out = wall(fn)
                runs[k].append(bars / t)
                if k.startswith("fit"):
                    prior = out
    res = {"bars": bars, "rounds": rounds}
    for k in calls:
        res[k] = {"bars_per_sec_runs": runs[k], "bars_per_sec_median": statistics.median(runs[k])}
    res["fit_over_encode"] = (res["fit_latent_prior_packed"]["bars_per_sec_median"]
                              / res["encode_songs"]["bars_per_sec_median"])
    res["prior"] = {"count": prior.count, "mean_norm": float(prior.mean.norm()),
                    "sqrt_trace_over_d": float(torch.trace(prior.cov) / D) ** 0.5, "shrinkage": prior.shrinkage}
    return res, prior


def time_draw(prior, songs_, bars, rounds):
    g = torch.Generator(device="cuda").manual_seed(5)
    prior.sample(bars, songs_, g)
    runs = [events_ms(lambda: prior.sample(bars, songs_, g))[0] for _ in range(rounds)]
    return {"songs": songs_, "bars": bars, "latents": songs_ * bars, "ms_runs": runs, "ms_median": statistics.median(runs)}


def norms(maker, model, prior, n):
    """illustration only: |z| of held-out encoded bars, of N(0, I) draws and of prior draws"""
    held = maker.encode_songs(model, songs(n // 4, 1, 6)).reshape(-1, D)
    g = torch.Generator(device="cuda").manual_seed(7)
    out = {}
    for name, z in (("held_out_encoded", held), ("randn", torch.randn(n, D, device="cuda", generator=g)),
                    ("prior_draws", prior.sample(n, 1, g).view(-1, D))):
        nz = z.double().norm(dim=1)
        out[name] = {"n": int(nz.numel()), "norm_mean": float(nz.mean()), "norm_std": float(nz.std())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunk", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--fit-bars", type=int, default=65536)
    ap.add_argument("--draw-songs", type=int, default=8192)
    ap.add_argument("--draw-bars", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_latent_prior: needs a CUDA device; nothing is measured without one")
    P = importlib.import_module(PKG + ".prior")
    maker = importlib.import_module(PKG + ".maker_bar")
    packed = importlib.import_module(PKG + ".data.packed")
    Model = importlib.import_module(PKG + ".graph.model").Model
    res = {"card": card(), "moments_kernel": time_kernel(P, args.chunk, args.iters)}
    model = Model().cuda().eval()
    enc = time_encode_pass(model, args.chunk, args.rounds)
    res["encode_pass"] = enc
    res["kernel_share_of_encode_pass"] = res["moments_kernel"]["ms_per_launch"] / enc["ms_median"]
    res["fit"], prior = time_fit(P, maker, packed, model, args.fit_bars, args.rounds)
    res["draw"] = time_draw(prior, args.draw_songs, args.draw_bars, args.rounds)
    res["norms_illustration"] = norms(maker, model, prior, args.chunk)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
