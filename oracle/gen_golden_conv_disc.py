#!/usr/bin/env python
"""Generate tests/golden/golden_conv_disc_v1.<i>.pt by running the reference's convolutional BarDiscriminator (UNMODIFIED) and
its Refiner on CPU.  TEST INFRASTRUCTURE; build container only (needs /root/reference):

    python oracle/gen_golden_conv_disc.py

The Refiner cannot execute as written: layer1 produces 2 channels and layer2's Conv2d is declared with 1 input channel
(graph/refiner.py:12 vs :19; its own comments :16,:23 give the intended shapes).  No reference source is edited: the
instance is patched in memory -- ``layer2[0] = nn.Conv2d(2, 8, kernel_size=4, padding=2)`` -- which is the one-line fix
SURVEY.md section 8(f) N1 names; everything else runs as the reference wrote it."""
import os
import sys
from collections import OrderedDict

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("BARVAE_REFERENCE", "/root/reference")
sys.path.insert(0, HERE)
sys.path.insert(0, REF)

import barvae_oracle as O  # noqa: E402
import disc_oracle as D  # noqa: E402
from golden_io import save_golden  # noqa: E402

torch.set_num_threads(8)


def run(module, sd, x, training, target_ones=True):
    module.load_state_dict(sd)
    module.train(training)
    module.zero_grad()
    x = x.clone().requires_grad_(True)
    out = module(x)
    if target_ones:
        loss = torch.nn.functional.binary_cross_entropy(out, torch.ones_like(out))      # DLoss (bar_loss.py:36-42)
    else:
        loss = (out * torch.linspace(0.5, 1.5, out.numel()).view_as(out)).mean()         # a fixed probe functional
    loss.backward()
    grads = OrderedDict((k, None if p.grad is None else p.grad.clone()) for k, p in module.named_parameters())
    buffers = OrderedDict((k, v.clone()) for k, v in module.state_dict().items() if "running" in k or "tracked" in k)
    small = OrderedDict((k, v) for k, v in grads.items() if v is None or v.numel() <= 4096)
    big = O.grad_digest(OrderedDict((k, v) for k, v in grads.items() if v is not None and v.numel() > 4096))
    return {"out": out.detach().clone(), "loss": loss.detach().clone(), "dx": x.grad.clone(), "grads": small,
            "grad_digest": big, "buffers_after": buffers}


def main():
    import torch.nn as nn
    from graph.bar_discriminator import BarDiscriminator
    from graph.refiner import Refiner
    from graph.weights_initializer import weights_init

    G = OrderedDict()
    G["meta"] = {"torch": torch.__version__, "reference": "KMU-AELAB-MusicProject/MusicGeneration_VAE-torch"}
    g = torch.Generator().manual_seed(123)
    # discriminator input: cat((pre_note, note), dim=2) -> [B,1,192,60] (agent/barGen_with_gan.py:485-486)
    x = (torch.rand(5, 1, 192, 60, generator=g) < 0.06).float()
    x[0] = torch.rand(1, 192, 60, generator=g)                                           # a generated (soft) bar pair too
    G["disc_x"] = x
    disc = BarDiscriminator()
    spec = D.bar_disc_spec()
    assert list(disc.state_dict().keys()) == list(spec.keys()), [a for a, b in zip(disc.state_dict(), spec) if a != b][:3]
    assert all(tuple(v.shape) == tuple(spec[k]) for k, v in disc.state_dict().items())
    for kind, seed in (("lively", 7), ("reference", 8)):
        sd = D.make_conv_state_dict(spec, seed, kind)
        G["bar_disc/%s/train" % kind] = run(disc, sd, x, True)
        G["bar_disc/%s/eval" % kind] = run(disc, sd, x, False)
    ref = Refiner()
    ref.layer2[0] = nn.Conv2d(2, 8, kernel_size=4, padding=2)                            # the in-memory fix (see docstring)
    ref.layer2[0].apply(weights_init)
    rspec = D.refiner_spec()
    assert list(ref.state_dict().keys()) == list(rspec.keys())
    assert all(tuple(v.shape) == tuple(rspec[k]) for k, v in ref.state_dict().items())
    xr = torch.rand(4, 1, 96, 60, generator=g)
    G["refiner_x"] = xr
    for kind, seed in (("lively", 9), ("reference", 10)):
        sd = D.make_conv_state_dict(rspec, seed, kind)
        G["refiner/%s/train" % kind] = run(ref, sd, xr, True, target_ones=False)
        G["refiner/%s/eval" % kind] = run(ref, sd, xr, False, target_ones=False)
    save_golden(G, "golden_conv_disc_v1")
    print("wrote tests/golden/golden_conv_disc_v1.*.pt")


if __name__ == "__main__":
    main()
