#!/usr/bin/env python
"""Generate tests/golden/*.pt by running the UNMODIFIED reference modules on CPU.

TEST INFRASTRUCTURE.  Run in the build container only (needs /root/reference):

    python oracle/gen_golden.py            # writes tests/golden/golden_v1.<i>.pt (oracle/golden_io.py)

The reference has no tests or golden vectors of its own (SURVEY.md section 4), so these
vectors -- outputs of the reference's own ``graph.*`` classes on seeded inputs and on
weights produced by ``barvae_oracle.make_state_dict`` -- are what pins the oracle.
Nothing under /root/reference is copied; the modules are imported from where they lie.

What is injected (and why), without editing any reference source:
  * ``Model.refiner`` is replaced by ``nn.Identity()`` -- graph/refiner.py:19 cannot execute.
  * ``Decoder.dropout`` is replaced by a module that applies pre-drawn keep-masks (scaled by
    1/0.7 like nn.Dropout(0.3)) so that train-mode outputs are reproducible anywhere.
  * ``Tensor.cuda`` / ``Tensor.type('torch.cuda.FloatTensor')`` are shimmed to CPU while
    graph/loss/bar_loss.py:Loss runs (it hard-codes CUDA, :20-21,31-32).
"""
import os
import sys
import time
from collections import OrderedDict

import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("BARVAE_REFERENCE", "/root/reference")
sys.path.insert(0, HERE)
sys.path.insert(0, REF)

import barvae_oracle as O  # noqa: E402
from golden_io import save_golden  # noqa: E402

torch.set_num_threads(8)


class MaskDrop(nn.Module):
    def __init__(self, masks):
        super().__init__()
        self.masks = list(masks)
        self.i = 0

    def forward(self, x):
        m = self.masks[self.i % len(self.masks)]
        self.i += 1
        return x * m / 0.7


class cpu_cuda_shim:
    """Let reference code that hard-codes CUDA run on CPU (bar_loss.py:20-21,31-32)."""

    def __enter__(self):
        self._cuda, self._type = torch.Tensor.cuda, torch.Tensor.type
        torch.Tensor.cuda = lambda s, *a, **k: s
        orig_type = self._type

        def _type(s, dtype=None, *a, **k):
            if isinstance(dtype, str):
                dtype = dtype.replace("torch.cuda.", "torch.")
            return orig_type(s, dtype, *a, **k)
        torch.Tensor.type = _type
        return self

    def __exit__(self, *exc):
        torch.Tensor.cuda, torch.Tensor.type = self._cuda, self._type


def check_spec(module, spec, name):
    sd = module.state_dict()
    assert list(sd.keys()) == list(spec.keys()), (name, set(sd) ^ set(spec))
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(spec[k]), (name, k, tuple(v.shape), spec[k])
    return len(sd)


def sub(sd, prefix):
    return OrderedDict((k[len(prefix):], v) for k, v in sd.items() if k.startswith(prefix))


def main():
    t0 = time.time()
    from graph.encoder import Encoder
    from graph.decoder import Decoder
    from graph.phrase_encoder import PhraseModel
    from graph.cbam import CBAM
    from graph.model import Model

    G = OrderedDict()
    G["meta"] = {"torch": torch.__version__, "reference": "KMU-AELAB-MusicProject/MusicGeneration_VAE-torch",
                 "generator": "oracle/gen_golden.py"}

    model = Model()
    model.refiner = nn.Identity()
    n_keys = check_spec(model, O.generator_spec(), "Model")
    G["meta"]["n_keys"] = n_keys
    G["meta"]["n_params"] = sum(p.numel() for p in model.parameters())
    print("spec ok: %d keys, %d params (%.1fs)" % (n_keys, G["meta"]["n_params"], time.time() - t0))
    check_spec(Encoder(O.ENC_LAYERS), O.encoder_spec(), "Encoder")
    check_spec(Decoder(O.DEC_LAYERS), O.decoder_spec(), "Decoder")
    check_spec(PhraseModel(O.ENC_LAYERS), O.phrase_model_spec(), "PhraseModel")

    B = 2
    for kind in ("lively", "reference"):
        seed_w, seed_x = (11, 21) if kind == "lively" else (12, 22)
        sd = O.make_state_dict(O.generator_spec(), seed_w, kind)
        model.load_state_dict(sd)
        note, pre_note, phrase, position = O.make_inputs(B, seed_x)
        case = {"seed_w": seed_w, "seed_x": seed_x, "B": B, "kind": kind}

        # --- encoder / phrase encoder forward + backward (graph/encoder.py, graph/phrase_encoder.py)
        g = torch.Generator().manual_seed(5)
        r = torch.randn(B, O.LATENT, generator=g)
        model.zero_grad()
        model.eval()
        z = model.encoder(note)
        (z * r).sum().backward()
        case["enc_z"] = z.detach().clone()
        case["enc_grad_digest"] = O.grad_digest(
            OrderedDict((k, p.grad) for k, p in model.named_parameters() if k.startswith("encoder.")))
        model.zero_grad()
        pz = model.phrase_encoder(phrase)
        (pz * r).sum().backward()
        case["phrase_z"] = pz.detach().clone()
        case["phrase_grad_digest"] = O.grad_digest(
            OrderedDict((k, p.grad) for k, p in model.named_parameters() if k.startswith("phrase_encoder.")))

        # --- decoder eval forward from fixed latents (graph/decoder.py:192-222)
        zz = torch.randn(B, O.LATENT, generator=g)
        pzz = torch.randn(B, O.LATENT, generator=g)
        pff = torch.randn(B, O.LATENT, generator=g)
        with torch.no_grad():
            case["dec_eval"] = model.decoder(zz, pzz, pff, position).clone()
            # eval path of Model.forward (graph/model.py:34-41): note slot carries the latent
            case["model_eval"] = model(zz, pre_note, phrase, position, False).clone()

        # --- full training forward/backward, both Loss modes (agent/barGen.py:308-333)
        masks = O.draw_dropout_masks(B, 77)
        from graph.loss.bar_loss import Loss
        for pre in (True, False):
            model.train()
            model.decoder.dropout = MaskDrop(masks)
            model.zero_grad()
            gen, z, pre_z, pf = model(note, pre_note, phrase, position)
            with cpu_cuda_shim():
                loss = Loss()(gen, note, pre)
            loss.backward()
            tag = "train_pre" if pre else "train_smooth"
            case[tag] = {"loss": loss.detach().clone(), "gen": gen.detach().clone(), "z": z.detach().clone(),
                         "pre_z": pre_z.detach().clone(), "pf": pf.detach().clone(),
                         "grad_digest": O.grad_digest(
                             OrderedDict((k, p.grad) for k, p in model.named_parameters()))}
            no_grad = [k for k, p in model.named_parameters() if p.grad is None]
            case[tag]["no_grad_keys"] = no_grad

        # --- two Adam steps (agent/barGen.py:61-62,332-333), lively only (keeps runtime down)
        if kind == "lively":
            model.load_state_dict(sd)
            opt = torch.optim.Adam(model.parameters(), lr=0.002)
            losses = []
            for step in range(2):
                model.decoder.dropout = MaskDrop(masks)
                opt.zero_grad()
                gen, _, _, _ = model(note, pre_note, phrase, position)
                with cpu_cuda_shim():
                    loss = Loss()(gen, note, True)
                loss.backward()
                opt.step()
                losses.append(loss.detach().clone())
            case["adam2"] = {"losses": torch.stack(losses),
                             "param_digest": O.grad_digest(model.state_dict())}
        model.decoder.dropout = nn.Dropout(p=0.3)
        G[kind] = case
        print("case %s done (%.1fs)" % (kind, time.time() - t0))

    # --- CBAM stand-alone (graph/cbam.py:55-68)
    g = torch.Generator().manual_seed(31)
    cb = CBAM(64)
    cb_sd = O.make_state_dict(OrderedDict(O._cbam_spec("", 64)), 41, "lively")
    cb.load_state_dict(cb_sd)
    x = torch.randn(2, 64, 12, 8, generator=g).requires_grad_(True)
    y = cb(x)
    w = torch.randn(y.shape, generator=g)
    (y * w).sum().backward()
    G["cbam"] = {"seed_w": 41, "x": x.detach().clone(), "w": w, "y": y.detach().clone(), "dx": x.grad.clone(),
                 "grad_digest": O.grad_digest(OrderedDict((k, p.grad) for k, p in cb.named_parameters()))}

    # --- Loss on adversarial probabilities (graph/loss/bar_loss.py:23-33)
    from graph.loss.bar_loss import Loss
    g = torch.Generator().manual_seed(51)
    probs = torch.rand(3, 1, 96, 60, generator=g)
    probs.view(-1)[:6] = torch.tensor([0.0, 1.0, 1e-30, 1 - 1e-7, 0.3, 0.30001])
    labels = (torch.rand(3, 1, 96, 60, generator=g) < 0.2).float()
    labels.view(-1)[:6] = torch.tensor([1.0, 0.0, 1.0, 0.0, 1.0, 1.0])
    with cpu_cuda_shim():
        L = Loss()
        G["loss"] = {"probs": probs, "labels": labels,
                     "pre": L(probs, labels, True).clone(), "smooth": L(probs, labels, False).clone()}

    # --- reparameterise + KL (old/graphs/models/bar_v1/encoder.py:60-63, old/graphs/losses/*.py)
    sys.path.insert(0, os.path.join(REF, "old"))
    from graphs.models.bar_v1.encoder import Encoder as OldEncoder
    from graphs.losses.loss import Loss as OldLoss
    g = torch.Generator().manual_seed(61)
    mean = torch.randn(4, O.LATENT, generator=g)
    logvar = torch.randn(4, O.LATENT, generator=g) * 0.5
    torch.manual_seed(99)
    z = OldEncoder.reparameterize(None, mean, logvar)
    torch.manual_seed(99)
    eps = torch.randn_like(mean)
    p = torch.full((4, 1, 96, 60), 0.25)
    t = torch.zeros(4, 1, 96, 60)
    with cpu_cuda_shim():
        total = OldLoss()(p, t, mean, logvar, torch.zeros(()))
        base = OldLoss()(p, t, torch.zeros_like(mean), torch.zeros_like(logvar), torch.zeros(()))
    G["vae_head"] = {"mean": mean, "logvar": logvar, "eps": eps, "z": z.clone(), "kl": (total - base).clone()}

    # --- sampling loop (maker_bar.py:32-44), S=1 song, music_length=2
    sd = O.make_state_dict(O.generator_spec(), 11, "lively")
    model.load_state_dict(sd)
    model.eval()
    music_length = 2
    g = torch.Generator().manual_seed(71)
    latents = torch.randn(music_length * 4, 1, O.LATENT, generator=g)
    outputs = []
    pre_phrase = torch.zeros(1, 1, 384, 60)
    pre_bar = torch.zeros(1, 1, 96, 60)
    phrase_idx = [330] + [i for i in range(music_length - 2, -1, -1)]
    k = 0
    first_probs = None
    with torch.no_grad():
        for idx in range(music_length):
            bar_set = []
            for _ in range(4):
                pre_bar = model(latents[k], pre_bar, pre_phrase, torch.tensor([phrase_idx[idx]]), False)
                if first_probs is None:
                    first_probs = pre_bar.clone()
                k += 1
                pre_bar = torch.gt(pre_bar, 0.3).float()
                bar_set.append(pre_bar.reshape(96, 60))
            ph = torch.cat(bar_set, dim=0)
            outputs.append(ph)
            pre_phrase = ph.reshape(1, 1, 384, 60)
    G["sample"] = {"seed_w": 11, "latents": latents, "roll": torch.cat(outputs, 0).to(torch.uint8),
                   "first_probs": first_probs, "music_length": music_length}

    save_golden(G, "golden_v1")
    print("wrote tests/golden/golden_v1.*.pt in %.1fs" % (time.time() - t0))


if __name__ == "__main__":
    main()
