"""CPU: the discriminator / model_with_gan oracle (oracle/disc_oracle.py) against goldens produced by the unmodified
reference classes (oracle/gen_golden_disc.py -> tests/golden/golden_disc_v1.pt)."""
import os
from collections import OrderedDict

import pytest
import torch
import torch.nn.functional as F

from golden_io import load_golden
from gpu_util import ROOT, pkg


@pytest.fixture(scope="module")
def gd():
    return torch.load(os.path.join(ROOT, "tests", "golden", "golden_disc_v1.pt"), map_location="cpu", weights_only=False)


def _run(fwd, spec, seed, kind, x, O, D):
    sd = OrderedDict((k, v.clone().requires_grad_(True)) for k, v in D.make_disc_state_dict(spec, seed, kind).items())
    x = x.clone().requires_grad_(True)
    out = fwd(x, sd)
    loss = F.binary_cross_entropy(out, torch.ones_like(out))
    loss.backward()
    return out.detach(), loss.detach(), x.grad, OrderedDict((k, v.grad) for k, v in sd.items())


@pytest.mark.parametrize("name", ["bar_z", "phrase_z", "feature"])
@pytest.mark.parametrize("kind,seed", [("lively", 5), ("reference", 6)])
def test_disc_oracle_vs_reference_golden(gd, oracle, name, kind, seed):
    import disc_oracle as D
    spec = D.feature_disc_spec() if name == "feature" else D.z_disc_spec()
    fwd = D.feature_disc_forward if name == "feature" else D.z_disc_forward
    out, loss, dx, grads = _run(fwd, spec, seed, kind, gd["x"], oracle, D)
    want = gd["%s/%s" % (name, kind)]
    assert torch.allclose(out, want["out"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(loss, want["loss"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(dx, want["dx"], rtol=1e-4, atol=1e-6 * float(want["dx"].abs().max() + 1e-30))
    dg = oracle.grad_digest(grads)
    for k, w in want["grad_digest"].items():
        assert torch.allclose(dg[k], w, rtol=1e-4, atol=1e-5 * float(w.abs().max() + 1e-30)), k


def test_model_with_gan_oracle_vs_reference_golden(gd, oracle):
    import disc_oracle as D
    sd = oracle.make_state_dict(oracle.generator_spec(), 11, "lively")
    batch = oracle.make_inputs(2, 31)
    with torch.no_grad():
        gen, z, pre_z, pf, zf = D.model_with_gan_forward(*batch, sd, True, None)
        gen2, zf2 = D.model_with_gan_forward(gd["gan/sample"]["latent"], batch[1], batch[2], batch[3], sd, False, None)
    w = gd["gan/train"]
    assert torch.allclose(gen, w["gen"], atol=2e-4) and torch.allclose(z, w["z"], rtol=2e-4, atol=2e-4)
    # the re-encoded feature depends on the thresholded bar: identical thresholding is part of the check
    assert torch.equal(D.fake_note(gen), D.fake_note(w["gen"]))
    assert torch.allclose(zf, w["z_fake"], rtol=2e-4, atol=2e-4)
    w2 = gd["gan/sample"]
    assert torch.allclose(gen2, w2["gen"], atol=2e-4) and torch.allclose(zf2, w2["z_fake"], rtol=2e-4, atol=2e-4)


def test_discriminator_mirrors_keep_reference_keys_and_refuse_cpu():
    import disc_oracle as D
    Z = pkg("graph.z_discriminator")
    Fd = pkg("graph.bar_discriminator_with_feature")
    for cls in (Z.BarZDiscriminator, Z.PhraseZDiscriminator):
        m = cls()
        assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == list(D.z_disc_spec().items())
        with pytest.raises(RuntimeError):
            m(torch.zeros(2, 1152))
    m = Fd.BarFeatureDiscriminator()
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == list(D.feature_disc_spec().items())
    G = pkg("graph.model_with_gan").Model()
    assert list(G.state_dict().keys()) == list(D.O.generator_spec().keys())


@pytest.fixture(scope="module")
def gc():
    return load_golden("golden_conv_disc_v1")


def _run_conv(fwd, spec, seed, kind, x, training, D, target_ones):
    sd = D.make_conv_state_dict(spec, seed, kind)
    leaves = OrderedDict((k, (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()))
                         for k, v in sd.items())
    x = x.clone().requires_grad_(True)
    out = fwd(x, leaves, training)
    if target_ones:
        loss = F.binary_cross_entropy(out, torch.ones_like(out))
    else:
        loss = (out * torch.linspace(0.5, 1.5, out.numel()).view_as(out)).mean()
    loss.backward()
    return out.detach(), loss.detach(), x.grad, leaves


@pytest.mark.parametrize("net", ["bar_disc", "refiner"])
@pytest.mark.parametrize("kind,seed", [("lively", 0), ("reference", 1)])
@pytest.mark.parametrize("training", [True, False])
def test_conv_disc_and_refiner_oracle_vs_reference_golden(gc, net, kind, seed, training):
    """oracle/disc_oracle.py bar_disc_forward / refiner_forward against the reference's BarDiscriminator (unmodified) and its
    Refiner with the in-memory layer2 fix (oracle/gen_golden_conv_disc.py): outputs, loss, input gradient, every parameter
    gradient and the BatchNorm buffers after the call, in training (batch statistics) and eval (running statistics) mode."""
    import disc_oracle as D
    if net == "bar_disc":
        spec, fwd, x, seed = D.bar_disc_spec(), D.bar_disc_forward, gc["disc_x"], 7 + seed
    else:
        spec, fwd, x, seed = D.refiner_spec(), D.refiner_forward, gc["refiner_x"], 9 + seed
    out, loss, dx, leaves = _run_conv(fwd, spec, seed, kind, x, training, D, net == "bar_disc")
    want = gc["%s/%s/%s" % (net, kind, "train" if training else "eval")]
    assert torch.allclose(out, want["out"], rtol=2e-4, atol=1e-5), float((out - want["out"]).abs().max())
    assert torch.allclose(loss, want["loss"], rtol=2e-4, atol=1e-6)
    tol = lambda w: dict(rtol=2e-3, atol=2e-4 * float(w.abs().max() + 1e-30))
    assert torch.allclose(dx, want["dx"], **tol(want["dx"]))
    for k, w in want["grads"].items():
        if w is None:
            assert leaves[k].grad is None, k
        else:
            assert torch.allclose(leaves[k].grad, w, **tol(w)), (k, float((leaves[k].grad - w).abs().max()), float(w.abs().max()))
    dg = __import__("barvae_oracle").grad_digest(OrderedDict((k, leaves[k].grad) for k in want["grad_digest"]))
    for k, w in want["grad_digest"].items():                                  # the tensors too large to store whole
        assert torch.allclose(dg[k], w, rtol=2e-3, atol=2e-4 * float(w.abs().max() + 1e-30)), k
    for k, w in want["buffers_after"].items():
        assert torch.allclose(leaves[k].float(), w.float(), rtol=1e-4, atol=1e-5), k
