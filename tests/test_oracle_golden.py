"""CPU: pin the oracle restatement (oracle/barvae_oracle.py) to outputs of the reference itself
(tests/golden/golden_v1.<i>.pt, produced by oracle/gen_golden.py from the reference's own modules)."""
from collections import OrderedDict

import pytest
import torch

from conftest import assert_close

TOL = dict(rtol=2e-4, atol=1e-6)     # fp32 CPU vs fp32 CPU, same library: reduction-order noise only
# Gradients: with the "lively" weights fp32 and fp64 agree to ~1e-3 per tensor, so the digests are held to 5e-3.
# With the reference's own N(-1,1) initialisation (graph/weights_initializer.py:5-23) the backward pass is
# ill-conditioned in fp32 (activations ~1e6, dead ReLUs, saturated gates): the SAME code run with 1 vs 8 CPU
# threads differs by >100 % on some tensors (measured: decoder.cbam.channel_attention.*, decoder.bn.bias), so
# for that initialisation only an order-of-magnitude check of the digests is meaningful; forward outputs and the
# loss stay tight for both.  See DESIGN.md "Parity tolerances".
GRAD_TOL = {"lively": dict(rtol=5e-3, floor_rel=1e-6), "reference": dict(rtol=3.0, floor_rel=1e-2)}


def _digest_close(got, want, what, rtol=2e-3, floor_rel=1e-6):
    """digest rows are [sum, abs-sum, sum-of-squares, samples...]; tensors whose gradient is analytically zero
    (e.g. a conv bias in front of an InstanceNorm) hold only rounding noise, hence the global absolute floor."""
    assert set(got) == set(want), (what, set(got) ^ set(want))
    floor = floor_rel * max(float(w[1]) for w in want.values())
    for k in want:
        g, w = got[k].double(), want[k].double()
        assert abs(g[1] - w[1]) <= rtol * abs(w[1]) + floor, (what, k, "abs-sum", float(g[1]), float(w[1]))
        assert abs(g[0] - w[0]) <= rtol * abs(w[1]) + floor, (what, k, "sum", float(g[0]), float(w[0]))
        assert abs(g[2] - w[2]) <= 2 * rtol * abs(w[2]) + floor * floor, (what, k, "sumsq", float(g[2]), float(w[2]))


@pytest.mark.parametrize("kind", ["lively", "reference"])
def test_encoders(golden, oracle, kind):
    O, c = oracle, golden[kind]
    sd = O.make_state_dict(O.generator_spec(), c["seed_w"], kind)
    note, pre_note, phrase, position = O.make_inputs(c["B"], c["seed_x"])
    r = torch.randn(c["B"], O.LATENT, generator=torch.Generator().manual_seed(5))
    leaves = OrderedDict((k, v.clone().requires_grad_(True)) for k, v in sd.items())
    z = O.encoder_forward(note, leaves, "encoder.")
    assert_close(z, c["enc_z"], what="enc_z", **TOL)
    (z * r).sum().backward()
    dg = O.grad_digest(OrderedDict((k, v.grad) for k, v in leaves.items() if k.startswith("encoder.")))
    _digest_close(dg, c["enc_grad_digest"], "enc_grad", **GRAD_TOL[kind])
    pz = O.phrase_model_forward(phrase, sd, "phrase_encoder.")
    assert_close(pz, c["phrase_z"], what="phrase_z", **TOL)


@pytest.mark.parametrize("kind", ["lively", "reference"])
def test_decoder_and_eval_path(golden, oracle, kind):
    O, c = oracle, golden[kind]
    sd = O.make_state_dict(O.generator_spec(), c["seed_w"], kind)
    note, pre_note, phrase, position = O.make_inputs(c["B"], c["seed_x"])
    g = torch.Generator().manual_seed(5)
    torch.randn(c["B"], O.LATENT, generator=g)
    zz = torch.randn(c["B"], O.LATENT, generator=g)
    pzz = torch.randn(c["B"], O.LATENT, generator=g)
    pff = torch.randn(c["B"], O.LATENT, generator=g)
    with torch.no_grad():
        assert_close(O.decoder_forward(zz, pzz, pff, position, sd, "decoder."), c["dec_eval"], what="dec_eval", **TOL)
        assert_close(O.model_forward(zz, pre_note, phrase, position, sd, False), c["model_eval"], what="model_eval",
                     **TOL)


@pytest.mark.parametrize("kind", ["lively", "reference"])
@pytest.mark.parametrize("pre", [True, False])
def test_train_forward_backward(golden, oracle, kind, pre):
    O, c = oracle, golden[kind]
    want = c["train_pre" if pre else "train_smooth"]
    sd = O.make_state_dict(O.generator_spec(), c["seed_w"], kind)
    batch = O.make_inputs(c["B"], c["seed_x"])
    masks = O.draw_dropout_masks(c["B"], 77)
    leaves = OrderedDict((k, v.clone().requires_grad_(True)) for k, v in sd.items())
    gen, z, pre_z, pf = O.model_forward(*batch, leaves, True, masks)
    loss = O.loss_forward(gen, batch[0], pre)
    loss.backward()
    assert_close(gen, want["gen"], what="gen", **TOL)
    assert_close(z, want["z"], what="z", **TOL)
    assert_close(pf, want["pf"], what="pf", **TOL)
    assert_close(loss, want["loss"], what="loss", rtol=1e-5, atol=1e-6)
    none = [k for k, v in leaves.items() if v.grad is None]
    assert sorted(none) == sorted(want["no_grad_keys"])          # the 4 unused bn1 gamma/beta (decoder.py:137,142)
    assert len(none) == 4
    dg = O.grad_digest(OrderedDict((k, v.grad) for k, v in leaves.items()))
    _digest_close(dg, want["grad_digest"], "grads", **GRAD_TOL[kind])


def test_adam_two_steps(golden, oracle):
    O, c = oracle, golden["lively"]
    sd = O.make_state_dict(O.generator_spec(), c["seed_w"], "lively")
    batch = O.make_inputs(c["B"], c["seed_x"])
    masks = O.draw_dropout_masks(c["B"], 77)
    m = OrderedDict((k, torch.zeros_like(v)) for k, v in sd.items())
    v = OrderedDict((k, torch.zeros_like(t)) for k, t in sd.items())
    losses = []
    for step in (1, 2):
        loss, _, _ = O.train_step(sd, batch, m, v, step, 0.002, masks, True)
        losses.append(loss)
    assert_close(torch.stack(losses), c["adam2"]["losses"], what="losses", rtol=1e-4, atol=1e-6)
    _digest_close(O.grad_digest(sd), c["adam2"]["param_digest"], "params", rtol=1e-4)


def test_cbam(golden, oracle):
    O, c = oracle, golden["cbam"]
    sd = O.make_state_dict(OrderedDict(O._cbam_spec("", 64)), c["seed_w"], "lively")
    x = c["x"].clone().requires_grad_(True)
    y = O.cbam(x, sd, "")
    (y * c["w"]).sum().backward()
    assert_close(y, c["y"], what="cbam y", **TOL)
    assert_close(x.grad, c["dx"], what="cbam dx", **TOL)


def test_loss(golden, oracle):
    O, c = oracle, golden["loss"]
    assert_close(O.loss_forward(c["probs"], c["labels"], True), c["pre"], what="loss pre", rtol=1e-6, atol=1e-6)
    assert_close(O.loss_forward(c["probs"], c["labels"], False), c["smooth"], what="loss smooth", rtol=1e-6, atol=1e-6)


def test_vae_head(golden, oracle):
    O, c = oracle, golden["vae_head"]
    assert_close(O.reparameterize(c["mean"], c["logvar"], c["eps"]), c["z"], what="reparam", rtol=1e-6, atol=1e-6)
    assert_close(O.kl_sum(c["mean"], c["logvar"]), c["kl"], what="kl", rtol=1e-4, atol=1e-3)


def test_sampling_loop(golden, oracle):
    O, c = oracle, golden["sample"]
    sd = O.make_state_dict(O.generator_spec(), c["seed_w"], "lively")
    with torch.no_grad():
        roll = O.sample_song(sd, c["latents"], c["music_length"])
    assert roll.shape == (1, c["music_length"] * 4 * 96, 60)
    assert torch.equal(roll[0].to(torch.uint8), c["roll"])


def test_emulation_exact_mode_is_the_oracle(oracle):
    """oracle/barvae_emul.py with every rounding switched off must BE the fp32 oracle: pins its hand-written norm-block
    backward (InstanceNorm projection on the saved normalised activation, CBAM routes taken at saved arg-max positions)
    against plain autograd through barvae_oracle.  Tensors below 1e-6 of the gradient norm (biases in front of an
    InstanceNorm: analytically zero) are rounding noise on both sides."""
    import barvae_emul as E
    from collections import OrderedDict
    O = oracle
    sd = O.make_state_dict(O.generator_spec(), 11, "lively")
    batch = O.make_inputs(2, 21)
    masks = O.draw_dropout_masks(2, 77)
    leaves = OrderedDict((k, v.clone().requires_grad_(True)) for k, v in sd.items())
    og = O.model_forward(*batch, leaves, True, masks)[0]
    ol = O.loss_forward(og, batch[0], True)
    ol.backward()
    with E.exact():
        el, egen, ez, eg = E.train_grads(sd, batch, masks)
    assert float((egen - og.detach()).abs().max()) < 1e-4
    assert abs(float(el) - float(ol)) < 1e-5 * abs(float(ol))
    gnorm = sum(float(v.grad.norm()) ** 2 for v in leaves.values() if v.grad is not None) ** 0.5
    for k, v in leaves.items():
        if v.grad is None:
            assert eg[k] is None, k
            continue
        n = float(v.grad.norm())
        if n < 1e-6 * gnorm:
            assert float(eg[k].norm()) < 1e-6 * gnorm, k
            continue
        # (fp32 on the CPU is itself not reproducible across thread counts on the smallest tensors: absolute floor)
        e = float((eg[k] - v.grad).norm())
        assert e < 2e-2 * n or e < 2e-5 * gnorm, (k, e / n, e / gnorm)
    # and the rounded mode differs from the oracle only by bf16-sized forward changes
    l2, gen2, _, _ = E.train_grads(sd, batch, masks)
    assert float((gen2 - og.detach()).abs().max()) < 6e-2
