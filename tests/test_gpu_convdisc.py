"""GPU: the convolutional BarDiscriminator (graph/bar_discriminator.py) and the Refiner (graph/refiner.py, with the layer2
fix) through libbarvae.so -- bvae_conv_gemm / bvae_wgrad_gemm + bvae_bn_forward / bvae_bn_backward -- against the CPU oracle
(oracle/disc_oracle.py, pinned to the reference classes' own outputs by tests/test_disc_cpu.py) and against the committed
reference goldens directly.
Arithmetic: bf16 GEMM operands / stored activations, fp32 accumulation, fp32 raw conv outputs in front of every BatchNorm,
fp32 statistics.  Tolerances ("lively" weights): output probability |err| <= 2e-2, loss 2e-2 rel (measured 5e-4 / 2e-4) against
the fp32 oracle AND the reference's own golden outputs; input gradient <= 6e-2 and every parameter gradient <= 1e-1
rel-Frobenius against the oracle evaluated at the storage precision (measured: 2.2e-2 / 6.1e-2 in training mode, 8e-4 / 2e-5
in eval mode; values go to gpurun_out/parity_report.jsonl);
BatchNorm running statistics after the call 2e-3.  Reference-init weights (N(-1,1) everywhere, BatchNorm gammas included):
forward only."""
from collections import OrderedDict

import pytest
import torch
import torch.nn.functional as F

from golden_io import load_golden
from gpu_util import pkg, rel_fro, report

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gc():
    return load_golden("golden_conv_disc_v1")


class _Storage:
    """the CUDA path's storage precision (oracle/barvae_emul.py: bf16 value / gradient roundings)"""
    import barvae_emul as _E
    q, gq, wq = staticmethod(_E.q), staticmethod(_E.gq), staticmethod(_E.wq)


def _oracle(fwd, sd, x, training, ones, prec=None):
    leaves = OrderedDict((k, (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()))
                         for k, v in sd.items())
    x = x.clone().requires_grad_(True)
    out = fwd(x, leaves, training) if prec is None else fwd(x, leaves, training, prec)
    loss = F.binary_cross_entropy(out, torch.ones_like(out)) if ones else \
        (out * torch.linspace(0.5, 1.5, out.numel()).view_as(out)).mean()
    loss.backward()
    return out.detach(), float(loss), x.grad, leaves


@pytest.mark.parametrize("net", ["bar_disc", "refiner"])
@pytest.mark.parametrize("training", [True, False])
def test_conv_nets_forward_backward_vs_oracle(gc, net, training):
    import disc_oracle as D
    if net == "bar_disc":
        cls, spec, fwd, x, seed = pkg("graph.bar_discriminator").BarDiscriminator, D.bar_disc_spec(), D.bar_disc_forward, gc["disc_x"], 7
    else:
        cls, spec, fwd, x, seed = pkg("graph.refiner").Refiner, D.refiner_spec(), D.refiner_forward, gc["refiner_x"], 9
    sd = D.make_conv_state_dict(spec, seed, "lively")
    # Gradients are compared with the oracle evaluated at the CUDA path's storage precision: both nets end in BatchNorm ->
    # global average pool, whose backward pass cancels (dy - mean(dy) - xhat mean(dy xhat) with a spatially constant dy), so
    # rounding ONLY the weights to bf16 inside the fp32 oracle already moves dx by 18 % and single tensors by 7-100 % while the
    # output moves 3e-4 (measured, tools/ note in DESIGN.md section 7).  Outputs / loss / buffers are held against fp32.
    want_out, want_loss, _, leaves32 = _oracle(fwd, sd, x, training, net == "bar_disc")
    _, _, want_dx, leaves = _oracle(fwd, sd, x, training, net == "bar_disc", _Storage)
    gold = gc["%s/lively/%s" % (net, "train" if training else "eval")]
    m = cls()
    assert list(m.state_dict().keys()) == list(spec.keys())                 # the reference's parameter AND buffer names
    m.load_state_dict(sd)
    m = m.cuda().train(training)
    xg = x.cuda().requires_grad_(True)
    out = m(xg)
    if net == "bar_disc":
        loss = pkg("graph.loss.bar_loss").DLoss()(out, torch.ones_like(out))
    else:
        loss = (out * torch.linspace(0.5, 1.5, out.numel(), device="cuda").view_as(out)).mean()
    loss.backward()
    torch.cuda.synchronize()
    errs = {"out_maxabs": float((out.detach().cpu() - want_out).abs().max()),
            "out_vs_reference_golden": float((out.detach().cpu() - gold["out"]).abs().max()),
            "loss_rel": abs(float(loss) - want_loss) / abs(want_loss), "dx": rel_fro(xg.grad, want_dx)}
    worst = 0.0
    for k, p in m.named_parameters():
        if leaves[k].grad is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k    # ConvModule.bn1 of the isBasic block: unused
            continue
        if net == "refiner" and training and k in ("layer1.0.bias", "layer2.0.bias"):
            # a bias in front of a batch-statistics BatchNorm: analytically zero gradient -- exactly zero here, fp32
            # rounding noise in the oracle (graph/_smallnet.py conv(bias_grad=False))
            gmax = max(float(v.grad.abs().max()) for v in leaves32.values() if v.grad is not None)
            assert float(p.grad.abs().max()) == 0.0 and float(leaves32[k].grad.abs().max()) < 1e-4 * gmax, k
            continue
        errs[k] = rel_fro(p.grad, leaves[k].grad)
        worst = max(worst, errs[k])
    bufs = {k: v for k, v in m.state_dict().items() if "running" in k}
    berr = max(float((v.cpu() - leaves32[k]).abs().max() / (leaves32[k].abs().max() + 1e-6)) for k, v in bufs.items())
    nbt = all(int(v) == int(leaves32[k]) for k, v in m.state_dict().items() if "tracked" in k)
    report(test="conv_net", net=net, training=training, out_maxabs=errs["out_maxabs"], out_vs_golden=errs["out_vs_reference_golden"],
           loss_rel=errs["loss_rel"], dx=errs["dx"], worst_param_grad=worst, running_stats=berr)
    assert errs["out_maxabs"] < 2e-2 and errs["out_vs_reference_golden"] < 2e-2 and errs["loss_rel"] < 2e-2, errs
    assert errs["dx"] < 6e-2 and worst < 1e-1, {k: v for k, v in errs.items() if isinstance(v, float) and v > 3e-2}
    assert berr < 2e-3 and nbt, berr


@pytest.mark.parametrize("net", ["bar_disc", "refiner"])
def test_conv_nets_reference_init_forward(gc, net):
    """reference initialisation (N(-1,1) convolution, Linear AND BatchNorm weights, fresh running statistics): forward against
    the reference's golden outputs and against the storage-precision oracle.  One case is held to the latter only: the
    Refiner in EVAL mode with fresh running statistics normalises nothing, its activations grow to ~1e3 and bf16 storage of
    them moves the pre-sigmoid values by O(1) -- a state no trained model is in (one training step updates the statistics)."""
    import disc_oracle as D
    if net == "bar_disc":
        cls, spec, fwd, x, seed = pkg("graph.bar_discriminator").BarDiscriminator, D.bar_disc_spec(), D.bar_disc_forward, gc["disc_x"], 8
    else:
        cls, spec, fwd, x, seed = pkg("graph.refiner").Refiner, D.refiner_spec(), D.refiner_forward, gc["refiner_x"], 10
    for training in (True, False):
        sd = D.make_conv_state_dict(spec, seed, "reference")
        m = cls()
        m.load_state_dict(sd)
        m = m.cuda().train(training)
        with torch.no_grad():
            out = m(x.cuda())
            emu = fwd(x, OrderedDict((k, v.clone()) for k, v in sd.items()), training, _Storage)
        want = gc["%s/reference/%s" % (net, "train" if training else "eval")]["out"]
        e, e2 = float((out.cpu() - want).abs().max()), float((out.cpu() - emu).abs().max())
        report(test="conv_net_reference_init", net=net, training=training, out_maxabs=e, out_vs_storage_precision_oracle=e2)
        assert e2 < 3e-2, (net, training, e2)
        assert e < 3e-2 or (net == "refiner" and not training), (net, training, e)


def test_frozen_discriminator_still_propagates_input_gradient(gc):
    """agent/barGen_with_gan.py:506-528: the generator step runs the discriminator with requires_grad=False on all of its
    parameters and backpropagates into the generated bar"""
    import disc_oracle as D
    m = pkg("graph.bar_discriminator").BarDiscriminator()
    m.load_state_dict(D.make_conv_state_dict(D.bar_disc_spec(), 7, "lively"))
    m = m.cuda().train()
    for p in m.parameters():
        p.requires_grad = False
    x = gc["disc_x"].cuda().requires_grad_(True)
    F.binary_cross_entropy(m(x), torch.ones(5, 1, device="cuda")).backward()
    assert x.grad is not None and float(x.grad.abs().sum()) > 0
    assert all(p.grad is None for p in m.parameters())


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


_SMALL_CONVS = [(1, 8, (3, 1), (2, 1), (1, 0), 192, 12), (8, 16, (3, 1), (2, 1), (1, 0), 96, 12), (16, 16, 1, 1, 0, 48, 12),
                (16, 32, 3, 2, 1, 48, 12), (32, 64, 3, 2, 1, 24, 6), (1, 8, 3, (2, 1), 1, 192, 1), (8, 8, 3, (2, 1), 1, 96, 1),
                (1, 8, (1, 4), (1, 2), (0, 1), 192, 60), (8, 8, (4, 1), (2, 1), (1, 0), 192, 30), (16, 8, 1, 1, 0, 96, 30),
                (8, 8, 3, 1, 1, 96, 30), (8, 16, 3, 2, 1, 96, 30), (1, 2, 4, 1, 2, 96, 60), (2, 8, 4, 1, 2, 48, 30),
                (32, 32, 1, 1, 0, 12, 1)]


@pytest.mark.parametrize("spec", _SMALL_CONVS, ids=lambda s: "%dto%d_k%s_s%s" % (s[0], s[1], s[2], s[3]))
@pytest.mark.parametrize("act", [False, True])
def test_small_channel_conv_ops_vs_torch(spec, act):
    """every convolution shape of the BarDiscriminator / Refiner through graph/_smallnet.conv (forward, weight gradient,
    data gradient: csrc/conv_small.cu for < 32 channels, the tcgen05 kernels otherwise) against torch.nn.functional on the
    same bf16-representable operands: fp32 outputs 1e-5, bf16 outputs / gradients 4e-3 (one bf16 rounding)"""
    import torch.nn as nn
    S = pkg("graph._smallnet")
    cin, cout, k, s, p, H, W = spec
    torch.manual_seed(1)
    m = nn.Conv2d(cin, cout, k, s, p, bias=False).cuda()
    x = torch.randn(3, cin, H, W, device="cuda").to(torch.bfloat16).float().requires_grad_(True)
    with torch.no_grad():
        m.weight.copy_(m.weight.to(torch.bfloat16).float())
    ref = m(x)
    if act:
        ref = F.relu(ref)
    g = torch.randn_like(ref).to(torch.bfloat16).float()
    ref.backward(g)
    rw, rx = m.weight.grad.clone(), x.grad.clone()
    m.weight.grad = None
    x2 = x.detach().permute(0, 2, 3, 1).contiguous().requires_grad_(True)
    out = S.conv(x2, m, act=act, out_f32=not act)
    out.backward(g.permute(0, 2, 3, 1).contiguous().to(out.dtype))
    e = (_rel(out.permute(0, 3, 1, 2).float(), ref), _rel(m.weight.grad, rw), _rel(x2.grad.permute(0, 3, 1, 2), rx))
    assert e[0] < (4e-3 if act else 1e-5) and e[1] < 1e-4 and e[2] < 4e-3, e


@pytest.mark.parametrize("cin,cout,H,W", [(8, 2, 24, 15), (2, 1, 48, 30)])
def test_small_channel_transposed_conv_vs_torch(cin, cout, H, W):
    import torch.nn as nn
    S = pkg("graph._smallnet")
    torch.manual_seed(2)
    m = nn.ConvTranspose2d(cin, cout, 4, 2, 1, bias=False).cuda()
    x = torch.randn(3, cin, H, W, device="cuda").to(torch.bfloat16).float().requires_grad_(True)
    with torch.no_grad():
        m.weight.copy_(m.weight.to(torch.bfloat16).float())
    ref = m(x)
    g = torch.randn_like(ref).to(torch.bfloat16).float()
    ref.backward(g)
    rw, rx = m.weight.grad.clone(), x.grad.clone()
    m.weight.grad = None
    x2 = x.detach().permute(0, 2, 3, 1).contiguous().requires_grad_(True)
    out = S.conv(x2, m)
    out.backward(g.permute(0, 2, 3, 1).contiguous())
    e = (_rel(out.permute(0, 3, 1, 2).float(), ref), _rel(m.weight.grad, rw), _rel(x2.grad.permute(0, 3, 1, 2), rx))
    assert e[0] < 1e-5 and e[1] < 1e-4 and e[2] < 4e-3, e


@pytest.mark.parametrize("C", [1, 2, 8, 16, 64])
@pytest.mark.parametrize("act,training,xf32", [(False, True, True), (True, True, True), (True, False, True), (False, True, False)])
def test_batch_norm_op_vs_torch(C, act, training, xf32):
    """bvae_bn_forward / bvae_bn_backward against nn.BatchNorm2d (+ReLU): output and dx within one bf16 rounding, dgamma /
    dbeta and the updated running statistics to fp32 precision"""
    import copy
    import torch.nn as nn
    S = pkg("graph._smallnet")
    torch.manual_seed(3)
    bn = nn.BatchNorm2d(C, momentum=0.01).cuda().train(training)
    with torch.no_grad():
        bn.weight.normal_(1, 0.3)
        bn.bias.normal_(0, 0.3)
        bn.running_mean.normal_(0, 0.2)
        bn.running_var.uniform_(0.5, 1.5)
    bn2 = copy.deepcopy(bn)
    x = torch.randn(4, C, 24, 15, device="cuda") * 2 + 3
    if not xf32:
        x = x.to(torch.bfloat16).float()
    x.requires_grad_(True)
    ref = bn(x)
    if act:
        ref = F.relu(ref)
    g = torch.randn_like(ref).to(torch.bfloat16).float()
    ref.backward(g)
    x2 = x.detach().permute(0, 2, 3, 1).contiguous()
    if not xf32:
        x2 = x2.to(torch.bfloat16)
    x2.requires_grad_(True)
    out = S.batch_norm(x2, bn2, act=act)
    out.backward(g.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16))
    assert _rel(out.permute(0, 3, 1, 2).float(), ref) < 4e-3 and _rel(x2.grad.permute(0, 3, 1, 2).float(), x.grad) < 4e-3
    assert _rel(bn2.weight.grad, bn.weight.grad) < 1e-4 and _rel(bn2.bias.grad, bn.bias.grad) < 1e-4
    assert _rel(bn2.running_mean, bn.running_mean) < 1e-5 and _rel(bn2.running_var, bn.running_var) < 1e-5
    assert int(bn2.num_batches_tracked) == int(bn.num_batches_tracked)
