"""GPU (B200) kernel-level parity, all through the C ABI of libbarvae.so (ctypes).

Floating-point kernels: the comparison is against plain PyTorch fp32 ops on the same device, on inputs that are
already bf16-representable, so the only differences are accumulation order and the bf16 rounding of stored outputs.
Tolerances are stated per test."""
import math

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from gpu_util import nchw, nhwc, pkg, rel_fro, report

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16
# the PyTorch side of every comparison must be true fp32 (cuDNN/cuBLAS default to TF32 for convs on this GPU)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def _bf(t):
    return t.to(BF16).float()


LAYERS = [
    # kind, cin, cout, kernel, stride, padding, output_padding, H, W          (reference site)
    ("conv", 64, 64, (3, 3), (1, 1), (1, 1), (0, 0), 12, 10),                # encodingBlock.py:74-77
    ("conv", 64, 128, (3, 3), (2, 2), (1, 1), (0, 0), 24, 15),               # encodingBlock.py:107 (odd width)
    ("conv", 32, 32, (1, 4), (1, 2), (0, 1), (0, 0), 12, 60),                # encodingBlock.py:14
    ("conv", 32, 32, (4, 1), (2, 1), (1, 0), (0, 0), 96, 30),                # encodingBlock.py:45
    ("conv", 1, 32, (4, 1), (2, 1), (1, 0), (0, 0), 96, 60),                 # encodingBlock.py:12 (C_in = 1)
    ("conv", 1, 32, (1, 4), (1, 2), (0, 1), (0, 0), 96, 60),                 # encodingBlock.py:43
    ("conv", 256, 128, (1, 1), (1, 1), (0, 0), (0, 0), 6, 5),                # decoder.py:79
    ("convT", 128, 64, (1, 3), (1, 3), (0, 0), (0, 0), 1, 1),                # decoder.py:43 (k == stride)
    ("convT", 64, 64, (6, 1), (6, 1), (0, 0), (0, 0), 1, 3),                 # decoder.py:45
    ("convT", 128, 64, (4, 4), (2, 2), (1, 1), (0, 1), 6, 3),                # decoder.py:116 (odd output width)
    ("convT", 64, 32, (4, 4), (2, 2), (1, 1), (0, 0), 12, 15),               # decoder.py:73
    ("convT", 64, 32, (3, 3), (2, 2), (1, 1), (1, 1), 12, 15),               # decoder.py:76
]


@pytest.mark.parametrize("spec", LAYERS, ids=lambda s: "%s_%dto%d_k%dx%d_s%dx%d" % (s[0], s[1], s[2], *s[3], *s[4]))
@pytest.mark.parametrize("impl", ["simt", "tc"])
def test_gemm_layer(spec, impl):
    """forward / data-gradient / weight-gradient of one layer vs torch.nn.functional (fp32).
    Tolerance: rel-Frobenius 2e-3 (fp32 outputs; operands are bf16-exact, so this is accumulation-order noise)."""
    eng = pkg("engine")
    lib = pkg("_lib")
    kind, cin, cout, k, s, p, op, H, W = spec
    if impl == "tc" and cin == 1:
        impl = "auto"            # C_in = 1 stems: dedicated streaming kernels (stem.cu), nothing for a tensor core to do
    _run_gemm_layer(spec, impl, 3)


BIG_LAYERS = [
    ("conv", 128, 256, (3, 3), (2, 2), (1, 1), (0, 0), 24, 15, 9),           # several M tiles, N tile 256
    ("conv", 256, 256, (3, 3), (1, 1), (1, 1), (0, 0), 12, 8, 11),           # boxes spanning several samples
    ("conv", 512, 1024, (3, 3), (2, 2), (1, 1), (0, 0), 6, 4, 7),            # 4 N tiles, K = 4608
    ("conv", 2048, 1024, (1, 1), (1, 1), (0, 0), (0, 0), 6, 3, 5),           # decoder.fit1
    ("conv", 2304, 1152, (1, 1), (1, 1), (0, 0), (0, 0), 1, 1, 130),         # Linear 2304 -> 1152 (N tile 192)
    ("convT", 2304, 1024, (6, 1), (6, 1), (0, 0), (0, 0), 1, 1, 33),         # decoder.time.time
    ("convT", 1024, 512, (4, 4), (2, 2), (1, 1), (0, 1), 6, 3, 6),           # decoder.layers.0.deConv1
    ("convT", 128, 64, (3, 3), (2, 2), (1, 1), (1, 1), 48, 30, 2),           # decoder.layers.3.deConv2
    ("conv", 64, 64, (3, 3), (1, 1), (1, 1), (0, 0), 48, 30, 4),             # encoder.layers.0
    ("conv", 32, 32, (1, 4), (1, 2), (0, 1), (0, 0), 192, 60, 2),            # phrase stem (KB = 32, SWIZZLE_64B)
    ("conv", 32, 32, (1, 4), (1, 2), (0, 1), (0, 0), 192, 60, 7),            # resident weights without halo (>= 296 tiles)
    # halo mode (one shared-memory tile per output tile, taps = row-shifted descriptors; needs >= 296 tiles)
    ("conv", 64, 64, (3, 3), (1, 1), (1, 1), (0, 0), 48, 30, 26),            # padded width 32, 4 rows per tile
    ("conv", 64, 64, (3, 3), (1, 1), (1, 1), (0, 0), 20, 60, 30),            # padded width 62, 2 rows per tile
    ("conv", 64, 64, (3, 3), (1, 1), (1, 1), (0, 0), 21, 13, 100),           # ragged: width 15, 8 rows, H % 8 != 0
    ("conv", 64, 64, (1, 4), (1, 1), (0, 1), (0, 0), 40, 30, 30),            # asymmetric taps, output narrower than input
]


@pytest.mark.parametrize("spec", BIG_LAYERS, ids=lambda s: "%s_%dto%d_k%dx%d_B%d" % (s[0], s[1], s[2], *s[3], s[9]))
def test_gemm_layer_tc_big(spec):
    """the tcgen05 kernels at multi-tile sizes (several M / N tiles, long K loops, split-K weight gradients)"""
    _run_gemm_layer(spec[:9], "tc", spec[9])


def _run_gemm_layer(spec, impl, B):
    eng = pkg("engine")
    lib = pkg("_lib")
    kind, cin, cout, k, s, p, op, H, W = spec
    torch.manual_seed(1)
    if kind == "conv":
        m = nn.Conv2d(cin, cout, k, s, p, bias=True).cuda()
    else:
        m = nn.ConvTranspose2d(cin, cout, k, s, p, output_padding=op, bias=True).cuda()
    with torch.no_grad():
        m.weight.copy_(_bf(torch.randn_like(m.weight) * 0.2))
        m.bias.copy_(_bf(torch.randn_like(m.bias)))
    g = pkg("graph.encodingBlock").gemm_of(m)
    x = _bf(torch.randn(B, cin, H, W, device="cuda")).requires_grad_(True)
    ref = m(x)
    OH, OW = ref.shape[2], ref.shape[3]
    assert (OH, OW) == g.out_hw(H, W)
    dyt = _bf(torch.randn_like(ref))
    ref.backward(dyt)
    ref_dx, ref_dw, ref_db = x.grad.clone(), m.weight.grad.clone(), m.bias.grad.clone()
    m.weight.grad = None
    m.bias.grad = None

    eng.set_impl({"simt": lib.IMPL_SIMT, "tc": lib.IMPL_TC, "auto": lib.IMPL_AUTO}[impl])
    try:
        xa = eng.Act(nhwc(x.detach()).to(BF16), B, H, W, cin)
        y = eng.Act.empty(B, OH, OW, cout, dtype=torch.float32)
        y.t.fill_(float("nan"))
        g.forward(xa, y)
        e_f = rel_fro(nchw(y.t), ref)
        dya = eng.Act(nhwc(dyt).to(BF16), B, OH, OW, cout)
        dx = eng.Act.empty(B, H, W, cin, dtype=torch.float32)
        dx.t.fill_(float("nan"))
        g.dgrad(dya, dx)
        e_d = rel_fro(nchw(dx.t), ref_dx)
        g.wgrad(xa, dya)
        g.bias_grad(dya)
        e_w = rel_fro(m.weight.grad, ref_dw)
        e_b = rel_fro(m.bias.grad, ref_db)
        # bf16 output + fused epilogue: bias, ReLU, addend, mask
        y2 = eng.Act.empty(B, OH, OW, cout)
        g.forward(xa, y2, act=True, slope=0.01)
        e_a = rel_fro(nchw(y2.t.float()), F.leaky_relu(ref, 0.01))
        add = eng.Act(torch.randn(B, H, W, cin, device="cuda").to(BF16), B, H, W, cin)
        msk = eng.Act(torch.randn(B, H, W, cin, device="cuda").to(BF16), B, H, W, cin)
        dx2 = eng.Act.empty(B, H, W, cin)
        g.dgrad(dya, dx2, addend=add, mask=msk, mask_slope=0.01)
        want = (ref_dx + nchw(add.t.float())) * torch.where(nchw(msk.t.float()) > 0, 1.0, 0.01)
        e_m = rel_fro(nchw(dx2.t.float()), want)
    finally:
        eng.set_impl(lib.IMPL_AUTO)
    report(test="gemm_layer", impl=impl, B=B, spec=str(spec), fwd=e_f, dgrad=e_d, wgrad=e_w, bias=e_b, act=e_a, mask=e_m)
    assert e_f < 2e-3 and e_d < 2e-3 and e_w < 2e-3 and e_b < 2e-3, (e_f, e_d, e_w, e_b)
    assert e_a < 6e-3 and e_m < 6e-3, (e_a, e_m)        # bf16 output rounding (2^-9 per element)


def _torch_block(y, gamma, beta, cb, res_mode, slope, res):
    """fp32 reference of the fused norm block, NCHW (the same ops the reference modules call)."""
    u = F.instance_norm(y, None, None, gamma, beta, True, 0.01, 1e-5)
    if cb is None:
        out = u
    else:
        w1, w2, wsp = cb
        a = F.conv2d(F.relu(F.conv2d(F.adaptive_avg_pool2d(u, 1), w1)), w2)
        m = F.conv2d(F.relu(F.conv2d(F.adaptive_max_pool2d(u, 1), w1)), w2)
        u1 = u * torch.sigmoid(a + m)
        sa = torch.cat([u1.mean(1, keepdim=True), u1.max(1, keepdim=True)[0]], 1)
        c = u1 * torch.sigmoid(F.conv2d(sa, wsp, padding=1))
        out = {1: u + c, 2: (res + c) if res is not None else c, 3: c}[res_mode]
    return F.leaky_relu(out, slope) if slope != 0 else F.relu(out)


@pytest.mark.parametrize("C,H,W", [(32, 48, 30), (64, 12, 8), (128, 24, 15), (512, 6, 4), (1024, 3, 2), (64, 96, 60),
                                   (64, 48, 30), (64, 192, 30), (256, 12, 8), (512, 24, 4), (1024, 12, 2)])
@pytest.mark.parametrize("mode", ["plain", "self", "ext"])
@pytest.mark.parametrize("raw", ["f32", "bf16"])
def test_norm_block(C, H, W, mode, raw):
    """InstanceNorm(+CBAM)(+residual)+act, forward and backward, vs PyTorch fp32 autograd.
    Tolerance: rel-Frobenius 1e-2 on activations and gradients (bf16 storage of uhat / out / dy; a single ReLU
    mask flip on the 3x2 maps is already 0.7 %)."""
    if raw == "bf16" and (C, H, W) not in [(64, 12, 8), (128, 24, 15)]:
        pytest.skip("bf16 raw input covered on two shapes")
    _run_norm_block(C, H, W, mode, raw)


# ---- every kernel-variant switch that ships (include/barvae.h: bvae_set_option) gets the same parity treatment ----------
NB_VARIANTS = [("BVAE_NB_MLP", 0), ("BVAE_NB_MLP", 1), ("BVAE_NB_MODE", 1), ("BVAE_NB_MODE", 2), ("BVAE_NB_SPLIT", 0),
               ("BVAE_NB_FAST", 0), ("BVAE_NB_SMALL", 0)]


@pytest.mark.parametrize("opt", NB_VARIANTS, ids=lambda o: "%s=%d" % o)
def test_kernel_variants_norm_blocks(opt):
    """channel MLP inside / outside the per-sample kernels, cluster and per-sample kernels on every map size, unsplit
    reduction sweeps, the generic (non-restructured) sweeps, the per-sample small-map kernels with the batched MLP
    (BVAE_NB_SMALL=0: the round-2 default; any other non-default BVAE_NB_MLP / BVAE_NB_MODE selects them too): all shapes
    and residual modes of test_norm_block"""
    lib = pkg("_lib")
    with lib.option(*opt):
        assert lib.load().bvae_get_option(opt[0].encode(), -7) == opt[1]
        for C, H, W in [(32, 48, 30), (64, 12, 8), (128, 24, 15), (512, 6, 4), (1024, 3, 2), (64, 96, 60), (256, 12, 8)]:
            for mode in ("plain", "self", "ext"):
                _run_norm_block(C, H, W, mode, "f32")
    assert lib.load().bvae_get_option(opt[0].encode(), -7) == -7


@pytest.mark.parametrize("C,H,W", [(32, 48, 30), (64, 48, 30), (128, 24, 15), (256, 24, 15), (128, 96, 15), (64, 20, 13),
                                   (32, 16, 9), (128, 12, 11)])
@pytest.mark.parametrize("mode", ["plain", "self", "ext"])
def test_norm_block_per_sample_kernels(C, H, W, mode):
    """the per-sample nbs_* kernels on every channel count / lane geometry they take at training batch sizes (32 and 64
    channels: several pixels per warp; maps up to 1440 pixels), forced here at 3 samples; same bounds as test_norm_block"""
    lib = pkg("_lib")
    with lib.option("BVAE_NB_SMALL_N", 1), lib.option("BVAE_NB_SMALL_HW", 1440):
        _run_norm_block(C, H, W, mode, "f32")


def _run_norm_block(C, H, W, mode, raw):
    eng = pkg("engine")
    torch.manual_seed(C + H)
    B = 3
    dev = "cuda"
    slope = 0.01 if C == 32 else 0.0
    y = torch.randn(B, C, H, W, device=dev) * 2.0 + torch.randn(1, C, 1, 1, device=dev) * 3.0
    if raw == "bf16":
        y = _bf(y)
    gamma = (1 + 0.3 * torch.randn(C, device=dev)).requires_grad_(True)
    beta = (0.3 * torch.randn(C, device=dev)).requires_grad_(True)
    gamma.data[0] = -0.7                                     # negative gamma: max-pool of u follows min of y
    res_mode = {"plain": 0, "self": 1, "ext": 2}[mode]
    cb = None
    if mode != "plain":
        cb = ((torch.randn(C // 16, C, 1, 1, device=dev) * (2.0 / math.sqrt(C))).requires_grad_(True),
              (torch.randn(C, C // 16, 1, 1, device=dev) * (2.0 / math.sqrt(C // 16))).requires_grad_(True),
              (torch.randn(1, 2, 3, 3, device=dev) * 0.5).requires_grad_(True))
    res = _bf(torch.randn(B, C, H, W, device=dev)).requires_grad_(True) if mode == "ext" else None
    yr = y.clone().requires_grad_(True)
    ref = _torch_block(yr, gamma, beta, cb, res_mode, slope, res)
    dout = _bf(torch.randn_like(ref))
    ref.backward(dout)

    params = [gamma, beta] + (list(cb) if cb else [])
    ref_grads = [p.grad.clone() for p in params]
    for p in params:
        p.grad = None
    nb = eng.NormBlock(C, gamma, beta, cb, res_mode, slope)
    ya = eng.Act(nhwc(y).to(torch.float32 if raw == "f32" else BF16), B, H, W, C)
    out = eng.Act.empty(B, H, W, C)
    ra = eng.Act(nhwc(res.detach()).to(BF16), B, H, W, C) if res is not None else None
    ctx = nb.forward(ya, out, ra)
    e_out = rel_fro(nchw(out.t.float()), ref)
    dy = eng.Act.empty(B, H, W, C)
    dres = eng.Act.empty(B, H, W, C) if res is not None else None
    nb.backward(ctx, eng.Act(nhwc(dout).to(BF16), B, H, W, C), dy, dres)
    e_dy = rel_fro(nchw(dy.t.float()), yr.grad)
    errs = {"out": e_out, "dy": e_dy}
    if res is not None:
        errs["dres"] = rel_fro(nchw(dres.t.float()), res.grad)
    names = ["dgamma", "dbeta", "dw1", "dw2", "dwsp"]
    for nme, p, rg in zip(names, params, ref_grads):
        errs[nme] = rel_fro(p.grad, rg)
    report(test="norm_block", C=C, H=H, W=W, mode=mode, raw=raw, **errs)
    bad = {k: v for k, v in errs.items() if not v < (2e-2 if k in ('dw1', 'dw2', 'dwsp') else 1e-2)}
    assert not bad, errs


def test_fit_sigmoid_bce():
    """fit2 + sigmoid + BCE forward/backward (decoder.py:175,220; bar_loss.py:23-33) vs torch fp32.
    Tolerance: 1e-5 relative on the loss, 3e-3 rel-Frobenius on gradients (dx is stored in bf16)."""
    lib = pkg("_lib")
    L = lib.lib()
    torch.manual_seed(3)
    B, H, W, C = 3, 96, 60, 64
    rows = B * H * W
    x = _bf(torch.randn(rows, C, device="cuda")).requires_grad_(True)
    w = (torch.randn(C, device="cuda") * 0.5).requires_grad_(True)
    t = (torch.rand(rows, device="cuda") < 0.1).float()
    for smoothing in (0, 1):
        for p in (x, w):
            p.grad = None
        logits = x @ w
        p_ref = torch.sigmoid(logits)
        tt = t
        if smoothing:
            O = __import__("barvae_oracle")
            prior = torch.tensor(O.PITCH_PRIOR, device="cuda") * 0.08
            tt = (t.view(-1, 60) * 0.82 + 0.1 / 60 + prior).view(-1)
        ref_loss = F.binary_cross_entropy(p_ref, tt)
        ref_loss.backward()
        xb = x.detach().to(BF16).contiguous()
        recon = torch.empty(rows, device="cuda")
        lg = torch.empty(rows, device="cuda")
        st = lib.stream_ptr()
        lib.check(L.bvae_fit_sigmoid_fwd(xb.data_ptr(), C, w.data_ptr(), rows, C, lg.data_ptr(), recon.data_ptr(), st))
        acc = torch.zeros(2, device="cuda")
        lib.check(L.bvae_bce_fwd(recon.data_ptr(), t.data_ptr(), rows, smoothing, acc.data_ptr(), st))
        miss = float(((t - (p_ref > 0.3).float()) > 1e-4).float().sum())
        dx = torch.empty(rows, C, device="cuda", dtype=BF16)
        dw = torch.zeros(C, device="cuda")
        lib.check(L.bvae_fit_sigmoid_bce_bwd(xb.data_ptr(), C, w.data_ptr(), recon.data_ptr(), t.data_ptr(), None,
                                             1.0 / rows, smoothing, rows, C, dx.data_ptr(), C, dw.data_ptr(), st))
        e = dict(recon=rel_fro(recon, p_ref), loss=abs(float(acc[0]) - float(ref_loss)) / float(ref_loss),
                 miss=abs(float(acc[1]) - miss), dx=rel_fro(dx.float(), x.grad), dw=rel_fro(dw, w.grad))
        report(test="fit_sigmoid_bce", smoothing=smoothing, **e)
        assert e["recon"] < 1e-5 and e["loss"] < 1e-5 and e["miss"] <= 2 and e["dx"] < 3e-3 and e["dw"] < 1e-4, e


def test_bce_clamp_edges(golden, oracle):
    """the -100 log clamp and the 0.3 / 1e-4 thresholds on adversarial probabilities; golden from the reference Loss."""
    Loss = pkg("graph.loss.bar_loss").Loss
    c = golden["loss"]
    p, t = c["probs"].cuda(), c["labels"].cuda()
    for pre, key in ((True, "pre"), (False, "smooth")):
        got = float(Loss()(p, t, pre))
        want = float(c[key])
        report(test="bce_clamp", pre=pre, got=got, want=want)
        assert abs(got - want) <= 1e-5 * abs(want), (got, want)


def test_reparam_kl(golden):
    """reparameterise + KL vs the golden produced by old/graphs/models/bar_v1/encoder.py:60-63 and loss.py:16."""
    M = pkg("graph.model")
    c = golden["vae_head"]
    mu = c["mean"].cuda().requires_grad_(True)
    lv = c["logvar"].cuda().requires_grad_(True)
    eps = c["eps"].cuda()
    z = M.reparameterize(mu, lv, eps)
    kl = M.kl_divergence(mu, lv)
    assert rel_fro(z, c["z"]) < 1e-6
    assert abs(float(kl) - float(c["kl"])) < 1e-4 * abs(float(c["kl"]))
    g = torch.randn_like(z)
    ((z * g).sum() + 0.5 * kl).backward()
    mu2 = c["mean"].cuda().requires_grad_(True)
    lv2 = c["logvar"].cuda().requires_grad_(True)
    z2 = mu2 + eps * torch.exp(0.5 * lv2)
    kl2 = -0.5 * torch.sum(1 + lv2 - mu2.pow(2) - lv2.exp())
    ((z2 * g).sum() + 0.5 * kl2).backward()
    assert rel_fro(mu.grad, mu2.grad) < 1e-5 and rel_fro(lv.grad, lv2.grad) < 1e-5


def test_flat_adam():
    """fused flat Adam vs torch.optim.Adam (agent/barGen.py:61-62), 3 steps.  Tolerance 1e-6 relative."""
    eng = pkg("engine")
    torch.manual_seed(5)
    net = nn.Sequential(nn.Linear(37, 53), nn.Linear(53, 11)).cuda()
    ref = nn.Sequential(nn.Linear(37, 53), nn.Linear(53, 11)).cuda()
    ref.load_state_dict(net.state_dict())
    flat = eng.flatten(net)
    opt = torch.optim.Adam(ref.parameters(), lr=0.002)
    for step in range(1, 4):
        x = torch.randn(19, 37, device="cuda")
        flat.attach_grads()
        net(x).pow(2).mean().backward()
        opt.zero_grad()
        ref(x).pow(2).mean().backward()
        opt.step()
        eng.adam_step(flat, 0.002, step)
        for a, b in zip(net.parameters(), ref.parameters()):
            assert rel_fro(a, b) < 1e-6


def test_pack_plan_matches_single_packs():
    """bvae_pack_plan_run (one launch for every contraction weight) must write bit-identical bf16 operands to the
    per-layer bvae_pack_weight launches, for conv / transposed conv / linear layouts and ragged sizes."""
    eng = pkg("engine")
    torch.manual_seed(11)
    mods = nn.ModuleList([nn.Conv2d(64, 128, 3), nn.ConvTranspose2d(128, 64, 4, 2, 1), nn.Linear(200, 72, bias=False),
                          nn.Conv2d(8, 24, (1, 4)), nn.ConvTranspose2d(96, 40, (6, 1), (6, 1)),
                          nn.Conv2d(1, 32, (4, 1))]).cuda()
    layers = [eng.GemmLayer("conv", mods[0].weight, None, (3, 3), (1, 1), (1, 1)),
              eng.GemmLayer("convT", mods[1].weight, None, (4, 4), (2, 2), (1, 1)),
              eng.GemmLayer("linear", mods[2].weight),
              eng.GemmLayer("conv", mods[3].weight, None, (1, 4), (1, 2), (0, 1)),
              eng.GemmLayer("convT", mods[4].weight, None, (6, 1), (6, 1), (0, 0)),
              eng.GemmLayer("conv", mods[5].weight, None, (4, 1), (2, 1), (1, 0))]
    flat = eng.flatten(mods)
    want = [(l.w_fwd().clone(), l.w_dgrad().clone()) for l in layers]
    plan = eng.PackPlan(flat)
    assert len(plan.items) == 2 * len(layers) and plan.valid()
    for l in layers:
        l._wf.zero_()
        l._wd.zero_()
    plan.run()
    torch.cuda.synchronize()
    for l, (wf, wd) in zip(layers, want):
        assert torch.equal(l._wf, wf) and torch.equal(l._wd, wd)
        assert l._wf_key == l._key() and l._wd_key == l._key()
    # after an optimiser step the plan refreshes the same buffers in place
    flat.attach_grads()
    flat.grad.normal_()
    bufs = [(l._wf, l._wd) for l in layers]
    eng.adam_step(flat, 0.01, 1)
    for l, (bf, bd) in zip(layers, bufs):
        assert l.w_fwd() is bf and l.w_dgrad() is bd
        ref_f = l._pack(l.Cout, l.Cin, l.f_src, l.f_perm)
        ref_d = l._pack(l.Cin, l.Cout, l.d_src, l.d_perm)
        assert torch.equal(bf, ref_f) and torch.equal(bd, ref_d)


def test_norm_block_inference_mode_skips_saved_activation():
    """engine.saving(False): the norm-block forward gets uhat = NULL and must produce the same block output without
    writing it (every forward variant: tiled / fast / small-map); backward of such a pass is refused"""
    eng = pkg("engine")
    torch.manual_seed(4)
    for (N, H, W, Cc, cbam) in [(3, 24, 15, 64, True), (3, 24, 15, 64, False), (2, 6, 3, 512, True), (5, 12, 8, 256, True),
                                (2, 48, 30, 32, True)]:
        gamma = torch.nn.Parameter(torch.randn(Cc, device="cuda") * 0.5 + 1)
        beta = torch.nn.Parameter(torch.randn(Cc, device="cuda") * 0.1)
        cb = None
        if cbam:
            cb = (torch.nn.Parameter(torch.randn(Cc // 16, Cc, 1, 1, device="cuda") * 0.1),
                  torch.nn.Parameter(torch.randn(Cc, Cc // 16, 1, 1, device="cuda") * 0.1),
                  torch.nn.Parameter(torch.randn(1, 2, 3, 3, device="cuda") * 0.1))
        nb = eng.NormBlock(Cc, gamma, beta, cb, 1 if cbam else 0, 0.0)
        y = eng.Act(torch.randn(N, H, W, Cc, device="cuda"), N, H, W, Cc)
        o1, o2 = eng.Act.empty(N, H, W, Cc), eng.Act.empty(N, H, W, Cc)
        c1 = nb.forward(y, o1)
        with eng.saving(False):
            c2 = nb.forward(y, o2)
        torch.cuda.synchronize()
        assert c1["uhat"] is not None and c2["uhat"] is None
        e = rel_fro(o2.t.float(), o1.t.float())
        assert e < 2e-3, ((N, H, W, Cc, cbam), e)          # same kernels, same inputs: only atomics order differs
        with pytest.raises(RuntimeError):
            nb.backward(c2, eng.Act.empty(N, H, W, Cc), eng.Act.empty(N, H, W, Cc))
