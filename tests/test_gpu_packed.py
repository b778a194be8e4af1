"""GPU: bit-packed piano-roll kernels (csrc/bits.cu) against the numpy oracle -- bit-exact -- and the packed training
entry point against the fp32-input one."""
import os
import sys

import numpy as np
import pytest
import torch

from gpu_util import ROOT, pkg, rel_fro, report

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import bits_oracle as BO  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,n_f32", [(8, 8), (1, 1), (13, 8), (13, 13), (5760, 0), (5760 * 3 + 5, 5760),
                                     (5760 * 3 + 5, 5760 * 3 + 5), (512 * 5760, 256 * 5760)])
def test_unpack_bits_bit_exact(n, n_f32):
    P = pkg("data.packed")
    r = np.random.RandomState(n % 9973)
    cells = (r.rand(n) < 0.3).astype(np.float32)
    bits = torch.from_numpy(BO.pack(cells)).cuda()
    pad = 64                                                  # canaries behind the outputs: nothing may be written there
    ob = torch.full((n + pad,), 7.0, device="cuda", dtype=torch.bfloat16)
    of = torch.full((n_f32 + pad,), 7.0, device="cuda", dtype=torch.float32)
    P.unpack_bits(bits, n, ob, of if n_f32 else None, n_f32)
    torch.cuda.synchronize()
    assert np.array_equal(ob[:n].float().cpu().numpy(), BO.unpack(bits.cpu().numpy(), n))
    assert bool((ob[n:] == 7.0).all())
    if n_f32:
        assert np.array_equal(of[:n_f32].cpu().numpy(), cells[:n_f32])
    assert bool((of[n_f32:] == 7.0).all())
    P.unpack_bits(bits, n, None, of if n_f32 else torch.empty(8, device="cuda"), n_f32)    # fp32-only call
    torch.cuda.synchronize()
    assert np.array_equal(of[:n_f32].cpu().numpy(), cells[:n_f32]) and bool((of[n_f32:] == 7.0).all())


@pytest.mark.parametrize("n", [1, 7, 8, 9, 5760, 5760 * 5 + 3])
@pytest.mark.parametrize("thr", [0.3, 0.5])
def test_threshold_pack_bit_exact(n, thr):
    P = pkg("data.packed")
    g = torch.Generator().manual_seed(n)
    p = torch.rand(n, generator=g)
    p[::5] = thr                                              # exactly on the threshold: strict > (maker_bar.py:39)
    bits, hard = P.threshold_pack(p.cuda(), thr, want_bits=True, want_float=True)
    torch.cuda.synchronize()
    wb, wh = BO.threshold_pack(p.numpy(), thr)
    assert np.array_equal(bits.cpu().numpy(), wb)
    assert np.array_equal(hard.cpu().numpy(), wh)
    only_bits, none = P.threshold_pack(p.cuda(), thr)
    assert none is None and np.array_equal(only_bits.cpu().numpy(), wb)


def test_roundtrip_at_bench_size():
    """BASELINE configs[1] size (512 bars + phrases = 17.7 M cells): pack(unpack(bits)) == bits, and the popcount of the
    bits equals the sum of the expanded cells (size-independent properties; the oracle loop is not run at this size)"""
    P = pkg("data.packed")
    B = 512
    nbytes = B * 4320
    g = torch.Generator(device="cuda").manual_seed(5)
    bits = torch.randint(0, 256, (nbytes,), device="cuda", dtype=torch.uint8, generator=g)
    cells = torch.empty(nbytes * 8, device="cuda", dtype=torch.float32)
    cells_b = torch.empty(nbytes * 8, device="cuda", dtype=torch.bfloat16)
    P.unpack_bits(bits, nbytes * 8, cells_b, cells, nbytes * 8)
    back, _ = P.threshold_pack(cells, 0.5)
    assert torch.equal(back, bits)
    assert torch.equal(cells_b.float(), cells)
    lut = torch.tensor([bin(i).count("1") for i in range(256)], device="cuda")
    assert int(lut[bits.long()].sum()) == int(cells.sum().item())


def test_packed_batch_to_device_matches_float_inputs():
    P = pkg("data.packed")
    O = __import__("barvae_oracle")
    note, pre, phrase, pos = O.make_inputs(5, 13)
    pb = P.PackedBatch.from_arrays(note, pre, phrase, pos, pin=True)
    side = torch.cuda.Stream()
    for stream in (None, side):
        n32, bars, ph, p, dbits = pb.to_device(torch.device("cuda", 0), stream)
        torch.cuda.synchronize()
        assert torch.equal(n32.cpu(), note) and torch.equal(p.cpu(), pos)
        assert torch.equal(bars.float().cpu(), torch.cat((note, pre), 0))
        assert torch.equal(ph.float().cpu(), phrase)
        assert bars.dtype == torch.bfloat16 and ph.dtype == torch.bfloat16 and n32.dtype == torch.float32


def test_model_forward_from_packed_equals_float_path():
    """the stems read bf16 {0,1} either way (inputs checked bit-exact above), so the only difference between the two
    input routes is the run-to-run floor of the forward itself (fp32 statistics atomics -> bf16 re-rounding downstream;
    measured 2.5e-3 on z): the comparison is against that floor, measured by running the float route twice"""
    P = pkg("data.packed")
    O = __import__("barvae_oracle")
    Model = pkg("graph.model").Model
    sd = O.make_state_dict(O.generator_spec(), 11, "lively")
    model = Model()
    model.load_state_dict(sd)
    model = model.cuda().eval()
    batch = O.make_inputs(3, 17)
    pb = P.PackedBatch.from_arrays(*batch)
    with torch.no_grad():
        gen0, z0, pz0, pf0 = model(*(t.cuda() for t in batch))
        gen0b, z0b, pz0b, pf0b = model(*(t.cuda() for t in batch))
        n32, bars, ph, pos, dbits = pb.to_device(torch.device("cuda", 0), None)
        gen1, z1, pz1, pf1 = model(bars[:3], bars[3:], ph, pos)
    torch.cuda.synchronize()
    fz, fp, fg = rel_fro(z0b, z0), rel_fro(pf0b, pf0), float((gen0b - gen0).abs().max())
    ez, ep, eg = rel_fro(z1, z0), rel_fro(pf1, pf0), float((gen1 - gen0).abs().max())
    report(test="packed_forward", z_rel=ez, pf_rel=ep, gen_maxabs=eg, floor_z=fz, floor_pf=fp, floor_gen=fg)
    assert ez < 3 * fz + 3e-3 and rel_fro(pz1, pz0) < 3 * rel_fro(pz0b, pz0) + 3e-3 and ep < 3 * fp + 3e-3, (ez, fz, ep, fp)
    assert eg < 3 * fg + 3e-2, (eg, fg)


def test_trainer_step_from_packed_matches_step_from_host():
    """two optimisation steps from bits vs from pinned fp32 tensors: same first-step loss up to the forward's run-to-run
    floor (identical inputs and weights; fp32 statistics atomics) and the same parameters within the run-to-run floor
    used by test_trainer_stream_and_segment_paths_agree"""
    P = pkg("data.packed")
    O = __import__("barvae_oracle")
    Model = pkg("graph.model").Model
    Trainer = pkg("trainer").GeneratorTrainer
    sd = O.make_state_dict(O.generator_spec(), 21, "lively")
    hb = O.make_inputs(4, 9)
    hbatch = tuple(t.pin_memory() for t in hb)
    pb = P.PackedBatch.from_arrays(*hb, pin=True)
    masks = tuple(m.cuda() for m in O.draw_dropout_masks(4, 5))

    def run(packed):
        model = Model()
        model.load_state_dict(sd)
        tr = Trainer(model.cuda().train(), lr=0.002)
        start = tr.flat.data.clone()
        losses = []
        for _ in range(2):
            loss = tr.step_from_packed(pb, masks) if packed else tr.step_from_host(*hbatch, masks)
            losses.append(float(loss))
        torch.cuda.synchronize()
        return tr.flat.data.clone(), start, losses

    # deterministic mode (include/barvae.h): the forward reductions run in a fixed order, so identical inputs and weights
    # give a BIT-identical first-step loss whichever way the batch reached the device; in the default mode the fp32
    # statistics atomics move it by up to ~1 % (it contains 0.005 x the count of cells on the wrong side of 0.3)
    lib = pkg("_lib")
    lib.set_deterministic(True)
    try:
        a, start, la = run(False)
        a2, _, _ = run(False)
        b, _, lb = run(True)
    finally:
        lib.set_deterministic(False)
    upd = (a - start).abs().mean().item()
    floor = (a2 - a).abs().mean().item() / upd
    e = (b - a).abs().mean().item() / upd
    report(test="trainer_packed", floor=floor, packed_vs_host=e, losses=[la, lb])
    assert lb[0] == la[0], (la, lb)
    assert e < 2 * floor + 0.05, (floor, e)
    assert abs(lb[1] - la[1]) < 0.1 * abs(la[1]), (la, lb)


def test_songs_to_host_packed_d2h():
    maker = pkg("maker_bar")
    g = torch.Generator(device="cuda").manual_seed(2)
    roll = (torch.rand(3, 2 * 4 * 96, 60, device="cuda", generator=g) < 0.1).float()
    host = maker.songs_to_host(roll)
    assert host.dtype == np.float32 and np.array_equal(host, roll.cpu().numpy())


def test_bargen_with_packed_input(tmp_path):
    """config.packed_input: the loader collates into PackedBatch (pinned by the DataLoader) and train_epoch steps from
    bits; same first-epoch loss as the fp32 loader on the same data and seed-fixed weights"""
    Config = pkg("config").Config
    BarGen = pkg("agent.barGen").BarGen
    P = pkg("data.packed")
    ds = pkg("data.bar_dataset").SyntheticBars(n_items=4, bars_per_item=2, batch_size=2, seed=3)

    def run(packed, sub):
        class Cfg(Config):
            root_path = str(tmp_path / sub)
            batch_size = 2
            packed_input = packed
        os.makedirs(Cfg.root_path, exist_ok=True)
        agent = BarGen(Cfg(), dataset=ds)
        sd = __import__("barvae_oracle").make_state_dict(__import__("barvae_oracle").generator_spec(), 11, "lively")
        agent.generator.load_state_dict(sd)
        b = agent.make_batch([ds[0], ds[1]])
        assert isinstance(b, P.PackedBatch) == packed
        torch.manual_seed(0)                         # same dropout draws in both runs (BarGen seeds randomly)
        torch.cuda.manual_seed_all(0)
        return agent.train_epoch()

    l_f, l_p = run(False, "f"), run(True, "p")
    report(test="bargen_packed", loss_float=l_f, loss_packed=l_p)
    assert l_p == l_p and abs(l_p - l_f) < 0.1 * abs(l_f), (l_f, l_p)


def test_adam_continues_from_reference_optimizer_state():
    """a torch.optim.Adam state_dict (the reference checkpoint's 'gen_optimizer1') loaded into the flat Adam: the next
    bvae_adam_step equals torch.optim.Adam's next step on the same gradient"""
    Model = pkg("graph.model").Model
    Trainer = pkg("trainer").GeneratorTrainer
    eng = pkg("engine")
    torch.manual_seed(3)
    model = Model().cuda()
    tr = Trainer(model, lr=0.002)
    flat = tr.flat
    clones = [torch.nn.Parameter(p.detach().clone()) for p in flat.params]
    opt = torch.optim.Adam(clones, lr=0.002)
    g = torch.Generator(device="cuda").manual_seed(1)

    def grads():
        return [torch.randn(c.shape, device="cuda", generator=g) * 1e-2 for c in clones]

    for c, gr in zip(clones, grads()):
        c.grad = gr
    opt.step()
    tr.load_state_dict(opt.state_dict())
    with torch.no_grad():
        for p, c in zip(flat.params, clones):
            p.copy_(c)
    g2 = grads()
    for c, gr in zip(clones, g2):
        c.grad = gr
    opt.step()
    flat.attach_grads(zero=True)
    for p, gr in zip(flat.params, g2):
        flat.grad_view(p).copy_(gr)
    tr.step_count += 1
    eng.adam_step(flat, tr.lr, tr.step_count, tr.betas, tr.eps, 1.0, repack=False)
    torch.cuda.synchronize()
    worst = max(float((p - c).abs().max()) for p, c in zip(flat.params, clones))
    report(test="adam_from_torch_state", worst_abs=worst)
    assert tr.step_count == 2 and worst < 2e-6, worst


@pytest.fixture
def deterministic_forward():
    """bvae_set_deterministic(1) for one test: fixed-order forward reductions, so two trainers that start from the same
    weights compute the same first-step loss bit for bit.  In the default mode the cross-CTA atomics of the InstanceNorm
    statistics spread a 3-bar loss by ~0.3 % from run to run, plus 0.005 for every cell that the noise moves across the
    0.3 threshold of the loss's count term (DESIGN.md section 7)."""
    lib = pkg("_lib")
    before = bool(lib.load().bvae_deterministic())
    lib.set_deterministic(True)
    yield
    lib.set_deterministic(before)


@pytest.mark.parametrize("packed", [False, True])
def test_prefetcher_hands_out_the_right_batches_while_steps_run(packed, deterministic_forward):
    """trainer.prefetch: 5 DISTINCT host batches (the last one smaller) through the two alternating device buffer sets
    with a training step running on each -- every DeviceBatch must equal its host batch bit for bit when it is handed
    out AND still after its step has been enqueued (the next copy must not overwrite a buffer that is in use), and the
    losses must match the sequential step_from_host loop on the same batches"""
    P = pkg("data.packed")
    O = __import__("barvae_oracle")
    Model = pkg("graph.model").Model
    Trainer = pkg("trainer").GeneratorTrainer
    sd = O.make_state_dict(O.generator_spec(), 21, "lively")
    sizes = [3, 3, 3, 3, 2]
    host = [O.make_inputs(b, 40 + i) for i, b in enumerate(sizes)]
    masks = [tuple(m.cuda() for m in O.draw_dropout_masks(b, 5 + i)) for i, b in enumerate(sizes)]
    feed = [P.PackedBatch.from_arrays(*hb, pin=True) if packed else tuple(t.pin_memory() for t in hb) for hb in host]

    def fresh():
        model = Model()
        model.load_state_dict(sd)
        return Trainer(model.cuda().train(), lr=0.002)

    tr = fresh()
    losses, snaps = [], []
    for i, db in enumerate(tr.prefetch(feed)):
        before = [t.clone() for t in db]
        loss = tr.step_batch(db, masks[i])
        snaps.append((before, [t.clone() for t in db], None if db.target is None else db.target.clone()))
        losses.append(loss)
    torch.cuda.synchronize()
    assert len(snaps) == len(host)
    for (before, after, target), hb in zip(snaps, host):
        for b, a, h in zip(before, after, hb):
            assert torch.equal(b.float().cpu(), h.float()) and torch.equal(a.float().cpu(), h.float())
        if packed:
            assert torch.equal(target.cpu(), hb[0]) and before[0].dtype == torch.bfloat16
    tr2 = fresh()
    want = [float(tr2.step_from_host(*(t.pin_memory() for t in hb), masks[i])) for i, hb in enumerate(host)]
    got = [float(l) for l in losses]
    report(test="prefetch_losses", packed=packed, got=got, want=want)
    assert abs(got[0] - want[0]) < 1e-2 * abs(want[0]), (got, want)
    assert all(abs(g - w) < 0.15 * abs(w) for g, w in zip(got, want)), (got, want)
    # the trainer reuses one prefetcher (one copy stream, one pair of buffer sets) across epochs
    assert tr.prefetch(feed) is tr.prefetch(feed)
