"""GPU (B200): the Bernoulli sampler (csrc/sample.cu) against the numpy oracle, the decoder's logits, and the sampling
loop's Bernoulli / primer modes.  Every assertion is deterministic: cells equal the oracle exactly, except -- on random
logits only -- where u lies within 8 ulps of the oracle's probability (numpy's float32 exp and the device's expf may
differ in the last bit).  The loop tests run with bvae_set_deterministic(1) (bit-reproducible forward, DESIGN.md
section 7), restored afterwards."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from gpu_util import PKG, ROOT, pkg, report

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import sample_oracle as SO  # noqa: E402

pytestmark = pytest.mark.gpu
CELLS = SO.BAR_CELLS


@pytest.fixture
def deterministic():
    lib = pkg("_lib")
    before = bool(lib.load().bvae_deterministic())
    lib.set_deterministic(True)
    yield
    lib.set_deterministic(before)


def _rows(bars):
    """the rows held against the oracle: all of them up to 512 bars, else the first / last 64 and 64 random ones"""
    if bars <= 512:
        return np.arange(bars)
    r = np.random.RandomState(bars)
    return np.unique(np.concatenate([np.arange(64), np.arange(bars - 64, bars), r.randint(0, bars, 64)]))


def _sample(logits, temperature, seed, song_base, bar_index, canary=7.0):
    """bernoulli_sample into a buffer with canaries behind the output; returns the output (host) and checks them"""
    n = logits.numel()
    buf = torch.full((n + 64,), canary, device="cuda")
    pkg("data.packed").bernoulli_sample(logits, temperature, seed, song_base, bar_index, out=buf[:n])
    tail = buf[n:].cpu()
    assert torch.all(tail == canary), "bernoulli_sample wrote behind its output"
    return buf[:n].view(-1, CELLS).cpu().numpy()


@pytest.mark.parametrize("bars,temperature", [(1, 1.0), (3, 0.5), (64, 2.0), (700, 1.0), (8192, 0.5), (8192, 2.0)])
def test_kernel_matches_oracle(bars, temperature):
    seed, base, k = 0x5eed0000abcd + bars, 1000 * bars, 13
    inv_t = float(np.float32(1.0 / temperature))
    rows = _rows(bars)
    # logits 0: p = 0.5 exactly on both sides -> bit-equal
    zeros = torch.zeros(bars, 1, 96, 60, device="cuda")
    got = _sample(zeros, temperature, seed, base, k)
    u = SO.uniforms(seed, base + rows, k)
    want = (u < np.float32(0.5)).astype(np.float32)
    assert np.array_equal(got[rows], want)
    assert set(np.unique(got).tolist()) <= {0.0, 1.0}
    # random logits: equal except within 8 ulps of p
    g = torch.Generator(device="cuda").manual_seed(bars)
    lg = torch.randn(bars, 1, 96, 60, device="cuda", generator=g) * 4
    got = _sample(lg, temperature, seed, base, k)
    lgh = lg.view(-1, CELLS).cpu().numpy()[rows]
    p = SO.probs(lgh, inv_t)
    want = (u < p).astype(np.float32)
    band = np.abs(u - p) <= 8 * np.spacing(p)
    diff = got[rows] != want
    report(test="bernoulli_kernel", bars=bars, temperature=temperature, mismatches=int(diff.sum()),
           in_band=int(band.sum()), cells=int(diff.size))
    assert not np.any(diff & ~band), int((diff & ~band).sum())


def test_song_base_splits_calls_exactly():
    g = torch.Generator(device="cuda").manual_seed(64)
    lg = torch.randn(64, 1, 96, 60, device="cuda", generator=g)
    one = _sample(lg, 1.3, 77, 0, 5)
    two = np.concatenate([_sample(lg[:32].contiguous(), 1.3, 77, 0, 5), _sample(lg[32:].contiguous(), 1.3, 77, 32, 5)])
    assert np.array_equal(one, two)


def test_extreme_logits():
    lg = torch.zeros(2, 1, 96, 60, device="cuda")
    flat = lg.view(-1)
    flat[0::3] = float("inf")
    flat[1::3] = float("-inf")
    flat[2::3] = float("nan")
    for t in (0.5, 1.0, 2.0):
        got = _sample(lg, t, 1, 0, 0).reshape(-1)
        assert np.all(got[0::3] == 1) and np.all(got[1::3] == 0) and np.all(got[2::3] == 0)


def test_argument_errors():
    L = pkg("_lib")
    lib = L.lib()
    x = torch.zeros(2 * CELLS + 8, device="cuda")
    y = torch.zeros(2 * CELLS + 8, device="cuda")
    st = L.stream_ptr()
    for inv_t in (0.0, -1.0, float("inf"), float("-inf"), float("nan")):
        assert lib.bvae_bernoulli_sample(x.data_ptr(), 1, inv_t, 0, 0, 0, y.data_ptr(), st) == 1
    assert lib.bvae_bernoulli_sample(x.data_ptr(), -1, 1.0, 0, 0, 0, y.data_ptr(), st) == 1
    assert lib.bvae_bernoulli_sample(x.data_ptr() + 4, 1, 1.0, 0, 0, 0, y.data_ptr(), st) == 2
    assert lib.bvae_bernoulli_sample(x.data_ptr(), 1, 1.0, 0, 0, 0, y.data_ptr() + 8, st) == 2
    assert lib.bvae_bernoulli_sample(x.data_ptr(), 0, 1.0, 0, 0, 0, y.data_ptr(), st) == 0
    torch.cuda.synchronize()
    assert torch.all(y == 0)
    packed = pkg("data.packed")
    for t in (0.0, -2.0, float("inf"), float("nan")):
        with pytest.raises(RuntimeError):
            packed.bernoulli_sample(x[:CELLS], t, 0, 0, 0)
    with pytest.raises(ValueError):
        packed.bernoulli_sample(x[:CELLS - 1], 1.0, 0, 0, 0)


# ---- decoder logits and the loop -------------------------------------------------------------------------------------
def _model(refiner=False):
    O = __import__("barvae_oracle")
    sd = O.make_state_dict(O.generator_spec(), 11, "lively")
    m = pkg("graph.model").Model(refiner=refiner)
    m.load_state_dict(sd, strict=not refiner)
    return m.cuda().eval()


def _latents(songs, music_length, seed=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(music_length * 4, songs, 1152, device="cuda", generator=g)


def test_forward_logits_matches_forward(deterministic):
    O = __import__("barvae_oracle")
    model = _model()
    _, pre_note, phrase, position = (t.cuda() for t in O.make_inputs(3, 21))
    z = _latents(3, 1)[0]
    with torch.no_grad():
        pre_z = model.encoder(pre_note)
        pf = model.phrase_encoder(phrase)
        probs = model.decoder(z, pre_z, pf, position)
        p2, logits = model.decoder.forward_logits(z, pre_z, pf, position)
    assert torch.equal(probs, p2)
    assert logits.shape == probs.shape and torch.isfinite(logits).all()
    torch.testing.assert_close(torch.sigmoid(logits), probs, rtol=1e-6, atol=1e-30)
    assert 0.0 < float((probs > 0.3).float().mean()) < 1.0             # lively weights: a bar with notes and rests
    with pytest.raises(RuntimeError):
        model.decoder.forward_logits(z, pre_z, pf, position)            # grad mode on
    model.train()
    with torch.no_grad(), pytest.raises(RuntimeError):
        model.decoder.forward_logits(z, pre_z, pf, position)            # training mode: dropout


S, L = 3, 3


def test_threshold_default_unchanged_by_sampler_arguments(deterministic):
    mb, model, lat = pkg("maker_bar"), _model(), _latents(S, L)
    a = mb.sample_songs(model, lat, L)
    b = mb.sample_songs(model, lat, L, sampler="threshold", seed=123, song_base=7, temperature=0.3)
    assert torch.equal(a, b)


@pytest.mark.parametrize("sampler", ["threshold", "bernoulli"])
@pytest.mark.parametrize("P", [1, 2])
def test_primer_continues_the_unprimed_run(deterministic, sampler, P):
    mb, model, lat = pkg("maker_bar"), _model(), _latents(S, L)
    kw = dict(sampler=sampler, seed=9, song_base=4, temperature=0.9)
    full = mb.sample_songs(model, lat, L, **kw)
    primer = full[:, :P * 384].clone()
    cont = mb.sample_songs(model, lat, L, primer=primer, **kw)
    report(test="primer_equivalence", sampler=sampler, P=P, cells_on=float(full.mean()))
    assert torch.equal(cont, full)


def test_bernoulli_seeds_and_primer_bars(deterministic):
    mb, model, lat = pkg("maker_bar"), _model(), _latents(S, L)
    a = mb.sample_songs(model, lat, L, sampler="bernoulli", seed=1)
    assert torch.equal(a, mb.sample_songs(model, lat, L, sampler="bernoulli", seed=1))
    b = mb.sample_songs(model, lat, L, sampler="bernoulli", seed=2)
    assert not torch.equal(a, b)
    thr = mb.sample_songs(model, lat, L)
    assert not torch.equal(a, thr)
    primer = ((torch.arange(384 * 60, device="cuda").view(384, 60) % 7) == 0).float()     # one primer for all songs
    c = mb.sample_songs(model, lat, L, sampler="bernoulli", seed=1, primer=primer)
    assert torch.equal(c[:, :384], primer.expand(S, -1, -1))
    assert not torch.equal(c[0, 384:], c[1, 384:])                    # songs draw from their own streams
    assert set(torch.unique(c).tolist()) <= {0.0, 1.0}


def test_bernoulli_with_refiner_raises():
    mb = pkg("maker_bar")
    model = _model(refiner=True)
    with pytest.raises(ValueError):
        mb.sample_songs(model, _latents(1, 2), 2, sampler="bernoulli")


@pytest.mark.parametrize("P", [0, 1])
def test_first_bar_is_the_oracle_draw_from_the_decoders_probabilities(deterministic, P):
    """temperature 1: the kernel's p is the decoder's probability bit for bit, so the first generated bar is exactly
    oracle_u(seed, song, k) < first_probs"""
    mb, model, lat = pkg("maker_bar"), _model(), _latents(S, L)
    seed, base = 0xfeedface12345678, 40
    primer = None if P == 0 else mb.sample_songs(model, lat, L)[:, :P * 384].clone()
    roll, first = mb.sample_songs(model, lat, L, True, sampler="bernoulli", seed=seed, song_base=base, primer=primer)
    k = 4 * P
    u = SO.uniforms(seed, base + np.arange(S), k)
    want = (u < first.view(S, CELLS).cpu().numpy()).astype(np.float32)
    got = roll[:, k * 96:(k + 1) * 96].reshape(S, CELLS).cpu().numpy()
    assert np.array_equal(got, want)


# ---- the script end to end -------------------------------------------------------------------------------------------
def _run_main(cwd, argv):
    env = dict(os.environ, BVAE_DETERMINISTIC="1", PYTHONPATH=ROOT)
    code = "import importlib, sys; importlib.import_module(%r).main(sys.argv[1:])" % (PKG + ".maker_bar")
    r = subprocess.run([sys.executable, "-c", code] + argv, cwd=str(cwd), env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


def test_main_end_to_end(tmp_path, deterministic):
    mb, midi = pkg("maker_bar"), pkg("midi")
    O = __import__("barvae_oracle")
    sd = O.make_state_dict(O.generator_spec(), 11, "lively")
    os.makedirs(tmp_path / "model")
    torch.save({"generator_state_dict": {"module." + k: v for k, v in sd.items()}},
               str(tmp_path / "model" / "checkpoint_10.pth.tar"))
    # default flags: the same file as sample_songs' default path
    out = _run_main(tmp_path, ["--music_length", "3", "--seed", "1"])
    assert "seed: 1" in out
    model = _model()
    g = torch.Generator(device="cuda").manual_seed(1)
    lat = torch.randn(12, 1, 1152, device="cuda", generator=g)
    roll = mb.songs_to_host(mb.sample_songs(model, lat, 3))[0]
    midi.write_midi(roll, str(tmp_path / "want.mid"))
    assert (tmp_path / "test.mid").read_bytes() == (tmp_path / "want.mid").read_bytes()
    # primer + Bernoulli: three different continuations of the same primer
    primer = roll[:384].copy()
    primer[-1, 30] = 1.0
    midi.write_midi(primer, str(tmp_path / "x.mid"))
    out = _run_main(tmp_path, ["--music_length", "3", "--seed", "2", "--primer", "x.mid", "--sampler", "bernoulli",
                               "--temperature", "0.8", "--songs", "3", "--out", "cont.mid"])
    assert "primer: 1 phrases" in out
    rolls = [midi.midi_to_roll(str(tmp_path / n), 3 * 384) for n in ("cont.mid", "cont_1.mid", "cont_2.mid")]
    for r in rolls:
        assert np.array_equal(r[:384], primer)
    assert not np.array_equal(rolls[0][384:], rolls[1][384:]) and not np.array_equal(rolls[1][384:], rolls[2][384:])
    assert not np.array_equal(rolls[0][384:], rolls[2][384:])
