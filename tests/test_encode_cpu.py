"""CPU: the per-bar score's oracle (pinned to closed forms, hand counts and torch's BCE-with-logits), latent
interpolation, MIDI loading for whole songs, and the argument checks of maker_bar.main's encode modes that run before
any device work."""
import math
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gpu_util import ROOT, pkg

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import score_oracle as SC  # noqa: E402

CELLS = SC.BAR_CELLS


# ---- score oracle ---------------------------------------------------------------------------------------------------
def test_oracle_logit_zero_is_ln2_per_cell():
    r = np.random.RandomState(0)
    target = (r.rand(3, CELLS) < 0.1).astype(np.float32)
    nll, counts, _ = SC.score(np.zeros((3, CELLS), np.float32), target, 1.0, 0.3)
    assert np.all(nll == CELLS * math.log(2.0))
    on = target.sum(1).astype(np.int64)
    assert np.array_equal(counts, np.stack([on, np.full(3, CELLS), on], 1))      # p = 0.5 > 0.3 everywhere


def test_oracle_infinite_and_nan_logits():
    lg = np.zeros((1, CELLS), np.float32)
    t = np.zeros((1, CELLS), np.float32)
    lg[0, :4] = [np.inf, np.inf, -np.inf, -np.inf]
    t[0, :4] = [1, 0, 1, 0]
    for k, want in enumerate([0.0, np.inf, np.inf, 0.0]):
        one = np.zeros((1, CELLS), np.float32)
        one[0, 0] = lg[0, k]
        tt = np.zeros((1, CELLS), np.float32)
        tt[0, 0] = t[0, k]
        nll, _, _ = SC.score(one, tt, 1.0, 0.3)
        rest = (CELLS - 1) * math.log(2.0)
        assert (nll[0] == np.inf) if want == np.inf else nll[0] == pytest.approx(rest, rel=1e-15)
    nan = np.zeros((1, CELLS), np.float32)
    nan[0, 7] = np.nan
    nll, counts, _ = SC.score(nan, np.ones((1, CELLS), np.float32), 1.0, -1.0)
    assert np.isnan(nll[0]) and counts[0, 1] == CELLS - 1       # NaN p is never predicted on, even at threshold -1


def test_oracle_temperature_divides_the_logits():
    r = np.random.RandomState(1)
    lg = (r.randn(2, CELLS) * 3).astype(np.float32)
    t = (r.rand(2, CELLS) < 0.2).astype(np.float32)
    for T in (0.5, 2.0, 4.0):                                    # powers of two: l / T is exact in float32
        a = SC.score(lg, t, 1.0 / T, 0.3)
        b = SC.score(lg / np.float32(T), t, 1.0, 0.3)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_oracle_against_torch_bce_with_logits():
    r = np.random.RandomState(2)
    lg = (r.randn(5, CELLS) * 5).astype(np.float32)
    t = (r.rand(5, CELLS) < 0.3).astype(np.float32)
    for inv_t in (1.0, 0.5, 2.0):
        nll, _, _ = SC.score(lg, t, inv_t, 0.3)
        l = torch.from_numpy(lg * np.float32(inv_t)).double()
        want = torch.stack([F.binary_cross_entropy_with_logits(l[b], torch.from_numpy(t[b]).double(),
                                                               reduction="sum") for b in range(5)])
        np.testing.assert_allclose(nll, want.numpy(), rtol=1e-12)


def test_oracle_hand_counted():
    lg = np.full((2, CELLS), -5.0, np.float32)                  # p = 0.0067: off
    t = np.zeros((2, CELLS), np.float32)
    lg[0, :10] = 3.0                                             # 10 predicted on
    t[0, 5:25] = 1.0                                             # 20 on, 5 of them predicted
    t[1, :3] = 2.0                                               # nonzero counts as 1
    _, counts, _ = SC.score(lg, t, 1.0, 0.3)
    assert counts.tolist() == [[5, 10, 20], [0, 0, 3]]
    _, counts, _ = SC.score(lg, t, 1.0, 0.999)                  # p(3) = 0.953 < 0.999
    assert counts.tolist() == [[0, 0, 20], [0, 0, 3]]


# ---- interpolation --------------------------------------------------------------------------------------------------
def _pair(K=6, D=1152, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(K, D, generator=g), torch.randn(K, D, generator=g)


@pytest.mark.parametrize("shape3", [False, True])
@pytest.mark.parametrize("steps", [2, 3, 7])
def test_interpolation_endpoints_are_exact(shape3, steps):
    mb = pkg("maker_bar")
    za, zb = _pair()
    if shape3:
        za, zb = za[:, None], zb[:, None]
    out = mb.interpolate_latents(za, zb, steps)
    assert out.shape == (6, steps, 1152) and out.dtype == za.dtype
    assert torch.equal(out[:, 0], za.reshape(6, 1152)) and torch.equal(out[:, -1], zb.reshape(6, 1152))


def test_interpolation_keeps_the_norm_between_orthogonal_vectors():
    mb = pkg("maker_bar")
    za, zb = _pair(K=4)
    zb = zb - (zb * za).sum(1, keepdim=True) / (za * za).sum(1, keepdim=True) * za      # orthogonal to za
    zb = zb * (za.norm(dim=1, keepdim=True) / zb.norm(dim=1, keepdim=True))              # same norm
    out = mb.interpolate_latents(za.double(), zb.double(), 9)
    n = out.norm(dim=2)
    torch.testing.assert_close(n, za.double().norm(dim=1, keepdim=True).expand(-1, 9), rtol=1e-6, atol=0)
    mid = out[:, 4]                                                                      # t = 1/2: on the bisector
    cos = (mid * za.double()).sum(1) / (mid.norm(dim=1) * za.double().norm(dim=1))
    torch.testing.assert_close(cos, torch.full_like(cos, math.cos(math.pi / 4)), rtol=1e-6, atol=0)


def test_interpolation_linear_fallback_without_nan():
    mb = pkg("maker_bar")
    za, _ = _pair(K=4)
    zb = torch.stack([za[0] * 3.0,               # parallel
                      -za[1],                    # antiparallel
                      torch.zeros(1152),         # zero
                      za[3]])                    # identical
    za = za.clone()
    za[2] = 0.0                                  # zero to zero in row 2 as well
    out = mb.interpolate_latents(za, zb, 5)
    assert torch.isfinite(out).all()
    t = torch.arange(5, dtype=torch.float64) / 4
    want = ((1 - t)[None, :, None] * za.double()[:, None] + t[None, :, None] * zb.double()[:, None]).float()
    torch.testing.assert_close(out, want, rtol=1e-6, atol=1e-6)
    one_zero = mb.interpolate_latents(za[:1], torch.zeros(1, 1152), 3)                   # one zero endpoint
    torch.testing.assert_close(one_zero[0, 1], za[0] * 0.5)


def test_interpolation_rejects_bad_arguments():
    mb = pkg("maker_bar")
    za, zb = _pair(K=2)
    for steps in (1, 0, -3, 2.5):
        with pytest.raises(ValueError):
            mb.interpolate_latents(za, zb, steps)
    for a, b in ((za, zb[:1]), (za[:, None], zb), (za[None], zb[None]), (za[:, None].expand(2, 2, 1152), zb)):
        with pytest.raises(ValueError):
            mb.interpolate_latents(a, b, 3)


# ---- MIDI -----------------------------------------------------------------------------------------------------------
def _roll(phrases, seed, last_step_note=True):
    r = np.random.RandomState(seed)
    roll = (r.rand(phrases * 384, 60) < 0.05).astype(np.float32)
    if last_step_note:
        roll[-1, 30] = 1.0                       # the file then covers all its phrases (MIDI has no end-of-roll mark)
    return roll


def test_load_roll(tmp_path):
    mb, midi = pkg("maker_bar"), pkg("midi")
    roll = _roll(3, 1)
    roll[5:9, 2] = 1.0
    path = str(tmp_path / "s.mid")
    midi.write_midi(roll, path, lowest_pitch=20)                # pitch 22 is below the window
    n_low = len([n for n in midi.roll_to_notes(roll, 20) if n[0] < midi.LOWEST_PITCH])
    want = np.zeros_like(roll)
    want[:, :53] = roll[:, 7:]
    got, P, dropped = mb.load_roll(path)
    assert P == 3 and dropped == n_low > 0 and np.array_equal(got, want)
    got2, P2, _ = mb.load_roll(path, phrases=2)
    assert P2 == 2 and np.array_equal(got2, want[:768])
    got5, P5, _ = mb.load_roll(path, phrases=5)                  # beyond the notes: silence
    assert P5 == 5 and np.array_equal(got5[:1152], want) and not got5[1152:].any()
    short = str(tmp_path / "short.mid")
    midi.write_midi(_roll(1, 2, last_step_note=False)[:100], short)
    got0, P0, _ = mb.load_roll(short)
    assert P0 == 0 and got0.shape == (0, 60)
    with pytest.raises(ValueError):
        mb.load_roll(path, phrases=-1)


def test_load_primer_is_load_roll_with_its_own_rule(tmp_path):
    mb, midi = pkg("maker_bar"), pkg("midi")
    roll = _roll(2, 3)
    path = str(tmp_path / "p.mid")
    midi.write_midi(roll, path)
    got, P, dropped = mb.load_primer(path, music_length=3)
    assert P == 2 and dropped == 0 and np.array_equal(got, mb.load_roll(path)[0])
    with pytest.raises(ValueError, match="need 1 <= P < music_length"):
        mb.load_primer(path, music_length=2)
    short = str(tmp_path / "short.mid")
    midi.write_midi(_roll(1, 2, last_step_note=False)[:100], short)
    with pytest.raises(ValueError, match="covers no whole"):
        mb.load_primer(short, music_length=3)


# ---- song API arguments that need no device -------------------------------------------------------------------------
class _Host(torch.nn.Module):
    """a module with one CPU parameter: enough for the argument checks, which run before any device work"""

    def __init__(self, refiner=None):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(1))
        self.refiner = refiner


def test_song_api_rejects_bad_rolls_and_the_refiner():
    mb = pkg("maker_bar")
    for roll in (np.zeros((383, 60)), np.zeros((384, 59)), np.zeros((0, 60)), np.zeros((0, 384, 60)),
                 np.zeros((1, 1, 384, 60)), np.full((384, 60), 0.5)):
        with pytest.raises(ValueError):
            mb.encode_songs(_Host(), roll)
        with pytest.raises(ValueError):
            mb.reconstruct_songs(_Host(), roll)
    with pytest.raises(ValueError):
        mb.encode_songs(_Host(), np.zeros((384, 60)), chunk=0)
    with pytest.raises(ValueError):                        # the Refiner outputs probabilities: no logits to score
        mb.reconstruct_songs(_Host(refiner=torch.nn.Identity()), np.zeros((384, 60)))


def test_score_bars_refuses_host_tensors():
    with pytest.raises(RuntimeError):
        pkg("data.packed").score_bars(torch.zeros(1, 1, 96, 60), torch.zeros(1, 1, 96, 60))


# ---- script arguments -----------------------------------------------------------------------------------------------
@pytest.fixture
def two_files(tmp_path):
    midi = pkg("midi")
    a, b, short = (str(tmp_path / n) for n in ("a.mid", "b.mid", "short.mid"))
    midi.write_midi(_roll(2, 4), a)
    midi.write_midi(_roll(3, 5), b)
    midi.write_midi(_roll(1, 6, last_step_note=False)[:100], short)
    return a, b, short


def test_main_rejects_bad_encode_arguments(two_files, monkeypatch):
    a, b, short = two_files

    def no_device(*args, **kw):
        raise AssertionError("the device was touched before the arguments were checked")
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    bad = [["--reconstruct", a, "--interpolate", a, b],
           ["--reconstruct", a, "--primer", a],
           ["--interpolate", a, b, "--primer", a],
           ["--reconstruct", a, "--songs", "2"],
           ["--interpolate", a, b, "--songs", "1"],
           ["--interpolate", a, b, "--steps", "1"],
           ["--interpolate", a, b, "--steps", "0"],
           ["--reconstruct", a, "--steps", "3"],
           ["--steps", "3"],
           ["--phrases", "1"],
           ["--reconstruct", a, "--phrases", "0"],
           ["--reconstruct", short],
           ["--interpolate", a, short],
           ["--interpolate", short, b],
           ["--interpolate", a],
           ["--reconstruct", a, "--temperature", "0"]]
    for argv in bad:
        with pytest.raises(SystemExit) as e:
            pkg("maker_bar").main(argv)
        assert e.value.code == 2, argv
