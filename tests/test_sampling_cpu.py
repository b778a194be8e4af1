"""CPU: the Bernoulli sampler's stream (oracle pinned to the Random123 known answers), primer loading and the argument
checks of the sampling loop and of maker_bar.main that run before any device work."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from gpu_util import ROOT, pkg

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import sample_oracle as SO  # noqa: E402

KAT = [  # Random123 kat_vectors, philox4x32_10: counter, key -> output
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
     (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff),
     (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    assert tuple(int(w) for w in SO.philox4x32_10(ctr, key)) == want


def test_philox_vectorised_equals_scalar():
    c = np.array([0, 1, 0xffffffff, 12345], dtype=np.uint64)
    got = SO.philox4x32_10((c, 7, c ^ np.uint64(0xabcdef), 3), (0x1234, 0xffff0000))
    for j in range(4):
        one = SO.philox4x32_10((int(c[j]), 7, int(c[j]) ^ 0xabcdef, 3), (0x1234, 0xffff0000))
        assert [int(w[j]) for w in got] == [int(w) for w in one]


def test_stream_layout():
    """cell i of bar k of song s is word i % 4 of the block for counter {i // 4, k, s lo, s hi}, key {seed lo, hi}"""
    seed, song, k = 0x0123456789abcdef, (5 << 32) + 9, 17
    u = SO.uniforms(seed, [song], k)[0]
    for i in (0, 1, 2, 3, 4, 2023, 5759):
        r = SO.philox4x32_10((i // 4, k, song & 0xffffffff, song >> 32), (seed & 0xffffffff, seed >> 32))[i % 4]
        assert u[i] == np.float32((int(r) >> 8) / 2.0 ** 24)
    assert u.dtype == np.float32 and 0.0 <= u.min() and u.max() < 1.0
    assert np.all(u * np.float32(2 ** 24) == np.floor(u * np.float32(2 ** 24)))      # multiples of 2^-24: exact


def test_oracle_same_inputs_same_bar_and_each_input_matters():
    base = SO.uniforms(3, [11], 2)
    assert np.array_equal(base, SO.uniforms(3, [11], 2))
    for other in (SO.uniforms(4, [11], 2), SO.uniforms(3, [12], 2), SO.uniforms(3, [11], 3),
                  SO.uniforms(3 + (1 << 32), [11], 2), SO.uniforms(3, [11 + (1 << 32)], 2)):
        assert (other != base).mean() > 0.99


def test_oracle_song_base_split_changes_nothing():
    r = np.random.RandomState(0)
    logits = r.randn(64, SO.BAR_CELLS).astype(np.float32) * 3
    u, p, cells = SO.sample(logits, 1.25, 99, 0, 6)
    u1, p1, c1 = SO.sample(logits[:32], 1.25, 99, 0, 6)
    u2, p2, c2 = SO.sample(logits[32:], 1.25, 99, 32, 6)
    assert np.array_equal(u, np.concatenate([u1, u2])) and np.array_equal(cells, np.concatenate([c1, c2]))


def test_oracle_extreme_logits():
    lg = np.zeros((1, SO.BAR_CELLS), dtype=np.float32)
    lg[0, :3] = [np.inf, -np.inf, np.nan]
    _, p, cells = SO.sample(lg, 1.0, 0, 0, 0)
    assert cells[0, 0] == 1 and cells[0, 1] == 0 and cells[0, 2] == 0
    assert np.all(p[0, 3:] == np.float32(0.5))


# ---- primer ---------------------------------------------------------------------------------------------------------
def _roll(phrases, seed, last_step_note=True):
    r = np.random.RandomState(seed)
    roll = (r.rand(phrases * 384, 60) < 0.05).astype(np.float32)
    if last_step_note:
        roll[-1, 30] = 1.0                       # the file then covers all its phrases (MIDI has no end-of-roll mark)
    return roll


def test_primer_midi_roundtrip(tmp_path):
    mb, midi = pkg("maker_bar"), pkg("midi")
    roll = _roll(2, 1)
    path = str(tmp_path / "p.mid")
    midi.write_midi(roll, path)
    got, P, dropped = mb.load_primer(path, music_length=4)
    assert P == 2 and dropped == 0 and np.array_equal(got, roll)
    got1, P1, _ = mb.load_primer(path, music_length=4, phrases=1)
    assert P1 == 1 and np.array_equal(got1, roll[:384])
    # a trailing silent phrase is not in the file; asking for it explicitly gives silence
    quiet = _roll(2, 2, last_step_note=False)
    quiet[384:] = 0
    midi.write_midi(quiet, path)
    got2, P2, _ = mb.load_primer(path, music_length=4, phrases=2)
    assert P2 == 2 and np.array_equal(got2, quiet)
    with pytest.raises(ValueError):
        mb.load_primer(path, music_length=4, phrases=4)


def test_primer_notes_outside_the_window_are_dropped(tmp_path):
    mb, midi = pkg("maker_bar"), pkg("midi")
    roll = _roll(1, 3)
    roll[10:20, 2] = 1.0                          # written at lowest_pitch 20: pitch 22 is below the window
    path = str(tmp_path / "low.mid")
    midi.write_midi(roll, path, lowest_pitch=20)
    n_low = len([n for n in midi.roll_to_notes(roll, 20) if n[0] < midi.LOWEST_PITCH])
    got, P, dropped = mb.load_primer(path, music_length=3)
    assert P == 1 and dropped == n_low > 0
    want = np.zeros_like(roll)
    want[:, :53] = roll[:, 7:]                    # pitch 27 + c lands in column c
    assert np.array_equal(got, want)


def test_primer_validation():
    mb = pkg("maker_bar")
    ok = np.zeros((384, 60), dtype=np.float32)
    assert mb.check_primer(ok, 3, 2) == 1
    assert mb.check_primer(torch.zeros(3, 768, 60), 3, 3) == 2
    assert mb.check_primer(torch.ones(768, 60, dtype=torch.uint8), 5, 3) == 2
    bad = [(np.zeros((383, 60)), 1, 3),              # not whole phrases
           (np.zeros((384, 59)), 1, 3),              # pitches
           (np.zeros((2, 384, 60)), 3, 3),           # songs
           (np.zeros((1, 1, 384, 60)), 1, 3),        # rank
           (np.zeros((0, 60)), 1, 3),                # P = 0
           (np.zeros((768, 60)), 1, 2),              # P >= music_length
           (np.full((384, 60), 0.5), 1, 3),          # not binary
           (np.full((384, 60), np.nan), 1, 3)]
    for primer, songs, L in bad:
        with pytest.raises(ValueError):
            mb.check_primer(primer, songs, L)


def test_sample_songs_rejects_bad_sampler_arguments():
    mb = pkg("maker_bar")
    lat = torch.zeros(8, 1, 1152)
    with pytest.raises(ValueError):
        mb.sample_songs(types.SimpleNamespace(refiner=None), lat, 2, sampler="nucleus")
    with pytest.raises(ValueError):                   # the Refiner outputs probabilities: no logits to draw from
        mb.sample_songs(types.SimpleNamespace(refiner=object()), lat, 2, sampler="bernoulli")
    with pytest.raises(ValueError):
        mb.sample_songs(types.SimpleNamespace(refiner=None), lat, 2, primer=torch.zeros(768, 60))


@pytest.mark.parametrize("argv", [["--temperature", "0"], ["--temperature", "-1"], ["--temperature", "nan"],
                                  ["--temperature", "inf"], ["--sampler", "topk"], ["--primer_phrases", "1"]])
def test_main_rejects_bad_arguments(argv):
    with pytest.raises(SystemExit):
        pkg("maker_bar").main(argv)


def test_main_rejects_bad_primer(tmp_path):
    midi = pkg("midi")
    path = str(tmp_path / "p.mid")
    midi.write_midi(_roll(2, 4), path)
    for argv in (["--music_length", "2"], ["--music_length", "4", "--primer_phrases", "0"],
                 ["--music_length", "4", "--primer_phrases", "4"]):
        with pytest.raises(SystemExit):
            pkg("maker_bar").main(argv + ["--primer", path])
    short = str(tmp_path / "short.mid")
    midi.write_midi(_roll(1, 5, last_step_note=False)[:100], short)     # covers no whole phrase
    with pytest.raises(SystemExit):
        pkg("maker_bar").main(["--primer", short])


def test_bernoulli_sample_refuses_host_tensors():
    with pytest.raises(RuntimeError):
        pkg("data.packed").bernoulli_sample(torch.zeros(1, 1, 96, 60), 1.0, 0, 0, 0)
