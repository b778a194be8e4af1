"""GPU (B200): the per-bar score (csrc/sample.cu, bvae_bar_score) against its numpy oracle, the decoder and the
training loss; the song-level API of maker_bar (encode_songs, reconstruct_songs, interpolate_latents) against the
explicit forward, the sampling loop and the fp32 CPU oracle; and the script's --reconstruct / --interpolate modes end to
end.  Model-level tests run with bvae_set_deterministic(1) (bit-reproducible forward, DESIGN.md section 7), restored
afterwards, and keep every exact comparison's passes below the 256-sample norm-block routing change (DESIGN.md 4.3)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from gpu_util import PKG, ROOT, pkg, report

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import score_oracle as SC  # noqa: E402

pytestmark = pytest.mark.gpu
CELLS = SC.BAR_CELLS


@pytest.fixture
def deterministic():
    lib = pkg("_lib")
    before = bool(lib.load().bvae_deterministic())
    lib.set_deterministic(True)
    yield
    lib.set_deterministic(before)


def _rows(bars):
    """the rows held against the oracle: all of them up to 700 bars, else the first / last 64 and 64 random ones"""
    if bars <= 700:
        return np.arange(bars)
    r = np.random.RandomState(bars)
    return np.unique(np.concatenate([np.arange(64), np.arange(bars - 64, bars), r.randint(0, bars, 64)]))


def _score(logits, target, temperature, threshold, canary=-7):
    """score_bars' kernel into buffers with canaries behind both outputs; returns host (nll, counts)"""
    bars = logits.numel() // CELLS
    nll = torch.full((bars + 16,), float(canary), device="cuda")
    counts = torch.full((bars * 3 + 16,), canary, dtype=torch.int32, device="cuda")
    L = pkg("_lib")
    L.check(L.lib().bvae_bar_score(logits.data_ptr(), target.data_ptr(), bars, 1.0 / temperature, threshold,
                                   nll.data_ptr(), counts.data_ptr(), L.stream_ptr()), "bar_score")
    nll, counts = nll.cpu(), counts.cpu()
    assert torch.all(nll[bars:] == canary) and torch.all(counts[bars * 3:] == canary), "bar_score wrote behind"
    return nll[:bars].numpy(), counts[:bars * 3].view(bars, 3).numpy()


def _data(bars, seed, scale=4.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    logits = torch.randn(bars, 1, 96, 60, device="cuda", generator=g) * scale
    # targets correlated with the logits, so that all four outcomes of (predicted, on) occur
    target = (torch.rand(bars, 1, 96, 60, device="cuda", generator=g) < torch.sigmoid(logits - 1.0)).float()
    return logits, target


# ---- the kernel -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("temperature", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("bars", [1, 3, 64, 700, 8192])
def test_kernel_matches_oracle(bars, temperature):
    logits, target = _data(bars, bars)
    rows = _rows(bars)
    lgh = logits.view(-1, CELLS).cpu().numpy()[rows]
    tgh = target.view(-1, CELLS).cpu().numpy()[rows]
    inv_t = float(np.float32(1.0 / temperature))
    for threshold in (0.3, 0.5):
        nll, counts = _score(logits, target, temperature, threshold)
        want_nll, want_counts, p = SC.score(lgh, tgh, inv_t, threshold)
        thr = np.float32(threshold)
        band = np.abs(p - thr) <= 8 * np.spacing(thr)                     # device expf may differ in the last bit
        slack = np.stack([(band & (tgh != 0)).sum(1), band.sum(1), np.zeros(len(rows), np.int64)], 1)
        diff = np.abs(counts[rows].astype(np.int64) - want_counts)
        report(test="bar_score_kernel", bars=bars, temperature=temperature, threshold=threshold,
               nll_max_rel=float(np.max(np.abs(nll[rows] - want_nll) / want_nll)), band_cells=int(band.sum()),
               count_mismatches=int(diff.sum()))
        np.testing.assert_allclose(nll[rows], want_nll, rtol=1e-5)
        assert np.all(diff <= slack)


def test_chunks_are_bit_identical_to_one_call():
    logits, target = _data(64, 5)
    whole = _score(logits, target, 1.3, 0.3)
    halves = [_score(logits[a:b].contiguous(), target[a:b].contiguous(), 1.3, 0.3) for a, b in ((0, 23), (23, 64))]
    assert np.array_equal(whole[0], np.concatenate([h[0] for h in halves]))
    assert np.array_equal(whole[1], np.concatenate([h[1] for h in halves]))


def test_infinite_and_nan_logits():
    logits = torch.zeros(5, 1, 96, 60, device="cuda")
    target = torch.zeros(5, 1, 96, 60, device="cuda")
    flat_l, flat_t = logits.view(5, CELLS), target.view(5, CELLS)
    flat_l[0, 0], flat_t[0, 0] = float("inf"), 1.0          # -> 0
    flat_l[1, 0], flat_t[1, 0] = float("inf"), 0.0          # -> +inf
    flat_l[2, 0], flat_t[2, 0] = float("-inf"), 1.0         # -> +inf
    flat_l[3, 0], flat_t[3, 0] = float("-inf"), 0.0         # -> 0
    flat_l[4, 0], flat_t[4, 0] = float("nan"), 1.0          # -> NaN, never predicted on
    rest = np.float32((CELLS - 1) * np.log(2.0))
    for temperature in (0.5, 1.0, 2.0):
        nll, counts = _score(logits, target, temperature, -1.0)                 # threshold -1: every non-NaN p is on
        np.testing.assert_allclose(nll[[0, 3]], [rest, rest], rtol=1e-5)
        assert np.isinf(nll[1]) and nll[1] > 0 and np.isinf(nll[2]) and nll[2] > 0 and np.isnan(nll[4])
        assert counts[:4, 1].tolist() == [CELLS] * 4 and counts[4].tolist() == [0, CELLS - 1, 1]
        assert counts[:, 0].tolist() == [1, 0, 1, 0, 0]


def test_argument_errors_leave_the_outputs_untouched():
    L = pkg("_lib")
    lib = L.lib()
    x = torch.zeros(2 * CELLS + 8, device="cuda")
    t = torch.zeros(2 * CELLS + 8, device="cuda")
    nll = torch.full((8,), 5.0, device="cuda")
    cnt = torch.full((16,), 5, dtype=torch.int32, device="cuda")
    st = L.stream_ptr()
    args = lambda **kw: dict(dict(lg=x.data_ptr(), tg=t.data_ptr(), bars=1, inv_t=1.0, thr=0.3, nll=nll.data_ptr(),
                                  cnt=cnt.data_ptr()), **kw)
    call = lambda a: lib.bvae_bar_score(a["lg"], a["tg"], a["bars"], a["inv_t"], a["thr"], a["nll"], a["cnt"], st)
    for inv_t in (0.0, -1.0, float("inf"), float("-inf"), float("nan")):
        assert call(args(inv_t=inv_t)) == 1
    for thr in (float("inf"), float("-inf"), float("nan")):
        assert call(args(thr=thr)) == 1
    assert call(args(bars=-1)) == 1
    assert call(args(lg=x.data_ptr() + 4)) == 2
    assert call(args(tg=t.data_ptr() + 8)) == 2
    assert call(args(nll=nll.data_ptr() + 2)) == 2
    assert call(args(cnt=cnt.data_ptr() + 1)) == 2
    assert call(args(bars=0)) == 0
    torch.cuda.synchronize()
    assert torch.all(nll == 5.0) and torch.all(cnt == 5)
    packed = pkg("data.packed")
    for temperature in (0.0, -2.0, float("inf"), float("nan")):
        with pytest.raises(RuntimeError):
            packed.score_bars(x[:CELLS], t[:CELLS], temperature)
    with pytest.raises(ValueError):
        packed.score_bars(x[:CELLS], t[:2 * CELLS])
    with pytest.raises(ValueError):
        packed.score_bars(x[:CELLS - 4], t[:CELLS - 4])


def test_against_the_training_loss():
    """on logits in [-4, 4]: nll / 5760 is bvae_bce_fwd's mean BCE on torch.sigmoid(logits), bar by bar"""
    L = pkg("_lib")
    g = torch.Generator(device="cuda").manual_seed(17)
    logits = torch.rand(6, 1, 96, 60, device="cuda", generator=g) * 8 - 4
    target = (torch.rand(6, 1, 96, 60, device="cuda", generator=g) < 0.3).float()
    nll, _ = pkg("data.packed").score_bars(logits, target)
    probs = torch.sigmoid(logits)
    for b in range(6):
        acc = torch.zeros(2, device="cuda")
        L.check(L.lib().bvae_bce_fwd(probs[b].data_ptr(), target[b].data_ptr(), CELLS, 0, acc.data_ptr(),
                                     L.stream_ptr()), "bce_fwd")
        assert abs(float(nll[b]) / CELLS - float(acc[0])) <= 1e-4 * float(acc[0])


# ---- the model ------------------------------------------------------------------------------------------------------
def _model(refiner=False):
    O = __import__("barvae_oracle")
    sd = O.make_state_dict(O.generator_spec(), 11, "lively")
    m = pkg("graph.model").Model(refiner=refiner)
    m.load_state_dict(sd, strict=not refiner)
    return m.cuda().eval()


def _songs(S, L, seed, density=0.05):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.rand(S, L * 384, 60, device="cuda", generator=g) < density).float()


def _items(song):
    """the teacher-forced items of songs [S, L*384, 60] in the dataset's layout (note, pre_note, pre_phrase, position),
    song-major, with the conditioning of the sampling loop"""
    S, L = song.shape[0], song.shape[1] // 384
    bars = song.view(S, 4 * L, 1, 96, 60)
    note, pre_note, pre_phrase, position = [], [], [], []
    phrase_idx = [330] + list(range(L - 2, -1, -1))
    for s in range(S):
        for k in range(4 * L):
            p = k // 4
            note.append(bars[s, k])
            pre_note.append(bars[s, k - 1] if k else torch.zeros_like(bars[s, k]))
            pre_phrase.append(song[s, (p - 1) * 384:p * 384].view(1, 384, 60) if p else torch.zeros(1, 384, 60,
                                                                                                    device="cuda"))
            position.append(phrase_idx[p])
    return (torch.stack(note), torch.stack(pre_note), torch.stack(pre_phrase),
            torch.tensor(position, device="cuda"))


def test_decoder_counts_at_temperature_one(deterministic):
    """T = 1: the kernel's p is the decoder's probability bit for bit, so the counts are those of (probs > 0.3)"""
    O = __import__("barvae_oracle")
    model = _model()
    note, pre_note, phrase, position = (t.cuda() for t in O.make_inputs(8, 31))
    g = torch.Generator(device="cuda").manual_seed(2)
    z = torch.randn(8, 1152, device="cuda", generator=g)
    with torch.no_grad():
        probs, logits = model.decoder.forward_logits(z, model.encoder(pre_note), model.phrase_encoder(phrase),
                                                     position)
    _, counts = pkg("data.packed").score_bars(logits, note, 1.0, 0.3)
    on = (probs > 0.3).view(8, CELLS)
    t = note.view(8, CELLS) != 0
    want = torch.stack([(on & t).sum(1), on.sum(1), t.sum(1)], 1).int()
    report(test="bar_score_decoder", predicted_on=int(want[:, 1].sum()), on=int(want[:, 2].sum()))
    assert 0 < int(want[:, 1].sum()) < 8 * CELLS
    assert torch.equal(counts, want)


def test_encode_songs_is_the_encoder_bar_by_bar(deterministic):
    mb, model = pkg("maker_bar"), _model()
    song = _songs(2, 2, 1)
    lat = mb.encode_songs(model, song)
    assert lat.shape == (8, 2, 1152) and lat.dtype == torch.float32
    with torch.no_grad():
        for s in range(2):
            for k in range(8):
                z = model.encoder(song[s, k * 96:(k + 1) * 96].view(1, 1, 96, 60))
                assert torch.equal(lat[k, s], z[0]), (s, k)
    assert torch.equal(mb.encode_songs(model, song, chunk=5), mb.encode_songs(model, song, chunk=64))
    assert torch.equal(mb.encode_songs(model, song[1]), lat[:, 1:])          # one song: [L*384, 60]


def test_reconstruct_is_the_explicit_forward(deterministic):
    mb, model = pkg("maker_bar"), _model()
    song = _songs(2, 3, 2)
    rec = mb.reconstruct_songs(model, song, return_logits=True)
    note, pre_note, pre_phrase, position = _items(song)
    with torch.no_grad():
        _, logits = model.decoder.forward_logits(model.encoder(note), model.encoder(pre_note),
                                                 model.phrase_encoder(pre_phrase), position)
    assert rec.logits.shape == (2, 12, 96, 60) and rec.nll.shape == (2, 12) and rec.counts.shape == (2, 12, 3)
    assert torch.equal(rec.logits.reshape(-1), logits.reshape(-1))
    assert torch.equal(rec.latents, mb.encode_songs(model, song))
    nll, counts = pkg("data.packed").score_bars(logits, note, 1.0, 0.3)
    assert torch.equal(rec.nll.reshape(-1), nll) and torch.equal(rec.counts.reshape(-1, 3), counts)
    rec2 = mb.reconstruct_songs(model, song, temperature=0.7, threshold=0.5, chunk=5)
    assert rec2.logits is None
    nll2, counts2 = pkg("data.packed").score_bars(logits, note, 0.7, 0.5)
    assert torch.equal(rec2.nll.reshape(-1), nll2) and torch.equal(rec2.counts.reshape(-1, 3), counts2)
    report(test="reconstruct_explicit", nll_per_bar=float(rec.nll.mean()), on=int(rec.counts[..., 2].sum()),
           tp=int(rec.counts[..., 0].sum()), predicted=int(rec.counts[..., 1].sum()))


@pytest.mark.parametrize("P", [0, 1, 2])
def test_reconstruct_is_the_sampling_loop_on_the_songs_own_latents(deterministic, P):
    """bar 4P, where the loop's pre_bar / pre_phrase are the song's own (its primer), decodes to the same bits"""
    mb, model = pkg("maker_bar"), _model()
    S, L = 2, 3
    song = _songs(S, L, 3)
    rec = mb.reconstruct_songs(model, song, return_logits=True)
    _, first = mb.sample_songs(model, mb.encode_songs(model, song), L, True,
                               primer=song[:, :P * 384] if P else None)
    note, pre_note, pre_phrase, position = (t.view(S, 4 * L, *t.shape[1:])[:, 4 * P] for t in _items(song))
    with torch.no_grad():
        probs, logits = model.decoder.forward_logits(model.encoder(note), model.encoder(pre_note),
                                                     model.phrase_encoder(pre_phrase), position)
    assert torch.equal(logits[:, 0], rec.logits[:, 4 * P])        # the teacher-forced bar ...
    assert torch.equal(first, probs)                              # ... and its probabilities are the loop's


def test_reconstruct_against_the_cpu_oracle(deterministic):
    O = __import__("barvae_oracle")
    sd = O.make_state_dict(O.generator_spec(), 11, "lively")
    mb, model = pkg("maker_bar"), _model()
    song = _songs(2, 2, 4)
    rec = mb.reconstruct_songs(model, song, return_logits=True)
    items = [t.cpu() for t in _items(song)]
    with torch.no_grad():
        gen = O.model_forward(*items, sd, True, None)[0]
    got = torch.sigmoid(rec.logits.reshape(-1, 1, 96, 60)).cpu()
    err = (got - gen).abs()
    report(test="reconstruct_oracle", max_abs=float(err.max()), mean_abs=float(err.mean()))
    assert float(err.max()) < 6e-2 and float(err.mean()) < 1e-2


def test_chunk_boundaries_at_the_benchmarked_size(deterministic):
    mb, model = pkg("maker_bar"), _model()
    song = _songs(512, 5, 5)
    a = mb.reconstruct_songs(model, song, chunk=8192)
    b = mb.reconstruct_songs(model, song, chunk=4096)
    report(test="reconstruct_chunks", bars=a.nll.numel(), nll_per_bar=float(a.nll.mean()))
    assert torch.equal(a.nll, b.nll) and torch.equal(a.counts, b.counts)


@pytest.mark.parametrize("sampler", ["threshold", "bernoulli"])
def test_interpolation_decodes_its_endpoints(deterministic, sampler):
    mb, model = pkg("maker_bar"), _model()
    L, N = 2, 4
    za = mb.encode_songs(model, _songs(1, L, 6)[0])
    zb = mb.encode_songs(model, _songs(1, L, 7, density=0.1)[0])
    z = mb.interpolate_latents(za, zb, N)
    assert z.shape == (4 * L, N, 1152)
    kw = dict(sampler=sampler, temperature=0.9, seed=21)
    songs = mb.sample_songs(model, z, L, **kw)
    assert torch.equal(songs[0], mb.sample_songs(model, za, L, **kw)[0])
    assert torch.equal(songs[N - 1], mb.sample_songs(model, zb, L, song_base=N - 1, **kw)[0])
    assert not torch.equal(songs[0], songs[N - 1])


def test_reconstruct_with_refiner_raises():
    mb = pkg("maker_bar")
    with pytest.raises(ValueError):
        mb.reconstruct_songs(_model(refiner=True), _songs(1, 1, 8)[0])


# ---- the script end to end -------------------------------------------------------------------------------------------
def _run_main(cwd, argv):
    env = dict(os.environ, BVAE_DETERMINISTIC="1", PYTHONPATH=ROOT)
    code = "import importlib, sys; importlib.import_module(%r).main(sys.argv[1:])" % (PKG + ".maker_bar")
    r = subprocess.run([sys.executable, "-c", code] + argv, cwd=str(cwd), env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


def test_main_reconstruct_and_interpolate(tmp_path, deterministic):
    mb, midi = pkg("maker_bar"), pkg("midi")
    O = __import__("barvae_oracle")
    sd = O.make_state_dict(O.generator_spec(), 11, "lively")
    os.makedirs(tmp_path / "model")
    torch.save({"generator_state_dict": {"module." + k: v for k, v in sd.items()}},
               str(tmp_path / "model" / "checkpoint_10.pth.tar"))
    model = _model()
    rolls = []
    for name, phrases, seed in (("a.mid", 2, 9), ("b.mid", 3, 10)):
        roll = _songs(1, phrases, seed)[0].cpu().numpy()
        roll[-1, 30] = 1.0                                  # the file covers all its phrases
        midi.write_midi(roll, str(tmp_path / name))
        rolls.append(mb.load_roll(str(tmp_path / name))[0])
    # --reconstruct: the free-running decode of the file's latents, and the teacher-forced score
    out = _run_main(tmp_path, ["--reconstruct", "a.mid", "--seed", "1", "--out", "rec.mid"])
    assert "reconstruct: 2 phrases from a.mid, 0 notes" in out
    want = mb.songs_to_host(mb.sample_songs(model, mb.encode_songs(model, rolls[0]), 2))[0]
    midi.write_midi(want, str(tmp_path / "want.mid"))
    assert (tmp_path / "rec.mid").read_bytes() == (tmp_path / "want.mid").read_bytes()
    line = mb.score_line(mb.reconstruct_songs(model, rolls[0]))
    assert line in out, (line, out)
    # --interpolate --steps 3: b is cut to a's two phrases; the first and last files are the endpoint decodes
    out = _run_main(tmp_path, ["--interpolate", "a.mid", "b.mid", "--steps", "3", "--out", "m.mid"])
    got = [midi.midi_to_roll(str(tmp_path / n), 2 * 384) for n in ("m.mid", "m_1.mid", "m_2.mid")]
    for i, r in ((0, rolls[0]), (2, rolls[1][:2 * 384])):
        want = mb.songs_to_host(mb.sample_songs(model, mb.encode_songs(model, r), 2))[0]
        assert np.array_equal(got[i], want), i
    assert not (tmp_path / "m_3.mid").exists()
