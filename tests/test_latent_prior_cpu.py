"""CPU: the latent prior's float64 oracle (pinned to numpy.cov and closed forms), the host finalisation and its errors,
the ridge, the prior file (round trip, format tag, encoder digest), the input helpers, and the argument checks of
maker_bar.main's --fit_prior / --latent_prior that run before any device work."""
import os
import sys

import numpy as np
import pytest
import torch

from gpu_util import ROOT, pkg

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import prior_oracle as PO  # noqa: E402


def _offset(n, d, seed):
    """latents like the reference initialisation's: mean 500, std 30, fp32"""
    return (500.0 + 30.0 * np.random.RandomState(seed).randn(n, d)).astype(np.float32)


# ---- the oracle --------------------------------------------------------------------------------------------------------
def test_oracle_matches_numpy_cov():
    z = _offset(50, 7, 1)
    mu, cov = PO.finalize(*PO.moments(z), 50)
    z64 = z.astype(np.float64)
    np.testing.assert_allclose(mu, z64.mean(0), rtol=1e-13)
    np.testing.assert_allclose(cov, np.cov(z64.T), rtol=1e-9, atol=1e-9 * np.abs(np.cov(z64.T)).max())


def test_oracle_sequential_order_is_chunk_invariant_and_agrees_with_blas():
    z = _offset(41, 5, 2)
    s, g = PO.moments_sequential(z)
    s1, g1 = PO.moments_sequential(z[:13])
    s2, g2 = PO.moments_sequential(z[13:], s1, g1)
    assert np.array_equal(s, s2) and np.array_equal(g, g2)
    sb, gb = PO.moments(z)
    np.testing.assert_allclose(s, sb, rtol=1e-14)
    np.testing.assert_allclose(g, gb, rtol=1e-14)
    assert not np.tril(g, -1).any()
    lower = np.full((5, 5), -7.25)
    assert np.array_equal(np.tril(PO.moments_sequential(z, None, lower)[1], -1), np.tril(lower, -1))


def test_oracle_closed_forms():
    a, b = np.array([1.0, 2.0, -3.0], np.float32), np.array([5.0, 2.0, 1.0], np.float32)
    mu, cov = PO.finalize(*PO.moments(np.stack([a, b])), 2)
    assert np.array_equal(mu, (a + b) / 2.0)
    dlt = (a - b).astype(np.float64)
    assert np.array_equal(cov, np.outer(dlt, dlt) / 2.0)
    z = np.array([[3, 1], [3, 2], [3, 5], [3, 8]], np.float32)       # a constant column has zero (co)variance
    mu, cov = PO.finalize(*PO.moments(z), 4)
    assert mu[0] == 3.0 and cov[0, 0] == 0.0 and cov[0, 1] == 0.0 and cov[1, 0] == 0.0
    assert cov[1, 1] == np.var(z[:, 1].astype(np.float64), ddof=1)


# ---- the host finalisation -------------------------------------------------------------------------------------------
def test_finalize_matches_oracle():
    P = pkg("prior")
    z = _offset(200, 9, 3)
    s, g = PO.moments(z)
    g_lower = g + np.tril(np.full((9, 9), 1e30), -1)                # the lower triangle is never read
    mu, cov = P.finalize_moments(s, g_lower, 200)
    want_mu, want_cov = PO.finalize(s, g, 200)
    assert np.array_equal(mu, want_mu) and np.array_equal(cov, want_cov)
    assert np.array_equal(cov, cov.T)


def test_finalize_errors():
    P = pkg("prior")
    s, g = PO.moments(_offset(5, 4, 4))
    with pytest.raises(ValueError, match="at least 2"):
        P.finalize_moments(s, g, 1)
    with pytest.raises(ValueError, match="at least 2"):
        P.finalize_moments(s, g, 0)
    for bad in (np.inf, np.nan):
        g2 = g.copy()
        g2[1, 2] = bad
        with pytest.raises(ValueError, match="not finite"):
            P.finalize_moments(s, g2, 5)
        s2 = s.copy()
        s2[0] = bad
        with pytest.raises(ValueError, match="not finite"):
            P.finalize_moments(s2, g, 5)
    zs, zg = PO.moments(np.zeros((6, 4), np.float32))                # silent bars: every latent the same
    with pytest.raises(ValueError, match="zero trace"):
        P.finalize_moments(zs, zg, 6)


def test_ridge_makes_rank_deficient_fits_usable():
    P = pkg("prior")
    z = _offset(3, 8, 5)                                             # 3 latents in 8 dimensions: rank 2
    mu, cov = P.finalize_moments(*PO.moments(z), 3)
    with pytest.raises(ValueError, match="shrinkage=0"):
        P.LatentPrior(mu, cov, 3, 0.0, "x").cholesky()
    L = P.LatentPrior(mu, cov, 3, 1e-3, "x").cholesky()
    want = PO.cholesky_ridge(cov, 1e-3)
    np.testing.assert_allclose(L.numpy(), want, rtol=1e-10, atol=1e-10 * np.abs(want).max())
    assert not np.triu(L.numpy(), 1).any()
    with pytest.raises(ValueError):
        P.LatentPrior(mu, cov, 3, -1.0, "x")


# ---- the prior file ---------------------------------------------------------------------------------------------------
class _Gen(torch.nn.Module):
    def __init__(self, seed):
        super().__init__()
        torch.manual_seed(seed)
        self.encoder = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 2))
        self.decoder = torch.nn.Linear(2, 2)


def _prior(model, d=6):
    P = pkg("prior")
    mu, cov = P.finalize_moments(*PO.moments(_offset(20, d, 6)), 20)
    return P.LatentPrior(mu, cov, 20, 2e-3, P.encoder_digest(model))


def test_save_load_round_trip(tmp_path):
    P = pkg("prior")
    m = _Gen(0)
    pr = _prior(m)
    path = str(tmp_path / "p.pt")
    P.save_latent_prior(pr, path)
    got = P.load_latent_prior(path, m)
    assert torch.equal(got.mean, pr.mean) and torch.equal(got.cov, pr.cov)
    assert (got.count, got.shrinkage, got.encoder_digest) == (20, 2e-3, pr.encoder_digest)
    assert got.mean.dtype == got.cov.dtype == torch.float64


def test_load_refuses_wrong_format_and_other_checkpoints(tmp_path):
    P = pkg("prior")
    m = _Gen(0)
    path = str(tmp_path / "p.pt")
    P.save_latent_prior(_prior(m), path)
    with pytest.raises(ValueError, match="refit"):
        P.load_latent_prior(path, _Gen(1))
    m2 = _Gen(0)
    with torch.no_grad():
        m2.decoder.weight.add_(1.0)                                  # only the bar encoder is hashed
    P.load_latent_prior(path, m2)
    with torch.no_grad():
        m2.encoder[1].bias[0] += 1e-6
    with pytest.raises(ValueError, match="refit"):
        P.load_latent_prior(path, m2)
    st = torch.load(path, weights_only=True)
    st["format"] = "something-else"
    torch.save(st, path)
    with pytest.raises(ValueError, match="not a latent prior"):
        P.load_latent_prior(path, m)
    torch.save({"mean": torch.zeros(2)}, path)
    with pytest.raises(ValueError, match="not a latent prior"):
        P.load_latent_prior(path, m)


def test_digest_covers_names_shapes_and_values():
    P = pkg("prior")
    a, b = _Gen(0), _Gen(0)
    assert P.encoder_digest(a) == P.encoder_digest(b)
    b.encoder = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 2))
    b.encoder.load_state_dict(a.encoder.state_dict())
    assert P.encoder_digest(a) == P.encoder_digest(b)
    b.encoder[0].weight.data = b.encoder[0].weight.data.double()
    assert P.encoder_digest(a) != P.encoder_digest(b)


# ---- input helpers and device-only entry points ---------------------------------------------------------------------
def test_bars_of_packed_reads_only_note_bits(tmp_path):
    P = pkg("prior")
    bits = np.random.RandomState(7).randint(0, 256, size=(10, 720)).astype(np.uint8)
    np.save(str(tmp_path / "note_bits.npy"), bits)
    parts = list(P.bars_of_packed(str(tmp_path), chunk=4))
    assert [p.shape for p in parts] == [(4, 720), (4, 720), (2, 720)]
    assert np.array_equal(np.concatenate(parts), bits)
    assert all(P._is_bit_rows(p) for p in parts)
    np.save(str(tmp_path / "note_bits.npy"), bits[:, :700])
    with pytest.raises(ValueError):
        list(P.bars_of_packed(str(tmp_path)))


def test_bars_of_midi(tmp_path):
    P, mb, midi = pkg("prior"), pkg("maker_bar"), pkg("midi")
    roll = (np.random.RandomState(8).rand(2 * 384, 60) < 0.05).astype(np.float32)
    roll[-1, 30] = 1.0
    midi.write_midi(roll, str(tmp_path / "a.mid"))
    midi.write_midi(roll[:100], str(tmp_path / "short.mid"))
    (got,) = list(P.bars_of_midi([str(tmp_path / "a.mid")]))
    assert got.shape == (8, 96, 60) and np.array_equal(got.reshape(-1, 60), mb.load_roll(str(tmp_path / "a.mid"))[0])
    with pytest.raises(ValueError, match="covers no whole"):
        list(P.bars_of_midi([str(tmp_path / "short.mid")]))


def test_device_entry_points_refuse_host_tensors():
    P = pkg("prior")
    with pytest.raises(RuntimeError):
        P.latent_moments(torch.zeros(3, 4), torch.zeros(4, dtype=torch.float64), torch.zeros(4, 4, dtype=torch.float64))
    pr = P.LatentPrior(np.zeros(3), np.eye(3), 5, 0.0, "x")
    with pytest.raises(RuntimeError):
        pr.sample(2, 2, torch.Generator())


# ---- script arguments -----------------------------------------------------------------------------------------------
def test_main_rejects_bad_prior_arguments(tmp_path, monkeypatch):
    midi = pkg("midi")
    roll = (np.random.RandomState(9).rand(2 * 384, 60) < 0.05).astype(np.float32)
    roll[-1, 30] = 1.0
    a = str(tmp_path / "a.mid")
    midi.write_midi(roll, a)
    np.save(str(tmp_path / "note_bits.npy"), np.zeros((4, 720), np.uint8))
    prior = str(tmp_path / "p.pt")
    with open(prior, "wb") as f:
        f.write(b"x")

    def no_device(*args, **kw):
        raise AssertionError("the device was touched before the arguments were checked")
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    bad = [["--latent_prior", prior, "--reconstruct", a],
           ["--latent_prior", prior, "--interpolate", a, a],
           ["--fit_prior", "o.pt", "--data", a, "--reconstruct", a],
           ["--fit_prior", "o.pt", "--data", a, "--interpolate", a, a],
           ["--fit_prior", "o.pt", "--data", a, "--primer", a],
           ["--fit_prior", "o.pt", "--data", a, "--latent_prior", prior],
           ["--fit_prior", "o.pt", "--data", a, "--songs", "2"],
           ["--data", a],
           ["--fit_prior", "o.pt"],
           ["--fit_prior", "o.pt", "--data", str(tmp_path / "missing.mid")],
           ["--fit_prior", "o.pt", "--data", prior],
           ["--fit_prior", "o.pt", "--data", str(tmp_path / "empty_dir_that_does_not_exist")],
           ["--latent_prior", str(tmp_path / "missing.pt")]]
    for argv in bad:
        with pytest.raises(SystemExit) as e:
            pkg("maker_bar").main(argv)
        assert e.value.code == 2, argv
