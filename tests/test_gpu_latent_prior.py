"""GPU (B200): the fp64 moment kernel (csrc/prior.cu, bvae_latent_moments) against its float64 oracle, bit for bit in
its summation order and across chunked calls; fit_latent_prior against float64 moments of encode_songs and across its
two input formats; the prior's draws; and maker_bar.main --fit_prior / --latent_prior end to end.  Model-level tests
run with bvae_set_deterministic(1), restored afterwards."""
import os
import sys

import numpy as np
import pytest
import torch

from gpu_util import ROOT, pkg, rel_fro, report
from test_gpu_encode import _model, _run_main, _songs

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import prior_oracle as PO  # noqa: E402

pytestmark = pytest.mark.gpu
CANARY = -7.25


@pytest.fixture
def deterministic():
    lib = pkg("_lib")
    before = bool(lib.load().bvae_deterministic())
    lib.set_deterministic(True)
    yield
    lib.set_deterministic(before)


def _offset(n, d, seed, ld=None):
    """reference-init-like latents (mean 500, std 30) as rows of pitch ``ld`` on the device: [n, d] view"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    buf = 500.0 + 30.0 * torch.randn(max(n, 1), ld or d, device="cuda", generator=g)
    return buf[:n, :d]


def _buffers(d, seed):
    """sum / gram with canaries behind both, nonzero starting values in the upper triangle and canaries below it"""
    r = np.random.RandomState(seed)
    s = np.concatenate([r.rand(d), np.full(16, CANARY)])
    g0 = np.triu(r.rand(d, d)) + np.tril(np.full((d, d), CANARY), -1)
    g = np.concatenate([g0.reshape(-1), np.full(16, CANARY)])
    return torch.from_numpy(s).cuda(), torch.from_numpy(g).cuda()


def _run(z, s, g, d):
    L = pkg("_lib")
    ld = z.stride(0) if z.shape[0] > 1 else d
    L.check(L.lib().bvae_latent_moments(z.data_ptr(), z.shape[0], d, ld, s.data_ptr(), g.data_ptr(), L.stream_ptr()),
            "latent_moments")


def _host(s, g, d):
    s, g = s.cpu().numpy(), g.cpu().numpy()
    assert np.all(s[d:] == CANARY) and np.all(g[d * d:] == CANARY), "latent_moments wrote behind its outputs"
    gm = g[:d * d].reshape(d, d)
    assert np.all(np.tril(gm, -1)[np.tril_indices(d, -1)] == CANARY), "latent_moments touched the lower triangle"
    return s[:d], gm


# ---- the kernel -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [37, 1152])
@pytest.mark.parametrize("n", [0, 1, 7, 8205])
def test_kernel_matches_oracle(n, d):
    ld = d + 3 if d == 37 else d                       # a row pitch wider than d for the small case
    z = _offset(n, d, n + d, ld)
    s, g = _buffers(d, n)
    s0, g0 = _host(s, g, d)
    _run(z, s, g, d)
    got_s, got_g = _host(s, g, d)
    zh = z.cpu().numpy()
    if n == 0:
        assert np.array_equal(got_s, s0) and np.array_equal(got_g, g0)
        return
    if d * d * n <= 37 * 37 * 8205:                     # the kernel's order exactly
        want_s, want_g = PO.moments_sequential(zh, s0, g0)
        assert np.array_equal(got_s, want_s) and np.array_equal(np.triu(got_g), np.triu(want_g))
    ms, mg = PO.moments(zh)
    want_s, want_g = s0 + ms, np.triu(g0) + mg
    up = np.triu_indices(d)
    err_g = float(np.max(np.abs(got_g[up] - want_g[up]) / np.abs(want_g[up])))
    err_s = float(np.max(np.abs(got_s - want_s) / np.abs(want_s)))
    report(test="latent_moments_kernel", n=n, d=d, gram_max_rel=err_g, sum_max_rel=err_s)
    assert err_g <= 1e-12 and err_s <= 1e-12, (err_g, err_s)


@pytest.mark.parametrize("d", [37, 1152])
def test_chunked_calls_are_bit_identical(d):
    z = _offset(8205, d, 3)
    one = _buffers(d, 1)
    _run(z, *one, d)
    again = _buffers(d, 1)
    _run(z, *again, d)
    parts = _buffers(d, 1)
    for i, j in ((0, 1), (1, 4096), (4096, 8205)):      # 1 + 4095 + 4109 rows
        _run(z[i:j], *parts, d)
    a, b, c = (_host(s, g, d) for s, g in (one, again, parts))
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(a[0], c[0]) and np.array_equal(a[1], c[1])


def test_error_codes():
    L = pkg("_lib")
    lib = L.lib()
    z = torch.zeros(8, 16, device="cuda")
    s = torch.zeros(17, dtype=torch.float64, device="cuda")
    g = torch.zeros(16 * 16 + 1, dtype=torch.float64, device="cuda")
    st = L.stream_ptr()
    assert lib.bvae_latent_moments(z.data_ptr(), -1, 16, 16, s.data_ptr(), g.data_ptr(), st) == 1
    assert lib.bvae_latent_moments(z.data_ptr(), 8, 0, 16, s.data_ptr(), g.data_ptr(), st) == 1
    assert lib.bvae_latent_moments(z.data_ptr(), 8, 16, 15, s.data_ptr(), g.data_ptr(), st) == 1
    assert lib.bvae_latent_moments(z.data_ptr() + 2, 4, 15, 16, s.data_ptr(), g.data_ptr(), st) == 2
    assert lib.bvae_latent_moments(z.data_ptr(), 8, 16, 16, s.data_ptr() + 4, g.data_ptr(), st) == 2
    assert lib.bvae_latent_moments(z.data_ptr(), 8, 16, 16, s.data_ptr(), g.data_ptr() + 4, st) == 2
    assert lib.bvae_latent_moments(z.data_ptr(), 0, 16, 16, s.data_ptr(), g.data_ptr(), st) == 0
    torch.cuda.synchronize()
    assert not s.any() and not g.any()
    P = pkg("prior")
    with pytest.raises(ValueError):
        P.latent_moments(z, s[:16].float(), g[:256].view(16, 16))
    with pytest.raises(ValueError):
        P.latent_moments(z.t(), s[:16], g[:256].view(16, 16))


# ---- the fit --------------------------------------------------------------------------------------------------------
def test_fit_matches_float64_moments_of_encode_songs(deterministic):
    mb, P = pkg("maker_bar"), pkg("prior")
    model = _model()
    roll = _songs(3, 3, 11)                               # 36 bars
    chunk = 16
    pr = P.fit_latent_prior(model, [roll.view(-1, 96, 60)], chunk=chunk)
    z = mb.encode_songs(model, roll, chunk=chunk).transpose(0, 1).reshape(-1, 1152).double()
    mu = z.mean(0)
    cov = torch.cov(z.T)
    err_mu = rel_fro(pr.mean, mu)
    err_cov = rel_fro(pr.cov, cov)
    report(test="fit_latent_prior", bars=z.shape[0], mean_rel_fro=err_mu, cov_rel_fro=err_cov,
           mean_over_std=float(mu.abs().mean() / cov.diagonal().sqrt().mean()))
    assert pr.count == 36 and err_mu <= 1e-12 and err_cov <= 1e-12, (err_mu, err_cov)
    assert pr.encoder_digest == P.encoder_digest(model)


def test_packed_and_cell_inputs_give_the_same_moments(deterministic, tmp_path):
    P, packed = pkg("prior"), pkg("data.packed")
    model = _model()
    cells = _songs(2, 5, 12).view(-1, 96, 60)             # 40 bars
    bits = packed.pack_cells(cells.cpu()).reshape(40, packed.BAR_BYTES)
    np.save(str(tmp_path / "note_bits.npy"), bits)
    chunk = 24
    a = P.fit_latent_prior(model, [cells[:24].cpu().numpy(), cells[24:]], chunk=chunk)
    b = P.fit_latent_prior(model, P.bars_of_packed(str(tmp_path), chunk), chunk=chunk)
    c = P.fit_latent_prior(model, [torch.from_numpy(bits)], chunk=chunk)
    assert a.count == b.count == c.count == 40
    for other in (b, c):
        assert torch.equal(a.mean, other.mean) and torch.equal(a.cov, other.cov)


# ---- the draws ------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def test_identity_prior_draws_bf16_of_the_normal_draw():
    P = pkg("prior")
    pr = P.LatentPrior(np.zeros(1152), np.eye(1152), 2, 0.0, "x")
    z = pr.sample(8, 5, _gen(4))
    eps = torch.randn(8, 5, 1152, device="cuda", generator=_gen(4))
    assert z.dtype == torch.float32 and z.shape == (8, 5, 1152) and z.is_cuda
    assert torch.equal(z, eps.bfloat16().float())


def _spd_prior(seed, shrinkage=1e-3):
    P = pkg("prior")
    r = np.random.RandomState(seed)
    a = r.randn(1152, 64) * 20.0
    cov = a @ a.T / 64 + np.diag(r.rand(1152) * 50 + 10)
    return P.LatentPrior(500.0 + 30.0 * r.randn(1152), cov, 10 ** 6, shrinkage, "x")


def test_fitted_prior_draw_matches_float64():
    pr = _spd_prior(5)
    z = pr.sample(40, 64, _gen(6))
    eps = torch.randn(40, 64, 1152, device="cuda", generator=_gen(6))
    L = pr.cholesky().numpy()
    want = PO.draw(pr.mean.numpy(), L, eps.cpu().numpy())
    err = rel_fro(z, torch.from_numpy(want))
    err_c = rel_fro(z.double().cpu() - pr.mean, torch.from_numpy(want) - pr.mean)
    report(test="prior_draw", rel_fro=err, centred_rel_fro=err_c)
    assert err <= 6e-3 and err_c <= 6e-3, (err, err_c)


def test_many_draws_reproduce_mean_and_covariance():
    """2^17 draws.  Per component the sample mean has std sqrt(cov_jj / N): every component must lie within 6 of
    those.  The sample covariance's expected rel-Frobenius error is sqrt((tr cov)^2 + |cov|_F^2) / (sqrt(N) |cov|_F)
    (Wishart second moments); it must stay below 1.5 times that plus 1e-2 for the bf16 operands."""
    pr = _spd_prior(7)
    N = 1 << 17
    z = pr.sample(128, N // 128, _gen(8)).view(N, 1152).double()
    mu = pr.mean.cuda()
    cov = torch.as_tensor(pr.cov + pr.shrinkage * torch.trace(pr.cov) / 1152 * torch.eye(1152, dtype=torch.float64)).cuda()
    zc = z - mu
    mean_hat = zc.mean(0)
    cov_hat = (zc.T @ zc) / N - torch.outer(mean_hat, mean_hat)
    z_score = float((mean_hat.abs() / (cov.diagonal() / N).sqrt()).max())
    expect = float(torch.sqrt(torch.trace(cov) ** 2 + (cov * cov).sum()) / (N ** 0.5 * cov.norm()))
    err = rel_fro(cov_hat, cov)
    report(test="prior_draw_statistics", draws=N, mean_max_z=z_score, cov_rel_fro=err, cov_expected_rel_fro=expect)
    assert z_score < 6.0, z_score
    assert err < 1.5 * expect + 1e-2, (err, expect)


# ---- the script end to end ------------------------------------------------------------------------------------------
def test_main_fit_prior_then_sample(tmp_path, deterministic):
    mb, midi, P = pkg("maker_bar"), pkg("midi"), pkg("prior")
    O = __import__("barvae_oracle")
    os.makedirs(tmp_path / "model")
    for number, seed in ((10, 11), (12, 13)):
        sd = O.make_state_dict(O.generator_spec(), seed, "lively")
        torch.save({"generator_state_dict": {"module." + k: v for k, v in sd.items()}},
                   str(tmp_path / "model" / ("checkpoint_%d.pth.tar" % number)))
    model = _model()
    roll = _songs(1, 2, 14)[0].cpu().numpy()
    roll[-1, 30] = 1.0
    midi.write_midi(roll, str(tmp_path / "a.mid"))
    os.makedirs(tmp_path / "packed")
    more = _songs(1, 3, 15)[0].cpu()
    np.save(str(tmp_path / "packed" / "note_bits.npy"),
            pkg("data.packed").pack_cells(more).reshape(12, pkg("data.packed").BAR_BYTES))
    out = _run_main(tmp_path, ["--fit_prior", "prior.pt", "--data", "a.mid", "packed"])
    assert "latent prior: 20 bars" in out and "-> prior.pt" in out, out
    prior = P.load_latent_prior(str(tmp_path / "prior.pt"), model)
    want = P.fit_latent_prior(model, list(P.bars_of_midi([str(tmp_path / "a.mid")])) + [more.view(-1, 96, 60)])
    assert torch.equal(prior.mean, want.mean) and torch.equal(prior.cov, want.cov)
    for extra in ([], ["--sampler", "bernoulli", "--temperature", "0.9", "--primer", "a.mid", "--music_length", "3"]):
        out = _run_main(tmp_path, ["--latent_prior", "prior.pt", "--seed", "5", "--out", "s.mid", "--songs", "2"]
                        + (extra or ["--music_length", "2"]))
        length = 3 if extra else 2
        g = torch.Generator(device="cuda").manual_seed(5)
        lat = prior.sample(length * 4, 2, g)
        kw = dict(sampler="bernoulli", temperature=0.9, primer=torch.from_numpy(mb.load_primer(
            str(tmp_path / "a.mid"), 3)[0]).cuda()) if extra else {}
        songs = mb.songs_to_host(mb.sample_songs(model, lat, length, seed=5, **kw))
        for i, name in enumerate(("s.mid", "s_1.mid")):
            midi.write_midi(songs[i], str(tmp_path / "want.mid"))
            assert (tmp_path / name).read_bytes() == (tmp_path / "want.mid").read_bytes(), (extra, name)
    # a prior fitted to another checkpoint is refused
    import subprocess
    env = dict(os.environ, BVAE_DETERMINISTIC="1", PYTHONPATH=ROOT)
    code = "import importlib, sys; importlib.import_module(%r).main(sys.argv[1:])" % (pkg("maker_bar").__name__)
    r = subprocess.run([sys.executable, "-c", code, "--model_number", "12", "--latent_prior", "prior.pt"],
                       cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "refit" in r.stderr, r.stdout + r.stderr
