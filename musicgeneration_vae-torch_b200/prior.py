"""A Gaussian prior fitted to the latents the bar encoder actually produces, to sample songs from.

``maker_bar.main`` and ``BarGen.generate`` draw every bar latent from N(0, I).  Nothing pulls the latents of a model
trained on BCE alone toward that distribution (under the reference initialisation z is about -520 +- 30 per component,
SURVEY.md section 0), so the decoder is then fed latents unlike any it saw in training.  The remedy for deterministic
and adversarial autoencoders (Ghosh et al., "From Variational to Deterministic Autoencoders", ICLR 2020) is to fit a
density to the encoded training data after training and sample from it; this module fits a full-covariance Gaussian.

The moments of millions of 1152-wide latents are accumulated on the device in fp64 by ``bvae_latent_moments``
(csrc/prior.cu) with a fixed per-element summation order, so the fit does not depend on how the bars are batched.  The
latents are far from centred (mean / std ~ 17), so ``gram / n - mu mu^T`` cancels about 8 bits; fp64 keeps more than
40 of the rest.  The mean and covariance are finalised on the host in float64.

With ``Model(vae_head=True)`` the encoder returns posterior means, so the fit is a fit of those means; N(0, I) is that
head's designed prior, and either can be sampled."""
from __future__ import annotations

import hashlib
import os

import numpy as np
import torch

from . import _lib

LATENT = 1152
FORMAT = "barvae-latent-prior-v1"


def latent_moments(z: torch.Tensor, sum: torch.Tensor, gram: torch.Tensor) -> None:
    """bvae_latent_moments: ``sum[j] += sum_i z[i][j]`` and ``gram[j][k] += sum_i z[i][j] z[i][k]`` for k >= j, in fp64
    and in increasing row order, on the current stream.  ``z`` [n, d] CUDA fp32 with unit column stride (its row stride
    is the library's ``ld``), ``sum`` [d] and ``gram`` [d, d] contiguous CUDA float64 on the same device.  The lower
    triangle of ``gram`` is neither read nor written."""
    if not (z.is_cuda and sum.is_cuda and gram.is_cuda):
        raise RuntimeError("latent_moments runs on the device (libbarvae.so); there is no CPU fallback")
    if not (z.device == sum.device == gram.device):
        raise ValueError("latent_moments: z, sum and gram must be on the same device")
    if z.dtype != torch.float32 or z.dim() != 2 or (z.shape[0] > 1 and z.stride(1) != 1):
        raise ValueError("latent_moments: z must be a 2-D fp32 tensor with contiguous rows")
    n, d = z.shape
    if sum.dtype != torch.float64 or not sum.is_contiguous() or tuple(sum.shape) != (d,):
        raise ValueError("latent_moments: sum must be a contiguous float64 tensor of shape [%d]" % d)
    if gram.dtype != torch.float64 or not gram.is_contiguous() or tuple(gram.shape) != (d, d):
        raise ValueError("latent_moments: gram must be a contiguous float64 tensor of shape [%d, %d]" % (d, d))
    ld = z.stride(0) if n > 1 else d
    _lib.check(_lib.lib().bvae_latent_moments(z.data_ptr(), n, d, ld, sum.data_ptr(), gram.data_ptr(),
                                              _lib.stream_ptr()), "latent_moments")


def finalize_moments(sum, gram, count):
    """``(mean [d], cov [d, d])`` float64 numpy from the accumulated moments: ``mu = sum / n``,
    ``cov = (gram_sym - n mu mu^T) / (n - 1)`` with ``gram_sym`` the upper triangle of ``gram`` mirrored.  Raises
    ValueError on n < 2, on non-finite moments and on a zero trace (a dataset of identical bars, e.g. all silent)."""
    n = int(count)
    if n < 2:
        raise ValueError("latent prior: need at least 2 bars to fit a covariance (got %d)" % n)
    s = np.asarray(sum, dtype=np.float64)
    g = np.triu(np.asarray(gram, dtype=np.float64))
    if not (np.isfinite(s).all() and np.isfinite(g).all()):
        raise ValueError("latent prior: the latent moments are not finite (the encoder produced inf or NaN)")
    g = g + np.triu(g, 1).T
    mu = s / n
    cov = (g - n * np.outer(mu, mu)) / (n - 1)
    if not np.isfinite(cov).all():
        raise ValueError("latent prior: the covariance is not finite")
    if not np.trace(cov) > 0:
        raise ValueError("latent prior: the covariance has zero trace: all %d bars encode to the same latent "
                         "(for example, a dataset of silent bars)" % n)
    return mu, cov


class LatentPrior:
    """N(``mean``, ``cov``) over one bar's latent, fitted to ``count`` encoded bars of the checkpoint whose bar encoder
    hashes to ``encoder_digest``.  ``mean`` [1152] and ``cov`` [1152, 1152] are float64 CPU tensors.  Draws use
    ``cov + shrinkage * (trace(cov) / d) * I``: the ridge makes rank-deficient fits (fewer bars than 1152) usable."""

    def __init__(self, mean, cov, count, shrinkage, encoder_digest):
        self.mean = torch.as_tensor(mean, dtype=torch.float64).cpu()
        self.cov = torch.as_tensor(cov, dtype=torch.float64).cpu()
        d = self.mean.shape[0]
        if self.mean.dim() != 1 or tuple(self.cov.shape) != (d, d):
            raise ValueError("LatentPrior: mean must be [d] and cov [d, d]")
        if not (float(shrinkage) >= 0 and np.isfinite(float(shrinkage))):
            raise ValueError("LatentPrior: shrinkage must be finite and >= 0 (got %r)" % (shrinkage,))
        self.count, self.shrinkage, self.encoder_digest = int(count), float(shrinkage), str(encoder_digest)
        self._chol = None
        self._linear = {}

    @property
    def dim(self) -> int:
        return self.mean.shape[0]

    def cholesky(self) -> torch.Tensor:
        """Lower Cholesky factor of ``cov + shrinkage * (trace(cov) / d) * I``, float64 on the host (cached)."""
        if self._chol is None:
            d = self.dim
            ridge = self.shrinkage * float(torch.trace(self.cov)) / d
            L, info = torch.linalg.cholesky_ex(self.cov + ridge * torch.eye(d, dtype=torch.float64))
            if int(info) != 0 or not bool(torch.isfinite(L).all()):
                raise ValueError("latent prior: the covariance is not positive definite with shrinkage=%g (the "
                                 "factorisation failed at column %d); refit with a larger shrinkage"
                                 % (self.shrinkage, int(info)))
            self._chol = L
        return self._chol

    def _gemm(self, device):
        """``nn.Linear(d, d)`` holding ``L`` and ``mean`` on ``device``: z = mean + L eps through the library's Linear
        path (``graph.encodingBlock.gemm_of``), the call the encoder's last layer makes."""
        lin = self._linear.get(device)
        if lin is None:
            lin = torch.nn.utils.skip_init(torch.nn.Linear, self.dim, self.dim, device=device)   # no RNG draw
            with torch.no_grad():
                lin.weight.copy_(self.cholesky().to(torch.float32))
                lin.bias.copy_(self.mean.to(torch.float32))
            lin.requires_grad_(False)
            self._linear[device] = lin
        return lin

    @torch.no_grad()
    def sample(self, bars: int, songs: int, generator: torch.Generator) -> torch.Tensor:
        """``[bars, songs, d]`` fp32 latents on the generator's device, the layout of ``sample_songs(latents=...)``:
        ``eps = torch.randn(bars, songs, d, generator=generator)`` -- drawn exactly as ``maker_bar.main`` draws N(0, I)
        latents -- then ``z = mean + L eps`` with bf16 operands, fp32 accumulation and ``mean`` added in fp32 in the
        epilogue."""
        from .engine import Act
        from .graph.encodingBlock import gemm_of
        dev = generator.device
        if dev.type != "cuda":
            raise RuntimeError("LatentPrior.sample runs on the device (libbarvae.so): pass a CUDA generator")
        d = self.dim
        eps = torch.randn(bars, songs, d, device=dev, generator=generator)
        N = bars * songs
        z = torch.empty(bars, songs, d, device=dev)
        if N:
            x = Act(eps.view(N, 1, 1, d).to(torch.bfloat16), N, 1, 1, d)
            gemm_of(self._gemm(dev)).forward(x, Act(z.view(N, 1, 1, d), N, 1, 1, d))
        return z

    def state(self) -> dict:
        return {"format": FORMAT, "mean": self.mean, "cov": self.cov, "count": self.count,
                "shrinkage": self.shrinkage, "encoder_digest": self.encoder_digest}


def encoder_digest(model) -> str:
    """SHA-256 over the bar encoder's ``state_dict`` tensors in key order: name, dtype, shape and bytes of each"""
    h = hashlib.sha256()
    for name, t in sorted(model.encoder.state_dict().items()):
        t = t.detach().cpu().contiguous().reshape(-1)
        h.update(("%s|%s|%s|" % (name, str(t.dtype), tuple(t.shape))).encode())
        h.update(t.view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


def save_latent_prior(prior: LatentPrior, path) -> None:
    torch.save(prior.state(), path)


def load_latent_prior(path, model) -> LatentPrior:
    """Read a prior written by ``save_latent_prior`` for use with ``model``.  Raises ValueError when the file is not a
    latent prior or was fitted to another checkpoint's encoder: its latents are then not the ones the prior describes."""
    st = torch.load(path, map_location="cpu", weights_only=True)
    if not isinstance(st, dict) or st.get("format") != FORMAT:
        raise ValueError("%s is not a latent prior (expected format %r)" % (path, FORMAT))
    prior = LatentPrior(st["mean"], st["cov"], st["count"], st["shrinkage"], st["encoder_digest"])
    if prior.encoder_digest != encoder_digest(model):
        raise ValueError("%s was fitted to a different checkpoint's encoder: refit it for this checkpoint "
                         "(maker_bar --fit_prior OUT.pt --data ...)" % (path,))
    return prior


# ---- bars to fit on ----------------------------------------------------------------------------------------------------
def bars_of_midi(paths):
    """Each file's whole phrases as ``[4P, 96, 60]`` float32 {0,1} bars (``maker_bar.load_roll``).  A file that covers no
    whole phrase raises ValueError."""
    from .maker_bar import PHRASE_STEPS, load_roll
    for path in paths:
        roll, P, _ = load_roll(path)
        if P == 0:
            raise ValueError("%s covers no whole %d-step phrase" % (path, PHRASE_STEPS))
        yield roll.reshape(4 * P, 96, 60)


def bars_of_packed(directory, chunk=8192):
    """Slices of at most ``chunk`` bars of a packed-array directory's ``note_bits.npy`` (``tools/pack_dataset.py``
    output): uint8 ``[n, 720]`` rows, 720 B per bar, read from the memory map without the phrase arrays."""
    from .data.packed import BAR_BYTES
    bits = np.load(os.path.join(directory, "note_bits.npy"), mmap_mode="r")
    if bits.dtype != np.uint8 or bits.ndim != 2 or bits.shape[1] != BAR_BYTES:
        raise ValueError("%s: note_bits.npy must be uint8 [n, %d], got %s %r" % (directory, BAR_BYTES, bits.dtype,
                                                                                bits.shape))
    chunk = int(chunk)
    if chunk < 1:
        raise ValueError("chunk must be >= 1 (got %r)" % (chunk,))
    for i in range(0, bits.shape[0], chunk):
        yield np.array(bits[i:i + chunk])               # a writable host copy of the slice


def _is_bit_rows(batch) -> bool:
    from .data.packed import BAR_BYTES
    return (getattr(batch, "dtype", None) in (np.uint8, torch.uint8) and getattr(batch, "ndim", 0) == 2
            and batch.shape[1] == BAR_BYTES)


@torch.no_grad()
def fit_latent_prior(model, bars, chunk=8192, shrinkage=1e-3) -> LatentPrior:
    """Fit N(mean, cov) to ``model.encoder``'s latents of ``bars``, an iterable of batches, each either {0,1} cells
    ``[n, 96, 60]`` (any dtype, host or device) or packed bit rows uint8 ``[n, 720]`` in ``numpy.packbits`` order (as
    ``note_bits.npy`` stores them).  Bit rows cross PCIe as bits and are expanded on the device straight into the bf16
    input of ``Encoder.encode``.  Each batch is encoded in passes of at most ``chunk`` bars and each pass's latents are
    added to fp64 moments on the device (``latent_moments``); the moments do not depend on how the bars are batched,
    the latents do only through the pass sizes.  ``shrinkage`` is stored for the draws (``LatentPrior.cholesky``).
    With ``Model(vae_head=True)`` this fits the posterior means."""
    from .data.packed import BAR_CELLS, unpack_bits
    from .maker_bar import _check_chunk, _encode_all
    chunk = _check_chunk(chunk)
    dev = next(model.parameters()).device
    enc = model.encoder
    was_training = model.training
    model.eval()
    s = torch.zeros(LATENT, dtype=torch.float64, device=dev)
    g = torch.zeros(LATENT, LATENT, dtype=torch.float64, device=dev)
    n = 0
    try:
        for batch in bars:
            if _is_bit_rows(batch):
                rows = torch.as_tensor(np.asarray(batch) if isinstance(batch, np.ndarray) else batch)
                for i in range(0, rows.shape[0], chunk):
                    part = rows[i:i + chunk]
                    k = part.shape[0]
                    x = torch.empty(k, 1, 96, 60, dtype=torch.bfloat16, device=dev)
                    unpack_bits(part.to(dev).contiguous(), k * BAR_CELLS, x, None, 0)
                    latent_moments(enc.encode(x), s, g)
                    n += k
                continue
            cells = torch.as_tensor(batch)
            if cells.dim() != 3 or tuple(cells.shape[1:]) != (96, 60):
                raise ValueError("fit_latent_prior: a batch must be {0,1} cells [n, 96, 60] or bit rows uint8 [n, 720], "
                                 "got %s %r" % (cells.dtype, tuple(cells.shape)))
            for i in range(0, cells.shape[0], chunk):
                part = cells[i:i + chunk].to(dev)
                if not bool(((part == 0) | (part == 1)).all()):
                    raise ValueError("fit_latent_prior: cells must be exactly 0 or 1")
                latent_moments(_encode_all(enc, part, chunk), s, g)
                n += part.shape[0]
    finally:
        model.train(was_training)
    mean, cov = finalize_moments(s.cpu().numpy(), g.cpu().numpy(), n)
    return LatentPrior(mean, cov, n, shrinkage, encoder_digest(model))
