"""float64 numpy restatement of the latent prior (csrc/prior.cu, musicgeneration_vae-torch_b200/prior.py).

moments_sequential: bvae_latent_moments' exact per-element order -- start from the given values, add the rows one at a
    time in increasing row order, each product formed in float64 (exact for fp32 inputs) -- so the kernel must match it
    bit for bit.  moments: the same sums through one float64 matrix product (BLAS order), for sizes where the
    sequential loop is slow.
finalize: mu = sum / n, cov = (gram_sym - n mu mu^T) / (n - 1), gram_sym the upper triangle mirrored.
cholesky_ridge: lower factor of cov + shrinkage * (trace(cov) / d) * I.
draw: mu + L eps."""
import numpy as np


def moments_sequential(z, sum0=None, gram0=None):
    """(sum [d], gram [d, d] upper triangle; lower triangle of gram0 passed through) in the kernel's order"""
    z = np.asarray(z, dtype=np.float32).astype(np.float64)
    n, d = z.shape
    s = np.zeros(d) if sum0 is None else np.array(sum0, dtype=np.float64)
    g = np.zeros((d, d)) if gram0 is None else np.array(gram0, dtype=np.float64)
    upper = np.triu(np.ones((d, d), dtype=bool))
    gu = g[upper]
    iu = np.nonzero(upper)
    for i in range(n):
        s += z[i]
        gu += z[i][iu[0]] * z[i][iu[1]]
    g[upper] = gu
    return s, g


def moments(z):
    """(sum [d], gram [d, d] upper triangle, zeros below) through one float64 product"""
    z = np.asarray(z, dtype=np.float32).astype(np.float64)
    return z.sum(0), np.triu(z.T @ z)


def finalize(s, gram_upper, n):
    g = np.triu(np.asarray(gram_upper, dtype=np.float64))
    g = g + np.triu(g, 1).T
    mu = np.asarray(s, dtype=np.float64) / n
    return mu, (g - n * np.outer(mu, mu)) / (n - 1)


def cholesky_ridge(cov, shrinkage):
    d = cov.shape[0]
    return np.linalg.cholesky(cov + shrinkage * np.trace(cov) / d * np.eye(d))


def draw(mu, L, eps):
    """eps [..., d] -> mu + L eps, float64"""
    return np.asarray(mu, dtype=np.float64) + np.asarray(eps, dtype=np.float64) @ np.asarray(L, dtype=np.float64).T
