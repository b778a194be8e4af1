"""CPU oracle for the per-bar score (csrc/sample.cu, bvae_bar_score)  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

For each bar of 5760 cells, with l = float32(logit * inv_temperature) and t = (target != 0):

    nll    = sum over cells of (t ? softplus(-l) : softplus(l)),   softplus(x) = max(x, 0) + log1p(exp(-|x|))
    counts = (#(p > threshold and t), #(p > threshold), #t),        p = sample_oracle.probs (float32)

``nll`` is summed in float64 (the device sums fp32 in a fixed order: parity within rtol 1e-5).  ``p`` is the float32
expression of the sampler's oracle, so counts are bit-exact wherever p is not within a few ulps of the threshold.
Only ``tests/`` imports this file.
"""
import numpy as np

import sample_oracle as SO

BAR_CELLS = SO.BAR_CELLS


def softplus(x):
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        return np.maximum(x, 0.0) + np.log1p(np.exp(-np.abs(x)))


def score(logits, target, inv_temperature, threshold):
    """logits, target: any shape of whole bars -> (nll [bars] float64, counts [bars, 3] int64, p [bars, 5760] float32)"""
    lg = np.asarray(logits, dtype=np.float32).reshape(-1, BAR_CELLS)
    t = np.asarray(target, dtype=np.float32).reshape(-1, BAR_CELLS) != 0
    l = (lg * np.float32(inv_temperature)).astype(np.float32)
    nll = np.where(t, softplus(-l.astype(np.float64)), softplus(l)).sum(axis=1)
    p = SO.probs(lg, inv_temperature)
    on = p > np.float32(threshold)
    counts = np.stack([(on & t).sum(1), on.sum(1), t.sum(1)], axis=1).astype(np.int64)
    return nll, counts, p
