"""CPU oracle for the Bernoulli sampler (csrc/sample.cu)  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Restates Philox4x32-10 (Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC'11; the
Random123 constants) in vectorised numpy -- 32x32 -> 64-bit products in uint64 -- and the sampler's stream layout:

    r = word (i % 4) of Philox4x32-10(counter = {i // 4, bar_index, song lo32, song hi32}, key = {seed lo32, hi32})
    u = float32((r >> 8) * 2^-24)                    (exact: 24 significant bits)
    p = 1 / (1 + exp(-(logit * inv_temperature)))    (float32)
    cell = u < p

for cell i (0..5759, C order of [96][60]) of bar ``bar_index`` of song ``song``.  Parity bar: ``u`` bit-exact; cells
bit-exact wherever ``|u - p|`` is not within a few ulps of ``p`` (numpy's float32 exp and the device's expf may differ
in the last bit).  Pinning: the Random123 known-answer vectors, checked in tests/test_sampling_cpu.py.  Only
``tests/`` imports this file.
"""
import numpy as np

BAR_CELLS = 96 * 60
M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
MASK = np.uint64(0xFFFFFFFF)
S32 = np.uint64(32)


def philox4x32_10(counter, key):
    """counter: 4 arrays (or ints) of uint32 words, key: 2; broadcast together.  Returns 4 uint32 arrays."""
    c = [np.asarray(w, dtype=np.uint64) & MASK for w in counter]
    k0, k1 = (np.asarray(w, dtype=np.uint64) & MASK for w in key)
    for r in range(10):
        p0 = M0 * c[0]                              # < 2^64: no wrap-around
        p1 = M1 * c[2]
        c = [((p1 >> S32) ^ c[1] ^ k0) & MASK, p1 & MASK, ((p0 >> S32) ^ c[3] ^ k1) & MASK, p0 & MASK]
        if r < 9:
            k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
    return [w.astype(np.uint32) for w in c]


def uniforms(seed: int, songs, bar_index: int) -> np.ndarray:
    """float32 u [len(songs), 5760] for bar ``bar_index`` of each song id in ``songs``"""
    song = np.asarray(songs, dtype=np.uint64).reshape(-1, 1)
    i = np.arange(BAR_CELLS, dtype=np.uint64).reshape(1, -1)
    seed = int(seed)
    words = philox4x32_10((i // np.uint64(4), int(bar_index) & 0xFFFFFFFF, song & MASK, song >> S32),
                          (seed & 0xFFFFFFFF, seed >> 32))
    w = np.stack(np.broadcast_arrays(*words), axis=0)                  # [4, songs, 5760]
    cells = np.arange(BAR_CELLS)
    r = w[cells % 4, :, cells].T                                        # word i % 4 of cell i
    return ((r >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)


def probs(logits, inv_temperature) -> np.ndarray:
    x = np.asarray(logits, dtype=np.float32) * np.float32(inv_temperature)
    with np.errstate(over="ignore"):
        return (np.float32(1) / (np.float32(1) + np.exp(-x))).astype(np.float32)


def sample(logits, inv_temperature, seed: int, song_base: int, bar_index: int):
    """logits [bars, 5760] (any shape with whole bars) -> (u [bars, 5760], p [bars, 5760], cells {0,1} float32)"""
    lg = np.asarray(logits, dtype=np.float32).reshape(-1, BAR_CELLS)
    u = uniforms(seed, np.arange(lg.shape[0], dtype=np.int64) + int(song_base), bar_index)
    p = probs(lg, inv_temperature)
    return u, p, (u < p).astype(np.float32)
