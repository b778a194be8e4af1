"""Bit-packed piano-roll batches (SURVEY.md section 8f N3).

The reference keeps every bar as fp32 on disk, in the loader and across PCIe (data/bar_dataset.py:22-25,
agent/barGen.py:134-141,302-306): 138 KB per training sample.  Cells are binary, so this module stores one bit per
cell -- ``numpy.packbits`` order: cells in C order, MSB first -- which is 4320 bytes per sample (32x less) and
lossless.  ``PackedBatch`` is one contiguous (pinned) uint8 buffer

    [ note: B*720 B | pre_note: B*720 B | pre_phrase: B*2880 B ]        + position [B] int64

that crosses PCIe in ONE copy and is expanded on the device by ``bvae_unpack_bits`` (csrc/bits.cu) straight into the
bf16 tensors the encoder stems read (note and pre_note land contiguously = the 2B-bar encoder batch) plus the fp32
copy of ``note`` the BCE loss uses as its target.  The generated bars of the sampling loop take the reverse route
(``threshold_pack``: torch.gt(bar, 0.3) of maker_bar.py:39 and the packing in one kernel; 720 B per bar D2H).

Host-side packing is loader work (numpy); everything on the device goes through libbarvae.so -- no fallback.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib

BAR_CELLS = 96 * 60            # config.py: one bar = 96 time steps x 60 pitches
PHRASE_CELLS = 384 * 60        # 4 bars
BAR_BYTES = BAR_CELLS // 8     # 720
PHRASE_BYTES = PHRASE_CELLS // 8


def pack_cells(x) -> np.ndarray:
    """{0,1}-valued array (any shape / dtype, numpy or CPU tensor) -> uint8 bits, numpy.packbits order.
    Raises ValueError if a cell is neither 0 nor 1: the packing must stay lossless."""
    a = x.numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    flat = np.ascontiguousarray(a).reshape(-1)
    b = flat.astype(np.uint8)
    if not np.array_equal(b, flat) or (b.size and b.max() > 1):
        raise ValueError("pack_cells: piano-roll cells must be exactly 0 or 1")
    return np.packbits(b)


def unpack_cells_host(bits: np.ndarray, shape) -> np.ndarray:
    """host inverse of pack_cells (used on the D2H side of the sampling loop and by loaders); float32 {0,1}"""
    n = int(np.prod(shape))
    return np.unpackbits(np.asarray(bits, dtype=np.uint8), count=n).astype(np.float32).reshape(shape)


class PackedBatch:
    """One training batch as bits.  ``bits`` is a uint8 CPU tensor (pinned when ``pin``), ``position`` int64."""

    def __init__(self, bits: torch.Tensor, position: torch.Tensor, batch: int):
        if bits.dtype != torch.uint8 or bits.numel() != batch * (2 * BAR_BYTES + PHRASE_BYTES):
            raise ValueError("PackedBatch: bits must be uint8 with %d bytes per bar" % (2 * BAR_BYTES + PHRASE_BYTES))
        self.bits, self.position, self.batch = bits, position, batch

    @classmethod
    def from_arrays(cls, note, pre_note, pre_phrase, position, pin: bool = False) -> "PackedBatch":
        B = int(np.asarray(position).shape[0]) if not isinstance(position, torch.Tensor) else position.shape[0]
        for name, t, cells in (("note", note, BAR_CELLS), ("pre_note", pre_note, BAR_CELLS),
                               ("pre_phrase", pre_phrase, PHRASE_CELLS)):
            n = t.numel() if isinstance(t, torch.Tensor) else np.asarray(t).size
            if n != B * cells:
                raise ValueError("PackedBatch: %s has %d cells, expected %d x %d" % (name, n, B, cells))
        bits = torch.from_numpy(np.concatenate([pack_cells(note), pack_cells(pre_note), pack_cells(pre_phrase)]))
        pos = position if isinstance(position, torch.Tensor) else torch.from_numpy(np.asarray(position))
        pos = pos.to(torch.long)
        if pin:
            bits, pos = bits.pin_memory(), pos.pin_memory()
        return cls(bits, pos, B)

    def pin_memory(self) -> "PackedBatch":
        """DataLoader(pin_memory=True) calls this on the collated batch"""
        return PackedBatch(self.bits.pin_memory(), self.position.pin_memory(), self.batch)

    @property
    def nbytes(self) -> int:
        return self.bits.numel() + self.position.numel() * self.position.element_size()

    def to_host_arrays(self):
        """(note, pre_note, pre_phrase, position) as float32 numpy arrays in the reference's shapes"""
        B, b = self.batch, self.bits.numpy()
        o1, o2 = B * BAR_BYTES, 2 * B * BAR_BYTES
        return (unpack_cells_host(b[:o1], (B, 1, 96, 60)), unpack_cells_host(b[o1:o2], (B, 1, 96, 60)),
                unpack_cells_host(b[o2:], (B, 1, 384, 60)), self.position.numpy())

    def to_device(self, device, phrase_stream=None):
        """H2D copy of the bits + expansion on the device.  Returns ``(note_f32, bars_bf16, phrase_bf16, position,
        dbits)``: note_f32 [B,1,96,60] fp32 (BCE target), bars_bf16 [2B,1,96,60] bf16 (= cat(note, pre_note): the
        encoder batch), phrase_bf16 [B,1,384,60] bf16.  With ``phrase_stream`` the phrase bits are expanded on that
        stream (the one the phrase encoder runs on) after it has waited for the copy; the caller must then keep
        ``dbits`` referenced until the main stream has joined ``phrase_stream`` again (the trainer holds it through the
        step) -- cheaper for the caching allocator than record_stream (DESIGN.md section 4.5)."""
        B = self.batch
        main = torch.cuda.current_stream(device)
        dbits = self.bits.to(device, non_blocking=True)
        pos = self.position.to(device, non_blocking=True)
        bars = torch.empty(2 * B, 1, 96, 60, device=device, dtype=torch.bfloat16)
        note = torch.empty(B, 1, 96, 60, device=device, dtype=torch.float32)
        phrase = torch.empty(B, 1, 384, 60, device=device, dtype=torch.bfloat16)
        nbar_bits = 2 * B * BAR_CELLS
        unpack_bits(dbits[:2 * B * BAR_BYTES], nbar_bits, bars, note, B * BAR_CELLS)
        if phrase_stream is None:
            unpack_bits(dbits[2 * B * BAR_BYTES:], B * PHRASE_CELLS, phrase, None, 0)
        else:
            phrase_stream.wait_stream(main)
            with torch.cuda.stream(phrase_stream):
                unpack_bits(dbits[2 * B * BAR_BYTES:], B * PHRASE_CELLS, phrase, None, 0)
        return note, bars, phrase, pos, dbits


# ---------------------------------------------------------------------------------------------------------------
# on-disk format: one .npz per item like the reference's (data/bar_dataset.py:22-25), cells stored as bits
# ---------------------------------------------------------------------------------------------------------------
PACKED_KEYS = ("note_bits", "pre_note_bits", "pre_phrase_bits", "position")


def pack_item(item) -> dict:
    """reference item ``{'note' [n,1,96,60], 'pre_note', 'pre_phrase' [n,1,384,60], 'position' [n]}`` -> packed item
    ``{'note_bits' [n,720] u8, 'pre_note_bits' [n,720] u8, 'pre_phrase_bits' [n,2880] u8, 'position' [n] i64}``.
    A bar is 5760 cells = 720 whole bytes, so rows stay per-bar and items concatenate along axis 0 like the
    reference's collate (agent/barGen.py:134-141) without touching a bit."""
    n = int(np.asarray(item["position"]).shape[0])
    return {"note_bits": pack_cells(item["note"]).reshape(n, BAR_BYTES),
            "pre_note_bits": pack_cells(item["pre_note"]).reshape(n, BAR_BYTES),
            "pre_phrase_bits": pack_cells(item["pre_phrase"]).reshape(n, PHRASE_BYTES),
            "position": np.asarray(item["position"]).astype(np.int64)}


def unpack_item(packed) -> dict:
    """inverse of pack_item (float32 arrays in the reference's shapes)"""
    n = packed["position"].shape[0]
    return {"note": unpack_cells_host(packed["note_bits"], (n, 1, 96, 60)),
            "pre_note": unpack_cells_host(packed["pre_note_bits"], (n, 1, 96, 60)),
            "pre_phrase": unpack_cells_host(packed["pre_phrase_bits"], (n, 1, 384, 60)),
            "position": np.asarray(packed["position"])}


def collate_packed(samples, pin: bool = False) -> PackedBatch:
    """DataLoader collate_fn for packed items: three byte-level concatenations written straight into the batch buffer"""
    B = sum(int(s["position"].shape[0]) for s in samples)
    bits = torch.empty(B * (2 * BAR_BYTES + PHRASE_BYTES), dtype=torch.uint8, pin_memory=pin)
    buf, off = bits.numpy(), 0
    for key, width in (("note_bits", BAR_BYTES), ("pre_note_bits", BAR_BYTES), ("pre_phrase_bits", PHRASE_BYTES)):
        for s in samples:
            a = np.asarray(s[key], dtype=np.uint8).reshape(-1)
            if a.size != int(s["position"].shape[0]) * width:
                raise ValueError("collate_packed: %s has %d bytes, expected %d per bar" % (key, a.size, width))
            buf[off:off + a.size] = a
            off += a.size
    pos = torch.from_numpy(np.concatenate([np.asarray(s["position"]).astype(np.int64) for s in samples]))
    return PackedBatch(bits, pos.pin_memory() if pin else pos, B)


class PackedNoteDataset(torch.utils.data.Dataset):
    """Directory of packed .npz items (written by ``convert_dataset`` / tools/pack_dataset.py): same item granularity
    and file names as the reference's NoteDataset (data/bar_dataset.py:9-25), 32x fewer bytes to read and collate."""

    def __init__(self, root_dir, config):
        import os
        self.dir = os.path.join(root_dir, getattr(config, "packed_data_path", config.data_path))
        self.file_list = sorted(f for f in os.listdir(self.dir) if f.endswith(".npz"))
        self.num_iterations = (len(self.file_list) + config.batch_size - 1) // config.batch_size

    def __len__(self):
        return len(self.file_list)

    def __getitem__(self, idx):
        import os
        with np.load(os.path.join(self.dir, self.file_list[idx])) as d:
            return {k: d[k] for k in PACKED_KEYS}


def convert_dataset(src_dir: str, dst_dir: str) -> int:
    """reference-format directory of .npz items -> packed directory (same file names); returns the number of bars"""
    import os
    os.makedirs(dst_dir, exist_ok=True)
    bars = 0
    for name in sorted(os.listdir(src_dir)):
        if not name.endswith(".npz"):
            continue
        with np.load(os.path.join(src_dir, name)) as d:
            item = pack_item({k: d[k] for k in ("note", "pre_note", "pre_phrase", "position")})
        np.savez(os.path.join(dst_dir, name), **item)
        bars += int(item["position"].shape[0])
    return bars


def convert_dataset_to_arrays(src_dir: str, dst_dir: str) -> int:
    """reference-format directory -> THREE flat arrays for memory-mapped loading: ``note_bits.npy [N,720]``,
    ``pre_note_bits.npy [N,720]``, ``pre_phrase_bits.npy [N,2880]`` (uint8) and ``position.npy [N]`` (int64), bars in
    file-name order.  4328 bytes per bar; a 1 M-bar corpus is 4.3 GB instead of 138 GB of fp32."""
    import os
    os.makedirs(dst_dir, exist_ok=True)
    parts = {k: [] for k in PACKED_KEYS}
    for name in sorted(os.listdir(src_dir)):
        if name.endswith(".npz"):
            with np.load(os.path.join(src_dir, name)) as d:
                item = d if "note_bits" in d.files else pack_item({k: d[k] for k in ("note", "pre_note", "pre_phrase",
                                                                                     "position")})
                for k in PACKED_KEYS:
                    parts[k].append(np.asarray(item[k]))
    for k in PACKED_KEYS:
        np.save(os.path.join(dst_dir, k + ".npy"), np.concatenate(parts[k], axis=0))
    return int(sum(p.shape[0] for p in parts["position"]))


class PackedMemmapDataset(torch.utils.data.Dataset):
    """Bars of ``convert_dataset_to_arrays`` memory-mapped from disk.  Indexing with an int gives one packed one-bar
    item (collate_packed-compatible); ``batch(indices)`` gathers a whole PackedBatch with three fancy-index reads -- no
    per-file open, no per-item Python work -- which is what keeps ONE loader process far ahead of a GPU."""

    def __init__(self, directory: str):
        import os
        self.arrays = {k: np.load(os.path.join(directory, k + ".npy"), mmap_mode="r") for k in PACKED_KEYS}
        n = self.arrays["position"].shape[0]
        if not (self.arrays["note_bits"].shape == (n, BAR_BYTES) and self.arrays["pre_note_bits"].shape == (n, BAR_BYTES)
                and self.arrays["pre_phrase_bits"].shape == (n, PHRASE_BYTES)):
            raise ValueError("PackedMemmapDataset: array shapes do not describe %d packed bars" % n)

    def __len__(self):
        return self.arrays["position"].shape[0]

    def __getitem__(self, idx):
        return {k: np.asarray(self.arrays[k][idx:idx + 1]) for k in PACKED_KEYS}

    def batch(self, indices, pin: bool = False) -> PackedBatch:
        idx = np.asarray(indices, dtype=np.int64)
        B = idx.shape[0]
        contiguous = B > 0 and bool(np.all(np.diff(idx) == 1))
        sel = slice(int(idx[0]), int(idx[0]) + B) if contiguous else np.sort(idx)      # sorted: one forward pass over the map
        order = None if contiguous else np.argsort(np.argsort(idx))                    # ... then back to the caller's order
        bits = torch.empty(B * (2 * BAR_BYTES + PHRASE_BYTES), dtype=torch.uint8, pin_memory=pin)
        buf, off = bits.numpy(), 0
        for key, width in (("note_bits", BAR_BYTES), ("pre_note_bits", BAR_BYTES), ("pre_phrase_bits", PHRASE_BYTES)):
            a = np.asarray(self.arrays[key][sel])
            if order is not None:
                a = a[order]
            buf[off:off + B * width] = a.reshape(-1)
            off += B * width
        pos = np.asarray(self.arrays["position"][sel])
        pos = torch.from_numpy(np.ascontiguousarray(pos if order is None else pos[order]).astype(np.int64))
        return PackedBatch(bits, pos.pin_memory() if pin else pos, B)

    def batches(self, batch_size: int, shuffle: bool = False, seed: int = 0, rank: int = 0, world: int = 1,
                pin: bool = False, drop_last: bool = False):
        """iterate PackedBatch; each rank takes a disjoint contiguous shard of the (optionally shuffled) bar order --
        the DistributedSampler semantics of agent/barGen_horovod.py:49-50"""
        n = len(self)
        order = np.random.RandomState(seed).permutation(n) if shuffle else np.arange(n)
        # every rank gets the same number of bars (hence of batches and of gradient all-reduces per epoch): the order is
        # padded by wrapping around, as torch's DistributedSampler does (parallel.shard_indices)
        per = (n + world - 1) // world if not drop_last else n // world
        if n > 0 and per * world > n:
            order = np.concatenate([order, order[np.arange(per * world - n) % n]])
        mine = order[rank * per:(rank + 1) * per]
        for i in range(0, len(mine), batch_size):
            idx = mine[i:i + batch_size]
            if drop_last and len(idx) < batch_size:
                break
            yield self.batch(idx, pin)


def unpack_bits(bits: torch.Tensor, nbits: int, out_bf16, out_f32, nbits_f32: int):
    """bvae_unpack_bits on the current stream (device tensors; outputs may be None)"""
    if not bits.is_cuda:
        raise RuntimeError("unpack_bits runs on the device (libbarvae.so); use unpack_cells_host for host arrays")
    assert bits.dtype == torch.uint8 and bits.is_contiguous() and bits.numel() * 8 >= nbits
    assert out_bf16 is None or (out_bf16.dtype == torch.bfloat16 and out_bf16.is_contiguous()
                                and out_bf16.numel() >= nbits)
    assert out_f32 is None or (out_f32.dtype == torch.float32 and out_f32.is_contiguous()
                               and out_f32.numel() >= nbits_f32)
    _lib.check(_lib.lib().bvae_unpack_bits(bits.data_ptr(), nbits, None if out_bf16 is None else out_bf16.data_ptr(),
                                           None if out_f32 is None else out_f32.data_ptr(), nbits_f32,
                                           _lib.stream_ptr()), "unpack_bits")


def threshold_pack(probs: torch.Tensor, threshold: float, want_bits: bool = True, want_float: bool = False):
    """bvae_threshold_pack: ``(bits uint8 [ceil(n/8)] | None, (probs > threshold).float() | None)``"""
    if not probs.is_cuda:
        raise RuntimeError("threshold_pack runs on the device (libbarvae.so); there is no CPU fallback")
    p = probs.contiguous().float()
    n = p.numel()
    bits = torch.empty((n + 7) // 8, device=p.device, dtype=torch.uint8) if want_bits else None
    out = torch.empty_like(p) if want_float else None
    _lib.check(_lib.lib().bvae_threshold_pack(p.data_ptr(), n, float(threshold),
                                              None if bits is None else bits.data_ptr(),
                                              None if out is None else out.data_ptr(), _lib.stream_ptr()),
               "threshold_pack")
    return bits, out


def bernoulli_sample(logits: torch.Tensor, temperature: float, seed: int, song_base: int, bar_index: int,
                     out: torch.Tensor = None) -> torch.Tensor:
    """bvae_bernoulli_sample: draw every cell of ``logits`` (contiguous CUDA fp32, rows of 5760 cells = one bar of song
    ``song_base + row``) as Bernoulli(sigmoid(logit / temperature)) from the counter-based stream of
    (seed, song, bar_index, cell).  Returns {0,1} fp32 of the same shape (``out`` if given)."""
    if not logits.is_cuda:
        raise RuntimeError("bernoulli_sample runs on the device (libbarvae.so); there is no CPU fallback")
    if logits.dtype != torch.float32 or not logits.is_contiguous() or logits.numel() % BAR_CELLS:
        raise ValueError("bernoulli_sample: logits must be a contiguous fp32 tensor of whole %d-cell bars" % BAR_CELLS)
    if not 0 <= int(seed) < 2 ** 64:
        raise ValueError("bernoulli_sample: seed must fit in 64 unsigned bits")
    t = float(temperature)
    inv_t = 1.0 / t if t > 0 else float("nan")      # the library rejects a non-finite / non-positive inverse
    if out is None:
        out = torch.empty_like(logits)
    elif out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != logits.numel() or not out.is_cuda:
        raise ValueError("bernoulli_sample: out must be a contiguous CUDA fp32 tensor like logits")
    _lib.check(_lib.lib().bvae_bernoulli_sample(logits.data_ptr(), logits.numel() // BAR_CELLS, inv_t, int(seed),
                                                int(song_base), int(bar_index), out.data_ptr(), _lib.stream_ptr()),
               "bernoulli_sample")
    return out


def score_bars(logits: torch.Tensor, target: torch.Tensor, temperature: float = 1.0, threshold: float = 0.3):
    """bvae_bar_score: the per-bar score of the {0,1} roll ``target`` under Bernoulli(sigmoid(logit / temperature)), the
    distribution ``bernoulli_sample`` draws from.  Both are contiguous CUDA fp32 tensors of the same number of whole
    5760-cell bars.  Returns ``(nll [N] fp32, counts [N, 3] int32)``: the negative log-likelihood of each bar in nats
    (binary_cross_entropy_with_logits with reduction='sum'), and per bar the cells with p > ``threshold`` that are on in
    the target, the cells with p > ``threshold``, and the cells on in the target."""
    if not (logits.is_cuda and target.is_cuda):
        raise RuntimeError("score_bars runs on the device (libbarvae.so); there is no CPU fallback")
    for name, t in (("logits", logits), ("target", target)):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() % BAR_CELLS:
            raise ValueError("score_bars: %s must be a contiguous fp32 tensor of whole %d-cell bars" % (name, BAR_CELLS))
    if target.numel() != logits.numel():
        raise ValueError("score_bars: logits and target must hold the same number of bars")
    t = float(temperature)
    inv_t = 1.0 / t if t > 0 else float("nan")      # the library rejects a non-finite / non-positive inverse
    bars = logits.numel() // BAR_CELLS
    nll = torch.empty(bars, dtype=torch.float32, device=logits.device)
    counts = torch.empty(bars, 3, dtype=torch.int32, device=logits.device)
    _lib.check(_lib.lib().bvae_bar_score(logits.data_ptr(), target.data_ptr(), bars, inv_t, float(threshold),
                                         nll.data_ptr(), counts.data_ptr(), _lib.stream_ptr()), "score_bars")
    return nll, counts
