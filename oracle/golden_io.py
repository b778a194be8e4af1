"""Golden dicts stored as shards: consecutive top-level entries of one dict, each shard one ``torch.save`` file of at most
SHARD_BYTES, so that no committed vector file grows past 1 MB.  ``load_golden`` merges the shards back into the dict the
generator built."""
import glob
import io
import os

import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
SHARD_BYTES = 900_000


def _shards(name):
    paths = glob.glob(os.path.join(GOLDEN_DIR, glob.escape(name) + ".*.pt"))
    return sorted(paths, key=lambda p: int(os.path.basename(p)[len(name) + 1:-3]))


def _nbytes(obj):
    buf = io.BytesIO()
    torch.save(obj, buf)
    return buf.tell()


def save_golden(obj, name):
    """write ``obj`` (a dict) as tests/golden/<name>.<i>.pt; one top-level entry larger than a shard is an error"""
    for p in _shards(name):
        os.remove(p)
    shards, cur, size = [], {}, 0
    for k, v in obj.items():
        n = _nbytes({k: v})
        if n > SHARD_BYTES:
            raise ValueError("golden entry %r is %d bytes; split it into smaller top-level entries" % (k, n))
        if cur and size + n > SHARD_BYTES:
            shards.append(cur)
            cur, size = {}, 0
        cur[k] = v
        size += n
    shards.append(cur)
    for i, s in enumerate(shards):
        torch.save(s, os.path.join(GOLDEN_DIR, "%s.%d.pt" % (name, i)))


def load_golden(name):
    paths = _shards(name)
    if not paths:
        raise FileNotFoundError("no golden shards %s.*.pt under %s" % (name, GOLDEN_DIR))
    out = {}
    for p in paths:
        out.update(torch.load(p, map_location="cpu", weights_only=False))
    return out
