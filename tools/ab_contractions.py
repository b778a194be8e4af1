"""Bit-level A/B of the contraction kernels between two builds of libbarvae.so, and the record of which kernel each
parity case launches.

Every LAYERS / BIG_LAYERS case of tests/test_gpu_kernels.py runs through the same dispatch as its parity test (tcgen05;
the C_in = 1 stems through the automatic choice) on the same seeded inputs, and one JSON line per (case, output) is
written: the kernel name bvae_last_kernel() reports after the call, the number of launches the call made (2 for a
weight gradient = the packed-scratch reduction followed by wgrad_unpack_kernel) and a SHA-256 of the output bytes.
Outputs: fp32 forward, bf16 forward with the activation, fp32 data gradient, bf16 data gradient with addend and mask,
and the weight gradient twice -- with BVAE_DETERMINISTIC semantics (one split per tile: one ordered accumulation per
element, so bit-exact between builds) and in the default mode (pixel splits reduced with float atomics: its hash is
recorded but not compared; the line shows which reduction the default dispatch picks).  The C_in = 1 stems' weight
gradient (stem_wgrad_kernel) accumulates with float atomics in both modes, so it is not compared either.

    BVAE_LIB_PATH=/path/to/other/libbarvae.so python tools/ab_contractions.py --out a.jsonl
    python tools/ab_contractions.py --out b.jsonl
    python tools/ab_contractions.py --compare a.jsonl b.jsonl
"""
import argparse
import hashlib
import json
import os
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_sampling import card  # noqa: E402
from gpu_util import nhwc, pkg  # noqa: E402
from test_gpu_kernels import BF16, BIG_LAYERS, LAYERS, _bf  # noqa: E402


def sha(t):
    return hashlib.sha256(t.detach().contiguous().view(torch.uint8).cpu().numpy().tobytes()).hexdigest()


def run_case(spec, impl, B, emit):
    eng, lib = pkg("engine"), pkg("_lib")
    kind, cin, cout, k, s, p, op, H, W = spec
    torch.manual_seed(1)
    if kind == "conv":
        m = nn.Conv2d(cin, cout, k, s, p, bias=True).cuda()
    else:
        m = nn.ConvTranspose2d(cin, cout, k, s, p, output_padding=op, bias=True).cuda()
    with torch.no_grad():
        m.weight.copy_(_bf(torch.randn_like(m.weight) * 0.2))
        m.bias.copy_(_bf(torch.randn_like(m.bias)))
    g = pkg("graph.encodingBlock").gemm_of(m)
    OH, OW = g.out_hw(H, W)
    x = _bf(torch.randn(B, cin, H, W, device="cuda"))
    dyt = _bf(torch.randn(B, cout, OH, OW, device="cuda"))
    add = eng.Act(torch.randn(B, H, W, cin, device="cuda").to(BF16), B, H, W, cin)
    msk = eng.Act(torch.randn(B, H, W, cin, device="cuda").to(BF16), B, H, W, cin)
    xa = eng.Act(nhwc(x).to(BF16), B, H, W, cin)
    dya = eng.Act(nhwc(dyt).to(BF16), B, OH, OW, cout)

    def call(name, fn, out):
        torch.cuda.synchronize()
        n0 = lib.launch_count()
        fn()
        torch.cuda.synchronize()
        emit(name, lib.last_kernel(), lib.launch_count() - n0, out)

    def empty(N, H_, W_, C_, dtype):
        a = eng.Act.empty(N, H_, W_, C_, dtype=dtype)
        a.t.fill_(float("nan"))
        return a

    eng.set_impl({"tc": lib.IMPL_TC, "auto": lib.IMPL_AUTO}[impl])
    try:
        y = empty(B, OH, OW, cout, torch.float32)
        call("fwd_f32", lambda: g.forward(xa, y), y.t)
        y2 = empty(B, OH, OW, cout, BF16)
        call("fwd_bf16_act", lambda: g.forward(xa, y2, act=True, slope=0.01), y2.t)
        dx = empty(B, H, W, cin, torch.float32)
        call("dgrad_f32", lambda: g.dgrad(dya, dx), dx.t)
        dx2 = empty(B, H, W, cin, BF16)
        call("dgrad_bf16_add_mask", lambda: g.dgrad(dya, dx2, addend=add, mask=msk, mask_slope=0.01), dx2.t)
        for name, det in (("wgrad_deterministic", True), ("wgrad_default", False)):
            m.weight.grad = None
            lib.set_deterministic(det)
            try:
                call(name, lambda: g.wgrad(xa, dya), None)
            finally:
                lib.set_deterministic(False)
            emit.last["sha256"] = sha(m.weight.grad)
    finally:
        eng.set_impl(lib.IMPL_AUTO)


def record(out_path):
    lines = [dict(card(), lib=os.path.relpath(pkg("_lib").LIB_PATH, ROOT))]

    def emit(output, kernel, launches, t):
        exact = output != "wgrad_default" and not kernel.startswith("stem_wgrad")
        emit.last = dict(case=case, output=output, kernel=kernel, launches=launches, exact=exact)
        if t is not None:
            emit.last["sha256"] = sha(t)
        lines.append(emit.last)

    pkg("_lib").lib()
    for spec in LAYERS:
        case = "%s_%dto%d_k%dx%d_s%dx%d_%dx%d_B3" % (spec[0], spec[1], spec[2], *spec[3], *spec[4], spec[7], spec[8])
        run_case(spec, "auto" if spec[1] == 1 else "tc", 3, emit)
    for spec in BIG_LAYERS:
        case = "%s_%dto%d_k%dx%d_s%dx%d_%dx%d_B%d" % (spec[0], spec[1], spec[2], *spec[3], *spec[4], spec[7], spec[8], spec[9])
        run_case(spec[:9], "tc", spec[9], emit)
    with open(out_path, "w") as f:
        for l in lines:
            f.write(json.dumps(l) + "\n")
    print("%d outputs of %d cases -> %s" % (len(lines) - 1, len(LAYERS) + len(BIG_LAYERS), out_path))


def compare(a_path, b_path):
    """bit-identity of every exact output and the same kernel on every line; prints the differences"""
    a, b = ([json.loads(l) for l in open(p)][1:] for p in (a_path, b_path))
    key = lambda r: (r["case"], r["output"])
    bd = {key(r): r for r in b}
    bad = 0
    for r in a:
        o = bd.pop(key(r), None)
        if o is None or r["kernel"] != o["kernel"] or r["launches"] != o["launches"] or (r["exact"] and r["sha256"] != o["sha256"]):
            bad += 1
            print("DIFF", json.dumps(r), "|", json.dumps(o))
    bad += len(bd)
    for r in bd.values():
        print("ONLY IN", b_path, json.dumps(r))
    print("%d lines compared, %d exact outputs, %d differences" % (len(a), sum(r["exact"] for r in a), bad))
    return bad == 0


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="write the record of this build (BVAE_LIB_PATH picks the library)")
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"))
    args = ap.parse_args()
    if args.compare:
        sys.exit(0 if compare(*args.compare) else 1)
    record(args.out)
