"""ctypes binding of libbarvae.so (the C ABI declared in include/barvae.h).

There is NO CPU or PyTorch fallback: if the shared library is missing, or the device is not sm_100 (B200),
every entry point raises.  PyTorch is used only for device memory, streams and torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BVAE_LIB_PATH") or os.path.join(_HERE, "libbarvae.so")    # (override: A/B builds of the library)
MAX_TAPS = 16
MAX_PHASES = 6
IMPL_AUTO, IMPL_SIMT, IMPL_TC = 0, 1, 2

c_i32, c_f32, c_vp, c_i64 = C.c_int32, C.c_float, C.c_void_p, C.c_int64


class ConvDesc(C.Structure):
    """struct bvae_conv_desc (include/barvae.h)."""
    _fields_ = [("x", c_vp), ("w", c_vp), ("y", c_vp), ("bias", c_vp), ("addend", c_vp), ("mask", c_vp),
                ("stats", c_vp),
                ("N", c_i32), ("H", c_i32), ("W", c_i32), ("C", c_i32), ("x_pitch", c_i32),
                ("Cout", c_i32), ("w_pitch", c_i32), ("ntaps", c_i32),
                ("dy", c_i32 * MAX_TAPS), ("dx", c_i32 * MAX_TAPS),
                ("sy", c_i32), ("sx", c_i32), ("QH", c_i32), ("QW", c_i32),
                ("OH", c_i32), ("OW", c_i32), ("y_pitch", c_i32),
                ("osy", c_i32), ("osx", c_i32), ("ooy", c_i32), ("oox", c_i32),
                ("add_pitch", c_i32), ("mask_pitch", c_i32), ("act", c_i32), ("out_f32", c_i32),
                ("slope", c_f32), ("mask_slope", c_f32),
                ("nphase", c_i32), ("ph_ntaps", c_i32 * MAX_PHASES), ("ph_ooy", c_i32 * MAX_PHASES),
                ("ph_oox", c_i32 * MAX_PHASES), ("ph_QH", c_i32 * MAX_PHASES), ("ph_QW", c_i32 * MAX_PHASES)]


class WgradDesc(C.Structure):
    """struct bvae_wgrad_desc."""
    _fields_ = [("a", c_vp), ("s", c_vp), ("dw", c_vp), ("scratch", c_vp),
                ("N", c_i32), ("AH", c_i32), ("AW", c_i32), ("Ca", c_i32), ("a_pitch", c_i32),
                ("SH", c_i32), ("SW", c_i32), ("Cs", c_i32), ("s_pitch", c_i32),
                ("sy", c_i32), ("sx", c_i32), ("ntaps", c_i32), ("T", c_i32),
                ("dy", c_i32 * MAX_TAPS), ("dx", c_i32 * MAX_TAPS), ("tap_idx", c_i32 * MAX_TAPS)]


class NbDesc(C.Structure):
    """struct bvae_nb_desc."""
    _fields_ = [("N", c_i32), ("H", c_i32), ("W", c_i32), ("C", c_i32),
                ("y_pitch", c_i32), ("out_pitch", c_i32), ("res_pitch", c_i32), ("dout_pitch", c_i32),
                ("dy_pitch", c_i32), ("dres_pitch", c_i32),
                ("has_cbam", c_i32), ("Cr", c_i32), ("res_mode", c_i32), ("y_f32", c_i32),
                ("stats_fused", c_i32), ("slope", c_f32), ("eps", c_f32),
                ("y", c_vp), ("uhat", c_vp), ("out", c_vp), ("stats", c_vp), ("res", c_vp),
                ("gamma", c_vp), ("beta", c_vp), ("w1", c_vp), ("w2", c_vp), ("wsp", c_vp),
                ("nc", c_vp), ("nc_idx", c_vp), ("sa", c_vp), ("cidx", c_vp), ("gs", c_vp),
                ("dout", c_vp), ("dy", c_vp), ("dres", c_vp),
                ("dgamma", c_vp), ("dbeta", c_vp), ("dw1", c_vp), ("dw2", c_vp), ("dwsp", c_vp),
                ("bwd_nc", c_vp), ("bwd_px", c_vp), ("bwd_h", c_vp)]


class BnDesc(C.Structure):
    """struct bvae_bn_desc."""
    _fields_ = [("P", c_i64),
                ("C", c_i32), ("x_pitch", c_i32), ("y_pitch", c_i32), ("dy_pitch", c_i32), ("dx_pitch", c_i32),
                ("x_f32", c_i32), ("y_f32", c_i32), ("dy_f32", c_i32), ("act", c_i32), ("training", c_i32),
                ("slope", c_f32), ("eps", c_f32), ("momentum", c_f32),
                ("x", c_vp), ("y", c_vp), ("gamma", c_vp), ("beta", c_vp), ("running_mean", c_vp), ("running_var", c_vp),
                ("save", c_vp), ("scratch", c_vp), ("dy", c_vp), ("dx", c_vp), ("dgamma", c_vp), ("dbeta", c_vp)]


class PackJob(C.Structure):
    """mirror of bvae_pack_job (include/barvae.h)"""
    _fields_ = [("src", c_vp), ("dst", c_vp), ("R", c_i32), ("T", c_i32), ("Cc", c_i32), ("dst_pitch", c_i32),
                ("sr", c_i64), ("sc", c_i64), ("perm", c_i32 * MAX_TAPS)]


_lib = None
_dev_checked = False

# every symbol include/barvae.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("bvae_version", C.c_int, []),
    ("bvae_last_error", C.c_char_p, []),
    ("bvae_launch_count", C.c_uint64, []),
    ("bvae_launch_count_reset", None, []),
    ("bvae_launch_count_add", None, [C.c_uint64]),
    ("bvae_device_ok", C.c_int, []),
    ("bvae_last_kernel", C.c_char_p, []),
    ("bvae_set_deterministic", None, [C.c_int]),
    ("bvae_deterministic", C.c_int, []),
    ("bvae_set_option", None, [C.c_char_p, C.c_int]),
    ("bvae_get_option", C.c_int, [C.c_char_p, C.c_int]),
    ("bvae_conv_gemm", C.c_int, [C.POINTER(ConvDesc), C.c_int, c_vp]),
    ("bvae_conv_stats_ok", C.c_int, [C.POINTER(ConvDesc)]),
    ("bvae_wgrad_gemm", C.c_int, [C.POINTER(WgradDesc), C.c_int, c_vp]),
    ("bvae_pack_weight", C.c_int, [c_vp, c_vp, C.c_int, C.c_int, C.c_int, c_i64, c_i64, C.POINTER(c_i32), C.c_int,
                                   c_vp]),
    ("bvae_pack_plan_create", C.c_int, [C.POINTER(PackJob), C.c_int, C.POINTER(c_vp)]),
    ("bvae_pack_plan_run", C.c_int, [c_vp, c_vp]),
    ("bvae_pack_plan_destroy", None, [c_vp]),
    ("bvae_colsum", C.c_int, [c_vp, C.c_int, c_i64, C.c_int, C.c_int, c_vp, c_vp]),
    ("bvae_nb_forward", C.c_int, [C.POINTER(NbDesc), c_vp]),
    ("bvae_nb_backward", C.c_int, [C.POINTER(NbDesc), c_vp]),
    ("bvae_fit_sigmoid_fwd", C.c_int, [c_vp, C.c_int, c_vp, c_i64, C.c_int, c_vp, c_vp, c_vp]),
    ("bvae_bce_fwd", C.c_int, [c_vp, c_vp, c_i64, C.c_int, c_vp, c_vp]),
    ("bvae_bce_bwd", C.c_int, [c_vp, c_vp, c_i64, C.c_int, c_f32, c_vp, c_vp]),
    ("bvae_fit_sigmoid_bce_bwd", C.c_int, [c_vp, C.c_int, c_vp, c_vp, c_vp, c_vp, c_f32, C.c_int, c_i64, C.c_int,
                                           c_vp, C.c_int, c_vp, c_vp]),
    ("bvae_reparam_kl_fwd", C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    ("bvae_reparam_kl_bwd", C.c_int, [c_vp, c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_i64, c_vp]),
    ("bvae_adam_step", C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_f32, C.c_int, c_f32, c_vp]),
    ("bvae_adam_hyper", None, [c_f32, c_f32, c_f32, c_f32, C.c_int, c_f32, c_vp]),
    ("bvae_adam_step_dev", C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    ("bvae_adam_hyper_upload", C.c_int, [c_f32, c_f32, c_f32, c_f32, C.c_int, c_f32, c_vp, c_vp]),
    ("bvae_f32_to_bf16", C.c_int, [c_vp, c_vp, c_i64, c_vp]),
    ("bvae_unpack_bits", C.c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    ("bvae_threshold_pack", C.c_int, [c_vp, c_i64, c_f32, c_vp, c_vp, c_vp]),
    ("bvae_bernoulli_sample", C.c_int, [c_vp, c_i64, c_f32, C.c_uint64, c_i64, c_i32, c_vp, c_vp]),
    ("bvae_bar_score", C.c_int, [c_vp, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp, c_vp]),
    ("bvae_latent_moments", C.c_int, [c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_vp]),
    ("bvae_bn_scratch_floats", C.c_int, [C.c_int]),
    ("bvae_bn_forward", C.c_int, [C.POINTER(BnDesc), c_vp]),
    ("bvae_bn_backward", C.c_int, [C.POINTER(BnDesc), c_vp]),
]


def load():
    """Load libbarvae.so and bind every symbol (no device needed).  Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libbarvae.so is not built (%s): run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or `make -C musicgeneration_vae-torch_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)     # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def lib():
    """The library, after checking once that the current CUDA device is a B200 (sm_100)."""
    global _dev_checked
    l = load()
    if not _dev_checked:
        if not torch.cuda.is_available():
            raise RuntimeError("libbarvae needs a CUDA device (sm_100a); none is visible and there is no CPU fallback")
        torch.cuda.current_device()     # make sure the primary context exists before the library queries it
        if not l.bvae_device_ok():
            raise RuntimeError("libbarvae: " + l.bvae_last_error().decode())
        _dev_checked = True
    return l


def check(rc: int, what: str = ""):
    if rc != 0:
        raise RuntimeError("libbarvae %s failed (code %d): %s" % (what, rc, load().bvae_last_error().decode()))


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(load().bvae_launch_count())


def reset_launch_count():
    load().bvae_launch_count_reset()


def set_deterministic(flag: bool):
    """bvae_set_deterministic (include/barvae.h): fixed-order forward reductions, one split per weight-gradient tile"""
    load().bvae_set_deterministic(1 if flag else 0)


def last_kernel() -> str:
    return load().bvae_last_kernel().decode()


class option:
    """``with option("BVAE_NB_FAST", 0): ...`` -- a kernel-variant switch (bvae_set_option) for the duration of the block"""

    def __init__(self, name: str, value: int):
        self.name, self.value = name.encode(), int(value)

    def __enter__(self):
        load().bvae_set_option(self.name, self.value)
        return self

    def __exit__(self, *exc):
        load().bvae_set_option(self.name, -1)
        return False
