import importlib
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

PKG = "musicgeneration_vae-torch_b200"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    from golden_io import load_golden
    return load_golden("golden_v1")


@pytest.fixture(scope="session")
def oracle():
    import barvae_oracle
    return barvae_oracle


@pytest.fixture(scope="session")
def pkg():
    return importlib.import_module(PKG)


def assert_close(a, b, rtol, atol, what=""):
    a = a.detach().float().cpu()
    b = b.detach().float().cpu()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    err = (a - b).abs()
    tol = atol + rtol * b.abs()
    bad = err > tol
    if bad.any():
        i = torch.argmax(err - tol)
        raise AssertionError("%s: %d/%d out of tol (rtol=%g atol=%g); worst |a-b|=%g at %d (a=%g b=%g); "
                             "rel-fro=%g" % (what, int(bad.sum()), bad.numel(), rtol, atol, float(err.flatten()[i]),
                                             int(i), float(a.flatten()[i]), float(b.flatten()[i]),
                                             float((a - b).norm() / (b.norm() + 1e-30))))


def rel_fro(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))
