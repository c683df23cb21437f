import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import __graft_entry__ as entry  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def pkg():
    return entry.load_pkg()


@pytest.fixture(scope="session")
def po():
    mod = entry.load_oracle()
    mod.build()
    return mod


@pytest.fixture(scope="session")
def port(po):
    return po.Port()


@pytest.fixture(scope="session")
def ref(po):
    if not po.have_ref():
        pytest.skip("oracle/_ref/libofdm_ref.so not built (reference tree absent)")
    return po.Ref()


@pytest.fixture(scope="session")
def lib(pkg):
    if not os.path.exists(pkg.binding.LIB_PATH):
        entry.build()
    return pkg.load_library()


@pytest.fixture(scope="session")
def ofdm(pkg, lib):
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    o = pkg.Ofdm(0, lib=lib)
    yield o
    o.close()


@pytest.fixture(scope="session")
def golden():
    out = {}
    for name in ("stage_vectors.npz", "chain_totals.npz"):
        with np.load(os.path.join(ROOT, "tests", "golden", name)) as z:
            out.update({k: z[k] for k in z.files})
    return out


def bits_and_noise(seed, n_frames, n_sym):
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2, (n_frames, 96 * n_sym), dtype=np.uint8)
    g = rng.standard_normal((n_frames, 160 + 80 * n_sym)).astype(np.float32)
    return bits, g
