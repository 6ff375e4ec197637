"""Shared fixtures.  `-m "not gpu"` runs here on CPU (oracle, emulator, ABI); `-m gpu` runs the
parity tests proper through the C ABI on a B200."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _make(target_dir, *args):
    subprocess.run(["make", "-s", "-C", target_dir, *args], check=True)


@pytest.fixture(scope="session")
def orc():
    """The plain-C oracle (test infrastructure)."""
    path = os.path.join(ROOT, "oracle", "liboracle.so")
    if not os.path.exists(path):
        _make(os.path.join(ROOT, "oracle"), "liboracle.so")
    lib = C.CDLL(path)
    for f in ("orc_compress_ctx", "orc_decompress_ctx", "orc_getitem", "orc_lz4_compress_fast", "orc_lz4_decompress_safe",
              "orc_blosclz_compress", "orc_blosclz_decompress", "orc_bitshuffle", "orc_bitunshuffle"):
        getattr(lib, f).restype = C.c_int
    return lib


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference (oracle/_ref, built only where its sources are at hand), or None.  Tests
    that take it run against the stored reference results in tests/golden/ and use it on top when present."""
    path = os.path.join(ROOT, "oracle", "_ref", "libblosc_ref.so")
    if not os.path.exists(path):
        return None
    lib = C.CDLL(path)
    for f in ("blosc_compress_ctx", "blosc_decompress_ctx", "blosc_getitem", "LZ4_compress_fast", "LZ4_decompress_safe",
              "blosclz_compress", "blosclz_decompress"):
        getattr(lib, f).restype = C.c_int
    return lib


@pytest.fixture(scope="session")
def emu():
    """CPU build of the library: real host code + device kernels inside the SIMT emulator."""
    _make(os.path.join(ROOT, "tests", "emu"), "all")
    lib = C.CDLL(os.path.join(ROOT, "tests", "emu", "_build", "libblosc_b200_emu.so"))
    for f in ("blosc_compress_ctx", "blosc_decompress_ctx", "blosc_getitem", "blosc_b200_filter", "emu_lz4_encode",
              "emu_lz4_decode", "emu_blz_encode", "emu_blz_decode"):
        getattr(lib, f).restype = C.c_int
    return lib


@pytest.fixture(scope="session")
def pkg():
    """The product: c-blosc_b200 over libblosc_b200.so (CUDA)."""
    import __graft_entry__ as g
    if not os.path.exists(g.LIB):
        g.build_product()
    return g.load_package()


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch
