import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def cplib():
    """libcenterpose_b200.so, built in-tree if missing (nvcc cross-compiles without a GPU)."""
    from centerpose_b200 import _lib, build
    if not _lib.lib_available():
        build.build()
    return _lib.load()


@pytest.fixture(scope="session")
def pose_host():
    """pose_core.h compiled for the host (test-only harness)."""
    import ctypes
    src = os.path.join(ROOT, "tests", "host", "pose_core_host.cpp")
    out_dir = os.path.join(ROOT, "tests", "host", "_build")
    so = os.path.join(out_dir, "libpose_core_host.so")
    hdr = os.path.join(ROOT, "centerpose_b200", "csrc", "pose_core.h")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        os.makedirs(out_dir, exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so, src])
    return ctypes.CDLL(so)
