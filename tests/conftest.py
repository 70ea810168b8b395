import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")
    # a fresh checkout has no built artefacts (they are git-ignored): build once instead of failing at import.
    # nvcc cross-compiles sm_100a without a GPU; on a box without nvcc the prebuilt files that travelled are used.
    import shutil
    import subprocess
    pkg = os.path.join(ROOT, "gpushare_device_plugin_b200")
    needed = [os.path.join(pkg, "libgpushare_b200.so"), os.path.join(pkg, "gsbd"), os.path.join(ROOT, "build", "h2_selftest"),
              os.path.join(ROOT, "oracle", "libprobe_oracle_c.so")]
    if not all(os.path.exists(p) for p in needed) and shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc"):
        if not all(os.path.exists(p) for p in needed):
            subprocess.run(["bash", os.path.join(ROOT, "build.sh")], check=True, cwd=ROOT)


@pytest.fixture
def tmp_path(tmp_path):
    """pytest's tmp_path, or, where that is too deep for the unix sockets the tests create in it (a socket's path may
    not exceed 107 bytes: a long TMPDIR or user name), a fresh short directory that is removed afterwards."""
    if len(str(tmp_path)) <= 72:
        yield tmp_path
        return
    import pathlib
    import shutil
    from gpushare_device_plugin_b200.testing import socket_dir
    d = socket_dir("gsb-test-")
    yield pathlib.Path(d)
    shutil.rmtree(d, ignore_errors=True)


@pytest.fixture(scope="session")
def gsb():
    """Initialised C-ABI device layer. GPU tests only; fails loudly (no CPU fallback exists)."""
    from gpushare_device_plugin_b200 import device
    device.init()
    yield device
    device.shutdown()


@pytest.fixture(scope="session")
def small_arena(gsb):
    """512 MiB arena on device 0 for the bit-exact comparisons against the numpy/C oracle."""
    nbytes = gsb.arena_create(0, max_bytes=512 << 20)
    assert nbytes == 512 << 20
    yield nbytes
    # the full-arena tests re-create the arena themselves


@pytest.fixture(scope="session")
def c_oracle():
    import ctypes as C
    path = os.path.join(ROOT, "oracle", "libprobe_oracle_c.so")
    lib = C.CDLL(path)
    lib.po_verify.restype = C.c_uint64
    return lib
