import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def native_lib():
    """Build (if stale) and load the product library.  Building needs nvcc only, not a GPU."""
    from gypsum_b200 import build, _native

    build.build()
    return _native.load()


@pytest.fixture(scope="session")
def emu_lib():
    """Host lane emulator (tests/emu): the product's lane-level device functions compiled for the CPU."""
    import ctypes

    from gypsum_b200 import build

    src = os.path.join(ROOT, "tests", "emu", "emu.cu")
    out = os.path.join(ROOT, "tests", "emu", "libgbemu.so")
    deps = [src] + [os.path.join(ROOT, "gypsum_b200", "csrc", f) for f in ("warp_fft.cuh", "fft32_gen.cuh", "cplx2.cuh", "gb_common.cuh", "tracker_core.cuh", "bits_core.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.run([build._nvcc(), "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-o", out, src], check=True,
                       capture_output=True)
    return ctypes.CDLL(out)
