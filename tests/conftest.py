"""pytest configuration: the `gpu` marker and shared fixtures.

`-m "not gpu"` runs on the CPU-only build container: oracle vs reference, golden
fixtures, host logic, the C-ABI surface, and the kernel bodies under the SIMT
emulator (tests/emu).  `-m gpu` runs on a B200 and drives the real kernels through
the C ABI, checking them against the oracle.
"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle_ref():
    """The reference's own compression.c/storage.c on liblz4/libzstd (oracle/_ref), built from the pg_cryogen
    sources PG_CRYOGEN_SRC names or prebuilt.  Without it oracle.ref makes the codec calls on liblz4/libzstd
    directly, and what needs the reference's storage.c is compared with its stored outputs (tests/golden)."""
    from oracle import ref
    src = os.environ.get("PG_CRYOGEN_SRC", "")
    if not ref.available() and src and os.path.exists(os.path.join(src, "compression.c")):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref"])
    if ref.available():
        ref.lib()
    return ref


@pytest.fixture(scope="session")
def oracle_port():
    from oracle import port
    port.build()
    port.lib()
    return port


@pytest.fixture(scope="session")
def gpu():
    """A libcryogpu context on cuda:0.  Fails (never skips) when the library or GPU is missing."""
    from pg_cryogen_b200 import CryoGPU
    g = CryoGPU(0)
    yield g
    g.close()
