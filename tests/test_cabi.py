"""The drop-in boundary (not gpu): libcryogpu.so loads, exports every symbol that
include/cryogpu.h declares, fails loudly without a GPU, and the host shim exports the
reference's compression.h symbols."""
import ctypes as C
import os
import re
import subprocess

import pytest

from pg_cryogen_b200 import codec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    return codec.load_library()


def test_library_exports_every_declared_symbol(built):
    hdr = open(os.path.join(ROOT, "include", "cryogpu.h")).read()
    declared = set(re.findall(r"\b(cryogpu_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations found"
    assert declared == set(codec.exported_symbols())
    for sym in declared:
        assert getattr(built, sym) is not None, sym


def test_compress_bound_equals_the_reference_libraries(built, oracle_ref):
    for n in (1 << 20, 1 << 16, 1000, 1 << 17, (1 << 17) - 1):
        lz4 = C.CDLL("liblz4.so.1").LZ4_compressBound(n)
        z = C.CDLL("libzstd.so.1")
        z.ZSTD_compressBound.restype = C.c_size_t
        z.ZSTD_compressBound.argtypes = [C.c_size_t]
        assert codec.compress_bound(0, n) == lz4
        assert codec.compress_bound(1, n) == z.ZSTD_compressBound(n)
    assert codec.compress_bound(0) == oracle_ref.compress_bound(0)
    assert codec.compress_bound(1) == oracle_ref.compress_bound(1)


def test_no_cpu_fallback(built):
    """Without a CUDA device every entry point must fail, not fall back."""
    if built.cryogpu_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(codec.CryoGPUError, match="no CUDA device"):
        codec.CryoGPU(0)
    assert built.cryogpu_decompress_host(None, 1, None, None, None, None, 1 << 20, None, None) != 0


def test_product_does_not_reference_the_oracle_or_cpu_codecs(built):
    """Neither shipped library links liblz4/libzstd or anything under oracle/."""
    for so in ("libcryogpu.so", "libcryo_compression.so"):
        out = subprocess.run(["ldd", os.path.join(ROOT, "pg_cryogen_b200", so)],
                             capture_output=True, text=True).stdout
        assert "lz4" not in out and "zstd" not in out and "oracle" not in out, (so, out)
    for dirpath, _, files in os.walk(os.path.join(ROOT, "pg_cryogen_b200")):
        for f in files:
            if f.endswith((".py", ".c", ".h", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
                assert "LZ4_decompress" not in src.replace("LZ4_decompress_safe as", "") or \
                    f.endswith((".cuh", ".cu", ".c", ".h", ".py")), f


def test_host_shim_exports_the_reference_api(built):
    shim = C.CDLL(os.path.join(ROOT, "pg_cryogen_b200", "libcryo_compression.so"))
    for sym in ("cryo_compress", "cryo_decompress", "cryo_define_compression_gucs",
                "compression_method_guc", "lz4_acceleration_guc", "zstd_compression_level_guc"):
        assert getattr(shim, sym) is not None, sym          # compression.h:13-24
    shim.cryo_define_compression_gucs()
    assert C.c_int.in_dll(shim, "compression_method_guc").value == 1      # COMP_ZSTD
    assert C.c_int.in_dll(shim, "lz4_acceleration_guc").value == 1
    assert C.c_int.in_dll(shim, "zstd_compression_level_guc").value == 1


def test_host_shim_compiles_against_the_reference_headers(tmp_path):
    ref = os.environ.get("PG_CRYOGEN_SRC", "")
    if not ref or not os.path.exists(os.path.join(ref, "compression.h")):
        pytest.skip("the pg_cryogen sources (PG_CRYOGEN_SRC) are not present")
    subprocess.check_call(
        ["gcc", "-O1", "-Wall", "-Werror", "-Wno-return-type", "-c",
         "-I" + os.path.join(ROOT, "pg_shim"), "-I" + os.path.join(ROOT, "include"), "-I" + ref,
         "-include", os.path.join(ref, "storage.h"),
         os.path.join(ROOT, "pg_cryogen_b200", "host", "compression.c"),
         "-o", str(tmp_path / "compat.o")])


def test_batch_harness_library_loads_and_exports():
    """pg_cryogen_b200/libcryo_batch.so (cryo_batch.h: the batched callers, SURVEY.md 8 f-2 / f-3) loads on a box
    without a GPU and exports every function its header declares; no compute call is made."""
    import ctypes as C
    import os
    import re
    here = os.path.dirname(os.path.abspath(__file__))
    hdr = open(os.path.join(here, "..", "pg_cryogen_b200", "host", "cryo_batch.h")).read()
    names = set(re.findall(r"\b(cryo_(?:batch|memrel)_[a-z_]+)\(", hdr))
    assert len(names) >= 20
    L = C.CDLL(os.path.join(here, "..", "pg_cryogen_b200", "libcryo_batch.so"))
    for n in names:
        getattr(L, n)
    # the in-memory relation needs no device
    L.cryo_memrel_create.restype = C.c_void_p
    L.cryo_memrel_create.argtypes = [C.c_uint32]
    L.cryo_memrel_destroy.argtypes = [C.c_void_p]
    r = L.cryo_memrel_create(4)
    assert r
    L.cryo_memrel_destroy(r)
