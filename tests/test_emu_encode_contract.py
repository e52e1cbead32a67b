"""The encoders' work loops under the SIMT emulator (tests/emu/emu_encode_multi.cpp), three blocks per batch and two
emulated CTAs sharing the work queue, in strided slots (CPU).  The subset of tests/test_gpu_encode_contract.py that
the emulator runs in about a minute: every stream passes the format checkers of tests/encode_check.py, nothing is
written past dst_cap, the source is not written, and a block's stream does not depend on the blocks beside it."""
import ctypes as C
import os

import numpy as np
import pytest

import encode_check as ec
import tuple_oracle
from pg_cryogen_b200 import COMP_LZ4, COMP_ZSTD

HERE = os.path.dirname(os.path.abspath(__file__))
SENTINEL = 0xA5
# every branch of lz4e_seg_count up to 128 KiB, short last segments, and zstd frames of two and three blocks
SIZES = [1, 13, 17, 63, 1023, 1025, 4099, 16383, 65537, 131077]


@pytest.fixture(scope="module")
def emu():
    L = tuple_oracle.build("libcryoemu_encode.so", ["g++", *tuple_oracle.EMU_CXXFLAGS, "-I" + os.path.join(HERE, "emu"),
                                                    "-shared", os.path.join(HERE, "emu", "emu_encode_multi.cpp")])
    L.emu_encode_multi.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p,
                                   C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]
    return L


def _aligned(shape, fill):
    nbytes = int(np.prod(shape))
    raw = np.full(nbytes + 16, fill, dtype=np.uint8)
    o = (-raw.ctypes.data) % 16
    return raw[o:o + nbytes].reshape(shape)


def _r16(v):
    return (v + 15) & ~15


def encode(emu, method, level, srcs, n):
    """srcs: [k, >= n] (each block followed by the padding its slot should hold).  Returns the streams; asserts
    status 0, the sentinels in [dst_cap, dst_stride) and an unchanged source."""
    k = len(srcs)
    ss, cap = _r16(n) + 4096, ec.compress_bound(method, n)
    ds = _r16(cap) + 4096
    src = _aligned((k, ss), 0)
    for i, s in enumerate(srcs):
        src[i] = s[:ss]
    before = ec.digest(src)
    dst = _aligned((k, ds), SENTINEL)
    sz = np.zeros(k, dtype=np.uint32)
    st = np.full(k, -1, dtype=np.int32)
    assert emu.emu_encode_multi(method, level, src.ctypes.data, ss, n, k, dst.ctypes.data, ds, cap, sz.ctypes.data,
                                st.ctypes.data, 2, 2) == 0
    assert (st == 0).all(), st
    assert (dst[:, cap:] == SENTINEL).all(), "written past dst_cap"
    assert ec.digest(src) == before, "the source was written"
    return [dst[i, :sz[i]].copy() for i in range(k)]


def _inputs(n, i):
    """three layouts, a different three for every size, each followed by 4 KiB that continue its pattern"""
    kinds = [ec.KINDS[(3 * i + j) % len(ec.KINDS)] for j in range(3)]
    return kinds, [ec.layout(kd, n, 7 + i, _r16(n) + 4096 - n) for kd in kinds]


@pytest.mark.parametrize("method,level", [(COMP_LZ4, 1), (COMP_ZSTD, 1)])
@pytest.mark.parametrize("n", SIZES)
def test_emu_encode_batch_in_strided_slots(emu, n, method, level):
    kinds, srcs = _inputs(n, SIZES.index(n))
    comp = encode(emu, method, level, srcs, n)
    for kd, c, s in zip(kinds, comp, srcs):
        try:
            ec.check(method, c, n, s[:n])
        except ec.StreamError as e:
            raise AssertionError(f"{kd} n={n}: {e}") from None
        if kd.startswith("run") and n >= 1024:
            assert len(c) <= ec.run_guard(method, n), (kd, n, len(c))
    # the same blocks one at a time, in another order: the same streams
    if n <= 16383:
        for i in (2, 0, 1):
            assert np.array_equal(encode(emu, method, level, [srcs[i]], n)[0], comp[i]), (kinds[i], n)


@pytest.mark.parametrize("method,level", [(COMP_LZ4, a) for a in ec.LZ4_ACCELS] + [(COMP_ZSTD, z) for z in ec.ZSTD_LEVELS])
def test_emu_encode_parameters(emu, method, level):
    for n, kinds in ((1025, ["run-ee", "text", "copies"]), (4099, ["sparse", "random", "run-00"])):
        srcs = [ec.layout(kd, n, 3, _r16(n) + 4096 - n) for kd in kinds]
        for kd, c, s in zip(kinds, encode(emu, method, level, srcs, n), srcs):
            try:
                ec.check(method, c, n, s[:n])
            except ec.StreamError as e:
                raise AssertionError(f"{kd} n={n} level {level}: {e}") from None


@pytest.mark.parametrize("method", [COMP_LZ4, COMP_ZSTD])
def test_emu_stream_does_not_depend_on_place_in_batch(emu, method):
    """Regression: several lanes of one warp stored their positions into the same hash-table slot at once, and CUDA
    leaves unspecified which store lands.  Under the emulator the winner followed the interleaving of the warps, so
    the same LZ4 block (copies, 16 383 bytes) came out as 1 872, 1 922 and 1 972 bytes at places 0, 1 and 2 of one
    batch.  Now the highest lane of each slot stores alone."""
    n = 16383
    src = ec.layout("copies", n, 7 + SIZES.index(n), _r16(n) + 4096 - n)
    comp = encode(emu, method, 1, [src] * 3, n)
    assert all(np.array_equal(c, comp[0]) for c in comp[1:]), [len(c) for c in comp]
    ec.check(method, comp[0], n, src[:n])
