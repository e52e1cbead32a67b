"""ctypes binding of oracle/_ref/libcryoref.so (TEST INFRASTRUCTURE ONLY).

Every call lands in the reference's own cryo_compress / cryo_decompress
(compression.c:125-159) or cryo_init_page / cryo_storage_insert (storage.c:15-50).

oracle/_ref is built from the pg_cryogen sources (oracle/Makefile, PG_CRYOGEN_SRC) or
kept prebuilt.  Where it is absent, the codec calls (compress, decompress, bounds,
versions) go straight to liblz4.so.1 / libzstd.so.1, which is all compression.c:61-159
does with them: the same entry points, arguments and failure tests.  That stand-in is
pinned to the reference's recorded outputs (tests/golden, tests/test_oracle.py).  The
reference's storage.c and GUC table have no stand-in: lib(), guc_defaults() and
build_block() need oracle/_ref, and the tests compare with stored outputs without it.
"""
from __future__ import annotations

import ctypes as C
import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

CRYO_BLCKSZ = 1 << 20
COMP_LZ4, COMP_ZSTD = 0, 1          # compression.h:7-11

_HERE = os.path.dirname(os.path.abspath(__file__))
_PATH = os.path.join(_HERE, "_ref", "libcryoref.so")
_lib = None


def available() -> bool:
    return os.path.exists(_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"{_PATH} missing: `make -C oracle ref PG_CRYOGEN_SRC=<pg_cryogen sources>`")
        L = C.CDLL(_PATH)
        L.oref_compress_bound.restype = C.c_uint64
        L.oref_compress_bound.argtypes = [C.c_int]
        L.oref_block_size.restype = C.c_uint64
        L.oref_compress_batch.restype = C.c_double
        L.oref_compress_batch.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                          C.c_uint64, C.c_void_p, C.c_int, C.c_int]
        L.oref_decompress_batch.restype = C.c_double
        L.oref_decompress_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_size_t, C.c_void_p, C.c_uint64, C.c_void_p,
                                            C.c_int, C.c_int]
        L.oref_versions.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.oref_define_gucs.argtypes = [C.POINTER(C.c_int)] * 3
        L.oref_init_page.argtypes = [C.c_void_p]
        L.oref_storage_insert.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32]
        L.oref_storage_insert.restype = C.c_int
        L.oref_storage_fetch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint32]
        L.oref_storage_fetch.restype = C.c_int
        _lib = L
    return _lib


_sys = None


def _syslibs():
    """liblz4.so.1 / libzstd.so.1 for the codec calls of compression.c:61-123 where oracle/_ref is absent."""
    global _sys
    if _sys is None:
        lz4, zstd = C.CDLL("liblz4.so.1"), C.CDLL("libzstd.so.1")
        lz4.LZ4_compress_fast.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        lz4.LZ4_decompress_safe.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        zstd.ZSTD_compressBound.restype = C.c_size_t
        zstd.ZSTD_compressBound.argtypes = [C.c_size_t]
        zstd.ZSTD_compress.restype = C.c_size_t
        zstd.ZSTD_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int]
        zstd.ZSTD_decompress.restype = C.c_size_t
        zstd.ZSTD_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        zstd.ZSTD_isError.argtypes = [C.c_size_t]
        _sys = lz4, zstd
    return _sys


def describe() -> str:
    if available():
        return "the reference's compression.c (oracle/_ref) on liblz4 / libzstd"
    return "liblz4 / libzstd called as the reference's compression.c calls them (oracle/_ref absent)"


def _run_ranges(fn, n: int, nthreads: int) -> float:
    """fn(begin, end) over n items split into nthreads contiguous ranges, as oracle/ref_driver.c does; seconds."""
    k = max(1, min(nthreads, n)) if n else 1
    ranges = [(n * t // k, n * (t + 1) // k) for t in range(k)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(k) as ex:
        list(ex.map(lambda r: fn(*r), ranges))
    return time.perf_counter() - t0


def versions() -> tuple[int, int]:
    if not available():
        lz4, zstd = _syslibs()
        return int(lz4.LZ4_versionNumber()), int(zstd.ZSTD_versionNumber())
    a, b = C.c_int(), C.c_int()
    lib().oref_versions(C.byref(a), C.byref(b))
    return a.value, b.value


def guc_defaults() -> tuple[int, int, int]:
    m, a, l = C.c_int(), C.c_int(), C.c_int()
    lib().oref_define_gucs(C.byref(m), C.byref(a), C.byref(l))
    return m.value, a.value, l.value


def compress_bound(method: int) -> int:
    if not available():
        lz4, zstd = _syslibs()
        return int(lz4.LZ4_compressBound(CRYO_BLCKSZ) if method == COMP_LZ4 else zstd.ZSTD_compressBound(CRYO_BLCKSZ))
    return int(lib().oref_compress_bound(method))


def _sys_compress(method, level_or_accel, blocks, dst, sizes, nthreads, reps) -> float:
    """compression.c:61-77 / :93-109 on each block: one call into the library, 0 is a failure."""
    if method not in (COMP_LZ4, COMP_ZSTD):
        raise ValueError("unknown compression method")
    lz4, zstd = _syslibs()
    bound = compress_bound(method)

    def work(begin, end):
        scratch = np.empty(bound, dtype=np.uint8)
        for _ in range(max(reps, 1)):
            for i in range(begin, end):
                out = (dst[i] if dst is not None else scratch).ctypes.data
                src = blocks[i].ctypes.data
                if method == COMP_LZ4:
                    r = lz4.LZ4_compress_fast(src, out, CRYO_BLCKSZ, bound, level_or_accel)
                else:
                    r = zstd.ZSTD_compress(out, bound, src, CRYO_BLCKSZ, level_or_accel)
                    r = 0 if zstd.ZSTD_isError(r) else r
                if r == 0:
                    raise RuntimeError("compression failed")
                sizes[i] = r
    return _run_ranges(work, blocks.shape[0], nthreads)


def _sys_decompress(methods, buf, offs, sizes, out, ok, nthreads, reps) -> float:
    """compression.c:79-91 / :111-123 on each block: a negative result (an error code) is false."""
    if not np.isin(methods, (COMP_LZ4, COMP_ZSTD)).all():
        raise ValueError("unknown compression method")
    lz4, zstd = _syslibs()

    def work(begin, end):
        for _ in range(max(reps, 1)):
            for i in range(begin, end):
                src, dst = buf.ctypes.data + int(offs[i]), out[i].ctypes.data
                if methods[i] == COMP_LZ4:
                    good = lz4.LZ4_decompress_safe(src, dst, int(sizes[i]), CRYO_BLCKSZ) >= 0
                else:
                    good = not zstd.ZSTD_isError(zstd.ZSTD_decompress(dst, CRYO_BLCKSZ, src, int(sizes[i])))
                ok[i] = 1 if good else 0
    return _run_ranges(work, len(sizes), nthreads)


def compress(method: int, level_or_accel: int, blocks: np.ndarray, nthreads: int = 1,
             reps: int = 1, keep: bool = True):
    """Compress [n, 1 MiB] uint8 blocks.  Returns (list of bytes-like arrays, seconds)."""
    blocks = np.ascontiguousarray(blocks, dtype=np.uint8).reshape(-1, CRYO_BLCKSZ)
    n = blocks.shape[0]
    bound = compress_bound(method)
    sizes = np.zeros(n, dtype=np.uint32)
    dst = np.empty((n, bound), dtype=np.uint8) if keep else None
    if not available():
        t = _sys_compress(method, level_or_accel, blocks, dst, sizes, nthreads, reps)
    else:
        t = lib().oref_compress_batch(method, level_or_accel, blocks.ctypes.data, n,
                                      dst.ctypes.data if keep else None, bound,
                                      sizes.ctypes.data, nthreads, reps)
    out = [dst[i, : sizes[i]].copy() for i in range(n)] if keep else None
    return out, sizes, t


def pack(chunks) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Concatenate compressed blocks, 16-byte aligned starts -> (buffer, offsets, sizes)."""
    sizes = np.array([len(c) for c in chunks], dtype=np.uint32)
    offs = np.zeros(len(chunks), dtype=np.uint64)
    p = 0
    for i, s in enumerate(sizes):
        offs[i] = p
        p += (int(s) + 15) & ~15
    buf = np.zeros(max(p, 16), dtype=np.uint8)
    for i, c in enumerate(chunks):
        buf[int(offs[i]): int(offs[i]) + len(c)] = np.frombuffer(bytes(c), dtype=np.uint8) \
            if not isinstance(c, np.ndarray) else c
    return buf, offs, sizes


def decompress(methods, buf: np.ndarray, offs: np.ndarray, sizes: np.ndarray,
               nthreads: int = 1, reps: int = 1, out: np.ndarray | None = None):
    """Returns (out [n, 1 MiB], ok [n] uint8, seconds)."""
    n = len(sizes)
    methods = np.ascontiguousarray(np.broadcast_to(np.asarray(methods, dtype=np.int32), (n,)))
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    sizes = np.ascontiguousarray(sizes, dtype=np.uint32)
    if out is None:
        out = np.zeros((n, CRYO_BLCKSZ), dtype=np.uint8)
    ok = np.zeros(n, dtype=np.uint8)
    if not available():
        t = _sys_decompress(methods, buf, offs, sizes, out, ok, nthreads, reps)
    else:
        t = lib().oref_decompress_batch(methods.ctypes.data, buf.ctypes.data, offs.ctypes.data,
                                        sizes.ctypes.data, n, out.ctypes.data, CRYO_BLCKSZ,
                                        ok.ctypes.data, nthreads, reps)
    return out, ok, t


def decompress_one(method: int, comp) -> tuple[np.ndarray, bool]:
    c = np.frombuffer(bytes(comp), dtype=np.uint8) if not isinstance(comp, np.ndarray) else comp
    buf, offs, sizes = pack([c])
    out, ok, _ = decompress([method], buf, offs, sizes)
    return out[0], bool(ok[0])


def build_block(tuples) -> np.ndarray:
    """Pack tuple images through the reference's cryo_init_page/cryo_storage_insert."""
    blk = np.empty(CRYO_BLCKSZ, dtype=np.uint8)
    L = lib()
    L.oref_init_page(blk.ctypes.data)
    for t in tuples:
        b = bytes(t)
        if L.oref_storage_insert(blk.ctypes.data, b, len(b)) < 0:
            raise ValueError("cryo_storage_insert returned -1")
    return blk
