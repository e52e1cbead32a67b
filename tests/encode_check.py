"""Checkers of what the encoders write (TEST INFRASTRUCTURE ONLY), and the seeded input layouts they are run on.

check_lz4 / check_zstd restate the format rules in plain Python and walk a stream before any decoder sees it, so
that a stream a lenient decoder would still accept (a match inside the last five bytes, a missing last-block flag)
is rejected too.  Then the system libraries and the plain-C restatement (oracle/port.py) must each restore the
block.  Shared by tests/test_emu_encode_contract.py (CPU) and tests/test_gpu_encode_contract.py (B200)."""
from __future__ import annotations

import ctypes as C
import hashlib

import numpy as np

from oracle import port
from pg_cryogen_b200 import COMP_LZ4, COMP_ZSTD, CRYO_BLCKSZ, blockgen as bg

MFLIMIT, LASTLITERALS = 12, 5          # LZ4 block format: the end-of-block rules
ZSTD_MAGIC = 0xFD2FB528
ZSTD_BLOCK_MAX = 128 << 10


class StreamError(AssertionError):
    """A stream breaks a rule of its format."""


_libs = None


def _syslibs():
    global _libs
    if _libs is None:
        lz4, zs = C.CDLL("liblz4.so.1"), C.CDLL("libzstd.so.1")
        lz4.LZ4_decompress_safe.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        zs.ZSTD_decompress.restype = C.c_size_t
        zs.ZSTD_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        zs.ZSTD_isError.argtypes = [C.c_size_t]
        zs.ZSTD_getFrameContentSize.restype = C.c_ulonglong
        zs.ZSTD_getFrameContentSize.argtypes = [C.c_void_p, C.c_size_t]
        zs.ZSTD_createDCtx.restype = C.c_void_p
        zs.ZSTD_freeDCtx.argtypes = [C.c_void_p]
        zs.ZSTD_decompressBegin.restype = C.c_size_t
        zs.ZSTD_decompressBegin.argtypes = [C.c_void_p]
        zs.ZSTD_nextSrcSizeToDecompress.restype = C.c_size_t
        zs.ZSTD_nextSrcSizeToDecompress.argtypes = [C.c_void_p]
        zs.ZSTD_decompressContinue.restype = C.c_size_t
        zs.ZSTD_decompressContinue.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        _libs = lz4, zs
    return _libs


def _u8(a) -> np.ndarray:
    return np.ascontiguousarray(np.frombuffer(bytes(a), dtype=np.uint8) if not isinstance(a, np.ndarray) else a,
                                dtype=np.uint8)


def compress_bound(method: int, n: int) -> int:
    """LZ4_compressBound / ZSTD_compressBound, as cryogpu_compress_bound states them"""
    if method == COMP_LZ4:
        return n + n // 255 + 16
    return n + (n >> 8) + (((128 << 10) - n) >> 11 if n < (128 << 10) else 0)


def lz4_walk(stream, n: int) -> int:
    """Walk the sequences of an LZ4 block that should decode to n bytes; raises StreamError on the first broken
    rule.  Returns the number of sequences."""
    s = bytes(stream)
    end, pos, out, nseq = len(s), 0, 0, 0
    while True:
        if pos >= end:
            raise StreamError(f"stream ends at byte {pos} without a closing literal run")
        token = s[pos]
        pos += 1
        nseq += 1
        ll = token >> 4
        if ll == 15:
            while True:
                if pos >= end:
                    raise StreamError("literal length extension runs past the stream")
                b = s[pos]
                pos += 1
                ll += b
                if b != 255:
                    break
        if pos + ll > end:
            raise StreamError(f"literal run of {ll} at byte {pos} runs past the stream")
        pos += ll
        out += ll
        if pos == end:                  # the last sequence: literals only
            if token & 15:
                raise StreamError("closing token has a match length")
            break
        if out > n - MFLIMIT:
            raise StreamError(f"match starts at {out}, after n - {MFLIMIT} = {n - MFLIMIT}")
        if pos + 2 > end:
            raise StreamError(f"offset at byte {pos} runs past the stream")
        off = s[pos] | s[pos + 1] << 8
        pos += 2
        if off == 0 or off > out:
            raise StreamError(f"offset {off} at output {out}")
        ml = token & 15
        if ml == 15:
            while True:
                if pos >= end:
                    raise StreamError("match length extension runs past the stream")
                b = s[pos]
                pos += 1
                ml += b
                if b != 255:
                    break
        out += ml + 4
        if pos == end:
            raise StreamError("the last sequence has a match")
        if out > n - LASTLITERALS:
            raise StreamError(f"match ends at {out}, inside the last {LASTLITERALS} bytes of {n}")
    if out != n:
        raise StreamError(f"stream decodes to {out} bytes, not {n}")
    return nseq


def check_lz4(stream, n: int, want) -> None:
    """The format walk, the bound, then liblz4 with capacity exactly n and the plain-C restatement."""
    c, want = _u8(stream), _u8(want)
    assert want.size == n
    if c.size > compress_bound(COMP_LZ4, n):
        raise StreamError(f"{c.size} bytes, above the bound {compress_bound(COMP_LZ4, n)}")
    lz4_walk(c, n)
    lz4, _ = _syslibs()
    out = np.zeros(n, dtype=np.uint8)
    got = lz4.LZ4_decompress_safe(c.ctypes.data, out.ctypes.data, c.size, n)
    if got != n or not np.array_equal(out, want):
        raise StreamError(f"LZ4_decompress_safe: {got} of {n} bytes, equal: {np.array_equal(out, want)}")
    got, out = port.lz4_decode(c, cap=n)
    if got != n or not np.array_equal(out, want):
        raise StreamError(f"oracle lz4_decode: {got} of {n} bytes")


def zstd_walk(frame, n: int) -> list[tuple[int, int, int]]:
    """Walk the header and the block headers of a zstd frame that should hold n bytes: one frame, single segment,
    no checksum, no dictionary, content size n, each block's content at most 128 KiB, the last-block flag on the
    last block only, nothing after it.  Returns (type, bytes, content) per block."""
    s = bytes(frame)
    if len(s) < 6 or int.from_bytes(s[:4], "little") != ZSTD_MAGIC:
        raise StreamError("no zstd magic")
    fhd = s[4]
    fcs_flag, single = fhd >> 6, (fhd >> 5) & 1
    if not single:
        raise StreamError("not a single-segment frame")
    if fhd & 0x08:
        raise StreamError("reserved bit set")
    if fhd & 0x04:
        raise StreamError("content checksum flag set")
    if fhd & 0x03:
        raise StreamError("dictionary id present")
    fsz = (1, 2, 4, 8)[fcs_flag]
    pos = 5 + fsz
    if pos > len(s):
        raise StreamError("frame header runs past the stream")
    fcs = int.from_bytes(s[5:pos], "little") + (256 if fsz == 2 else 0)
    if fcs != n:
        raise StreamError(f"frame content size {fcs}, not {n}")
    blocks = []
    while True:
        if pos + 3 > len(s):
            raise StreamError(f"block header at byte {pos} runs past the stream (no last block)")
        h = int.from_bytes(s[pos:pos + 3], "little")
        last, btype, bsize = h & 1, (h >> 1) & 3, h >> 3
        if btype == 3:
            raise StreamError("reserved block type")
        if bsize > ZSTD_BLOCK_MAX:
            raise StreamError(f"{('Raw', 'RLE', 'Compressed')[btype]} block of {bsize} bytes, above 128 KiB")
        nbytes = 1 if btype == 1 else bsize
        if pos + 3 + nbytes > len(s):
            raise StreamError(f"block at byte {pos} runs past the stream")
        blocks.append([btype, pos, nbytes, bsize if btype != 2 else None])
        pos += 3 + nbytes
        if last:
            break
    if pos != len(s):
        raise StreamError(f"{len(s) - pos} bytes after the last block")
    _zstd_block_contents(s, 5 + fsz, blocks, n)
    for k, b in enumerate(blocks):
        if b[3] > ZSTD_BLOCK_MAX:
            raise StreamError(f"block {k} holds {b[3]} bytes, above 128 KiB")
    if sum(b[3] for b in blocks) != n:
        raise StreamError(f"blocks hold {sum(b[3] for b in blocks)} bytes, not {n}")
    return [(b[0], b[2], b[3]) for b in blocks]


def _zstd_block_contents(s: bytes, hdr: int, blocks: list, n: int) -> None:
    """Fill in the bytes each Compressed block produces (blocks[k][3]), with libzstd's buffer-less decoder fed the
    header and then one block header and one block body per call, as the walk found them."""
    _, zs = _syslibs()
    c = np.frombuffer(s, dtype=np.uint8).copy()
    out = np.zeros(max(n, 1) + ZSTD_BLOCK_MAX, dtype=np.uint8)
    d = zs.ZSTD_createDCtx()
    op = 0

    def feed(at, size):
        if zs.ZSTD_nextSrcSizeToDecompress(d) != size:
            raise StreamError(f"libzstd expects {zs.ZSTD_nextSrcSizeToDecompress(d)} bytes at byte {at}, not {size}")
        r = zs.ZSTD_decompressContinue(d, out.ctypes.data + op, out.size - op, c.ctypes.data + at, size)
        if zs.ZSTD_isError(r):
            raise StreamError(f"libzstd rejects the {size} bytes at byte {at}")
        return int(r)
    try:
        zs.ZSTD_decompressBegin(d)
        feed(0, 5)
        feed(5, hdr - 5)
        for b in blocks:
            feed(b[1], 3)
            if b[2]:
                r = feed(b[1] + 3, b[2])
                op += r
                if b[3] is None:
                    b[3] = r
            elif b[3] is None:
                b[3] = 0
    finally:
        zs.ZSTD_freeDCtx(d)


def check_zstd(frame, n: int, want) -> None:
    """The header and block walk, the bound, then libzstd and the plain-C restatement."""
    c, want = _u8(frame), _u8(want)
    assert want.size == n
    if c.size > compress_bound(COMP_ZSTD, n):
        raise StreamError(f"{c.size} bytes, above the bound {compress_bound(COMP_ZSTD, n)}")
    zstd_walk(c, n)
    _, zs = _syslibs()
    fcs = zs.ZSTD_getFrameContentSize(c.ctypes.data, c.size)
    if fcs != n:
        raise StreamError(f"ZSTD_getFrameContentSize = {fcs}, not {n}")
    out = np.zeros(max(n, 1), dtype=np.uint8)
    got = zs.ZSTD_decompress(out.ctypes.data, n, c.ctypes.data, c.size)
    if zs.ZSTD_isError(got) or got != n or not np.array_equal(out[:n], want):
        raise StreamError(f"ZSTD_decompress: {got} of {n} bytes")
    got, out = port.zstd_decode(c, cap=n)
    if got != n or not np.array_equal(out[:n], want):
        raise StreamError(f"oracle zstd_decode: {got} of {n} bytes")


def check(method: int, stream, n: int, want) -> None:
    (check_lz4 if method == COMP_LZ4 else check_zstd)(stream, n, want)


def run_guard(method: int, n: int) -> int:
    """Most bytes a one-byte run of n >= 1024 may take: n / 200 + 64, and for LZ4 160 more, because every one of
    the (below 1 MiB, up to 16) segments of the GPU encoder keeps the end-of-block rules and closes with five
    literals, a token and an offset -- about 9 bytes a segment, which n / 200 does not cover below ~100 KiB"""
    return n // 200 + 64 + (160 if method == COMP_LZ4 else 0)


def digest(a) -> str:
    return hashlib.sha256(_u8(a).tobytes()).hexdigest()


# ---- input layouts ------------------------------------------------------------------------------------------------

SIZES = [1, 13, 16, 17, 63, 1023, 1025, 4099, 16383, 65535, 65536, 65537, 70001, 131077, 777777,
         CRYO_BLCKSZ - 1, CRYO_BLCKSZ, CRYO_BLCKSZ + 17, 3 * CRYO_BLCKSZ + 5]
KINDS = ["run-ee", "run-00", "random", "text", "copies", "tile65535", "tile65536", "tile65537", "sparse"]
LZ4_ACCELS = [0, 1, 2, 3, 9, 17, 65537, 2 ** 31 - 1, -7]
ZSTD_LEVELS = [-50, -5, -1, 0, 1, 3, 4, 19, 22]


def _copies(rng, total: int) -> np.ndarray:
    """runs, random bytes, four-letter text and copies taken from anywhere earlier (at any distance)"""
    out = np.empty(total, dtype=np.uint8)
    at = 0
    while at < total:
        kind = int(rng.integers(0, 5))
        if kind == 0:
            p = np.full(int(rng.integers(1, 5000)), int(rng.integers(0, 256)), dtype=np.uint8)
        elif kind == 1:
            p = rng.integers(0, 256, size=int(rng.integers(1, 400)), dtype=np.uint8)
        elif kind == 2:
            p = rng.integers(97, 101, size=int(rng.integers(1, 2000)), dtype=np.uint8)
        elif at > 16:
            src = int(rng.integers(0, at - 4))
            p = out[src: src + int(rng.integers(4, min(at - src, 3000) + 1))].copy()
        else:
            continue
        k = min(p.size, total - at)
        out[at: at + k] = p[:k]
        at += k
    return out


def _sparse(seed: int, total: int) -> np.ndarray:
    """the head and the tail of sparse cryo blocks (items, zero gap, tuples), cut to `total` bytes"""
    nblk = (total + CRYO_BLCKSZ - 1) // CRYO_BLCKSZ
    blk = np.concatenate([bg.make_block("S", "hex" if (seed + i) & 1 else "lowcard", seed + i) for i in range(nblk)])
    head = total // 3
    return np.concatenate([blk[:head], blk[blk.size - (total - head):]])


def layout(kind: str, n: int, seed: int, extra: int = 0) -> np.ndarray:
    """n + extra bytes of layout `kind`; the extra bytes continue the block's own pattern, so a read past n finds
    what looks like the rest of a match"""
    total = n + extra
    rng = np.random.default_rng([seed, n, KINDS.index(kind)])
    if kind == "run-ee":
        return np.full(total, 0xEE, dtype=np.uint8)
    if kind == "run-00":
        return np.zeros(total, dtype=np.uint8)
    if kind in ("random", "sparse"):
        blk = rng.integers(0, 256, size=n, dtype=np.uint8) if kind == "random" else _sparse(seed + n % 997, n)
        # the block's tail again: a match at the end of the block would run on into it
        return np.concatenate([blk, np.resize(blk[max(0, n - 4096):], extra)])
    if kind == "text":
        return rng.integers(97, 101, size=total, dtype=np.uint8)
    if kind == "copies":
        return _copies(rng, total)
    if kind.startswith("tile"):
        period = int(kind[4:])
        return np.resize(rng.integers(0, 256, size=period, dtype=np.uint8), total)
    raise ValueError(kind)
