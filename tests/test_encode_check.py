"""The encoder-output checkers of tests/encode_check.py (CPU): they pass what liblz4 / libzstd write and hand-made
streams that keep the rules, and reject hand-broken streams, each for the rule it breaks -- including streams a
lenient decoder would still restore."""
import ctypes as C

import numpy as np
import pytest

import encode_check as ec
from pg_cryogen_b200 import COMP_LZ4, COMP_ZSTD


def _ext(v):
    out = b""
    v -= 15
    while v >= 255:
        out += b"\xff"
        v -= 255
    return out + bytes([v])


def lz4_stream(seqs):
    """[(literals, offset, match length), ..., (literals, None, None)] -> an LZ4 block; a last entry with a match
    gives a block that ends on it"""
    out = b""
    for lit, off, ml in seqs:
        m = 0 if ml is None else ml - 4
        out += bytes([(min(len(lit), 15) << 4) | min(m, 15)])
        out += _ext(len(lit)) if len(lit) >= 15 else b""
        out += lit
        if off is not None:
            out += off.to_bytes(2, "little") + (_ext(m) if m >= 15 else b"")
    return out


def _expand(seqs):
    out = bytearray()
    for lit, off, ml in seqs:
        out += lit
        for _ in range(ml or 0):
            out.append(out[-off] if 0 < off <= len(out) else 0)
    return np.frombuffer(bytes(out), dtype=np.uint8)


A8 = b"abcdefgh"


def test_lz4_checker_accepts_liblz4_and_a_hand_made_block():
    lz4 = C.CDLL("liblz4.so.1")
    lz4.LZ4_compress_default.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    for kind, n in (("text", 70001), ("copies", 65537), ("run-00", 1025), ("random", 13)):
        src = ec.layout(kind, n, 3)
        dst = np.zeros(ec.compress_bound(COMP_LZ4, n), dtype=np.uint8)
        k = lz4.LZ4_compress_default(src.ctypes.data, dst.ctypes.data, n, dst.size)
        ec.check_lz4(dst[:k], n, src)
    seqs = [(A8, 8, 27), (b"abcde", None, None)]              # a match ending at n - 5 exactly
    ec.check_lz4(lz4_stream(seqs), 40, _expand(seqs))
    seqs = [(A8 * 3 + b"abcd", 8, 4), (A8, None, None)]         # a match starting at n - 12 exactly
    ec.check_lz4(lz4_stream(seqs), 40, _expand(seqs))
    seqs = [(b"a", 1, 300), (b"a" * 20, None, None)]           # length extensions on both sides
    ec.check_lz4(lz4_stream(seqs), 321, _expand(seqs))


@pytest.mark.parametrize("name,seqs,n,why", [
    ("match covers the last 5 bytes", [(A8, 8, 29), (b"abc", None, None)], 40, "inside the last 5"),
    ("match starts at n - 11", [(A8 * 3 + b"abcde", 8, 4), (b"bcdefgh", None, None)], 40, "after n - 12"),
    ("offset 0", [(A8, 0, 4), (A8 * 3 + b"abcd", None, None)], 40, "offset 0"),
    ("offset beyond the output", [(A8, 9, 4), (A8 * 3 + b"abcd", None, None)], 40, "offset 9"),
    ("final sequence with a match", [(A8, 8, 32)], 40, "last sequence has a match"),
    ("closing token one byte late", None, 40, None),
    ("stream one byte short", [(A8, 8, 20), (A8 + b"abcd", None, None)], 40, "past the stream"),
])
def test_lz4_checker_rejects_broken_blocks(name, seqs, n, why):
    if seqs is None:                    # a good block with a stray byte where its closing token should be
        good = [(A8, 8, 20), (A8 + b"abcd", None, None)]
        s = lz4_stream(good)
        at = len(lz4_stream(good[:1]))
        s = s[:at] + b"\x00" + s[at:]
        want = _expand(good)
    else:
        s = lz4_stream(seqs)
        want = np.resize(_expand(seqs), n)
        if name == "stream one byte short":
            s = s[:-1]
    with pytest.raises(ec.StreamError, match=why):
        ec.check_lz4(s, n, want)


def _zstd_frame(n, blocks, fcs=None, trailing=b""):
    """blocks: [(type, size, last, payload)] -> a single-segment frame with a 4-byte content size"""
    out = (0xFD2FB528).to_bytes(4, "little") + bytes([0xA0]) + (n if fcs is None else fcs).to_bytes(4, "little")
    for btype, size, last, payload in blocks:
        out += (last | btype << 1 | size << 3).to_bytes(3, "little") + payload
    return out + trailing


def test_zstd_checker_accepts_libzstd_and_a_hand_made_frame():
    zs = C.CDLL("libzstd.so.1")
    zs.ZSTD_compress.restype = C.c_size_t
    zs.ZSTD_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int]
    for kind, n, level in (("text", 300001, 3), ("copies", 65537, 1), ("run-ee", 1025, -5), ("random", 13, 1)):
        src = ec.layout(kind, n, 5)
        dst = np.zeros(ec.compress_bound(COMP_ZSTD, n), dtype=np.uint8)
        k = zs.ZSTD_compress(dst.ctypes.data, dst.size, src.ctypes.data, n, level)
        blocks = ec.zstd_walk(dst[:k], n)
        assert sum(b[2] for b in blocks) == n
        ec.check_zstd(dst[:k], n, src)
    raw = bytes(range(256)) * 400
    f = _zstd_frame(102400 + 1000, [(0, 102400, 0, raw[:102400]), (1, 1000, 1, b"\x07")])
    ec.check_zstd(f, 103400, np.frombuffer(raw[:102400] + b"\x07" * 1000, dtype=np.uint8))


def test_zstd_checker_rejects_broken_frames():
    raw = np.frombuffer(bytes(range(256)) * 600, dtype=np.uint8)
    good = [(0, 65536, 0, raw[:65536].tobytes()), (0, 65536, 1, raw[65536:131072].tobytes())]
    ec.check_zstd(_zstd_frame(131072, good), 131072, raw[:131072])
    cases = {
        "frame content size": _zstd_frame(131072, good, fcs=131071),
        "no last block": _zstd_frame(131072, [good[0], good[1][:2] + (0,) + good[1][3:]]),
        "above 128 KiB": _zstd_frame(140000, [(0, 140000, 1, raw[:140000].tobytes())]),
        "after the last block": _zstd_frame(131072, good, trailing=b"\x00"),
        "bytes after": _zstd_frame(131072, [good[0][:2] + (1,) + good[0][3:], good[1]]),   # last flag too early
    }
    for why, f in cases.items():
        n = 140000 if why == "above 128 KiB" else 131072
        with pytest.raises(ec.StreamError, match=why):
            ec.check_zstd(f, n, raw[:n])
    bad = bytearray(_zstd_frame(131072, good))
    bad[4] |= 0x04                                              # checksum flag
    with pytest.raises(ec.StreamError, match="checksum"):
        ec.check_zstd(bytes(bad), 131072, raw[:131072])


def test_bound_restatement_is_the_librarys():
    """The checkers' bound is cryogpu_compress_bound (libcryogpu.so loads without a GPU)."""
    from pg_cryogen_b200.codec import compress_bound
    for n in ec.SIZES + [(128 << 10) - 1, 128 << 10, 128 << 20]:
        for m in (COMP_LZ4, COMP_ZSTD):
            assert ec.compress_bound(m, n) == compress_bound(m, n), (m, n)


def test_layouts_are_seeded_and_continue_past_the_block():
    for kind in ec.KINDS:
        a = ec.layout(kind, 4099, 1, 4096)
        assert a.size == 4099 + 4096 and np.array_equal(a, ec.layout(kind, 4099, 1, 4096))
        assert np.array_equal(a[:4099], ec.layout(kind, 4099, 1)), kind
    t = ec.layout("tile65537", 70001, 2, 100)
    assert np.array_equal(t[65537:70101], t[:70101 - 65537])
