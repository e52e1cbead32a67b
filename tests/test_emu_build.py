"""The block-build kernel body (cryo_tuples.cuh: blk_build_block) under the SIMT emulator (tests/emu/emu_build.cpp),
launched as cryogpu.cu launches k_block_build, byte for byte against blockgen.pack_block (which the stored block
SHA-256 values pin to the reference's storage.c).  CPU only; tests/test_gpu_build_blocks.py runs the device calls."""
import ctypes as C
import os

import numpy as np
import pytest

import tuple_oracle
from golden_util import reference_block_sha256
from pg_cryogen_b200 import CRYO_BLCKSZ, blockgen as bg
from test_emu_tuples import emu_tuples

HERE = os.path.dirname(os.path.abspath(__file__))
FILL = 0xA5
NONE = 0xFFFFFFFFFFFFFFFF


@pytest.fixture(scope="module")
def emu():
    return tuple_oracle.build("libcryoemu_build.so", ["g++", *tuple_oracle.EMU_CXXFLAGS, "-I" + os.path.join(HERE, "emu"),
                                                      "-shared", os.path.join(HERE, "emu", "emu_build.cpp")])


# ---- shared with tests/test_gpu_build_blocks.py ----

def storage_split(lens, block_size=CRYO_BLCKSZ):
    """storage_insert's arithmetic (storage.c:26-50) over a stream of tuple lengths, a new block whenever one refuses:
    (block index, 1-based position) per tuple, as the batched writer hands out item pointers."""
    out, blk, lower, upper = [], 0, 8, block_size
    for ln in lens:
        if ln + 8 > upper - lower or (lower - 8) // 8 + 1 >= 291:
            blk, lower, upper = blk + 1, 8, block_size
            assert ln + 8 <= upper - lower, "tuple cannot fit an empty block"
        upper -= (ln + 7) & ~7
        lower += 8
        out.append((blk, (lower - 8) // 8))
    return out


def pack_entries(blocks, rng=None, lead=0):
    """Tuples per block (lists of bytes) -> (data, tup_off, tup_len, block_first) in the layout the tuple fetch returns.
    rng None: MAXALIGNed and back to back, as the writer appends them; else 0..15 bytes of junk before each tuple,
    so that tuples start at every alignment.  lead: bytes of junk before the first one."""
    parts, off, ln, bf, at = [bytes([0x5C]) * lead], [], [], [0], lead
    for tuples in blocks:
        for t in tuples:
            gap = int(rng.integers(0, 16)) if rng is not None else 0
            parts.append(bytes(rng.integers(0, 256, size=gap, dtype=np.uint8)) if gap else b"")
            at += gap
            off.append(at)
            ln.append(len(t))
            pad = ((len(t) + 7) & ~7) - len(t) if rng is None else 0
            parts.append(bytes(t) + bytes(pad))
            at += len(t) + pad
        bf.append(len(off))
    data = np.frombuffer(b"".join(parts), dtype=np.uint8).copy()
    return data, np.array(off, dtype=np.uint64), np.array(ln, dtype=np.uint32), np.array(bf, dtype=np.uint64)


def reference_blocks(blocks, block_size, monkeypatch=None):
    """blockgen.pack_block of every block; at another block size through its CRYO_BLCKSZ"""
    if block_size != CRYO_BLCKSZ:
        monkeypatch.setattr(bg, "CRYO_BLCKSZ", block_size)
    out = np.stack([bg.pack_block(list(t), out=np.zeros(block_size, np.uint8)) for t in blocks]) if blocks else \
        np.zeros((0, block_size), np.uint8)
    if block_size != CRYO_BLCKSZ:
        monkeypatch.undo()
    return out


def random_blocks(rng, block_size, nblocks):
    """Blocks of random tuples 0..9 000 bytes long, each filled until a random count or storage.c refuses the next"""
    blocks = []
    for _ in range(nblocks):
        want, cur, lower, upper = int(rng.integers(0, 60)), [], 8, block_size
        while len(cur) < want:
            ln = int(rng.integers(0, 9001)) if rng.random() < 0.3 else int(rng.integers(0, 200))
            if ln + 8 > upper - lower or len(cur) >= 290:
                break
            cur.append(bytes(rng.integers(0, 256, size=ln, dtype=np.uint8)))
            upper -= (ln + 7) & ~7
            lower += 8
        blocks.append(cur)
    return blocks


def filled_to_the_end(block_size, extra=0):
    """Tuples whose last one takes the whole gap (len + 8 == upper - lower); extra > 0: that many bytes too many"""
    t = [bytes([k + 1]) * (50 + 13 * k) for k in range(7)]
    lower, upper = 8 + 8 * len(t), block_size - sum((len(x) + 7) & ~7 for x in t)
    return t + [bytes([0xEE]) * (upper - lower - 8 + extra)]


# ---- emulator calls ----

def emu_build(emu, data, tup_off, tup_len, block_first, block_size, data_size=None, lead=3):
    """blocks [n, stride] (FILL where nothing was written) and status.  The data sit `lead` bytes past a 16-byte boundary."""
    n = block_first.size - 1
    stride = (block_size + 15) & ~15
    raw = np.full(data.size + 64, 0x77, dtype=np.uint8)
    at = (-raw.ctypes.data) % 16 + lead
    raw[at: at + data.size] = data
    buf = raw[at:]
    dst_raw = np.full(n * stride + 32, FILL, dtype=np.uint8)
    d0 = (-dst_raw.ctypes.data) % 16
    dst = dst_raw[d0: d0 + n * stride]
    st = np.full(max(n, 1), -1, dtype=np.int32)
    to = np.ascontiguousarray(tup_off, dtype=np.uint64)
    tl = np.ascontiguousarray(tup_len, dtype=np.uint32)
    bf = np.ascontiguousarray(block_first, dtype=np.uint64)
    rc = emu.emu_build_blocks(C.c_uint32(n), C.c_void_p(buf.ctypes.data),
                              C.c_uint64(data.size if data_size is None else data_size),
                              C.c_void_p(to.ctypes.data if to.size else 0), C.c_void_p(tl.ctypes.data if tl.size else 0),
                              C.c_void_p(bf.ctypes.data), C.c_uint32(block_size), C.c_void_p(dst.ctypes.data),
                              C.c_uint64(stride), C.c_void_p(st.ctypes.data))
    assert rc == 0
    return dst.reshape(n, stride), st[:n]


@pytest.mark.parametrize("block_size", [40_008, (1 << 16) + 8, 8_200])
def test_random_tuples_at_unaligned_offsets(emu, monkeypatch, block_size):
    rng = np.random.default_rng(block_size)
    blocks = random_blocks(rng, block_size, 10)
    blocks += [[], [bytes([k % 7]) * (k % 23) for k in range(290)], filled_to_the_end(block_size), []]
    want = reference_blocks(blocks, block_size, monkeypatch)
    assert [int(w[:4].view(np.uint32)[0]) for w in want[-3:-1]] == [8 + 8 * 290, 8 + 8 * 8]
    assert want[-2][:8].view(np.uint32)[0] == want[-2][:8].view(np.uint32)[1]      # no gap left
    for r in (rng, None):
        got, st = emu_build(emu, *pack_entries(blocks, r), block_size)
        assert (st == 0).all(), st
        assert np.array_equal(got[:, :block_size], want), np.flatnonzero((got[:, :block_size] != want).any(axis=1))


def test_reference_blocks_at_1mib(emu, oracle_ref):
    import hashlib
    cases = [(f"{k}_{p}_5", [bytes(r) for r in bg.make_tuples(k, p, 5)]) for k in "SMD" for p in ("hex", "lowcard")]
    cases += [("ragged_100", [bytes([i % 251]) * (25 + 7 * i) for i in range(100)]), ("empty", [])]
    got, st = emu_build(emu, *pack_entries([t for _, t in cases], np.random.default_rng(1)), CRYO_BLCKSZ)
    assert (st == 0).all()
    for (key, t), blk in zip(cases, got):
        assert hashlib.sha256(blk.tobytes()).hexdigest() == reference_block_sha256(oracle_ref, key, t), key


def test_rejections_write_nothing(emu, monkeypatch):
    bs = 16_392
    rng = np.random.default_rng(3)
    good = [bytes(rng.integers(0, 256, size=40, dtype=np.uint8)) for _ in range(5)]
    blocks = [good, [b"x"] * 291, filled_to_the_end(bs, extra=1), good, good, good, good, good]
    data, off, ln, bf = pack_entries(blocks, rng)
    off[bf[4] + 2] = data.size - 39                     # 40 bytes from 39 before the end: past data_size
    off[bf[5] + 4] = NONE                               # the fetch's "not found"
    ln[bf[6] + 1] = bs + 1                              # longer than a block
    got, st = emu_build(emu, data, off, ln, bf, bs)
    assert list(st) == [0, 2, 2, 0, 4, 4, 4, 0], st    # OUTPUT: item 291, one byte too many; FORMAT
    want = reference_blocks([good], bs, monkeypatch)[0]
    for i in range(8):
        if st[i] == 0:
            assert np.array_equal(got[i, :bs], want), i
        else:
            assert (got[i] == FILL).all(), i            # nothing written
    # entries that end exactly at data_size are fine; block_first going backwards is malformed
    ok = pack_entries([good], rng)
    assert emu_build(emu, *ok, bs)[1][0] == 0
    assert list(emu_build(emu, data, off, ln, np.array([0, 5, 3, 8], dtype=np.uint64), bs)[1]) == [0, 4, 0]


def test_round_trip_through_the_tuple_fetch(emu):
    """Built blocks, every item fetched back: the input entries, byte for byte."""
    bs = 65_544
    rng = np.random.default_rng(9)
    blocks = random_blocks(rng, bs, 12) + [filled_to_the_end(bs)]
    data, off, ln, bf = pack_entries(blocks, rng)
    built, st = emu_build(emu, data, off, ln, bf, bs)
    assert (st == 0).all()
    fdata, foff, flen, fbf, fst, need = emu_tuples(tuple_oracle.emu_lib(), built, bs)
    assert (fst == 0).all() and np.array_equal(fbf, bf) and np.array_equal(flen, ln)
    for e in range(ln.size):
        a, b = int(foff[e]), int(off[e])
        assert np.array_equal(fdata[a: a + ln[e]], data[b: b + ln[e]]), e
