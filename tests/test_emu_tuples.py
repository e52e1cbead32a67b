"""The tuple-fetch kernel bodies (cryo_tuples.cuh: select, scan, gather) under the SIMT emulator (tests/emu/emu_tuples.cpp),
launched as cryogpu.cu launches them, byte for byte against the restatement in tests/tuple_oracle.c
(cryo_oracle_block_tuples).  CPU only; tests/test_gpu_tuple_fetch.py runs the same comparison on the device."""
import ctypes as C

import numpy as np
import pytest

import tuple_oracle as opg

FILL = 0xA5


@pytest.fixture(scope="module")
def emu():
    return opg.emu_lib()


def _aligned(n, fill=0, dtype=np.uint8):
    item = np.dtype(dtype).itemsize
    raw = np.full(n + 64 // item, fill, dtype=dtype)
    at = ((-raw.ctypes.data) % 16) // item
    return raw[at: at + n]


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def emu_tuples(emu, blocks, block_size, sel=None, block_status=None, data_cap=None, tup_cap=None):
    n, stride = blocks.shape
    buf = _aligned(n * stride)
    buf[:] = blocks.reshape(-1)
    off, pos = opg.sel_arrays(sel, n)
    if data_cap is None or tup_cap is None:
        need = opg.block_tuples(blocks, sel, block_status, 0, 0, block_size)[5]
        data_cap = need[0] if data_cap is None else data_cap
        tup_cap = need[1] if tup_cap is None else tup_cap
    data = _aligned(max(data_cap, 1), FILL)
    to = np.full(max(tup_cap, 1), FILL * 0x0101010101010101, dtype=np.uint64)
    tl = np.full(max(tup_cap, 1), FILL * 0x01010101, dtype=np.uint32)
    bf = np.zeros(n + 1, dtype=np.uint64)
    st = np.zeros(n, dtype=np.int32)
    need = np.zeros(2, dtype=np.uint64)
    work = np.zeros(3 * (n + 1), dtype=np.uint64)
    bst = None if block_status is None else np.ascontiguousarray(block_status, dtype=np.int32)
    rc = emu.emu_tuples(_p(buf), C.c_uint64(stride), C.c_uint32(block_size), C.c_uint32(n), _p(bst), _p(off), _p(pos),
                        _p(data), C.c_uint64(data_cap), _p(to), _p(tl), C.c_uint64(tup_cap), _p(bf), _p(st), _p(need),
                        _p(work))
    assert rc == 0
    return data[:data_cap], to[:tup_cap], tl[:tup_cap], bf, st, (int(need[0]), int(need[1]))


def random_block(rng, block_size, stride, kind):
    """A decoded block of random layout: items at any alignment (overlaps allowed), 1 byte up to the whole data area."""
    blk = rng.integers(0, 256, size=stride, dtype=np.uint8)
    ntup = int(rng.integers(0, 40)) if kind != "many" else int(rng.integers(100, 300))
    lower = 8 + 8 * ntup + (int(rng.integers(1, 8)) if rng.random() < 0.2 else 0)
    lower = min(lower, block_size)
    upper = int(rng.integers(lower, block_size + 1))
    items = np.zeros((max(ntup, 1), 2), dtype=np.uint32)
    for k in range(ntup):
        if upper >= block_size:
            off, ln = block_size, 0
        elif k == 0 and rng.random() < 0.3:
            off, ln = upper, block_size - upper                     # the whole data area
        else:
            off = int(rng.integers(upper, block_size))
            ln = int(rng.integers(1, min(block_size - off, 9000) + 1)) if rng.random() < 0.7 else \
                int(rng.integers(1, min(block_size - off, 130) + 1))
        items[k] = off, ln
    blk[0:8] = np.array([lower, upper], dtype=np.uint32).view(np.uint8)
    room = max(0, min(ntup, (block_size - 8) // 8 - 1))
    blk[8: 8 + 8 * room] = items[:room].view(np.uint8).reshape(-1)
    if kind == "bad" and ntup:
        k = int(rng.integers(0, room)) if room else 0
        blk[8 + 8 * k: 12 + 8 * k] = np.frombuffer(np.uint32(block_size + 1).tobytes(), dtype=np.uint8)
    return blk


def random_selection(rng, blocks):
    sel = []
    for b in range(blocks.shape[0]):
        lower = int(blocks[b, 0:4].view(np.uint32)[0])
        nt = max(0, (lower - 1) // 8)
        choices = list(range(1, nt + 1)) or [1]
        k = int(rng.integers(0, 12))
        s = [int(rng.choice(choices)) for _ in range(k)]
        if rng.random() < 0.3:
            s.insert(int(rng.integers(0, len(s) + 1)), 0)
        if rng.random() < 0.3:
            s += [nt + 1, 0xFFFFFFFF]
        if s and rng.random() < 0.3:
            s += s[:3]                                              # repeats
        sel.append(s)
    return sel


def _check(got, want):
    names = ("data", "tup_off", "tup_len", "block_first", "status", "need")
    for name, g, w in zip(names, got, want):
        if isinstance(w, tuple):
            assert g == w, name
        else:
            assert np.array_equal(g, w), (name, np.flatnonzero(g != w)[:8])


@pytest.mark.parametrize("block_size", [1 << 16, 40_001, 8_200])
def test_emulated_tuple_fetch_equals_the_restatement(emu, block_size):
    rng = np.random.default_rng(2024 + block_size)
    stride = (block_size + 15) & ~15
    kinds = ["plain"] * 9 + ["bad", "many", "plain"]
    blocks = np.stack([random_block(rng, block_size, stride, k) for k in kinds])
    status = np.zeros(len(kinds), dtype=np.int32)
    status[[2, 7]] = [1, 9]                                         # failed in the decoder / the chain check
    for sel in (None, random_selection(rng, blocks)):
        want = opg.block_tuples(blocks, sel, status, block_size=block_size, fill=FILL)
        assert want[4][2] == 1 and want[4][7] == 9 and want[4][9] == 4
        got = emu_tuples(emu, blocks, block_size, sel, status)
        _check(got, want)
        # capacities that end inside the batch: every block from the first one that crosses on is OUTPUT
        dcap, tcap = want[5][0] // 2, want[5][1]
        _check(emu_tuples(emu, blocks, block_size, sel, status, dcap, tcap),
               opg.block_tuples(blocks, sel, status, dcap, tcap, block_size, fill=FILL))


def test_emulated_tuple_fetch_unaligned_items(emu):
    """Tuples at every offset mod 16 and of every length mod 16, both copy paths and the ragged ends."""
    bs = 4096
    blk = np.random.default_rng(5).integers(0, 256, size=bs, dtype=np.uint8)
    items = [(1024 + 67 * k + (k % 16), 1 + 13 * k) for k in range(40)]
    blk[0:8] = np.array([8 + 8 * len(items), 1024], dtype=np.uint32).view(np.uint8)
    blk[8: 8 + 8 * len(items)] = np.array(items, dtype=np.uint32).view(np.uint8).reshape(-1)
    blocks = np.stack([blk, blk])
    for sel in (None, [[3, 1, 0, 40, 41], list(range(40, 0, -1))]):
        _check(emu_tuples(emu, blocks, bs, sel), opg.block_tuples(blocks, sel, block_size=bs, fill=FILL))
