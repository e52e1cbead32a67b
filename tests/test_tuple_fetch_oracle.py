"""The restatement of the batched tuple fetch (tests/tuple_oracle.c, cryo_oracle_block_tuples) against the tuples
blockgen put into each block (storage.c:26-50 packing), against the reference's own cryo_storage_fetch (storage.c:55-68,
through oracle/_ref) where it is built, and on the selection and capacity edge cases the GPU and emulator tests rely on."""
import ctypes as C

import numpy as np
import pytest

import tuple_oracle as opg
from pg_cryogen_b200 import CRYO_BLCKSZ, blockgen as bg

ST_OK, ST_OUTPUT, ST_FORMAT = 0, 2, 4
NONE = 0xFFFFFFFFFFFFFFFF


def _empty_block():
    blk = np.zeros(CRYO_BLCKSZ, dtype=np.uint8)
    blk[0:8] = np.array([8, CRYO_BLCKSZ], dtype=np.uint32).view(np.uint8)   # cryo_init_page, storage.c:15-21
    return blk


def _table():
    tuples, blocks = [], []
    for i, (k, p) in enumerate((k, p) for k in bg.KINDS for p in bg.PAYLOADS):
        t = bg.make_tuples(k, p, 70 + i)
        tuples.append([t[j].tobytes() for j in range(t.shape[0])])
        blocks.append(bg.pack_block(t))
    reg = bg.regression_block(1, 290)
    tuples.append([reg[int(o): int(o) + int(n)].tobytes()
                   for o, n in reg[8: 8 + 8 * 290].view(np.uint32).reshape(-1, 2)])
    blocks.append(reg)
    tuples.append([])
    blocks.append(_empty_block())
    return tuples, np.stack(blocks)


def _tuple(data, to, tl, e):
    return data[int(to[e]): int(to[e]) + int(tl[e])].tobytes()


def test_every_item_is_the_tuple_that_was_inserted(oracle_ref):
    tuples, blocks = _table()
    data, to, tl, bf, st, need = opg.block_tuples(blocks)
    assert (st == ST_OK).all()
    assert need == (sum(bg.maxalign(len(t)) for ts in tuples for t in ts), sum(len(ts) for ts in tuples))
    assert list(np.diff(bf)) == [len(ts) for ts in tuples] and bf[-1] == need[1]
    for b, ts in enumerate(tuples):
        for j, t in enumerate(ts):
            e = int(bf[b]) + j
            assert to[e] % 8 == 0 and _tuple(data, to, tl, e) == t, (b, j)
            pad = data[int(to[e]) + len(t): int(to[e]) + bg.maxalign(len(t))]
            assert not pad.any()
    # entries are packed back to back
    assert np.array_equal(to[1:], to[:-1] + (tl[:-1].astype(np.uint64) + 7) // 8 * 8)
    if oracle_ref.available():
        L = oracle_ref.lib()
        out = np.zeros(CRYO_BLCKSZ, dtype=np.uint8)
        for b, ts in enumerate(tuples):
            blk = blocks[b].copy()
            for j in range(len(ts)):
                n = L.oref_storage_fetch(blk.ctypes.data, j + 1, out.ctypes.data, out.size)
                assert out[:n].tobytes() == _tuple(data, to, tl, int(bf[b]) + j), (b, j)


def test_selection_repeats_zero_and_missing_positions():
    tuples, blocks = _table()
    blocks = blocks[[0, 9, 4]]
    tuples = [tuples[0], tuples[9], tuples[4]]
    sel = [[3, 3, 290, 1, 291, 0xFFFFFFFF, 3], [0, 17, 0], [5]]
    data, to, tl, bf, st, need = opg.block_tuples(blocks, sel)
    assert (st == ST_OK).all() and list(bf) == [0, 7, 7 + 290 + 1 + 290, 7 + 290 + 1 + 290 + 1]
    want = [tuples[0][2], tuples[0][2], tuples[0][289], tuples[0][0], None, None, tuples[0][2]] + \
        tuples[1] + [tuples[1][16]] + tuples[1] + [tuples[2][4]]
    assert len(want) == need[1]
    for e, t in enumerate(want):
        if t is None:
            assert to[e] == NONE and tl[e] == 0
        else:
            assert _tuple(data, to, tl, e) == t, e
    assert need[0] == sum(bg.maxalign(len(t)) for t in want if t is not None)
    # a block with no items: a position beyond it is "not found", 0 selects nothing
    data, to, tl, bf, st, need = opg.block_tuples(np.stack([_empty_block()]), [[0, 1]])
    assert st[0] == ST_OK and need == (0, 1) and to[0] == NONE


def test_invalid_item_table_and_failed_blocks():
    _, blocks = _table()
    blocks = blocks[:4].copy()
    blocks[1, 8 + 8 * 5: 8 + 8 * 5 + 4] = np.frombuffer(np.uint32(CRYO_BLCKSZ - 10).tobytes(), dtype=np.uint8)  # item 6 crosses the end
    blocks[2, 0:4] = np.frombuffer(np.uint32(4).tobytes(), dtype=np.uint8)                                     # lower < 8
    data, to, tl, bf, st, need = opg.block_tuples(blocks, block_status=[0, 0, 0, 1])
    assert list(st) == [ST_OK, ST_FORMAT, ST_FORMAT, 1]
    assert list(bf) == [0, 290, 290, 290, 290]


@pytest.mark.parametrize("which", ["entries", "bytes"])
def test_capacity_overflow_at_every_block_boundary(which):
    _, blocks = _table()
    blocks = blocks[[0, 3, 10, 6, 9]]                   # the empty block sits in the middle
    sel = [[1, 2], [0], [1], [7, 7, 7], [0, 400]]
    full = opg.block_tuples(blocks, sel, fill=0x33)
    bf, (nbytes, nent) = full[3], full[5]
    sizes = np.where(full[1] == NONE, 0, (full[2].astype(np.uint64) + 7) // 8 * 8)
    bend = [int(sizes[: int(bf[b + 1])].sum()) for b in range(len(blocks))]       # byte end of each block
    bounds = [int(x) for x in bf] if which == "entries" else [0] + bend
    for k in range(len(blocks) + 1):
        for cap in sorted({bounds[k], max(bounds[k] - 1, 0)}):
            dcap, tcap = (nbytes, cap) if which == "entries" else (cap, nent)
            data, to, tl, bf2, st, need = opg.block_tuples(blocks, sel, data_cap=dcap, tup_cap=tcap, fill=0x33)
            assert need == (nbytes, nent) and np.array_equal(bf2, bf)
            for b in range(len(blocks)):
                lo, hi = int(bf[b]), int(bf[b + 1])
                fits = hi == lo or (hi <= tcap and bend[b] <= dcap)
                assert st[b] == (ST_OK if fits else ST_OUTPUT), (which, k, cap, b)
                if fits:
                    assert np.array_equal(to[lo:hi], full[1][lo:hi]) and np.array_equal(tl[lo:hi], full[2][lo:hi])
                else:
                    assert (to[lo:min(hi, tcap)] == 0x3333333333333333).all()       # nothing written
            # the blocks that fit are a prefix, and their bytes are the uncapped run's
            end = max([bend[b] for b in range(len(blocks)) if st[b] == ST_OK and bf[b + 1] > bf[b]], default=0)
            assert np.array_equal(data[:end], full[0][:end])
            assert (data[end:] == 0x33).all()
