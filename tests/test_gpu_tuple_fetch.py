"""-m gpu: the batched tuple fetch (cryogpu_tuples_device, cryogpu_decompress_tuples_host,
cryogpu_decompress_pages_tuples_host and cryo_batch_fetch_tuples) against the restatement in tests/tuple_oracle.c
(cryo_oracle_block_tuples, tests/test_tuple_fetch_oracle.py) and the tuples that were inserted."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import pages as opg
import tuple_oracle
from pg_cryogen_b200 import CRYO_BLCKSZ, blockgen as bg
from pg_cryogen_b200.codec import _sel_arrays

from gpu_util import decode_device
from test_emu_tuples import random_block, random_selection
from test_gpu_batch import RelOps

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
PAGE = 8192
NONE = 0xFFFFFFFFFFFFFFFF
KINDS = [("S", "hex"), ("M", "lowcard"), ("D", "hex"), ("S", "random"), ("M", "hex"), ("D", "lowcard")]


def _same(got, want, n_fields=6):
    for name, g, w in zip(("data", "tup_off", "tup_len", "block_first", "status", "need"), got[:n_fields], want):
        if isinstance(w, tuple):
            assert tuple(g) == w, name
        else:
            assert np.array_equal(np.asarray(g), w), (name, np.flatnonzero(np.asarray(g) != w)[:8])


def _device_fetch(gpu, blocks, block_size, stride, sel, block_status, fill=0xA5):
    """cryogpu_tuples_device on blocks uploaded to HBM; capacities from the restatement's need."""
    dev = torch.device("cuda", gpu.device)
    n = blocks.shape[0]
    need = tuple_oracle.block_tuples(blocks, sel, block_status, 0, 0, block_size)[5]
    d_blk = torch.from_numpy(np.ascontiguousarray(blocks)).to(dev)
    d_bst = None if block_status is None else torch.from_numpy(np.asarray(block_status, dtype=np.int32)).to(dev)
    off, pos = _sel_arrays(sel, n)
    d_off = None if off is None else torch.from_numpy(off.view(np.int64)).to(dev)
    d_pos = None if pos is None else torch.from_numpy(pos.view(np.int32)).to(dev)
    d_data = torch.full((max(need[0], 16),), fill, dtype=torch.uint8, device=dev)
    d_to = torch.full((max(need[1], 1),), -1, dtype=torch.int64, device=dev)
    d_tl = torch.full((max(need[1], 1),), -1, dtype=torch.int32, device=dev)
    d_bf = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    d_st = torch.full((n,), -1, dtype=torch.int32, device=dev)
    d_need = torch.zeros(2, dtype=torch.int64, device=dev)
    gpu.tuples_device(d_blk, stride, n, d_bst, d_off, d_pos, d_data, need[0], d_to, d_tl, need[1], d_bf, d_st, d_need,
                      block_size=block_size, stream=torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    nd = d_need.cpu().numpy().view(np.uint64)
    return (d_data.cpu().numpy()[: need[0]], d_to.cpu().numpy().view(np.uint64)[: need[1]],
            d_tl.cpu().numpy().view(np.uint32)[: need[1]], d_bf.cpu().numpy().view(np.uint64),
            d_st.cpu().numpy(), (int(nd[0]), int(nd[1])))


@pytest.mark.parametrize("method", [0, 1])
def test_device_call_on_decoded_blocks(gpu, oracle_ref, method):
    blocks = np.stack([bg.make_block(k, p, 300 + i) for i, (k, p) in enumerate(KINDS)] + [bg.regression_block(1, 290)])
    comp = [oracle_ref.compress(method, 1, b)[0][0] for b in blocks]
    comp[3] = comp[3][:-7]                                  # a truncated stream: its status passes through
    dec, osz, st = decode_device(gpu, [method] * len(comp), comp)
    assert st[3] != 0 and (np.delete(st, 3) == 0).all()
    dec[3] = 0                                              # what the decoder left there does not matter
    rng = np.random.default_rng(method)
    for sel in (None, [[int(x) for x in rng.integers(0, 292, size=40)] for _ in range(len(blocks))]):
        want = tuple_oracle.block_tuples(dec, sel, st, fill=0xA5)
        got = _device_fetch(gpu, dec, CRYO_BLCKSZ, CRYO_BLCKSZ, sel, st)
        _same(got, want)
        again = _device_fetch(gpu, dec, CRYO_BLCKSZ, CRYO_BLCKSZ, sel, st, fill=0x11)
        assert np.array_equal(again[0], got[0])            # pad bytes are written: the buffer is deterministic


@pytest.mark.parametrize("block_size", [1 << 16, 40_001])
def test_device_call_on_random_layouts(gpu, block_size):
    """Items at any alignment, 1 byte up to the whole data area, odd block sizes: both copy paths on the device."""
    rng = np.random.default_rng(block_size)
    stride = (block_size + 15) & ~15
    kinds = ["plain"] * 20 + ["bad", "many"] * 3
    blocks = np.stack([random_block(rng, block_size, stride, k) for k in kinds])
    status = np.zeros(len(kinds), dtype=np.int32)
    status[[4, 9]] = [1, 10]
    for sel in (None, random_selection(rng, blocks)):
        _same(_device_fetch(gpu, blocks, block_size, stride, sel, status),
              tuple_oracle.block_tuples(blocks, sel, status, block_size=block_size, fill=0xA5))


def test_host_call_from_streams(gpu, oracle_ref):
    blocks = [bg.make_block(k, p, 400 + i) for i, (k, p) in enumerate(KINDS)]
    bad = blocks[0].copy()
    bad[8 + 8 * 9: 8 + 8 * 9 + 4] = 0xFF                   # item 10 points outside the block
    blocks = np.stack(blocks + [bad])
    methods = [i & 1 for i in range(len(blocks))]
    comp = [oracle_ref.compress(m, 1, b)[0][0] for m, b in zip(methods, blocks)]
    comp.append(comp[1][:-5])
    methods.append(methods[1])
    dec = np.concatenate([blocks, np.zeros((1, CRYO_BLCKSZ), dtype=np.uint8)])
    bst = [0] * len(blocks) + [1]
    sel = [[1, 290, 5, 5], [0], [288, 289, 1], [2, 0, 7], [], [17, 400], [3], [1, 2]]
    for s in (None, sel):
        got = gpu.decompress_tuples_host(methods, comp, s)
        st = got[4]
        assert st[-2] == 4 and st[-1] not in (0, 2), st    # bad item table: FORMAT; truncated stream: the decoder's
        want = tuple_oracle.block_tuples(dec, s, [0] * len(blocks) + [int(st[-1])], fill=0)
        _same(got, want)
        h2d, d2h = gpu.last_transfer_bytes()
        n = len(comp)
        assert h2d >= sum(c.size for c in comp)
        assert d2h <= want[5][0] + 12 * want[5][1] + 32 * (n + 1) + 64, (d2h, want[5])
    # room for part of the batch: the blocks that cross it are OUTPUT, need is the whole batch's
    full = gpu.decompress_tuples_host(methods, comp, sel)
    part = gpu.decompress_tuples_host(methods, comp, sel, data_cap=int(full[1][int(full[3][3])]), tup_cap=int(full[5][1]))
    assert part[5] == full[5] and list(part[4][:3]) == [0, 0, 0] and part[4][3] == 2


def _relation(oracle_ref, rng):
    rel = np.zeros((900, PAGE), dtype=np.uint8)
    free = list(rng.permutation(np.arange(1, 900)))
    blocks = np.stack([bg.make_block(k, p, 500 + i) for i, (k, p) in enumerate(KINDS)])
    chains = []
    for i, b in enumerate(blocks):
        c = oracle_ref.compress(i & 1, 1, b)[0][0]
        ch = [int(free.pop()) for _ in range(opg.pages_needed(c.size))]
        assert opg.split(rel, ch, c, i & 1, 700 + i) == len(ch)
        chains.append(ch)
    return rel, blocks, chains, free


def test_pages_call_with_chain_errors(gpu, oracle_ref):
    rng = np.random.default_rng(7)
    rel, blocks, chains, free = _relation(oracle_ref, rng)
    rel[chains[5][2], 28:32] = 0xFF                         # cut: the walk stops at the third page
    ask = chains[:5] + [chains[5][:3], [int(free[0])], chains[2][1:], [], chains[0]]
    n = len(ask)
    dec = np.concatenate([blocks[:5], np.zeros((4, CRYO_BLCKSZ), dtype=np.uint8), blocks[:1]])
    sel = [[1, 2, 0], [290], [0], [5, 5, 5], [], [1], [1], [1], [1], [9, 291]]
    for s in (None, sel):
        got = gpu.decompress_pages_tuples_host(rel, ask, s)
        st, me, csz = got[4], got[6], got[7]
        assert list(st[5:9]) == [10, 8, 9, 8], st          # CHAIN, EMPTY_BLOCK, WRONG_START, EMPTY_BLOCK
        _same(got, tuple_oracle.block_tuples(dec, s, [0] * 5 + [10, 8, 9, 8, 0], fill=0))
        for i in (0, 1, 2, 3, 4, 9):
            err, m, size, _, _ = opg.gather(rel, ask[i][0])
            assert (me[i], csz[i]) == (m, size)


@pytest.fixture(scope="module")
def blib():
    L = C.CDLL(os.path.join(HERE, "..", "pg_cryogen_b200", "libcryo_batch.so"))
    L.cryo_memrel_create.restype = C.c_void_p
    L.cryo_memrel_create.argtypes = [C.c_uint32]
    L.cryo_memrel_ops.restype = RelOps
    L.cryo_memrel_ops.argtypes = [C.c_void_p]
    L.cryo_memrel_pages.restype = C.POINTER(C.c_uint8)
    L.cryo_memrel_pages.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    L.cryo_memrel_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_writer_create.restype = C.c_void_p
    L.cryo_batch_writer_create.argtypes = [C.c_void_p, C.POINTER(RelOps), C.c_int, C.c_int, C.c_int, C.c_uint32]
    L.cryo_batch_insert.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.cryo_batch_flush.argtypes = [C.c_void_p]
    L.cryo_batch_writer_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_fetch_tuples.argtypes = [C.c_void_p, C.POINTER(RelOps), C.c_void_p, C.c_void_p, C.c_int,
                                          C.POINTER(FetchResult)]
    L.cryo_fetch_result_free.argtypes = [C.POINTER(FetchResult)]
    return L


class FetchResult(C.Structure):
    _fields_ = [("err", C.POINTER(C.c_int)), ("xid", C.POINTER(C.c_uint32)), ("first", C.POINTER(C.c_uint64)),
                ("tuple", C.POINTER(C.c_void_p)), ("len", C.POINTER(C.c_uint32)), ("ntuples", C.c_uint64),
                ("calls", C.c_uint64), ("data_", C.c_void_p), ("tup_off_", C.c_void_p), ("tup_len_", C.c_void_p)]


@pytest.mark.parametrize("method", [0, 1])
def test_fetch_tuples_through_the_batched_caller(gpu, blib, method):
    plan = [("S", "hex", 5 * 290), ("M", "lowcard", 2 * 290), ("D", "hex", 288 + 40)]
    tuples = []
    for kind, pl, rows in plan:
        per = bg.KINDS[kind][0]
        for b0 in range(0, rows, per):
            t = bg.make_tuples(kind, pl, 600 + b0, min(per, rows - b0))
            tuples.extend(t[i].tobytes() for i in range(t.shape[0]))
    rel = blib.cryo_memrel_create(4000)
    ops = blib.cryo_memrel_ops(rel)
    w = blib.cryo_batch_writer_create(gpu.handle, C.byref(ops), method, 1, 3, 777)
    tids = []
    tb, tp = C.c_uint32(0), C.c_uint32(0)
    for t in tuples:
        assert blib.cryo_batch_insert(w, t, len(t), C.byref(tb), C.byref(tp)) == 0
        tids.append((tb.value, tp.value))
    assert blib.cryo_batch_flush(w) == 0
    blib.cryo_batch_writer_destroy(w)
    nb = C.c_uint32(0)
    relation = np.ctypeslib.as_array(blib.cryo_memrel_pages(rel, C.byref(nb)), shape=(4000, PAGE))
    firsts = sorted({b for b, _ in tids})
    by_block = {b: [t for t, (bb, _) in zip(tuples, tids) if bb == b] for b in firsts}
    # a block whose first page was never written (PageIsNew): EMPTY_BLOCK for its TIDs
    empty = firsts[-1]
    relation[empty] = 0
    # TIDs from the insert, shuffled, with repeats, positions that do not exist, a lossy page, and the errors of cache.c
    rng = np.random.default_rng(method)
    pick = [tids[int(i)] for i in rng.integers(0, len(tids), size=600)]
    pick += pick[:50] + [(firsts[0], 291), (firsts[6], 0xFFFFFFFF), (firsts[1], 0), (firsts[7], 0)]
    cont = opg.gather(relation, firsts[5])[4][1]            # the second page of an M block's chain
    pick += [(cont, 1), (0, 1), (nb.value + 3, 1)]
    order = rng.permutation(len(pick))
    pick = [pick[int(i)] for i in order]
    tb_arr = np.array([b for b, _ in pick], dtype=np.uint32)
    tp_arr = np.array([p for _, p in pick], dtype=np.uint32)
    res = FetchResult()
    assert blib.cryo_batch_fetch_tuples(gpu.handle, C.byref(ops), tb_arr.ctypes.data, tp_arr.ctypes.data, len(pick),
                                        C.byref(res)) == 0
    assert res.calls == 1
    for i, (b, p) in enumerate(pick):
        lo, hi = res.first[i], res.first[i + 1]
        if b == 0 or b >= nb.value or b == cont:
            assert res.err[i] == 2 and hi == lo, (b, p)     # CRYO_ERR_WRONG_STARTING_BLOCK
            continue
        if b == empty:
            assert res.err[i] == 3 and hi == lo             # CRYO_ERR_EMPTY_BLOCK
            continue
        assert res.err[i] == 0 and res.xid[i] == 777
        want = by_block[b] if p == 0 else [by_block[b][p - 1] if p <= len(by_block[b]) else None]
        assert hi - lo == len(want), (b, p)
        for j, t in enumerate(want):
            ptr, ln = res.tuple[lo + j], res.len[lo + j]
            if t is None:
                assert not ptr and ln == 0
            else:
                assert ptr % 8 == 0 and C.string_at(ptr, ln) == t, (b, p, j)
    blib.cryo_fetch_result_free(C.byref(res))
    blib.cryo_memrel_destroy(rel)


def test_headline_table_every_item(gpu, oracle_ref):
    """3 449 blocks (the 1M-row S/hex table), every item: chunking and global offsets."""
    blocks = bg.make_table_blocks(1_000_000, "S", "hex")
    assert blocks.shape[0] == 3449
    comp = oracle_ref.compress(0, 1, blocks, nthreads=os.cpu_count() or 1)[0]
    got = gpu.decompress_tuples_host(0, comp)
    _same(got, tuple_oracle.block_tuples(blocks))
    assert got[5] == (1_000_000 * 64, 1_000_000)
