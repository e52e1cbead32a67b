"""-m gpu: the batched callers (SURVEY.md 8 f-2, f-3) in pg_cryogen_b200/host/cryo_batch.c: COPY-style inserts
through the batched writer into an in-memory relation, then a sequential scan with read-ahead through the
batched cache.  Checked against the reference's storage.c (block images), its codec (oracle/_ref) and the
restatement of its page gather (oracle/cryo_pages.c)."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from oracle import pages as opg
from pg_cryogen_b200 import CRYO_BLCKSZ, blockgen as bg

import golden_util

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
PAGE = 8192


class RelOps(C.Structure):
    _fields_ = [("rel", C.c_void_p), ("nblocks", C.c_void_p), ("read_page", C.c_void_p), ("extend", C.c_void_p)]


@pytest.fixture(scope="module")
def lib():
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
    L.cryo_batch_writer_stats.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 3
    L.cryo_batch_writer_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_cache_create.restype = C.c_void_p
    L.cryo_batch_cache_create.argtypes = [C.c_void_p, C.c_int]
    L.cryo_batch_cache_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_cache_stats.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 3
    L.cryo_batch_read_data.argtypes = [C.c_void_p, C.POINTER(RelOps), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.cryo_batch_get_data.restype = C.POINTER(C.c_uint8)
    L.cryo_batch_get_data.argtypes = [C.c_void_p, C.c_int]
    L.cryo_batch_get_xid.restype = C.c_uint32
    L.cryo_batch_get_xid.argtypes = [C.c_void_p, C.c_int]
    L.cryo_batch_get_pg_nblocks.restype = C.c_uint32
    L.cryo_batch_get_pg_nblocks.argtypes = [C.c_void_p, C.c_int]
    L.cryo_batch_scan_begin.restype = C.c_void_p
    L.cryo_batch_scan_begin.argtypes = [C.c_void_p, C.POINTER(RelOps), C.c_int]
    L.cryo_batch_scan_next.restype = C.POINTER(C.c_uint8)
    L.cryo_batch_scan_next.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
    L.cryo_batch_scan_end.argtypes = [C.c_void_p]
    return L


@pytest.mark.parametrize("method", [0, 1])
def test_copy_then_seqscan_through_the_batched_callers(gpu, lib, oracle_ref, method):
    # rows of three kinds: 9 full blocks of S rows, 3 of M rows, 2 of D rows, and a partial last block
    plan = [("S", "hex", 9 * 290), ("M", "lowcard", 3 * 290), ("D", "hex", 2 * 288 + 17)]
    tuples = []
    for kind, pl, rows in plan:
        per = bg.KINDS[kind][0]
        for b0 in range(0, rows, per):
            t = bg.make_tuples(kind, pl, 900 + b0, min(per, rows - b0))
            tuples.extend(t[i] for i in range(t.shape[0]))
    rel = lib.cryo_memrel_create(6000)
    ops = lib.cryo_memrel_ops(rel)
    w = lib.cryo_batch_writer_create(gpu.handle, C.byref(ops), method, 1, 4, 555)
    tids = []
    tb, tp = C.c_uint32(0), C.c_uint32(0)
    for t in tuples:
        t = np.ascontiguousarray(t)
        assert lib.cryo_batch_insert(w, t.ctypes.data, t.size, C.byref(tb), C.byref(tp)) == 0
        tids.append((tb.value, tp.value))
    assert lib.cryo_batch_flush(w) == 0
    calls, blocks, pages = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    lib.cryo_batch_writer_stats(w, C.byref(calls), C.byref(blocks), C.byref(pages))
    assert blocks.value == 15 and calls.value == 4          # 4 + 4 + 4 + 3 blocks: one device call per batch, not per block
    lib.cryo_batch_writer_destroy(w)

    # what the reference's storage.c makes of the same tuples, block by block
    want_blocks, cur = [], []
    for t in tuples:
        try:
            blk = bg.pack_block(cur + [bytes(t)])
            cur.append(bytes(t))
        except ValueError:
            want_blocks.append(bg.pack_block(cur))
            cur = [bytes(t)]
    want_blocks.append(bg.pack_block(cur))
    assert len(want_blocks) == 15
    assert hashlib.sha256(want_blocks[0].tobytes()).hexdigest() == \
        golden_util.reference_block_sha256(oracle_ref, "S_hex_900", tuples[:290])

    # the relation on "disk": every chain reads back through the restated gather and the reference's codec
    nb = C.c_uint32(0)
    p = lib.cryo_memrel_pages(rel, C.byref(nb))
    relation = np.ctypeslib.as_array(p, shape=(nb.value, PAGE))
    assert nb.value == 1 + pages.value
    firsts = sorted({b for b, _ in tids})
    assert len(firsts) == 15
    for i, fb in enumerate(firsts):
        err, m, size, got, chain = opg.gather(relation, fb)
        assert err == opg.ERR_SUCCESS and m == method and got.size == size
        back, ok = oracle_ref.decompress_one(method, got)
        assert ok and np.array_equal(back, want_blocks[i]), i
    # item pointers: (first page of the block, 1-based position), pg_cryogen.c:648-650
    assert tids[0] == (firsts[0], 1) and tids[289] == (firsts[0], 290) and tids[290] == (firsts[1], 1)

    # sequential scan with read-ahead 6: 15 blocks in 3 device calls; every block, in block-number order
    cache = lib.cryo_batch_cache_create(gpu.handle, 8)
    scan = lib.cryo_batch_scan_begin(cache, C.byref(ops), 6)
    seen = []
    bno, xid, err = C.c_uint32(0), C.c_uint32(0), C.c_int(0)
    while True:
        d = lib.cryo_batch_scan_next(scan, C.byref(bno), C.byref(xid), C.byref(err))
        if not d:
            break
        seen.append((bno.value, np.ctypeslib.as_array(d, shape=(CRYO_BLCKSZ,)).copy()))
        assert xid.value == 555
    assert err.value == 0
    lib.cryo_batch_scan_end(scan)
    assert [b for b, _ in seen] == firsts
    for i, (_, blk) in enumerate(seen):
        assert np.array_equal(blk, want_blocks[i]), i
    lib.cryo_batch_cache_stats(cache, C.byref(calls), C.byref(blocks), C.byref(pages))
    assert calls.value == 3 and blocks.value == 15

    # index / bitmap scan: random blocks, hits and misses, and the errors of cache.c
    cont = opg.gather(relation, firsts[10])[4][1]           # the second page of a multi-page chain
    ask = np.array([firsts[3], firsts[14], firsts[13], firsts[3], cont, 0, nb.value + 5, firsts[7]], dtype=np.uint32)
    ent = np.zeros(ask.size, dtype=np.int32)
    errs = np.zeros(ask.size, dtype=np.int32)
    assert lib.cryo_batch_read_data(cache, C.byref(ops), ask.ctypes.data, ask.size, ent.ctypes.data, errs.ctypes.data) == 0
    assert list(errs) == [0, 0, 0, 0, 2, 2, 2, 0]          # a continuation page, the metapage, past the end: WRONG_STARTING_BLOCK
    for j in (0, 1, 2, 3, 7):
        d = lib.cryo_batch_get_data(cache, int(ent[j]))
        assert np.array_equal(np.ctypeslib.as_array(d, shape=(CRYO_BLCKSZ,)), want_blocks[firsts.index(int(ask[j]))])
        assert lib.cryo_batch_get_xid(cache, int(ent[j])) == 555
        assert lib.cryo_batch_get_pg_nblocks(cache, int(ent[j])) == len(opg.gather(relation, int(ask[j]))[4])
    lib.cryo_batch_cache_destroy(cache)
    lib.cryo_memrel_destroy(rel)
