"""-m gpu: cryo blocks built on the device from packed tuples -- cryogpu_build_blocks_device,
cryogpu_compress_tuples_pages_alloc_host and the batched writer on top of it -- against blockgen.pack_block (pinned to
the reference's storage.c by the stored block SHA-256 values) and against cryogpu_compress_pages_alloc_host on those
block images."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import pages as opg
from pg_cryogen_b200 import CRYO_BLCKSZ, blockgen as bg
from pg_cryogen_b200.codec import compress_bound, page_callbacks

from golden_util import reference_block_sha256
from gpu_util import decode_device
from test_emu_build import pack_entries, storage_split
from test_gpu_tuple_fetch import FetchResult, KINDS, blib  # noqa: F401 (blib: the fixture)

pytestmark = pytest.mark.gpu
PAGE = 8192
NONE = 0xFFFFFFFFFFFFFFFF


def _dev(gpu):
    return torch.device("cuda", gpu.device)


def device_build(gpu, data, tup_off, tup_len, block_first, block_size=CRYO_BLCKSZ, lead=5, fill=0xA5):
    """cryogpu_build_blocks_device with the data `lead` bytes past a 16-byte boundary.  Returns the blocks (a CUDA
    tensor [n, stride]) and the status."""
    dev = _dev(gpu)
    n = block_first.size - 1
    stride = (block_size + 15) & ~15
    d_raw = torch.zeros(data.size + lead + 16, dtype=torch.uint8, device=dev)
    d_raw[lead: lead + data.size] = torch.from_numpy(data).to(dev)
    d_to = torch.from_numpy(np.ascontiguousarray(tup_off, dtype=np.uint64).view(np.int64)).to(dev)
    d_tl = torch.from_numpy(np.ascontiguousarray(tup_len, dtype=np.uint32).view(np.int32)).to(dev)
    d_bf = torch.from_numpy(np.ascontiguousarray(block_first, dtype=np.uint64).view(np.int64)).to(dev)
    d_dst = torch.full((n, stride), fill, dtype=torch.uint8, device=dev)
    d_st = torch.full((n,), -1, dtype=torch.int32, device=dev)
    gpu.build_blocks_device(d_raw.data_ptr() + lead, data.size, d_to, d_tl, d_bf, n, d_dst, stride, d_st,
                            block_size=block_size, stream=torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    return d_dst, d_st.cpu().numpy()


def _sha(a) -> str:
    return hashlib.sha256(a.tobytes()).hexdigest()


def test_device_call_against_the_reference_blocks(gpu, oracle_ref):
    cases = [(f"{k}_{p}_5", [bytes(r) for r in bg.make_tuples(k, p, 5)]) for k in "SMD" for p in bg.PAYLOADS]
    cases += [("ragged_100", [bytes([i % 251]) * (25 + 7 * i) for i in range(100)]),
              ("S_hex_3448_80", [bytes(r) for r in bg.make_tuples("S", "hex", 3448, ntuples=80)]), ("empty", [])]
    for rng in (np.random.default_rng(11), None):
        got, st = device_build(gpu, *pack_entries([t for _, t in cases], rng))
        assert (st == 0).all(), st
        got = got.cpu().numpy()
        for (key, t), blk in zip(cases, got):
            assert _sha(blk) == reference_block_sha256(oracle_ref, key, t), key


def table_entries(nrows, kind="S", payload="hex"):
    """The packed tuples of an nrows-row table, as the writer appends them (numpy, no per-tuple loop)"""
    per, t_len = bg.KINDS[kind]
    nb = bg.table_block_count(nrows, kind)
    step = (t_len + 7) & ~7
    data = np.zeros((nrows, step), dtype=np.uint8)
    counts = [min(per, nrows - b * per) for b in range(nb)]
    for b in range(nb):
        data[b * per: b * per + counts[b], :t_len] = bg.make_tuples(kind, payload, b, counts[b])
    bf = np.zeros(nb + 1, dtype=np.uint64)
    bf[1:] = np.cumsum(counts)
    return (data.reshape(-1), np.arange(nrows, dtype=np.uint64) * np.uint64(step), np.full(nrows, t_len, np.uint32), bf)


def test_device_call_on_the_headline_table(gpu):
    """The whole 1M-row S/hex table (3 449 blocks), block for block against pack_block"""
    got, st = device_build(gpu, *table_entries(1_000_000), lead=0)
    assert got.shape[0] == 3449 and (st == 0).all()
    want = bg.make_table_blocks(1_000_000, "S", "hex")
    for lo in range(0, 3449, 512):
        g = got[lo: lo + 512].cpu().numpy()
        bad = np.flatnonzero((g != want[lo: lo + 512]).any(axis=1))
        assert bad.size == 0, lo + bad[:8]


@pytest.mark.parametrize("method", [0, 1])
def test_round_trip_through_the_fetch(gpu, oracle_ref, method):
    """Decode on the device, fetch every item, build again: the decoded blocks"""
    blocks = np.stack([bg.make_block(k, p, 40 + i) for i, (k, p) in enumerate(KINDS)] +
                      [bg.regression_block(1, 290), bg.pack_block([bytes([7]) * 9000, b"", b"abc"])])
    comp = [oracle_ref.compress(method, 1, b)[0][0] for b in blocks]
    dec, _, st = decode_device(gpu, [method] * len(comp), comp)
    assert (st == 0).all() and np.array_equal(dec, blocks)
    dev = _dev(gpu)
    n = len(blocks)
    d_dec = torch.from_numpy(dec).to(dev)
    ntup = sum(int(b[:4].view(np.uint32)[0] - 8) // 8 for b in blocks)
    d_data = torch.zeros(n * CRYO_BLCKSZ, dtype=torch.uint8, device=dev)
    d_to = torch.zeros(ntup, dtype=torch.int64, device=dev)
    d_tl = torch.zeros(ntup, dtype=torch.int32, device=dev)
    d_bf = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    d_fst = torch.full((n,), -1, dtype=torch.int32, device=dev)
    d_need = torch.zeros(2, dtype=torch.int64, device=dev)
    d_out = torch.full((n, CRYO_BLCKSZ), 0x3C, dtype=torch.uint8, device=dev)
    d_st = torch.full((n,), -1, dtype=torch.int32, device=dev)
    s = torch.cuda.current_stream(dev).cuda_stream
    gpu.tuples_device(d_dec, CRYO_BLCKSZ, n, None, None, None, d_data, d_data.numel(), d_to, d_tl, ntup, d_bf, d_fst, d_need,
                      stream=s)
    gpu.build_blocks_device(d_data, int(d_data.numel()), d_to, d_tl, d_bf, n, d_out, CRYO_BLCKSZ, d_st, stream=s)
    torch.cuda.synchronize(dev)
    assert (d_fst.cpu().numpy() == 0).all() and (d_st.cpu().numpy() == 0).all()
    assert torch.equal(d_out, d_dec)


def old_flush(gpu, method, level, images, relation, first_blkno, next_blkno, xid):
    """cryogpu_compress_pages_alloc_host on block images: the parent commit's flush"""
    n = images.shape[0]
    alloc, page_ptr, handed = page_callbacks(relation, next_blkno)
    srcp = (C.c_void_p * n)(*[images[i].ctypes.data for i in range(n)])
    first = np.ascontiguousarray(first_blkno, dtype=np.uint32)
    npg, csz, st = np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.full(n, -1, np.int32)
    assert gpu.lib.cryogpu_compress_pages_alloc_host(gpu.handle, n, method, level, srcp, images.shape[1], first.ctypes.data,
                                                     alloc, page_ptr, None, xid, npg.ctypes.data, csz.ctypes.data,
                                                     st.ctypes.data) == 0, gpu.lib.cryogpu_last_error()
    return npg, csz, st, handed


def mixed_blocks(seed, nblocks):
    out = []
    for i in range(nblocks):
        k, p = KINDS[i % len(KINDS)]
        out.append([bytes(r) for r in bg.make_tuples(k, p, seed + i, 1 + (37 * i) % bg.KINDS[k][0])])
    return out


def h2d_bound(blocks, chunk_counts, cap_pages):
    """Σ MAXALIGN(len) + 12 per entry + 8 per block + the block-number rows + 256 bytes per array per chunk"""
    tup = sum(((len(t) + 7) & ~7) + 12 for b in blocks for t in b)
    return tup + 8 * len(blocks) + sum(c * cap_pages * 4 for c in chunk_counts) + 256 * 5 * len(chunk_counts)


@pytest.mark.parametrize("method,level", [(0, 1), (1, 1), (1, 3)])
def test_host_call_equals_the_flush_of_block_images(gpu, method, level):
    blocks = mixed_blocks(70, 20)
    images = np.stack([bg.pack_block(t) for t in blocks])
    first = np.arange(1, 21, dtype=np.uint32)
    rel_old = np.zeros((3000, PAGE), dtype=np.uint8)
    rel_new = np.zeros((3000, PAGE), dtype=np.uint8)
    want = old_flush(gpu, method, level, images, rel_old, first, 21, 99)
    old_h2d = gpu.last_transfer_bytes()[0]
    got = gpu.compress_tuples_pages_host(method, level, *pack_entries(blocks), rel_new, first, 21, 99)
    assert (got[2] == 0).all(), got[2]
    for name, g, w in zip(("npages", "comp_size", "status", "block numbers"), got, want):
        assert np.array_equal(np.asarray(g), np.asarray(w)), name
    assert np.array_equal(rel_new, rel_old)
    h2d = gpu.last_transfer_bytes()[0]
    assert h2d <= h2d_bound(blocks, [20], opg.pages_needed(compress_bound(method))) < old_h2d, (h2d, old_h2d)


def test_chunks_transfer_bytes_and_failures(gpu):
    """300 blocks cross PG_HOST_CHUNK (128); one block with a "not found" entry fails alone"""
    blocks = [[bytes(r) for r in bg.make_tuples("S", "hex", 900 + i, 290 - (i % 50))] for i in range(300)]
    data, off, ln, bf = pack_entries(blocks)
    cap_pages = opg.pages_needed(compress_bound(0))
    first = np.arange(1, 301, dtype=np.uint32)
    rel = np.zeros((2000, PAGE), dtype=np.uint8)
    npg, csz, st, handed = gpu.compress_tuples_pages_host(0, 1, data, off, ln, bf, rel, first, 301, 5)
    assert (st == 0).all() and len(handed) == int(npg.sum()) - 300
    h2d, _ = gpu.last_transfer_bytes()
    assert h2d <= h2d_bound(blocks, [128, 128, 44], cap_pages), h2d
    assert h2d < 300 * 32 * 1024                        # against 1 MiB per block for images
    # block 7 fails; the others are as the flush of their images, with the same block numbers
    off[int(bf[7]) + 3] = NONE
    rel_new = np.zeros((2000, PAGE), dtype=np.uint8)
    got = gpu.compress_tuples_pages_host(0, 1, data, off, ln, bf, rel_new, first, 301, 5)
    assert got[2][7] == 4 and got[0][7] == 0 and (np.delete(got[2], 7) == 0).all()
    assert not rel_new[8].any()                         # its reserved first page is not written
    keep = [i for i in range(300) if i != 7]
    rel_old = np.zeros((2000, PAGE), dtype=np.uint8)
    want = old_flush(gpu, 0, 1, np.stack([bg.pack_block(blocks[i]) for i in keep]), rel_old, first[keep], 301, 5)
    assert got[3] == want[3]
    assert np.array_equal(got[0][keep], want[0]) and np.array_equal(got[1][keep], want[1])
    assert np.array_equal(rel_new, rel_old)


def test_argument_errors(gpu):
    L, h = gpu.lib, gpu.handle
    data, off, ln, bf = pack_entries([[b"abc"]])
    alloc, page_ptr, _ = page_callbacks(np.zeros((4, PAGE), np.uint8), 2)
    out = np.zeros(4, np.uint32)
    st = np.zeros(4, np.int32)
    first = np.ones(1, np.uint32)

    def call(method=0, block_size=CRYO_BLCKSZ, bf_=bf, npages=out.ctypes.data, off_=off.ctypes.data):
        return L.cryogpu_compress_tuples_pages_alloc_host(h, 1, method, 1, data.ctypes.data, data.size, off_, ln.ctypes.data,
                                                          bf_.ctypes.data, block_size, first.ctypes.data, alloc, page_ptr,
                                                          None, 1, npages, out.ctypes.data, st.ctypes.data)
    assert call(method=5) == -4                         # CRYOGPU_E_METHOD
    assert call(block_size=CRYO_BLCKSZ - 4) == -2       # not a multiple of 8
    assert call(npages=None) == -2 and call(off_=None) == -2
    assert call(bf_=np.array([1, 0], np.uint64)) == -2  # block_first going backwards
    assert L.cryogpu_compress_tuples_pages_alloc_host(None, 1, 0, 1, data.ctypes.data, data.size, off.ctypes.data,
                                                      ln.ctypes.data, bf.ctypes.data, CRYO_BLCKSZ, first.ctypes.data, alloc,
                                                      page_ptr, None, 1, out.ctypes.data, out.ctypes.data, st.ctypes.data) == -2
    dev = _dev(gpu)
    d = torch.zeros(1 << 20, dtype=torch.uint8, device=dev)
    d8 = torch.zeros(16, dtype=torch.int64, device=dev)
    for bs, dst, stride in ((1020, d, 1024), (1024, d[1:], 1024), (1024, d, 1000), (1024, d, 1032)):
        assert L.cryogpu_build_blocks_device(h, 1, d.data_ptr(), 16, d8.data_ptr(), d8.data_ptr(), d8.data_ptr(), bs,
                                             dst.data_ptr(), stride, d8.data_ptr(), None) == -2, (bs, stride)
    assert L.cryogpu_build_blocks_device(h, 1, d.data_ptr(), 16, None, d8.data_ptr(), d8.data_ptr(), 1024, d.data_ptr(),
                                         1024, d8.data_ptr(), None) == -2
    assert L.cryogpu_build_blocks_device(h, 0, None, 0, None, None, None, 1024, None, 1024, None, None) == 0


def test_writer_end_to_end(gpu, blib):
    """Mixed lengths, tuples over 8 KiB and one that exactly fills its block, through cryo_batch_writer into cryo_memrel:
    the parent's item pointers, the pages of the flush of pack_block images, every tuple back by its TID."""
    rng = np.random.default_rng(4)
    tuples = []
    for i in range(6):
        k, p = KINDS[i]
        tuples += [bytes(r) for r in bg.make_tuples(k, p, 80 + i, 150 + 20 * i)]
        tuples += [bytes(rng.integers(0, 256, size=int(rng.integers(8193, 40000)), dtype=np.uint8)) for _ in range(3)]
    # a tuple that takes exactly the room left in its block (len + 8 == upper - lower)
    split = storage_split([len(t) for t in tuples])
    cur = [len(t) for t, (b, _) in zip(tuples, split) if b == split[-1][0]]
    room = CRYO_BLCKSZ - sum((x + 7) & ~7 for x in cur) - 8 - 8 * len(cur)
    assert room >= 8 and len(cur) < 290
    tuples += [bytes([0xAB]) * (room - 8), b"after the full block"]
    split = storage_split([len(t) for t in tuples])
    assert split[-1] == (split[-2][0] + 1, 1) and split[-2][1] == len(cur) + 1
    nblocks = split[-1][0] + 1
    batch = 3

    rel = blib.cryo_memrel_create(8000)
    ops = blib.cryo_memrel_ops(rel)
    blib.cryo_batch_writer_stats.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 3
    w = blib.cryo_batch_writer_create(gpu.handle, C.byref(ops), 1, 1, batch, 321)
    tids = []
    tb, tp = C.c_uint32(0), C.c_uint32(0)
    for t in tuples:
        assert blib.cryo_batch_insert(w, t, len(t), C.byref(tb), C.byref(tp)) == 0
        tids.append((tb.value, tp.value))
    assert blib.cryo_batch_flush(w) == 0
    h2d_last = gpu.last_transfer_bytes()[0]
    calls, nb_, pages = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    blib.cryo_batch_writer_stats(w, C.byref(calls), C.byref(nb_), C.byref(pages))
    blib.cryo_batch_writer_destroy(w)
    assert nb_.value == nblocks and calls.value == (nblocks + batch - 1) // batch
    # item pointers: storage_insert's arithmetic, and one first page per block
    firsts = [tids[[b for b, _ in split].index(k)][0] for k in range(nblocks)]
    assert [(firsts[b], p) for b, p in split] == tids

    # the parent's writer over the same tuples: block images, flushed `batch` at a time, pages numbered as it did
    per_block = [[t for t, (b, _) in zip(tuples, split) if b == k] for k in range(nblocks)]
    nbv = C.c_uint32(0)
    relation = np.ctypeslib.as_array(blib.cryo_memrel_pages(rel, C.byref(nbv)), shape=(8000, PAGE))
    want = np.zeros((8000, PAGE), dtype=np.uint8)
    nxt = 1
    for lo in range(0, nblocks, batch):
        ks = list(range(lo, min(lo + batch, nblocks)))
        assert [firsts[k] for k in ks] == list(range(nxt, nxt + len(ks)))
        nxt += len(ks)
        npg, _, st, handed = old_flush(gpu, 1, 1, np.stack([bg.pack_block(per_block[k]) for k in ks]), want,
                                       [firsts[k] for k in ks], nxt, 321)
        assert (st == 0).all()
        nxt += len(handed)
    assert nbv.value == nxt and np.array_equal(relation[:nxt], want[:nxt])
    last = per_block[(nblocks - 1) // batch * batch:]
    assert h2d_last <= h2d_bound(last, [len(last)], opg.pages_needed(compress_bound(1))), h2d_last

    # every tuple back by its TID
    tb_arr = np.array([b for b, _ in tids], dtype=np.uint32)
    tp_arr = np.array([p for _, p in tids], dtype=np.uint32)
    res = FetchResult()
    assert blib.cryo_batch_fetch_tuples(gpu.handle, C.byref(ops), tb_arr.ctypes.data, tp_arr.ctypes.data, len(tids),
                                        C.byref(res)) == 0
    for i, t in enumerate(tuples):
        assert res.err[i] == 0 and res.xid[i] == 321 and res.first[i + 1] - res.first[i] == 1
        assert C.string_at(res.tuple[res.first[i]], res.len[res.first[i]]) == t, i
    blib.cryo_fetch_result_free(C.byref(res))
    blib.cryo_memrel_destroy(rel)
