"""-m gpu: the page-chain calls on the device (cryogpu_{de,}compress_pages_{device,host},
cryogpu_compress_pages_alloc_host, cryogpu_decompress_pages_tuples_host) against the restated split and gather
(oracle/pages.py), the gather rules of tests/caller_model.py and the codecs.

  gather edges      streams of exact compressed sizes around every page boundary and the compressed-size bound, in
                    chains written by the reference's split; the decode must be what cryogpu_decompress_device gives
                    for the same stream, above the bound CHAIN
  split edges       compressed sizes T - 1, T, T + 1 at each boundary T, every page against the split of the stream
  chunks            batches around the 128-block chunk of the host calls, failing blocks at 127 and 128, a chunk of
                    empty chain lists, pageable / pinned / mixed destinations and sources, odd block sizes
  header fields     junk in the fields the gather does not read changes nothing; each field it reads, changed, gives
                    the restated gather's error
"""
import ctypes as C

import numpy as np
import pytest
import torch

import caller_model as cm
import tuple_oracle
from decode_vectors import _lz4_len, lz4_block, raw, zstd_frame
from gpu_util import decode_device, encode_device
from oracle import pages as opg
from oracle import ref
from pg_cryogen_b200 import CRYO_BLCKSZ
from pg_cryogen_b200.codec import ALLOC_PAGE_FN, PAGE_PTR_FN, compress_bound, pages_needed
from test_emu_tuples import random_block

pytestmark = pytest.mark.gpu
PAGE = 8192
FIRST, CONT = PAGE - 48, PAGE - 32
MAXC = max(ref.compress_bound(0), ref.compress_bound(1))
EDGES = [1, 15, 16, 17, FIRST - 1, FIRST, FIRST + 1] + [FIRST + CONT * k + d for k in (1, 2, 3) for d in (-1, 0, 1)]


def _rb(rng, k):
    return rng.integers(0, 256, size=k, dtype=np.uint8).tobytes()


def exact_streams(rng, T):
    """[(method, stream)] of exactly T bytes: a literal-only LZ4 block and / or a zstd frame of Raw blocks"""
    out = []
    for L in range(max(0, T - T // 255 - 4), T + 1):
        if 1 + L + (len(_lz4_len(L - 15)) if L >= 15 else 0) == T:
            out.append((0, lz4_block([], _rb(rng, L))[0]))
            break
    for L in range(max(0, T - 40 - 3 * (T // (128 << 10))), T + 1):
        data = _rb(rng, L)
        s = zstd_frame([raw(data[i:i + (128 << 10)]) for i in range(0, max(L, 1), 128 << 10)])[0]
        if s.size == T:
            out.append((1, s))
            break
        if s.size > T:
            break
    assert out, T
    return out


def _chains(rng, streams, spare=40):
    """the streams written by the reference's split into a relation, pages scattered -> (rel, chains, free pages)"""
    total = sum(opg.pages_needed(s.size) for _, s in streams)
    rel = np.zeros((total + spare + 1, PAGE), dtype=np.uint8)
    free = [int(x) for x in rng.permutation(np.arange(1, rel.shape[0]))]
    chains = []
    for i, (m, s) in enumerate(streams):
        ch = [free.pop() for _ in range(opg.pages_needed(s.size))]
        assert opg.split(rel, ch, s, m, 900 + i) == len(ch)
        chains.append(ch)
    return rel, chains, free


def _dev(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def pages_device(gpu, rel, chains, block_size=CRYO_BLCKSZ, rng=None, comp_size=True):
    """cryogpu_decompress_pages_device with the pages in HBM: every page of the chains in a permuted slot, stale pages
    between them -> (out, out_size, status, methods, comp_size or None)"""
    dev = torch.device("cuda", gpu.device)
    flat = [b for ch in chains for b in ch]
    n = len(chains)
    nslot = 2 * len(flat) + 3
    perm = rng.permutation(nslot)[: len(flat)]
    pages = rng.integers(0, 256, size=(nslot, PAGE), dtype=np.uint8)           # stale bytes in the unused slots
    pages[perm] = rel[flat]
    coff = np.zeros(n + 1, dtype=np.uint32)
    coff[1:] = np.cumsum([len(ch) for ch in chains])
    stride = (block_size + 15) & ~15
    d_pages, d_slot = _dev(pages, dev), _dev(perm.astype(np.int32), dev)
    d_blk, d_coff = _dev(np.array(flat + [0], dtype=np.uint32).view(np.int32), dev), _dev(coff.view(np.int32), dev)
    d_out = torch.full((n, stride), 0x5A, dtype=torch.uint8, device=dev)
    d_osz, d_st, d_me, d_cs = (torch.full((n,), -1, dtype=torch.int32, device=dev) for _ in range(4))
    s = torch.cuda.current_stream(dev).cuda_stream
    rc = gpu.lib.cryogpu_decompress_pages_device(gpu.handle, n, d_pages.data_ptr(), d_slot.data_ptr(), d_blk.data_ptr(),
                                                 d_coff.data_ptr(), max(len(flat), 1), d_out.data_ptr(), stride, block_size,
                                                 d_osz.data_ptr(), d_st.data_ptr(), d_me.data_ptr(),
                                                 d_cs.data_ptr() if comp_size else None, s or 1)
    assert rc == 0, gpu.lib.cryogpu_last_error()
    torch.cuda.synchronize(dev)
    cs = d_cs.cpu().numpy().view(np.uint32)
    return (d_out.cpu().numpy()[:, :block_size], d_osz.cpu().numpy().view(np.uint32), d_st.cpu().numpy(),
            d_me.cpu().numpy(), cs if comp_size else None)


def _same_decode(got, want, i):
    (o, osz, st), (wo, wosz, wst) = got, want
    assert st == wst, (i, st, wst)
    if st == 0:
        assert osz == wosz and np.array_equal(o[:osz], wo[:wosz]), i
    else:
        assert osz == 0 or st == wst, i


def test_gather_at_page_edges(gpu):
    rng = np.random.default_rng(1)
    streams = [ms for T in EDGES + [MAXC, MAXC + 1] for ms in exact_streams(rng, T)]
    sizes = [s.size for _, s in streams]
    assert set(sizes) == set(EDGES + [MAXC, MAXC + 1])
    rel, chains, _ = _chains(rng, streams)
    for i, ch in enumerate(chains):           # the reference's gather reads the stream back whole
        err, m, size, got, chain = opg.gather(rel, ch[0])
        assert err == 0 and size == sizes[i] and chain == ch and np.array_equal(got, streams[i][1]), i
    in_bound = [i for i, s in enumerate(sizes) if s <= MAXC]
    w_out, w_osz, w_st = decode_device(gpu, [streams[i][0] for i in in_bound], [streams[i][1] for i in in_bound])
    want = {i: (w_out[k], w_osz[k], w_st[k]) for k, i in enumerate(in_bound)}
    out, osz, st, me, cs = gpu.decompress_pages_host(rel, chains)
    # on the device: slots permuted, one block's chain named twice, stale pages between the slots, d_comp_size NULL
    twice = chains + [chains[len(chains) // 2]]
    d = pages_device(gpu, rel, twice, rng=rng)
    dn = pages_device(gpu, rel, twice, rng=rng, comp_size=False)
    assert dn[4] is None
    for i, (m, s) in enumerate(streams):
        for o, z, t, mm, c in ((out, osz, st, me, cs), d, (dn[0], dn[1], dn[2], dn[3], cs)):
            assert mm[i] == m, i
            if s.size > MAXC:
                assert t[i] == cm.ST_CHAIN and z[i] == 0 and c[i] == 0, (i, t[i])
                continue
            assert c[i] == s.size, i
            _same_decode((o[i], z[i], t[i]), want[i], i)
    j = len(chains) // 2
    assert d[2][-1] == d[2][j] and d[1][-1] == d[1][j] and np.array_equal(d[0][-1][: d[1][j]], d[0][j][: d[1][j]])


def test_split_at_page_edges(gpu):
    """Random prefixes before zeros, swept so that every edge T is hit at T - 1, T and T + 1 by the device encoders;
    every page is the reference's split of the stream cryogpu_compress_device makes of the same block."""
    rng = np.random.default_rng(2)
    dev = torch.device("cuda", gpu.device)
    edges = [T for T in EDGES if T >= FIRST - 1]
    noise = rng.integers(0, 256, size=CRYO_BLCKSZ, dtype=np.uint8)

    def blocks_for(prefixes):
        b = np.zeros((len(prefixes), CRYO_BLCKSZ), dtype=np.uint8)
        for k, p in enumerate(prefixes):
            b[k, :p] = noise[:p]
        return b

    hit = {T: set() for T in edges}
    for method in (0, 1):
        probe, _ = encode_device(gpu, method, 1, blocks_for(edges))
        prefixes = sorted({max(0, T - (probe[k].size - T)) + d for k, T in enumerate(edges) for d in range(-24, 24)})
        blocks = blocks_for(prefixes)
        streams, sst = encode_device(gpu, method, 1, blocks)
        assert (sst == 0).all()
        n = len(prefixes)
        mincap = pages_needed(compress_bound(method))
        for cap in (mincap, mincap + 3):
            blk = np.arange(1, n * cap + 1, dtype=np.uint32).reshape(n, cap)
            d_src = _dev(blocks, dev)
            d_blk = _dev(blk.view(np.int32), dev)
            d_pages = torch.full((n * cap, PAGE), 0xA5, dtype=torch.uint8, device=dev)
            d_np, d_cs, d_st = (torch.full((n,), -1, dtype=torch.int32, device=dev) for _ in range(3))
            s = torch.cuda.current_stream(dev).cuda_stream
            rc = gpu.lib.cryogpu_compress_pages_device(gpu.handle, n, method, 1, d_src.data_ptr(), CRYO_BLCKSZ, CRYO_BLCKSZ,
                                                       d_blk.data_ptr(), cap, 4242, d_pages.data_ptr(), d_np.data_ptr(),
                                                       d_cs.data_ptr(), d_st.data_ptr(), s or 1)
            assert rc == 0
            torch.cuda.synchronize(dev)
            pages = d_pages.cpu().numpy().reshape(n, cap, PAGE)
            npg, cs, st = d_np.cpu().numpy(), d_cs.cpu().numpy(), d_st.cpu().numpy()
            assert (st == 0).all()
            for k in range(n):
                assert cs[k] == streams[k].size and npg[k] == opg.pages_needed(cs[k]), k
                want = np.zeros((cap + 1, PAGE), dtype=np.uint8)
                opg.split(want, blk[k, : npg[k]] - blk[k, 0] + 1, streams[k], method, 4242)
                # the split writes block numbers relative to this row; the device's are the row's own
                row = pages[k, : npg[k]].copy()
                for j in range(npg[k]):
                    assert cm.u32(row[j], 24) == blk[k, 0]
                    assert cm.u32(row[j], 28) == (blk[k, j + 1] if j + 1 < npg[k] else cm.INVALID)
                    row[j, 24:32] = want[1 + j, 24:32]
                assert np.array_equal(row, want[1: 1 + npg[k]]), (method, cap, k)
                assert (pages[k, npg[k]:] == 0xA5).all(), (method, cap, k)      # unused pages keep their stale bytes
                for T in (int(cs[k]) - 1, int(cs[k]), int(cs[k]) + 1):
                    if T in hit:
                        hit[T].add(int(cs[k]) - T)
    missing = {T: sorted({-1, 0, 1} - h) for T, h in hit.items() if {-1, 0, 1} - h}
    assert not missing, missing


# ---- chunks and destinations -------------------------------------------------------------------------------------------

def encode_strided(gpu, method: int, blocks: np.ndarray, block_size: int):
    """cryogpu_compress_device at level 1 on [n, block_size] blocks, each in a slot of 16-byte stride"""
    dev = torch.device("cuda", gpu.device)
    n, stride = blocks.shape[0], (block_size + 15) & ~15
    src = np.zeros((n, stride), dtype=np.uint8)
    src[:, :block_size] = blocks
    bound = compress_bound(method, block_size)
    dstride = (bound + 15) & ~15
    d_src = _dev(src, dev)
    d_dst = torch.zeros((n, dstride), dtype=torch.uint8, device=dev)
    d_sz, d_st = (torch.full((n,), -1, dtype=torch.int32, device=dev) for _ in range(2))
    gpu.compress_device(method, 1, d_src, stride, d_dst, dstride, dstride, d_sz, d_st, n, block_size=block_size,
                        stream=torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    sz, out = d_sz.cpu().numpy().view(np.uint32), d_dst.cpu().numpy()
    return [out[i, : sz[i]].copy() for i in range(n)], d_st.cpu().numpy()


def lib_compress(method: int, data: np.ndarray) -> np.ndarray:
    """liblz4 / libzstd, as compression.c calls them, at any block size"""
    lz4, zstd = ref._syslibs()
    src = np.ascontiguousarray(data)
    dst = np.zeros(src.size + src.size // 200 + 1024, dtype=np.uint8)
    if method == 0:
        r = lz4.LZ4_compress_fast(src.ctypes.data, dst.ctypes.data, src.size, dst.size, 1)
    else:
        r = zstd.ZSTD_compress(dst.ctypes.data, dst.size, src.ctypes.data, src.size, 1)
    assert r > 0
    return dst[:r].copy()


class Pinned:
    """host memory from cryogpu_host_alloc, as numpy"""

    def __init__(self, gpu, nbytes):
        self.gpu, self.p = gpu, gpu.lib.cryogpu_host_alloc(nbytes)
        assert self.p
        self.a = np.ctypeslib.as_array(C.cast(self.p, C.POINTER(C.c_uint8)), shape=(nbytes,))

    def free(self):
        self.gpu.lib.cryogpu_host_free(self.p)


def _blocks(rng, n, block_size):
    """decoded blocks with valid item tables (zeros between lower and upper: they compress)"""
    out = np.zeros((n, block_size), dtype=np.uint8)
    for i in range(n):
        b = random_block(rng, block_size, block_size, "plain" if i % 9 else "many")
        lower, upper = (int(x) for x in b[:8].view(np.uint32))
        b[lower:upper] = 0
        out[i] = b
    return out


CHUNK_CASES = [(127, 1 << 20), (128, 65537), (129, 40001), (300, 65537), (300, 40001)]


@pytest.mark.parametrize("n,block_size", CHUNK_CASES)
def test_decompress_pages_host_chunks(gpu, n, block_size):
    rng = np.random.default_rng(n + block_size)
    plain = _blocks(rng, n, block_size)
    methods = [int(x) for x in rng.integers(0, 2, size=n)]
    streams = [(m, lib_compress(m, plain[i])) for i, m in enumerate(methods)]
    rel, chains, _ = _chains(rng, streams)
    fail = {}
    for i in (127, 128):
        if i < n and i == 127 and len(chains[i]) > 1:
            chains[i] = chains[i][:-1]                          # the walk ended early: CHAIN
            fail[i] = "chain"
        elif i < n:
            rel[chains[i][0], 36:40] = np.frombuffer(np.uint32(9).tobytes(), dtype=np.uint8)     # unknown method
            fail[i] = "method"
    if n > 256:
        for i in range(256, n):
            chains[i] = []                                      # a whole chunk of empty chain lists
    flat = [b for ch in chains for b in ch]
    coff = np.zeros(n + 1, dtype=np.uint32)
    coff[1:] = np.cumsum([len(ch) for ch in chains])
    blk = np.array(flat + [0], dtype=np.uint32)
    pagep = (C.c_void_p * max(len(flat), 1))(*[rel[b].ctypes.data for b in flat])
    w_unknown = decode_device(gpu, [9], [streams[0][1]])[2][0]
    # destinations: chunk 0 starts pinned with pageable ones in it, chunk 1 starts pageable with pinned ones in it
    pinned = Pinned(gpu, n * block_size)
    page_out = np.full((n, block_size), 0x77, dtype=np.uint8)
    pin_out = pinned.a.reshape(n, block_size)
    pin_out[:] = 0x77
    use_pin = [(i // 128 % 2 == 0) == (i % 3 != 1) for i in range(n)]
    dst = [pin_out[i] if use_pin[i] else page_out[i] for i in range(n)]
    try:
        dstp = (C.c_void_p * n)(*[d.ctypes.data for d in dst])
        osz = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        me = np.full(n, -1, dtype=np.int32)
        cs = np.full(n, 7, dtype=np.uint32)
        assert gpu.lib.cryogpu_decompress_pages_host(gpu.handle, n, pagep, blk.ctypes.data, coff.ctypes.data, dstp,
                                                     block_size, osz.ctypes.data, st.ctypes.data, me.ctypes.data,
                                                     cs.ctypes.data) == 0
        for i in range(n):
            if not chains[i]:
                assert (st[i], osz[i], me[i], cs[i]) == (cm.ST_EMPTY_BLOCK, 0, 0, 0), i
            elif fail.get(i) == "chain":
                assert (st[i], osz[i], me[i], cs[i]) == (cm.ST_CHAIN, 0, methods[i], 0), i
            elif fail.get(i) == "method":
                assert (st[i], me[i], cs[i]) == (w_unknown, 9, streams[i][1].size) and st[i] != 0, i
            else:
                assert (st[i], osz[i], me[i], cs[i]) == (0, block_size, methods[i], streams[i][1].size), i
                assert np.array_equal(dst[i], plain[i]), i
        # the same chains, tuples out (sel None: every item); failed blocks pass their status through
        got = gpu.decompress_pages_tuples_host(rel, chains, None, block_size=block_size)
        dec = plain.copy()
        dec[st != 0] = 0
        want = tuple_oracle.block_tuples(dec, None, st, block_size=block_size)
        for name, g, w in zip(("data", "tup_off", "tup_len", "block_first", "status", "need"), got[:6], want):
            assert (tuple(g) == w) if isinstance(w, tuple) else np.array_equal(np.asarray(g), w), name
        assert list(got[6]) == list(me) and list(got[7]) == list(cs)
    finally:
        pinned.free()


@pytest.mark.parametrize("n,block_size", CHUNK_CASES)
def test_compress_pages_host_chunks(gpu, n, block_size):
    rng = np.random.default_rng(3 * n + block_size)
    plain = _blocks(rng, n, block_size)
    for method in (0, 1):
        streams, sst = encode_strided(gpu, method, plain, block_size)
        assert (sst == 0).all()
        cap = pages_needed(compress_bound(method, block_size))
        # cryogpu_compress_pages_host: the caller's reserved rows, pages where they live
        rel = np.full((n * cap + 1, PAGE), 0xA5, dtype=np.uint8)
        blknos = (1 + rng.permutation(n * cap)).astype(np.uint32).reshape(n, cap)
        npg, cs, st = gpu.compress_pages_host(method, 1, plain, rel, blknos, created_xid=99, block_size=block_size)
        assert (st == 0).all()
        want = np.full_like(rel, 0xA5)
        for i in range(n):
            assert cs[i] == streams[i].size and npg[i] == opg.pages_needed(cs[i]), i
            opg.split(want, blknos[i, : npg[i]], streams[i], method, 99)
        assert np.array_equal(rel, want), method
        # cryogpu_compress_pages_alloc_host: first pages given, the others from alloc, block by block, page by page;
        # sources pinned in chunk 0 (with pageable ones in it) and pageable in chunk 1 (with pinned ones in it)
        pinned = Pinned(gpu, n * block_size)
        try:
            pin_src = pinned.a.reshape(n, block_size)
            pin_src[:] = plain
            src = [pin_src[i] if (i // 128 % 2 == 0) == (i % 4 != 2) else plain[i] for i in range(n)]
            first = np.arange(1, n + 1, dtype=np.uint32)
            rel2 = np.zeros((n * cap + 1, PAGE), dtype=np.uint8)
            handed = []

            def alloc(_a):
                handed.append(n + 1 + len(handed))
                return handed[-1]
            fa, fp = ALLOC_PAGE_FN(alloc), PAGE_PTR_FN(lambda _a, b: rel2[b].ctypes.data if b < rel2.shape[0] else None)
            srcp = (C.c_void_p * n)(*[s.ctypes.data for s in src])
            npg2, cs2, st2 = np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.full(n, -1, np.int32)
            assert gpu.lib.cryogpu_compress_pages_alloc_host(gpu.handle, n, method, 1, srcp, block_size, first.ctypes.data,
                                                             fa, fp, None, 77, npg2.ctypes.data, cs2.ctypes.data,
                                                             st2.ctypes.data) == 0
        finally:
            pinned.free()
        assert (st2 == 0).all() and list(cs2) == [s.size for s in streams] and list(npg2) == list(npg)
        want2, nxt = np.zeros_like(rel2), n + 1
        for i in range(n):
            chain = [int(first[i])] + list(range(nxt, nxt + int(npg2[i]) - 1))
            nxt += int(npg2[i]) - 1
            opg.split(want2, chain, streams[i], method, 77)
        assert handed == list(range(n + 1, nxt)), "alloc was not called block by block, page by page"
        assert np.array_equal(rel2, want2), method


# ---- header fields ---------------------------------------------------------------------------------------------------

def test_header_fields(gpu, oracle_ref):
    rng = np.random.default_rng(4)
    from pg_cryogen_b200 import blockgen as bg
    blocks = [bg.make_block("M", "hex", 40), bg.make_block("M", "lowcard", 41)]
    streams = [(m, oracle_ref.compress(m, 1, b)[0][0]) for m, b in zip((0, 1), blocks)]
    rel, chains, free = _chains(rng, streams)
    assert all(len(ch) >= 3 for ch in chains)
    junk = rel.copy()
    for ch in chains:
        for k, p in enumerate(ch):
            for off, w in ((0, 8), (8, 2), (12, 2), (16, 2), (18, 2)):     # pd_lsn, pd_checksum, pd_lower, special, version
                junk[p, off:off + w] = rng.integers(0, 256, size=w, dtype=np.uint8)
            if k == 0:
                junk[p, 44:46] = rng.integers(0, 256, size=2, dtype=np.uint8)   # npages
                junk[p, 32:36] = rng.integers(0, 256, size=4, dtype=np.uint8)   # created_xid
    clean = gpu.decompress_pages_host(rel, chains)
    assert (clean[2] == 0).all() and all(np.array_equal(clean[0][i], blocks[i]) for i in range(2))
    for got in (gpu.decompress_pages_host(junk, chains), pages_device(gpu, junk, chains, rng=rng)):
        for a, b in zip(got, clean):
            assert np.array_equal(a, b)

    def put(r, p, off, v, w=4):
        r[p, off:off + w] = np.frombuffer(int(v).to_bytes(w, "little"), dtype=np.uint8)

    ch0 = chains[0]
    cases = [("pd_upper", lambda r: put(r, ch0[0], 14, 0, 2)),
             ("first", lambda r: put(r, ch0[0], 24, ch0[1])),
             ("first of page 2", lambda r: put(r, ch0[1], 24, ch0[2])),
             ("next", lambda r: put(r, ch0[0], 28, free[0])),
             ("next of page 2", lambda r: put(r, ch0[1], 28, cm.INVALID)),
             ("method", lambda r: put(r, ch0[0], 36, 5)),
             ("compressed_size + 1", lambda r: put(r, ch0[0], 40, streams[0][1].size + 1)),
             ("compressed_size - 1", lambda r: put(r, ch0[0], 40, streams[0][1].size - 1)),
             ("compressed_size beyond the chain", lambda r: put(r, ch0[0], 40, len(ch0) * CONT + 200)),
             ("compressed_size beyond the bound", lambda r: put(r, ch0[0], 40, MAXC + 1))]
    for name, change in cases:
        r = rel.copy()
        change(r)
        want = cm.Outcome(r, r.shape[0], ch0[0]).err
        assert want != cm.ERR_SUCCESS, name
        for got in (gpu.decompress_pages_host(r, chains), pages_device(gpu, r, chains, rng=rng)):
            assert cm.fetch_error(got[2][0]) == want, (name, got[2][0], want)
            assert got[2][1] == 0 and np.array_equal(got[0][1], blocks[1]), name
