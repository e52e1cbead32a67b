"""A plain-Python model of the reference's callers around the codec (TEST INFRASTRUCTURE ONLY), for the scenarios of
tests/batch_scenarios.py that run pg_cryogen_b200/host/cryo_batch.c on the CPU stand-in and on the device.

  gather       pg_gather_block's rules (csrc/cryo_pages.cuh) over a relation [npages, 8192]: the reference's gather
               (cache.c:151-176, oracle/cryo_pages.c) follows `next` until compressed_size is covered and never reads
               npages; the device also checks `first` on every page and bounds compressed_size
  decode       liblz4 / libzstd, the calls compression.c:79-123 makes; a block is read when it decodes to CRYO_BLCKSZ
  cache        cryo_read_data (cache.c:244-297) request by request, with cryo_batch.c's LRU and per-call stamp
  scan         cryo_getnextslot's block loop (pg_cryogen.c:253-291) over the iterator of scan_iterator.c
  writer       cryo_storage_insert's counters (storage.c:26-50) and cryo_preserve's page allocation (pg_cryogen.c:588-805)
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from oracle import ref

BLCKSZ = 1 << 20
PAGE = 8192
INVALID = 0xFFFFFFFF
ERR_SUCCESS, ERR_DECOMPRESSION_FAILED, ERR_WRONG_STARTING_BLOCK, ERR_EMPTY_BLOCK, ERR_CACHE_IS_FULL = range(5)
# the device's per-block status (include/cryogpu.h) -> CryoError, as fetch_error in cryo_batch.c maps it
ST_OK, ST_EMPTY_BLOCK, ST_WRONG_START, ST_CHAIN = 0, 8, 9, 10


def fetch_error(status: int) -> int:
    return {ST_OK: ERR_SUCCESS, ST_EMPTY_BLOCK: ERR_EMPTY_BLOCK,
            ST_WRONG_START: ERR_WRONG_STARTING_BLOCK}.get(int(status), ERR_DECOMPRESSION_FAILED)


def u16(page, off: int) -> int:
    return int(page[off]) | int(page[off + 1]) << 8


def u32(page, off: int) -> int:
    return int(np.frombuffer(page[off:off + 4].tobytes(), dtype="<u4")[0])


def pages_needed(size: int) -> int:
    """cryo_pages_needed, pg_cryogen.c:692-704"""
    return 1 if size <= PAGE - 48 else 1 + (size - (PAGE - 48) + PAGE - 32 - 1) // (PAGE - 32)


def max_csize() -> int:
    """the compressed-size bound the device puts on a chain: the larger of the libraries' bounds for 1 MiB"""
    return max(ref.compress_bound(0), ref.compress_bound(1))


def gather(rel: np.ndarray, nrel: int, b: int):
    """-> (status, method, compressed_size, stream or None, chain) of the block whose first page is b (0 < b < nrel)"""
    pg = rel[b]
    if u16(pg, 14) == 0:
        return ST_EMPTY_BLOCK, 0, 0, None, [b]
    if u32(pg, 24) != b:
        return ST_WRONG_START, 0, 0, None, [b]
    method, cs = u32(pg, 36), u32(pg, 40)
    chain, need, cur = [b], pages_needed(cs), b
    while len(chain) < min(need, 132):
        cur = u32(rel[cur], 28)
        if cur == INVALID or cur >= nrel:
            break
        chain.append(cur)
    if cs > max_csize() or len(chain) < need or any(u32(rel[p], 24) != b for p in chain):
        return ST_CHAIN, method, cs, None, chain
    parts, left = [], cs
    for k, p in enumerate(chain):
        hdr = 48 if k == 0 else 32
        take = min(PAGE - hdr, left)
        parts.append(rel[p, hdr:hdr + take])
        left -= take
    return ST_OK, method, cs, np.concatenate(parts), chain


def ref_decode(method: int, stream: np.ndarray):
    """the block compression.c:79-123 makes of the stream, or None when it fails or is not CRYO_BLCKSZ bytes"""
    if method not in (0, 1):
        return None
    lz4, zstd = ref._syslibs()
    src = np.ascontiguousarray(stream, dtype=np.uint8)
    out = np.zeros(BLCKSZ, dtype=np.uint8)
    if method == 0:
        r = lz4.LZ4_decompress_safe(src.ctypes.data, out.ctypes.data, src.size, BLCKSZ)
    else:
        r = zstd.ZSTD_decompress(out.ctypes.data, BLCKSZ, src.ctypes.data, src.size)
        r = -1 if zstd.ZSTD_isError(r) else r
    return out if r == BLCKSZ else None


class Outcome:
    """what reading the block that starts at b gives: err, the decoded block, created_xid and the chain the reader
    walked (cache.c:39-40: pg_nblocks, pg_blocks)"""

    def __init__(self, rel: np.ndarray, nrel: int, b: int):
        self.data, self.xid, self.chain = None, 0, []
        if b == 0 or b >= nrel:
            self.err = ERR_WRONG_STARTING_BLOCK
            return
        st, method, _, stream, self.chain = gather(rel, nrel, b)
        if st == ST_OK:
            self.data = ref_decode(method, stream)
            st = ST_OK if self.data is not None else -1
        self.err = fetch_error(st)
        if self.err == ERR_SUCCESS:
            self.xid = u32(rel[b], 32)


class CacheModel:
    """cryo_read_data for n block numbers at a time, request by request, over nslots slots"""

    def __init__(self, rel: np.ndarray, nrel: int, nslots: int):
        self.rel, self.nrel = rel, nrel
        self.slot = [None] * nslots             # [block, ts] or None
        self.clock = self.calls = self.blocks = self.hits = 0
        self._outcome = {}

    def outcome(self, b: int) -> Outcome:
        if b not in self._outcome:
            self._outcome[b] = Outcome(self.rel, self.nrel, b)
        return self._outcome[b]

    def _take(self, stamp: int):
        """a free slot, else the least recently used one this call has not touched (cache.c:184-230)"""
        best = None
        for i, s in enumerate(self.slot):
            if s is None:
                return i
            if s[1] < stamp and (best is None or s[1] < self.slot[best][1]):
                best = i
        return best

    def read_data(self, blocknos):
        """-> [(err, entry)] per request"""
        self.clock += 1
        stamp = self.clock
        res, first_miss, misses = [], {}, []
        for i, b in enumerate(blocknos):
            if b == 0 or b >= self.nrel:                    # cache.c:256-260
                res.append([ERR_WRONG_STARTING_BLOCK, -1])
                continue
            if b in first_miss:                             # a repeat of this call's miss: its outcome, not a hit
                res.append(None)
                continue
            e = next((k for k, s in enumerate(self.slot) if s is not None and s[0] == b), None)
            if e is not None:
                self.slot[e][1] = stamp
                self.hits += 1
                res.append([ERR_SUCCESS, e])
                continue
            e = self._take(stamp)
            if e is None:
                res.append([ERR_CACHE_IS_FULL, -1])        # cache.c:272-273
                continue
            self.slot[e] = [b, stamp]
            first_miss[b] = i
            misses.append(i)
            res.append([ERR_SUCCESS, e])
        if misses:
            self.calls += 1
            self.blocks += len(misses)
        for i in misses:
            o = self.outcome(blocknos[i])
            if o.err != ERR_SUCCESS:
                self.slot[res[i][1]] = None                 # cache.c:283-286
                res[i] = [o.err, -1]
        return [tuple(r) if r is not None else tuple(res[first_miss[blocknos[i]]]) for i, r in enumerate(res)]


def scan(rel: np.ndarray, nrel: int):
    """The blocks a sequential scan returns, in order, and (err, block) of the error that ends it (None at the end):
    pages of an earlier block's chain are not starting pages, EMPTY_BLOCK is skipped (pg_cryogen.c:268-272)"""
    excluded, out = set(), []
    for b in range(1, nrel):
        if b in excluded:
            continue
        pg = rel[b]
        if u16(pg, 14) != 0 and u32(pg, 24) == b:
            need, nb, k = pages_needed(u32(pg, 40)), u32(pg, 28), 1
            while k < need and nb != INVALID and nb < nrel:
                excluded.add(nb)
                nb = u32(rel[nb], 28)
                k += 1
        o = Outcome(rel, nrel, b)
        if o.err == ERR_EMPTY_BLOCK:
            continue
        if o.err != ERR_SUCCESS:
            return out, (o.err, b)
        out.append(b)
    return out, None


class WriterModel:
    """cryo_batch_insert / cryo_batch_flush: which block each tuple goes to, its item pointer, and the page numbers
    the relation hands out (a block's first page when it is started, pg_cryogen.c:588-601; the others when its batch
    is flushed, block by block, pages_needed(compressed_size) - 1 each, pg_cryogen.c:737-759)"""

    def __init__(self, batch: int):
        self.batch = batch
        self.blocks = []            # per block: [first page, [tuples], [further pages]]; pages are set by allocate()
        self.queued, self.cur = [], None
        self.lower = self.upper = 0
        self.items = []             # per insert: (block index, pos) or None (the writer returned -1)
        self.events = []            # ("start", block) / ("flush", [blocks]) in the order they happen

    def _start(self):
        self.blocks.append([None, [], None])
        self.cur = len(self.blocks) - 1
        self.lower, self.upper = 8, BLCKSZ
        self.events.append(("start", self.cur))

    def _insert(self, t: bytes) -> int:
        if len(t) + 8 > self.upper - self.lower or (self.lower - 8) // 8 + 1 >= 291:
            return -1
        self.upper -= (len(t) + 7) & ~7
        self.blocks[self.cur][1].append(t)
        self.lower += 8
        return (self.lower - 8) // 8

    def insert(self, t: bytes):
        if self.cur is None:
            self._start()
        pos = self._insert(t)
        if pos < 0:
            self.queued.append(self.cur)
            self.cur = None
            if len(self.queued) == self.batch:
                self.events.append(("flush", self.queued))
                self.queued = []
            self._start()
            pos = self._insert(t)
            if pos < 0:
                self.items.append(None)
                return
        self.items.append((self.cur, pos))

    def flush(self):
        q = self.queued + ([self.cur] if self.cur is not None else [])
        if q:
            self.events.append(("flush", q))
        self.queued, self.cur = [], None

    def allocate(self, csize_of, first: int = 1):
        """Replay the page allocation from page `first` on; csize_of(page) is the compressed_size the written first
        page holds.  Sets every block's pages and returns the page numbers in the order they were handed out."""
        page, order = first, []
        for kind, what in self.events:
            if kind == "start":
                self.blocks[what][0] = page
                order.append(page)
                page += 1
                continue
            for k in what:
                extra = list(range(page, page + pages_needed(csize_of(self.blocks[k][0])) - 1))
                self.blocks[k][2] = extra
                order += extra
                page += len(extra)
        return order

    def tids(self):
        """the item pointers of the inserts (first page of the block, position), None for a -1; after allocate()"""
        return [None if it is None else (self.blocks[it[0]][0], it[1]) for it in self.items]


def block_items(block: np.ndarray):
    """(lower, upper, [(off, len)]) of a decoded cryo block (storage.h:69-86)"""
    w = block[: 8].view("<u4")
    lower, upper = int(w[0]), int(w[1])
    n = (lower - 1) // 8 if lower else 0
    it = block[8: 8 + 8 * n].view("<u4").reshape(-1, 2)
    return lower, upper, [(int(o), int(l)) for o, l in it]


def c_u8(ptr, n: int) -> np.ndarray:
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(n,))
