"""The scenarios of the batched callers in pg_cryogen_b200/host/cryo_batch.c (TEST INFRASTRUCTURE ONLY), run by
tests/test_batch_callers.py on the CPU stand-in of the codec calls (tests/cryogpu_stub.c) and by
tests/test_gpu_batch_callers.py on libcryo_batch.so and the device.  Every result is checked against the model of the
reference's callers in tests/caller_model.py, the restated gather and the reference's codec.

  cache    relations of cryo blocks of every blockgen kind and both methods, with faulty blocks among them; seeded
           sequences of cryo_batch_read_data calls with repeats, hits and misses mixed
  scan     the sequential scan with read-ahead over chains laid out the way the batched writer lays them out
  writer   COPY through the batched writer at the edges of storage.c's counters, every page checked
  fetch    the TID fetch over the faulty relation
"""
from __future__ import annotations

import ctypes as C
import functools
import os

import numpy as np

import caller_model as cm
import tuple_oracle
from oracle import pages as opg
from oracle import ref
from pg_cryogen_b200 import blockgen as bg

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PAGE, BLCKSZ = cm.PAGE, cm.BLCKSZ
XID = 4711


class RelOps(C.Structure):
    _fields_ = [("rel", C.c_void_p), ("nblocks", C.c_void_p), ("read_page", C.c_void_p), ("extend", C.c_void_p)]


class FetchResult(C.Structure):
    _fields_ = [("err", C.POINTER(C.c_int)), ("xid", C.POINTER(C.c_uint32)), ("first", C.POINTER(C.c_uint64)),
                ("tuple", C.POINTER(C.c_void_p)), ("len", C.POINTER(C.c_uint32)), ("ntuples", C.c_uint64),
                ("calls", C.c_uint64), ("data_", C.c_void_p), ("tup_off_", C.c_void_p), ("tup_len_", C.c_void_p)]


_NBLOCKS = C.CFUNCTYPE(C.c_uint32, C.c_void_p)
_READ = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_uint32)
_EXTEND = C.CFUNCTYPE(C.c_uint32, C.c_void_p)


class Relation:
    """the buffer manager as CryoRelOps sees it, over pages [cap, 8192]: nblocks, read_page, extend (a zeroed page)"""

    def __init__(self, pages: np.ndarray, nblocks: int):
        self.pages, self.n = pages, nblocks
        self.base = pages.ctypes.data
        self._cb = (_NBLOCKS(lambda _r: self.n), _READ(self._read), _EXTEND(self._extend))
        self.ops = RelOps(None, *[C.cast(f, C.c_void_p) for f in self._cb])

    def _read(self, _r, b):
        return self.base + b * PAGE if b < self.n else None

    def _extend(self, _r):
        if self.n >= self.pages.shape[0]:
            return cm.INVALID
        self.pages[self.n] = 0
        self.n += 1
        return self.n - 1


def bind(L):
    """the argument types of cryo_batch.h on a library that has it"""
    P = C.c_void_p
    for name, res, args in (
            ("cryo_batch_cache_create", P, [P, C.c_int]), ("cryo_batch_cache_destroy", None, [P]),
            ("cryo_batch_read_data", C.c_int, [P, C.POINTER(RelOps), P, C.c_int, P, P]),
            ("cryo_batch_get_data", P, [P, C.c_int]), ("cryo_batch_get_xid", C.c_uint32, [P, C.c_int]),
            ("cryo_batch_get_pg_nblocks", C.c_uint32, [P, C.c_int]),
            ("cryo_batch_get_pg_blocks", C.POINTER(C.c_uint32), [P, C.c_int]),
            ("cryo_batch_cache_stats", None, [P] + [C.POINTER(C.c_uint64)] * 3),
            ("cryo_batch_scan_begin", P, [P, C.POINTER(RelOps), C.c_int]),
            ("cryo_batch_scan_next", P, [P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_int)]),
            ("cryo_batch_scan_end", None, [P]),
            ("cryo_batch_fetch_tuples", C.c_int, [P, C.POINTER(RelOps), P, P, C.c_int, C.POINTER(FetchResult)]),
            ("cryo_fetch_result_free", None, [C.POINTER(FetchResult)]),
            ("cryo_batch_writer_create", P, [P, C.POINTER(RelOps), C.c_int, C.c_int, C.c_int, C.c_uint32]),
            ("cryo_batch_insert", C.c_int, [P, P, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
            ("cryo_batch_flush", C.c_int, [P]),
            ("cryo_batch_writer_stats", None, [P] + [C.POINTER(C.c_uint64)] * 3),
            ("cryo_batch_writer_destroy", None, [P])):
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    return L


def stub_library():
    """cryo_batch.c built against the CPU stand-in of its five libcryogpu calls (tests/cryogpu_stub.c), once per
    process, into a temporary directory"""
    src = [os.path.join(HERE, "cryogpu_stub.c"), os.path.join(ROOT, "pg_cryogen_b200", "host", "cryo_batch.c"),
           os.path.join(ROOT, "oracle", "cryo_oracle.c"), os.path.join(HERE, "tuple_oracle.c")]
    inc = ["include", "pg_cryogen_b200/host", "oracle", "pg_shim"]
    return bind(tuple_oracle.build("libcryo_batch_stub.so", [
        "gcc", "-O2", "-fPIC", "-Wall", "-Wno-unused-function", "-std=c11", "-shared",
        *["-I" + os.path.join(ROOT, d) for d in inc], *src, "-l:liblz4.so.1", "-l:libzstd.so.1"]))


class Backend:
    """a cryo_batch library and the context its calls take (None for the stand-in)"""

    def __init__(self, lib, ctx):
        self.L, self.ctx = lib, ctx


# ---- relations -----------------------------------------------------------------------------------------------------

KINDS = [(k, p) for k in "SMD" for p in bg.PAYLOADS]
FAULTS = ("unwritten", "cut", "foreign", "corrupt", "method", "npages0", "npages1", "npagesFFFF")


def _put(rel, b, off, v, width=4):
    rel[b, off:off + width] = np.frombuffer(int(v).to_bytes(width, "little"), dtype=np.uint8)


@functools.lru_cache(maxsize=None)
def relation(seed: int, nblocks: int, faults: tuple, batch: int = 4):
    """A relation of nblocks cryo blocks (every blockgen kind, both methods, a few small and all-zero ones) written the
    way the batched writer lays them out: per batch of `batch` blocks the first pages, then the further pages block by
    block.  faults: which of FAULTS to plant, each on its own block.  -> (pages [n, 8192], n, {fault: block}, firsts)"""
    rng = np.random.default_rng(seed)
    plain, methods = [], []
    for j in range(nblocks):
        kind, pl = KINDS[j % len(KINDS)]
        if j % 11 == 5:
            plain.append(np.zeros(BLCKSZ, dtype=np.uint8))
        else:
            nt = None if j % 7 else int(rng.integers(1, 40))
            plain.append(bg.make_block(kind, pl, seed * 1000 + j, ntuples=nt))
        methods.append(int(rng.integers(0, 2)))
    comp = [ref.compress(m, 1, b)[0][0] for m, b in zip(methods, plain)]
    if "unwritten" in faults:
        comp[nblocks // 2] = None                       # a reserved first page the flush never wrote
    total = 1 + sum(1 if c is None else opg.pages_needed(c.size) for c in comp)
    rel = np.zeros((total, PAGE), dtype=np.uint8)
    page, firsts, chains = 1, [], [None] * nblocks
    for b0 in range(0, nblocks, batch):
        idx = range(b0, min(b0 + batch, nblocks))
        for i in idx:
            firsts.append(page)
            chains[i] = [page]
            page += 1
        for i in idx:
            if comp[i] is not None:
                k = opg.pages_needed(comp[i].size) - 1
                chains[i] += list(range(page, page + k))
                page += k
                assert opg.split(rel, chains[i], comp[i], methods[i], XID + i) == len(chains[i])
    assert page == total
    # the faults, each on a block of its own (multi-page where the fault needs it), late in the relation
    multi = [i for i in range(nblocks) if comp[i] is not None and len(chains[i]) >= 4][::-1]
    where = {}
    if "unwritten" in faults:
        where["unwritten"] = firsts[nblocks // 2]
    for f in sorted(FAULTS[1:], key=lambda f: f != "corrupt"):    # the corrupt block last in the relation
        if f not in faults:
            continue
        i = multi.pop(0)
        ch, where[f] = chains[i], chains[i][0]
        if f == "cut":
            _put(rel, ch[1], 28, cm.INVALID)            # the walk ends after two pages
        elif f == "foreign":
            other = next(c for c in chains if c is not None and c is not ch and len(c) >= 3)
            _put(rel, ch[1], 28, other[2])              # `next` names a page of another block's chain
        elif f == "corrupt":
            # a stream byte the reference's decoder rejects (a byte of the first page's payload)
            for pos in rng.permutation(min(comp[i].size, PAGE - 48)):
                rel[ch[0], 48 + pos] ^= 0x5A
                st, m, _, stream, _ = cm.gather(rel, total, ch[0])
                if cm.ref_decode(m, stream) is None:
                    break
                rel[ch[0], 48 + pos] ^= 0x5A
            else:
                raise AssertionError("no byte of the stream breaks it")
        elif f == "method":
            _put(rel, ch[0], 36, 7)                     # an unknown compression method in the header
        else:
            _put(rel, ch[0], 44, {"npages0": 0, "npages1": 1, "npagesFFFF": 0xFFFF}[f], 2)
    rel.setflags(write=False)
    return rel, total, where, firsts, chains


def _writable(rel: np.ndarray) -> np.ndarray:
    return np.array(rel)


# ---- cache -----------------------------------------------------------------------------------------------------------

def _pick(rng, pool, call):
    """a block number for the next request: a repeat within the call, a recent block (a likely hit), or any of pool"""
    r = rng.random()
    if call and r < 0.25:
        return call[int(rng.integers(0, len(call)))]
    return pool[int(rng.integers(0, len(pool)))]


def run_cache(be: Backend, nslots: int, seed: int, ncalls: int = 36):
    pages, n, where, firsts, chains = relation(1, 40, FAULTS)
    rel = Relation(_writable(pages), n)
    model = cm.CacheModel(pages, n, nslots)
    conts = [ch[1] for ch in chains if len(ch) > 1][:3]
    bad = list(where.values()) + conts + [0, n, n + 7]
    rng = np.random.default_rng([seed, nslots])
    L = be.L
    cache = L.cryo_batch_cache_create(be.ctx, nslots)
    assert cache
    try:
        recent = []
        for k in range(ncalls):
            length = int(rng.integers(1, nslots + 4))
            pool = (recent[-2 * nslots:] or firsts) if rng.random() < 0.4 else firsts + bad
            call = []
            for _ in range(length):
                call.append(int(_pick(rng, pool if rng.random() < 0.8 else bad, call)))
            recent += call
            ask = np.array(call, dtype=np.uint32)
            ent = np.full(len(call), -7, dtype=np.int32)
            errs = np.full(len(call), -7, dtype=np.int32)
            assert L.cryo_batch_read_data(cache, C.byref(rel.ops), ask.ctypes.data, len(call), ent.ctypes.data,
                                          errs.ctypes.data) == 0
            want = model.read_data(call)
            assert [int(e) for e in errs] == [w[0] for w in want], (k, call, list(errs), want)
            assert [int(e) for e in ent] == [w[1] for w in want], (k, call, list(ent), want)
            for i, b in enumerate(call):
                if errs[i] != cm.ERR_SUCCESS:
                    continue
                o = model.outcome(b)
                e = int(ent[i])
                assert all(ent[j] == e for j in range(len(call)) if call[j] == b)      # one entry per block
                assert np.array_equal(cm.c_u8(L.cryo_batch_get_data(cache, e), BLCKSZ), o.data), (k, i, b)
                assert L.cryo_batch_get_xid(cache, e) == o.xid
                nb = L.cryo_batch_get_pg_nblocks(cache, e)
                assert nb == len(o.chain) and list(L.cryo_batch_get_pg_blocks(cache, e)[:nb]) == o.chain, (b, nb)
            st = [C.c_uint64(0) for _ in range(3)]
            L.cryo_batch_cache_stats(cache, *[C.byref(s) for s in st])
            assert [s.value for s in st] == [model.calls, model.blocks, model.hits], k
    finally:
        L.cryo_batch_cache_destroy(cache)
    return model


def repeat_case(be: Backend):
    """read_data([b, b]) for a reserved page never written, a corrupt block and a good one, in one call and after a
    hit: each request gets its block's outcome, and one slot"""
    pages, n, where, firsts, _ = relation(1, 40, FAULTS)
    rel = Relation(_writable(pages), n)
    good = firsts[1]
    L = be.L
    for nslots in (1, 2, 4):
        model = cm.CacheModel(pages, n, nslots)
        cache = L.cryo_batch_cache_create(be.ctx, nslots)
        try:
            for call in ([where["unwritten"]] * 2, [where["corrupt"], good, where["corrupt"]], [good, good],
                         [where["npages0"], where["npages0"], good], [good, where["cut"], where["cut"], good]):
                ask = np.array(call, dtype=np.uint32)
                ent = np.full(len(call), -7, dtype=np.int32)
                errs = np.full(len(call), -7, dtype=np.int32)
                assert L.cryo_batch_read_data(cache, C.byref(rel.ops), ask.ctypes.data, len(call), ent.ctypes.data,
                                              errs.ctypes.data) == 0
                want = model.read_data(call)
                assert [(int(e), int(x)) for e, x in zip(errs, ent)] == want, (nslots, call)
            st = [C.c_uint64(0) for _ in range(3)]
            L.cryo_batch_cache_stats(cache, *[C.byref(s) for s in st])
            assert [s.value for s in st] == [model.calls, model.blocks, model.hits]
        finally:
            L.cryo_batch_cache_destroy(cache)


# ---- scan ------------------------------------------------------------------------------------------------------------

def run_scan(be: Backend, nslots: int, readahead: int):
    pages, n, where, _, _ = relation(2, 36, ("unwritten", "corrupt", "npages0", "npages1", "npagesFFFF"), 3)
    rel = Relation(_writable(pages), n)
    want, end = cm.scan(pages, n)
    assert end is not None and end[0] == cm.ERR_DECOMPRESSION_FAILED and end[1] == where["corrupt"]
    assert where["unwritten"] < end[1] and where["unwritten"] not in want
    L = be.L
    cache = L.cryo_batch_cache_create(be.ctx, nslots)
    scan = L.cryo_batch_scan_begin(cache, C.byref(rel.ops), readahead)
    try:
        got = []
        bno, xid, err = C.c_uint32(0), C.c_uint32(0), C.c_int(-7)
        while True:
            d = L.cryo_batch_scan_next(scan, C.byref(bno), C.byref(xid), C.byref(err))
            if not d:
                break
            o = cm.Outcome(pages, n, bno.value)
            assert o.err == cm.ERR_SUCCESS and np.array_equal(cm.c_u8(d, BLCKSZ), o.data), bno.value
            assert xid.value == o.xid
            got.append(bno.value)
        assert got == want
        assert (err.value, bno.value) == end
    finally:
        L.cryo_batch_scan_end(scan)
        L.cryo_batch_cache_destroy(cache)


# ---- writer ----------------------------------------------------------------------------------------------------------

def writer_tuples(model: cm.WriterModel, seed: int, big: int):
    """Tuples at the edges of storage.c's counters, fed to the model as they are made (the exact fits depend on the
    counters): 1 byte up to the 290-item limit and one past it, 8 191 bytes, a tuple that leaves upper - lower exactly
    len + 8 and one a byte longer, a tuple no empty block takes, and `big` tuples of 1 MiB - 16 bytes."""
    rng = np.random.default_rng(seed)
    out = []

    def add(t):
        out.append(t)
        model.insert(t)

    rb = lambda k: rng.integers(0, 256, size=k, dtype=np.uint8).tobytes()     # noqa: E731
    for i in range(291):
        add(bytes([i & 0xFF]))                          # 290 items fill a block; the 291st starts the next
    for i in range(3):
        add(rb(8191))
    add(rb(model.upper - model.lower - 8))              # upper - lower == len + 8: the tuple fits exactly
    add(b"z")                                           # nothing is left: a new block
    add(rb(model.upper - model.lower - 7))              # one byte too long: a new block
    add(rb(BLCKSZ - 15))                                # too large for an empty block: -1
    for i in range(130):
        add(rb(8191))
    for i in range(big):
        # a random prefix, then a pattern: chains of one page up to many
        k = int(rng.integers(0, 3 * PAGE)) if i % 5 else int(rng.integers(0, BLCKSZ - 16))
        body = rb(k) + bytes([(i * 7 + j) & 0xFF for j in range(61)]) * ((BLCKSZ - 16 - k) // 61 + 1)
        add(body[: BLCKSZ - 16])
    add(rb(BLCKSZ - 16))
    add(bytes(range(200)))
    return out


def run_writer(be: Backend, method: int, batch: int, big: int):
    model = cm.WriterModel(batch)
    tuples = writer_tuples(model, 31 * batch + method, big)
    model.flush()
    cap = 1 + len(model.blocks) * cm.pages_needed(cm.max_csize())
    rel = Relation(np.zeros((cap, PAGE), dtype=np.uint8), 1)
    L = be.L
    w = L.cryo_batch_writer_create(be.ctx, C.byref(rel.ops), method, 1, batch, XID)
    assert w
    got = []
    tb, tp = C.c_uint32(0), C.c_uint32(0)
    try:
        for t in tuples:
            rc = L.cryo_batch_insert(w, t, len(t), C.byref(tb), C.byref(tp))
            assert rc in (0, -1)
            got.append((tb.value, tp.value) if rc == 0 else None)
        assert L.cryo_batch_flush(w) == 0
        st = [C.c_uint64(0) for _ in range(3)]
        L.cryo_batch_writer_stats(w, *[C.byref(s) for s in st])
    finally:
        L.cryo_batch_writer_destroy(w)
    pages, n = rel.pages, rel.n
    order = model.allocate(lambda b: cm.u32(pages[b], 40))
    assert got == model.tids()
    assert order == list(range(1, n)), "pages were handed out in another order"
    nflush = sum(1 for e in model.events if e[0] == "flush")
    assert [s.value for s in st] == [nflush, len(model.blocks), n - 1]
    want = np.zeros_like(pages[:n])
    for i, (first, tups, extra) in enumerate(model.blocks):
        err, m, size, stream, chain = opg.gather(pages[:n], first)
        assert err == opg.ERR_SUCCESS and m == method and chain == [first] + extra, i
        assert cm.u32(pages[first], 32) == XID
        back = cm.ref_decode(method, stream)
        assert back is not None and np.array_equal(back, bg.pack_block(tups)), i
        opg.split(want, chain, stream, method, XID)
    bad = np.flatnonzero((pages[:n] != want).any(axis=1))
    assert bad.size == 0, f"pages differ from the split of their streams (or are not zero): {bad[:8]}"
    return model


# ---- TID fetch -------------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def _fetch_want(b: int, pos: int):
    """(err, xid, [tuple bytes or None]) the fetch must give for (b, pos), from the model and tuple_oracle"""
    pages, n, *_ = relation(1, 40, FAULTS)
    o = cm.Outcome(pages, n, b)
    if o.err != cm.ERR_SUCCESS:
        return o.err, 0, []
    data, to, tl, bf, st, _ = tuple_oracle.block_tuples(o.data[None], [[pos]])
    if st[0] != 0:
        return cm.fetch_error(int(st[0])), 0, []
    return cm.ERR_SUCCESS, o.xid, [None if off == 0xFFFFFFFFFFFFFFFF else data[off:off + ln].tobytes()
                                   for off, ln in zip(to, tl)]


def run_fetch(be: Backend, seed: int):
    pages, n, where, firsts, chains = relation(1, 40, FAULTS)
    rel = Relation(_writable(pages), n)
    rng = np.random.default_rng(seed)
    bad = list(where.values()) + [next(ch[1] for ch in chains if len(ch) > 1), 0, n, n + 9]
    pick = []
    for _ in range(300):
        b = firsts[int(rng.integers(0, len(firsts)))] if rng.random() < 0.8 else bad[int(rng.integers(0, len(bad)))]
        r = rng.random()
        pos = 0 if r < 0.05 else int(rng.integers(290, 300)) if r < 0.1 else 0xFFFFFFFF if r < 0.12 \
            else int(rng.integers(1, 41))
        pick.append((b, pos))
    pick += pick[:40] + [(b, 1) for b in bad]
    pick = [pick[int(i)] for i in rng.permutation(len(pick))]
    tb = np.array([b for b, _ in pick], dtype=np.uint32)
    tp = np.array([p for _, p in pick], dtype=np.uint32)
    res = FetchResult()
    assert be.L.cryo_batch_fetch_tuples(be.ctx, C.byref(rel.ops), tb.ctypes.data, tp.ctypes.data, len(pick),
                                        C.byref(res)) == 0
    try:
        for i, (b, p) in enumerate(pick):
            err, xid, tups = _fetch_want(b, p)
            lo, hi = res.first[i], res.first[i + 1]
            assert res.err[i] == err, (b, p, res.err[i], err)
            assert hi - lo == len(tups), (b, p)
            if err != cm.ERR_SUCCESS:
                continue
            assert res.xid[i] == xid
            for j, t in enumerate(tups):
                ptr, ln = res.tuple[lo + j], res.len[lo + j]
                if t is None:
                    assert not ptr and ln == 0, (b, p)
                else:
                    assert ptr % 8 == 0 and C.string_at(ptr, ln) == t, (b, p, j)
        kinds = {_fetch_want(b, p)[0] for b, p in pick}
        assert kinds >= {cm.ERR_SUCCESS, cm.ERR_DECOMPRESSION_FAILED, cm.ERR_WRONG_STARTING_BLOCK, cm.ERR_EMPTY_BLOCK}
    finally:
        be.L.cryo_fetch_result_free(C.byref(res))
