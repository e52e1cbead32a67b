"""-m gpu: the encoders' contract on the device, beyond heap-tuple blocks.

Every call here puts its blocks in strided slots: a source slot of roundup16(n) + 4 KiB whose padding continues the
block's own pattern (a read past n finds what looks like more of a match), and a destination slot of
roundup16(bound) + 4 KiB with dst_cap = cryogpu_compress_bound exactly, pre-filled with a sentinel.  After every call:
every status is 0, every stream passes the format checkers of tests/encode_check.py (the end-of-block rules, the
block headers, the bound, then liblz4 / libzstd and the plain-C restatement restore the block), nothing is written
past dst_cap and the source is unchanged.  Then: a block's stream is the same alone and inside large shuffled mixed
batches, the device decoder reads every stream back, and the host calls (two lanes, pinned, pageable and mixed
sources, multi-context, page chains) write what the device call writes.  No ratio is asserted beyond the bound and
one cheap guard on one-byte runs (DESIGN.md section 1 promises its tolerance for heap-tuple blocks only)."""
import ctypes as C

import numpy as np
import pytest
import torch

import encode_check as ec
from oracle import pages as opg
from pg_cryogen_b200 import COMP_LZ4, COMP_ZSTD, CRYO_BLCKSZ, CryoGPU
from pg_cryogen_b200.codec import compress_bound, pages_needed

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5
PAD = 4096


def _r16(v):
    return (v + 15) & ~15


def _slots(srcs, n):
    """[k, roundup16(n) + PAD] source slots: each block followed by the continuation of its pattern"""
    ss = _r16(n) + PAD
    out = np.empty((len(srcs), ss), dtype=np.uint8)
    for i, s in enumerate(srcs):
        out[i] = s[:ss] if s.size >= ss else np.resize(s, ss)
    return out


def encode(gpu, method, level, slots, n):
    """cryogpu_compress_device over the source slots [k, src_stride].  Returns the streams; asserts status 0, the
    sentinels in [dst_cap, dst_stride) of every slot and an unchanged source."""
    k, ss = slots.shape
    cap = compress_bound(method, n)
    ds = _r16(cap) + PAD
    dev = torch.device("cuda", gpu.device)
    d_src = torch.from_numpy(slots).to(dev)
    d_dst = torch.full((k, ds), SENTINEL, dtype=torch.uint8, device=dev)
    d_sz = torch.full((k,), -1, dtype=torch.int32, device=dev)
    d_st = torch.full((k,), -1, dtype=torch.int32, device=dev)
    gpu.compress_device(method, level, d_src, ss, d_dst, ds, cap, d_sz, d_st, k, block_size=n,
                        stream=torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    st = d_st.cpu().numpy()
    assert (st == 0).all(), st
    dst = d_dst.cpu().numpy()
    assert (dst[:, cap:] == SENTINEL).all(), "written past dst_cap"
    assert ec.digest(d_src.cpu().numpy()) == ec.digest(slots), "the source was written"
    sz = d_sz.cpu().numpy().view(np.uint32)
    return [dst[i, :sz[i]].copy() for i in range(k)]


def decode(gpu, methods, streams, n):
    """cryogpu_decompress_device into slots of roundup16(n) bytes -> (out [k, n], out_size, status)"""
    from pg_cryogen_b200.codec import pack_chunks
    k = len(streams)
    buf, offs, sizes = pack_chunks(streams)
    dev = torch.device("cuda", gpu.device)
    stride = _r16(n)
    d_dst = torch.full((k, stride), 0x5A, dtype=torch.uint8, device=dev)
    d_osz = torch.full((k,), -1, dtype=torch.int32, device=dev)
    d_st = torch.full((k,), -1, dtype=torch.int32, device=dev)
    gpu.decompress_device(torch.from_numpy(np.asarray(methods, dtype=np.int32)).to(dev), torch.from_numpy(buf).to(dev),
                          torch.from_numpy(offs.view(np.int64)).to(dev), torch.from_numpy(sizes.view(np.int32)).to(dev),
                          d_dst, stride, d_osz, d_st, k, block_size=n, stream=torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    return d_dst.cpu().numpy()[:, :n], d_osz.cpu().numpy().view(np.uint32), d_st.cpu().numpy()


def _check_all(method, level, kinds, streams, slots, n):
    for kd, c, s in zip(kinds, streams, slots):
        try:
            ec.check(method, c, n, s[:n])
        except ec.StreamError as e:
            raise AssertionError(f"{kd} n={n} method {method} level {level}: {e}") from None
        if kd.startswith("run") and n >= 1024:
            assert len(c) <= ec.run_guard(method, n), (kd, n, method, len(c))


@pytest.mark.parametrize("n", ec.SIZES)
def test_every_layout_in_strided_slots_and_back_through_the_device(gpu, n):
    kinds = ec.KINDS
    slots = _slots([ec.layout(kd, n, 1, PAD + 16) for kd in kinds], n)
    lz = encode(gpu, COMP_LZ4, 1, slots, n)
    _check_all(COMP_LZ4, 1, kinds, lz, slots, n)
    zs = encode(gpu, COMP_ZSTD, 1, slots, n)
    _check_all(COMP_ZSTD, 1, kinds, zs, slots, n)
    # one batch of mixed methods through the device decoder
    order = np.random.default_rng(n).permutation(2 * len(kinds))
    streams = [(lz + zs)[i] for i in order]
    methods = [COMP_LZ4 if i < len(kinds) else COMP_ZSTD for i in order]
    out, osz, st = decode(gpu, methods, streams, n)
    assert (st == 0).all(), st
    assert (osz == n).all(), osz
    for j, i in enumerate(order):
        assert np.array_equal(out[j], slots[i % len(kinds), :n]), (kinds[i % len(kinds)], n, methods[j])


PARAM_SIZES = [17, 1025, 65537, 131077, CRYO_BLCKSZ + 17]
PARAM_KINDS = ["run-ee", "text", "copies", "sparse", "tile65537"]


@pytest.mark.parametrize("method,level", [(COMP_LZ4, a) for a in ec.LZ4_ACCELS] + [(COMP_ZSTD, z) for z in ec.ZSTD_LEVELS])
def test_every_acceleration_and_level(gpu, method, level):
    for n in PARAM_SIZES:
        slots = _slots([ec.layout(kd, n, 2, PAD + 16) for kd in PARAM_KINDS], n)
        _check_all(method, level, PARAM_KINDS, encode(gpu, method, level, slots, n), slots, n)


def _mixed(n, count):
    """count distinct blocks of every layout, in slots"""
    return _slots([ec.layout(ec.KINDS[i % len(ec.KINDS)], n, 100 + i, PAD + 16) for i in range(count)], n)


@pytest.mark.parametrize("n", [65537, CRYO_BLCKSZ + 17])
@pytest.mark.parametrize("method", [COMP_LZ4, COMP_ZSTD])
def test_stream_does_not_depend_on_the_batch(gpu, method, n):
    """Both encoders hand out (block, segment) work items from one queue to persistent CTAs: a block's stream is
    the same alone and inside two shuffled batches of more than 3 x SM-count mixed blocks."""
    uniq = _mixed(n, 18)
    alone = [encode(gpu, method, 1, uniq[i:i + 1], n)[0] for i in range(len(uniq))]
    nsm = torch.cuda.get_device_properties(gpu.device).multi_processor_count
    reps = -(-3 * nsm // len(uniq)) + 1
    for seed in (1, 2):
        idx = np.random.default_rng(seed).permutation(np.tile(np.arange(len(uniq)), reps))
        comp = encode(gpu, method, 1, uniq[idx], n)
        for j, i in enumerate(idx):
            assert np.array_equal(comp[j], alone[i]), (ec.KINDS[i % len(ec.KINDS)], i, j, seed)
    for i in range(len(uniq)):
        ec.check(method, alone[i], n, uniq[i, :n])


def _host_compress(gpu, method, srcs, n, multi_ctx=None):
    """cryogpu_compress_host (or _host_multi over the contexts given) with every destination pre-filled with the
    sentinel; asserts nothing is written past dst_size[i].  srcs: per block a pointer into a buffer the caller
    keeps alive."""
    k = len(srcs)
    cap = compress_bound(method, n)
    dst = np.full((k, cap + 64), SENTINEL, dtype=np.uint8)
    srcp = (C.c_void_p * k)(*srcs)
    dstp = (C.c_void_p * k)(*[dst[i].ctypes.data for i in range(k)])
    sz = np.zeros(k, dtype=np.uint32)
    st = np.full(k, -1, dtype=np.int32)
    if multi_ctx is None:
        rc = gpu.lib.cryogpu_compress_host(gpu.handle, k, method, 1, srcp, n, dstp, cap, sz.ctypes.data, st.ctypes.data)
    else:
        arr = (C.c_void_p * len(multi_ctx))(*[c.handle for c in multi_ctx])
        rc = gpu.lib.cryogpu_compress_host_multi(arr, len(multi_ctx), k, method, 1, srcp, n, dstp, cap, sz.ctypes.data,
                                                 st.ctypes.data)
    assert rc == 0, gpu.lib.cryogpu_last_error().decode()
    assert (st == 0).all(), st
    for i in range(k):
        assert (dst[i, sz[i]:] == SENTINEL).all(), ("written past dst_size", i)
    return [dst[i, :sz[i]].copy() for i in range(k)]


class _Pinned:
    """cryogpu_host_alloc'd copy of [k, n] blocks"""

    def __init__(self, lib, blocks):
        self.lib, k, n = lib, *blocks.shape
        self.p = lib.cryogpu_host_alloc(k * n)
        assert self.p
        self.a = np.ctypeslib.as_array((C.c_uint8 * (k * n)).from_address(self.p)).reshape(k, n)
        self.a[:] = blocks

    def ptr(self, i):
        return self.p + i * self.a.shape[1]

    def free(self):
        self.lib.cryogpu_host_free(self.p)


@pytest.mark.parametrize("n,count", [(CRYO_BLCKSZ, 300), (65537, 4200)])
@pytest.mark.parametrize("method", [COMP_LZ4, COMP_ZSTD])
def test_compress_host_two_lanes_and_mixed_sources(gpu, method, n, count):
    """More than one chunk per call (chunk_blocks: 128 at 1 MiB, 2 047 at 65 537 bytes), so both lanes and both
    halves of the scratch area are in flight; pageable, pinned and mixed sources (the call looks at src[0] only).
    Every variant writes the device call's streams."""
    uniq = _mixed(n, 24)
    idx = np.random.default_rng(count).integers(0, len(uniq), size=count)
    want_u = encode(gpu, method, 1, uniq, n)
    blocks = np.ascontiguousarray(uniq[idx, :n])
    pinned = _Pinned(gpu.lib, blocks)
    try:
        pageable = [blocks[i].ctypes.data for i in range(count)]
        pin = [pinned.ptr(i) for i in range(count)]
        variants = {"pageable": pageable, "pinned": pin, "pinned first": [pin[0]] + pageable[1:],
                    "pageable first": [pageable[0]] + pin[1:]}
        for name, srcs in variants.items():
            got = _host_compress(gpu, method, srcs, n)
            for j, i in enumerate(idx):
                assert np.array_equal(got[j], want_u[i]), (name, j)
    finally:
        pinned.free()


@pytest.mark.parametrize("method", [COMP_LZ4, COMP_ZSTD])
def test_compress_host_multi_matches_compress_host(gpu, method):
    n = 777777
    blocks = np.ascontiguousarray(_mixed(n, 21)[:, :n])
    ptrs = [blocks[i].ctypes.data for i in range(len(blocks))]
    want = _host_compress(gpu, method, ptrs, n)
    for nctx in (1, 2):
        if nctx > int(gpu.lib.cryogpu_device_count()):
            continue
        ctxs = [CryoGPU(i) for i in range(nctx)]
        try:
            got = _host_compress(gpu, method, ptrs, n, multi_ctx=ctxs)
        finally:
            for c in ctxs:
                c.close()
        for i in range(len(blocks)):
            assert np.array_equal(got[i], want[i]), (nctx, i)


@pytest.mark.parametrize("n", [65537, 777777])
@pytest.mark.parametrize("method", [COMP_LZ4, COMP_ZSTD])
def test_page_chains_hold_the_device_streams(gpu, method, n):
    slots = _mixed(n, 12)
    want = encode(gpu, method, 1, slots, n)
    blocks = np.ascontiguousarray(slots[:, :n])
    k = len(blocks)
    cap = pages_needed(compress_bound(method, n))
    rel = np.full((k * cap + 4, opg.PAGE), SENTINEL, dtype=np.uint8)
    blknos = np.random.default_rng(n).permutation(np.arange(1, rel.shape[0]))[: k * cap].astype(np.uint32).reshape(k, cap)
    npg, csz, st = gpu.compress_pages_host(method, 1, blocks, rel, blknos, created_xid=77, block_size=n)
    assert (st == 0).all(), st
    for i in range(k):
        err, m, size, got, chain = opg.gather(rel, int(blknos[i, 0]), cap=cap * opg.PAGE)
        assert err == opg.ERR_SUCCESS and m == method and size == csz[i], (i, err, m, size)
        assert chain == [int(x) for x in blknos[i, :npg[i]]]
        assert np.array_equal(got, want[i]), i
