"""-m gpu: the decoders' contract on the device, on every route a batch can take.

A batch of at most 2 x SM-count blocks takes the CTA-per-block LZ4 decoder and the pipeline's CTA executor; a larger
one takes the warp LZ4 decoder (which hands blocks over LZ4W_BUDGET sequences to the CTA one), the pipeline's
per-frame choice of executor, its raw / RLE stage, the early pass and the jobs.  So every case runs twice: below
2 x SM and at 2 x SM + 1 or more, with a count that is not a multiple of ZP_G = 8.

Every call goes through decode(): the streams sit in one source buffer at offsets that cycle through every residue
mod 16, with bait between them (0xFF bytes, or the head of the next stream), the last one ending at the buffer's end
rounded up to 16.  The destination stride is roundup16(block_size) + 4 KiB, pre-filled with a sentinel.  After
every call: each block's status, out_size and bytes against the plain-C restatement (tests/decode_vectors.py
verdict(), as tools/emu_fuzz.py judges), the sentinels in [block_size, stride) of every block whatever its status,
and an unchanged source.  [out_size, block_size) of a failed block is not checked: the header promises nothing there.

Run as a script (python tests/test_gpu_decode_contract.py OUT.json), it decodes one mixed batch through
cryogpu_decompress_host and writes a digest per block: the route knobs are read once per process, so
test_route_knobs_agree runs it in fresh processes under each setting."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import decode_vectors as dv            # noqa: E402
import encode_check as ec              # noqa: E402
from pg_cryogen_b200 import COMP_LZ4, COMP_ZSTD, CRYO_BLCKSZ, CryoGPU   # noqa: E402
from pg_cryogen_b200 import blockgen as bg  # noqa: E402

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5
PAD = 4096
MiB = 1 << 20


def _r16(v):
    return (v + 15) & ~15


def place(streams, seed=0):
    """One source buffer: stream i at an offset = i mod 16, bait in front of it (0xFF, or the head of stream i + 1),
    the last stream ending at the buffer's end rounded up to 16.  Returns (buffer, offsets, sizes)."""
    k = len(streams)
    offs, parts, pos = np.zeros(k, dtype=np.uint64), [], 0
    for i, s in enumerate(streams):
        gap = (i % 16 - pos) % 16 + 16 * (1 + (i + seed) % 3)
        if (i + seed) % 2:
            bait = np.full(gap, 0xFF, dtype=np.uint8)
        else:
            nxt = streams[(i + 1) % k]
            bait = np.resize(nxt[:gap], gap) if nxt.size else np.full(gap, 0xFF, dtype=np.uint8)
        parts += [bait, np.asarray(s, dtype=np.uint8)]
        offs[i] = pos + gap
        pos += gap + len(s)
    parts.append(np.full(_r16(pos) - pos, 0xFF, dtype=np.uint8))
    buf = np.concatenate(parts)
    return buf, offs, np.array([len(s) for s in streams], dtype=np.uint32)


def decode(gpu, methods, streams, n):
    """cryogpu_decompress_device over place()d streams into strided, sentinel-filled slots.  Returns (out [k, n],
    out_size, status); asserts the sentinels and the source."""
    import torch
    k = len(streams)
    buf, offs, sizes = place(streams, seed=k)
    dev = torch.device("cuda", gpu.device)
    stride = _r16(n) + PAD
    d_src = torch.from_numpy(buf).to(dev)
    d_dst = torch.full((k, stride), SENTINEL, dtype=torch.uint8, device=dev)
    d_osz = torch.full((k,), -1, dtype=torch.int32, device=dev)
    d_st = torch.full((k,), -1, dtype=torch.int32, device=dev)
    gpu.decompress_device(torch.from_numpy(np.asarray(methods, dtype=np.int32)).to(dev), d_src,
                          torch.from_numpy(offs.view(np.int64)).to(dev), torch.from_numpy(sizes.view(np.int32)).to(dev),
                          d_dst, stride, d_osz, d_st, k, block_size=n, stream=torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    tail = d_dst[:, n:]
    bad = (tail != SENTINEL).any(dim=1).nonzero().flatten().tolist()
    assert not bad, f"written past block_size in blocks {bad[:8]}"
    assert torch.equal(d_src.cpu(), torch.from_numpy(buf)), "the source was written"
    out = d_dst[:, :n].cpu().numpy()
    return out, d_osz.cpu().numpy().view(np.uint32), d_st.cpu().numpy()


def judge(out, osz, st, want, n, tags):
    """want[j]: decode_vectors.verdict() of the block's stream, or its bytes"""
    for j, w in enumerate(want):
        if w is not None and w.size == n:
            assert st[j] == 0 and osz[j] == n, (tags[j], int(st[j]), int(osz[j]))
            if not np.array_equal(out[j], w):
                raise AssertionError((tags[j], "bytes differ at", int(np.argmax(out[j] != w))))
        else:
            assert dv.accepts(w, n, int(st[j]), int(osz[j]), out[j]), (tags[j], int(st[j]), int(osz[j]))


def counts(gpu):
    import torch
    nsm = torch.cuda.get_device_properties(gpu.device).multi_processor_count
    large = 2 * nsm + 1
    if large % 8 == 0:
        large += 1
    return nsm, large


def both_routes(gpu, items, n, seed, check_routes=None):
    """items: (method, stream, want, tag).  One batch below 2 x SM (the items, as many as fit), one at 2 x SM + 1 or more
    (the items repeated, shuffled).  check_routes(gpu, batch items) runs after the large call."""
    nsm, large = counts(gpu)
    rng = np.random.default_rng(seed)
    small = items[: 2 * nsm]
    total = max(large, len(items) + 1)
    idx = rng.permutation(np.resize(np.arange(len(items)), total + (total % 8 == 0)))
    for batch in (small, [items[i] for i in idx]):
        out, osz, st = decode(gpu, [b[0] for b in batch], [b[1] for b in batch], n)
        judge(out, osz, st, [b[2] for b in batch], n, [b[3] for b in batch])
        if check_routes is not None and len(batch) > 2 * nsm:
            check_routes(gpu, batch)


# ---- 1. sizes x producers ------------------------------------------------------------------------------------------

PRODUCERS = dv.LZ4_PRODUCERS + dv.ZSTD_PRODUCERS


@pytest.mark.parametrize("n", ec.SIZES + [5 * MiB])
def test_sizes_and_producers(gpu, n):
    """Every layout kind of tests/encode_check.py, each written by two of the producers (liblz4 at accelerations 1, 9,
    65 537 and LZ4_compress_HC; libzstd at levels -5, 1, 3, 9, 19, 22; the pairing turns with the size), both methods
    in every batch.  At 5 MiB LZ4 is above LZ4C_MAXCAP and only the warp kernel runs; beyond 1 MiB + 17 levels 19 and
    22 are replaced by 9 and 3 to keep the compression time down."""
    si = (ec.SIZES + [5 * MiB]).index(n)
    items = []
    for r in range(2):
        for i, kind in enumerate(ec.KINDS):
            blk = ec.layout(kind, n, 10 + r)
            p = PRODUCERS[(i + si + 5 * r) % len(PRODUCERS)]
            if n > CRYO_BLCKSZ + 17 and p[0] == "zstd" and p[1] >= 19:
                p = ("zstd", 9 if p[1] == 19 else 3)
            m, s = dv.produce(p, blk)
            items.append((m, s, blk, f"{kind}/{p[0]}{p[1]}"))

    def routes(g, batch):
        blocks, cta = g.lz4_route_stats()
        if n > 4 * MiB - 1:
            assert blocks == 0 and cta == 0, (blocks, cta)      # not routed: the warp kernel alone
    both_routes(gpu, items, n, seed=n, check_routes=routes)


# ---- 2. crafted vectors --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [65791, 300017])
def test_crafted_vectors_on_both_routes(gpu, n):
    """The vectors of tests/decode_vectors.py, with libzstd frames at levels <= 3 beside them.  In the large batch:
    blocks over LZ4W_BUDGET sequences go to the CTA kernel and no other; the 17-block and window-2^28 frames are the
    pipeline's only fallbacks (and the window-2^28 frame is rejected); libzstd frames at level <= 3 are not.  A dense
    frame's placement depends on the room left in the pool: only its bytes are asserted, in the second batch, with the
    rule-breaking vectors and the checksum deviation (DESIGN.md section 1: a content checksum is skipped, not verified:
    a wrong one is accepted)."""
    vs = dv.vectors(n)
    lib = []
    for i, kind in enumerate(["copies", "sparse", "text"]):
        blk = ec.layout(kind, n, 30 + i)
        for lv in (-5, 1, 3):
            lib.append((COMP_ZSTD,) + (dv.produce(("zstd", lv), blk)[1], blk, f"{kind}/zstd{lv}"))
    routed = [(v.method, v.stream, v.plain, v.name) for v in vs if v.plain is not None and v.route != "dense"]
    routed += [(v.method, v.stream, None, v.name) for v in vs if v.name == "zstd-window-28"]
    routed += lib

    def routes(g, batch):
        _, cta = g.lz4_route_stats()
        assert cta == sum(1 for b in batch if b[3].startswith("lz4-seqs-3073")), cta
        frames, fallback = g.zstd_pipeline_stats()
        assert frames == sum(1 for b in batch if b[0] == COMP_ZSTD), frames
        want = sum(1 for b in batch if b[3] in ("zstd-17-blocks", "zstd-window-28"))
        assert fallback == want, (fallback, want)
    both_routes(gpu, routed, n, seed=n, check_routes=routes)

    bad, plan = dv.zstd_frame([dv.raw(bytes(range(16)))] + dv._fill_rle(16, n), checksum="bad")
    rest = [(v.method, v.stream, v.plain if v.plain is not None else dv.verdict(v.method, v.stream, n), v.name)
            for v in vs if v.plain is None or v.route == "dense"]
    rest += [(COMP_ZSTD, bad, dv._u8(plan), "zstd-checksum-bad")] + lib[:3]
    both_routes(gpu, rest, n, seed=n + 1)


# ---- 3. sequence pool exhaustion -----------------------------------------------------------------------------------

def test_sequence_pool_exhaustion(gpu):
    """Dense frames (about 349 000 sequences a MiB against a pool of cap / 8 + 64 per frame): stage 1 declines the
    frames past the pool's end in atomic order and the fallback decodes them.  First a large batch of dense frames
    only, then dense frames shuffled among heap-tuple frames."""
    nsm, large = counts(gpu)
    dense = [dv.dense_frame(CRYO_BLCKSZ, seed) for seed in range(3)]
    items = [(COMP_ZSTD, f, dv._u8(p), f"dense{i}") for i, (f, p) in enumerate(dense)]
    out, osz, st = decode(gpu, [COMP_ZSTD] * large, [items[i % 3][1] for i in range(large)], CRYO_BLCKSZ)
    judge(out, osz, st, [items[i % 3][2] for i in range(large)], CRYO_BLCKSZ, [items[i % 3][3] for i in range(large)])
    frames, fallback = gpu.zstd_pipeline_stats()
    assert frames == large and fallback > 0, (frames, fallback)
    heap = []
    for i in range(6):
        blk = bg.make_block("S", "hex" if i % 2 else "lowcard", 60 + i)
        heap.append((COMP_ZSTD, dv.produce(("zstd", 1), blk)[1], blk, f"heap{i}"))
    idx = np.random.default_rng(3).permutation(large)
    batch = [heap[i % len(heap)] if i % 3 == 0 else items[i % 3] for i in idx]      # two dense frames in three
    out, osz, st = decode(gpu, [b[0] for b in batch], [b[1] for b in batch], CRYO_BLCKSZ)
    judge(out, osz, st, [b[2] for b in batch], CRYO_BLCKSZ, [b[3] for b in batch])
    assert gpu.zstd_pipeline_stats()[1] > 0


# ---- 4. corrupt neighbours -----------------------------------------------------------------------------------------

def test_corrupt_neighbours(gpu):
    """The mutation corpus the emulator test runs (decode_vectors.corpus()), shuffled into large batches: about a
    third of the frames mutated.  Intact frames bit-exact, mutated ones the restatement's verdict, no sentinel
    touched."""
    nsm, large = counts(gpu)
    cap = dv.CORPUS_CAP
    items = [(m, s, b if b is not None else dv.verdict(m, s, cap), t) for m, s, b, t in dv.corpus()]
    for seed in (1, 2):
        idx = np.random.default_rng(seed).permutation(np.resize(np.arange(len(items)), large + 8 * seed))
        batch = [items[i] for i in idx]
        out, osz, st = decode(gpu, [b[0] for b in batch], [b[1] for b in batch], cap)
        judge(out, osz, st, [b[2] for b in batch], cap, [b[3] for b in batch])


# ---- 5. batch and route independence -------------------------------------------------------------------------------

def _mixed_items(n=300017):
    items = [(v.method, v.stream, v.name) for v in dv.vectors(n) if v.route != "dense"]
    for i, kind in enumerate(["copies", "sparse", "text", "random"]):
        blk = ec.layout(kind, n, 40 + i)
        for p in (("lz4", 1), ("zstd", 1), ("zstd", 19)):
            items.append(dv.produce(p, blk) + (f"{kind}/{p[0]}{p[1]}",))
    return items, n


def _digest(out, osz, st):
    """ok, size and bytes of a decoded block; "failed" for a rejected one (which status, and how far it got, is the
    decoder's own)"""
    return [f"ok:{int(z)}:" + hashlib.sha256(o[:z].tobytes()).hexdigest()[:16] if s == 0 else "failed"
            for o, z, s in zip(out, osz, st)]


def test_batch_independence(gpu):
    """Each stream alone, then inside two shuffled mixed batches of more than 3 x SM-count: the same status, size
    and bytes."""
    items, n = _mixed_items()
    nsm, _ = counts(gpu)
    alone = [_digest(*decode(gpu, [m], [s], n))[0] for m, s, _ in items]
    for seed in (1, 2):
        idx = np.random.default_rng(seed).permutation(np.resize(np.arange(len(items)), 3 * nsm + 5 * seed))
        out, osz, st = decode(gpu, [items[i][0] for i in idx], [items[i][1] for i in idx], n)
        got = _digest(out, osz, st)
        for j, i in enumerate(idx):
            assert got[j] == alone[i], (items[i][2], got[j], alone[i])


KNOBS = [{}, {"CRYOGPU_LZ4_KERNEL": "warp"}, {"CRYOGPU_LZ4_KERNEL": "cx"}, {"CRYOGPU_ZSTD_KERNEL": "warp"},
         {"CRYOGPU_ZSTD_EXEC": "warp"}, {"CRYOGPU_ZSTD_EXEC": "cx"}]


def test_route_knobs_agree(gpu, tmp_path):
    """One mixed batch of more than 2 x SM blocks in a fresh process per setting of the route switches: the per-block
    digests of status, size and bytes are the same under every one."""
    res = []
    for k, env in enumerate(KNOBS):
        path = tmp_path / f"knobs{k}.json"
        r = subprocess.run([sys.executable, os.path.abspath(__file__), str(path), str(counts(gpu)[1] + 12)],
                           env={**os.environ, **env},
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, (env, r.stdout[-2000:], r.stderr[-2000:])
        res.append(json.loads(path.read_text()))
    for env, got in zip(KNOBS[1:], res[1:]):
        diff = [j for j, (a, b) in enumerate(zip(res[0], got)) if a != b]
        assert len(got) == len(res[0]) and not diff, (env, diff[:8])


def _knobs_case(path, count):
    gpu = CryoGPU(0)
    items, n = _mixed_items()
    idx = np.random.default_rng(5).permutation(np.resize(np.arange(len(items)), count))
    out, osz, st = gpu.decompress_host([items[i][0] for i in idx], [items[i][1] for i in idx], block_size=n)
    want = [dv.verdict(items[i][0], items[i][1], n) for i in idx]
    judge(out, osz, st, want, n, [items[i][2] for i in idx])
    with open(path, "w") as f:
        json.dump(_digest(out, osz, st), f)
    gpu.close()


# ---- 6. host calls at odd sizes ------------------------------------------------------------------------------------

def _host(gpu, methods, streams, n, dst, multi=False):
    """cryogpu_decompress_host (or _host_multi on this context) into the rows of dst [k, >= n]"""
    import ctypes as C
    k = len(streams)
    me = np.asarray(methods, dtype=np.int32)
    srcp = (C.c_void_p * k)(*[s.ctypes.data for s in streams])
    sizes = np.array([s.size for s in streams], dtype=np.uint32)
    dstp = (C.c_void_p * k)(*[dst.ctypes.data + i * dst.strides[0] for i in range(k)])
    osz = np.zeros(k, dtype=np.uint32)
    st = np.full(k, -1, dtype=np.int32)
    if multi:
        arr = (C.c_void_p * 1)(gpu.handle)
        rc = gpu.lib.cryogpu_decompress_host_multi(arr, 1, k, me.ctypes.data, srcp, sizes.ctypes.data, dstp, n,
                                                   osz.ctypes.data, st.ctypes.data)
    else:
        rc = gpu.lib.cryogpu_decompress_host(gpu.handle, k, me.ctypes.data, srcp, sizes.ctypes.data, dstp, n,
                                             osz.ctypes.data, st.ctypes.data)
    assert rc == 0, gpu.lib.cryogpu_last_error().decode()
    return osz, st


@pytest.mark.parametrize("n,count", [(65537, 4200), (777777, 400), (CRYO_BLCKSZ + 17, 300)])
def test_host_calls_at_odd_sizes(gpu, n, count):
    """At least three chunks (128 MiB / block_size blocks each) with one failed block per chunk.  Sparse blocks, so
    only the non-zero 4 KiB pages travel, and the ragged tail page always does.  Pageable memory pre-filled with stale
    bytes, pinned memory, cryogpu_set_zero_by_unmap on, and _host_multi: each writes what the device call writes."""
    uniq = []
    for i in range(6):
        # mostly zero pages, so that the sparse return runs, with bytes in the first page, one page inside and the
        # ragged tail page
        blk = np.zeros(n, dtype=np.uint8)
        rng = np.random.default_rng([n, i])
        for at in (0, (n // 2) & ~4095, n - 1 - (n - 1) % 4096):
            blk[at: at + 1 + i * 7] = rng.integers(1, 256, size=len(blk[at: at + 1 + i * 7]), dtype=np.uint8)
        uniq.append(dv.produce([("lz4", 1), ("zstd", 1), ("zstd", 3)][i % 3], blk) + (blk,))
    chunk = (128 << 20) // n
    assert count > 2 * chunk
    idx = np.random.default_rng(n).integers(0, len(uniq), size=count)
    methods = [uniq[i][0] for i in idx]
    streams = [uniq[i][1] for i in idx]
    bad = uniq[1][1].copy()
    bad[0] ^= 0xFF                                  # no zstd magic
    assert dv.verdict(COMP_ZSTD, bad, n) is None
    for c in range(0, count, chunk):
        methods[c + 5], streams[c + 5] = COMP_ZSTD, bad
    out, osz, st = decode(gpu, methods, streams, n)
    want = [None if j % chunk == 5 else uniq[i][2] for j, i in enumerate(idx)]
    judge(out, osz, st, want, n, [f"block {j}" for j in range(count)])

    def same(name, got, gosz, gst):
        assert np.array_equal(gst, st) and np.array_equal(gosz, osz), name
        ok = st == 0
        assert np.array_equal(got[ok, :n], out[ok]), name
        assert (got[:, n:] == 0x77).all(), (name, "written past block_size")

    try:
        stale = np.full((count, n + 64), 0x77, dtype=np.uint8)
        same("pageable", stale, *_host(gpu, methods, streams, n, stale))
        stale[:] = 0x77
        assert gpu.lib.cryogpu_set_zero_by_unmap(gpu.handle, 1) == 0
        same("zero by unmap", stale, *_host(gpu, methods, streams, n, stale))
        assert gpu.lib.cryogpu_set_zero_by_unmap(gpu.handle, 0) == 0
        stale[:] = 0x77
        same("host_multi", stale, *_host(gpu, methods, streams, n, stale, multi=True))
        del stale
        import ctypes as C
        size = count * (n + 64)
        p = gpu.lib.cryogpu_host_alloc(size)
        assert p
        try:
            pin = np.ctypeslib.as_array((C.c_uint8 * size).from_address(p)).reshape(count, n + 64)
            pin[:] = 0x77
            same("pinned", pin, *_host(gpu, methods, streams, n, pin))
        finally:
            gpu.lib.cryogpu_host_free(p)
    finally:
        gpu.lib.cryogpu_set_zero_by_unmap(gpu.handle, 0)


if __name__ == "__main__":
    _knobs_case(sys.argv[1], int(sys.argv[2]))
