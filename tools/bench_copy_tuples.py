"""COPY flush on a B200: a whole table's cryo blocks compressed into relation pages, three ways.

  images     cryogpu_compress_pages_alloc_host on pinned 1 MiB block images built on the host (the flush before the
             blocks were built on the device)
  tuples     cryogpu_compress_tuples_pages_alloc_host on the same tuples, packed and pinned, as the batched writer holds
             them: the device builds the blocks, only the tuple bytes and their entries go over the bus
  reference  the reference's codec (oracle.ref: compression.c on liblz4 / libzstd) on all cores over the block images
             (the time of cryo_compress alone; building the images on the host is not in it)

The two device paths write into the C in-memory relation of host/cryo_batch.c (alloc = its extend, page_ptr = its
read_page), every block's first page reserved beforehand.  They are alternated, each a median of --reps after a warm-up,
at 64 and 512 blocks per call.  Also: the batched writer end to end (cryo_batch_insert_many + cryo_batch_flush, 64
blocks per call), k_block_build alone (torch.profiler) with its algorithmic bytes over its time, and where a 64-block
call of each device path spends its time (torch.profiler: H2D copies, the block build, the encoder, the page split, D2H
copies; the rest of the wall time is host work: callbacks, page copies, waits).  Prints one JSON document (and writes
--out).

    python tools/bench_copy_tuples.py --out /tmp/r04_copy_from_tuples.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from oracle import ref  # noqa: E402
from pg_cryogen_b200 import CRYO_BLCKSZ, CryoGPU, blockgen as bg  # noqa: E402
from bench_tuple_fetch import card  # noqa: E402

HBM_DATASHEET_TBPS = 7.7        # NVIDIA's HGX B200 data sheet, one GPU; not a measured figure


class RelOps(C.Structure):
    _fields_ = [("rel", C.c_void_p), ("nblocks", C.c_void_p), ("read_page", C.c_void_p), ("extend", C.c_void_p)]


def batch_lib():
    L = C.CDLL(os.path.join(ROOT, "pg_cryogen_b200", "libcryo_batch.so"))
    L.cryo_memrel_create.restype = C.c_void_p
    L.cryo_memrel_create.argtypes = [C.c_uint32]
    L.cryo_memrel_ops.restype = RelOps
    L.cryo_memrel_ops.argtypes = [C.c_void_p]
    L.cryo_memrel_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_writer_create.restype = C.c_void_p
    L.cryo_batch_writer_create.argtypes = [C.c_void_p, C.POINTER(RelOps), C.c_int, C.c_int, C.c_int, C.c_uint32]
    L.cryo_batch_insert_many.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]
    L.cryo_batch_flush.argtypes = [C.c_void_p]
    L.cryo_batch_writer_stats.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 3
    L.cryo_batch_writer_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_writer_flush_seconds.restype = C.c_double
    L.cryo_batch_writer_flush_seconds.argtypes = [C.c_void_p]
    return L


def pinned(gpu, nbytes, dtype=np.uint8):
    p = gpu.lib.cryogpu_host_alloc(max(nbytes, 16))
    assert p, "cryogpu_host_alloc failed"
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(nbytes, 16),))[:nbytes].view(dtype), p


class Table:
    """A table of one block kind: its tuples (packed, pinned), its block images (pinned), its entries"""

    def __init__(self, gpu, kind, payload, rows):
        per, t_len = bg.KINDS[kind]
        self.kind, self.payload, self.rows, self.t_len = kind, payload, rows, t_len
        self.n = bg.table_block_count(rows, kind)
        step = (t_len + 7) & ~7
        self.tuples = np.concatenate([bg.make_tuples(kind, payload, b, min(per, rows - b * per)) for b in range(self.n)])
        self.data, self._pd = pinned(gpu, rows * step)
        self.data.reshape(rows, step)[:, :t_len] = self.tuples
        self.off, self._po = pinned(gpu, rows * 8, np.uint64)
        self.off[:] = np.arange(rows, dtype=np.uint64) * np.uint64(step)
        self.len, self._pl = pinned(gpu, rows * 4, np.uint32)
        self.len[:] = t_len
        self.bf = np.minimum(np.arange(self.n + 1, dtype=np.uint64) * np.uint64(per), np.uint64(rows))
        self.images, self._pi = pinned(gpu, self.n * CRYO_BLCKSZ)
        self.images = self.images.reshape(self.n, CRYO_BLCKSZ)
        bg.make_table_blocks(rows, kind, payload, out=self.images)
        self.srcp = (C.c_void_p * self.n)(*[self.images[i].ctypes.data for i in range(self.n)])

    def free(self, gpu):
        for p in (self._pd, self._po, self._pl, self._pi):
            gpu.lib.cryogpu_host_free(p)


def flush_table(gpu, L, t, path, method, level, per_call):
    """One flush of the whole table in calls of per_call blocks into a fresh relation: (seconds, h2d, d2h, pages)"""
    rel = L.cryo_memrel_create(t.n * 140 + 16)
    ops = L.cryo_memrel_ops(rel)
    extend = C.CFUNCTYPE(C.c_uint32, C.c_void_p)(ops.extend)
    first = np.array([extend(ops.rel) for _ in range(t.n)], dtype=np.uint32)
    npg = np.zeros(t.n, np.uint32)
    csz = np.zeros(t.n, np.uint32)
    st = np.full(t.n, -1, np.int32)
    h2d = d2h = 0
    a, b = C.c_uint64(0), C.c_uint64(0)
    t0 = time.perf_counter()
    for lo in range(0, t.n, per_call):
        k = min(per_call, t.n - lo)
        if path == "images":
            rc = gpu.lib.cryogpu_compress_pages_alloc_host(
                gpu.handle, k, method, level, C.addressof(t.srcp) + 8 * lo, CRYO_BLCKSZ,
                first.ctypes.data + 4 * lo, ops.extend, ops.read_page, ops.rel, 7, npg.ctypes.data + 4 * lo,
                csz.ctypes.data + 4 * lo, st.ctypes.data + 4 * lo)
        else:
            rc = gpu.lib.cryogpu_compress_tuples_pages_alloc_host(
                gpu.handle, k, method, level, t.data.ctypes.data, t.data.size, t.off.ctypes.data, t.len.ctypes.data,
                t.bf.ctypes.data + 8 * lo, CRYO_BLCKSZ, first.ctypes.data + 4 * lo, ops.extend, ops.read_page, ops.rel, 7,
                npg.ctypes.data + 4 * lo, csz.ctypes.data + 4 * lo, st.ctypes.data + 4 * lo)
        assert rc == 0, gpu.lib.cryogpu_last_error()
        gpu.lib.cryogpu_last_transfer_bytes(gpu.handle, C.byref(a), C.byref(b))
        h2d += a.value
        d2h += b.value
    sec = time.perf_counter() - t0
    assert (st == 0).all(), np.unique(st)
    L.cryo_memrel_destroy(rel)
    return sec, h2d, d2h, int(npg.sum()), csz.copy()


def compare_paths(gpu, L, t, method, level, per_call, reps):
    """images and tuples alternated; both write the same compressed sizes"""
    res = {"images": [], "tuples": []}
    sizes = {}
    for r in range(reps + 1):
        for path in ("images", "tuples") if r % 2 == 0 else ("tuples", "images"):
            sec, h2d, d2h, pages, csz = flush_table(gpu, L, t, path, method, level, per_call)
            sizes[path] = csz
            if r:
                res[path].append(sec)
            res[path + "_bytes"] = {"h2d": h2d, "d2h": d2h, "pages": pages}
    assert np.array_equal(sizes["images"], sizes["tuples"]), "the two paths compressed different blocks"
    block_bytes = t.n * CRYO_BLCKSZ
    out = {}
    for path in ("images", "tuples"):
        s = float(np.median(res[path]))
        out[path] = dict(res[path + "_bytes"], seconds=s, reps=[round(x, 6) for x in res[path]],
                         GBps_of_block_data=block_bytes / s / 1e9, h2d_per_block=res[path + "_bytes"]["h2d"] / t.n)
    out["speedup_tuples_over_images"] = out["images"]["seconds"] / out["tuples"]["seconds"]
    return out


def reference(t, method, level, reps):
    threads = os.cpu_count() or 1
    ref.compress(method, level, t.images[: min(64, t.n)], nthreads=threads)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        ref.compress(method, level, t.images, nthreads=threads)
        ts.append(time.perf_counter() - t0)
    s = float(np.median(ts))
    return {"seconds": s, "threads": threads, "GBps_of_block_data": t.n * CRYO_BLCKSZ / s / 1e9, "codec": ref.describe()}


def writer_end_to_end(gpu, L, t, method, level):
    rel = L.cryo_memrel_create(t.n * 140 + 16)
    ops = L.cryo_memrel_ops(rel)
    w = L.cryo_batch_writer_create(gpu.handle, C.byref(ops), method, level, 64, 7)
    t0 = time.perf_counter()
    rc = L.cryo_batch_insert_many(w, t.tuples.ctypes.data, t.t_len, t.rows)
    rc = rc or L.cryo_batch_flush(w)
    sec = time.perf_counter() - t0
    assert rc == 0
    calls, blocks, pages = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    L.cryo_batch_writer_stats(w, C.byref(calls), C.byref(blocks), C.byref(pages))
    flush = L.cryo_batch_writer_flush_seconds(w)
    L.cryo_batch_writer_destroy(w)
    L.cryo_memrel_destroy(rel)
    return {"seconds_with_inserts": sec, "flush_seconds": flush, "device_calls": calls.value, "blocks": blocks.value,
            "pages": pages.value, "GBps_of_block_data_with_inserts": blocks.value * CRYO_BLCKSZ / sec / 1e9,
            "GBps_of_block_data_flush_calls": blocks.value * CRYO_BLCKSZ / flush / 1e9}


def _cuda_events(prof):
    """(name, device microseconds) of every CUDA kernel and copy in a profile"""
    out = []
    for ev in prof.events():
        if ev.device_type.name == "CUDA":
            out.append((ev.name, ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time))
    return out


def build_kernel(gpu, t, reps):
    """k_block_build alone on the table's tuples in HBM: median device time and algorithmic bytes over it"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda", gpu.device)
    d_data = torch.from_numpy(t.data.copy()).to(dev)
    d_to = torch.from_numpy(t.off.view(np.int64).copy()).to(dev)
    d_tl = torch.from_numpy(t.len.view(np.int32).copy()).to(dev)
    d_bf = torch.from_numpy(t.bf.view(np.int64).copy()).to(dev)
    d_dst = torch.empty((t.n, CRYO_BLCKSZ), dtype=torch.uint8, device=dev)
    d_st = torch.empty(t.n, dtype=torch.int32, device=dev)
    s = torch.cuda.current_stream(dev).cuda_stream

    def call():
        gpu.build_blocks_device(d_data, t.data.size, d_to, d_tl, d_bf, t.n, d_dst, CRYO_BLCKSZ, d_st, stream=s)
    call()
    torch.cuda.synchronize(dev)
    assert (d_st.cpu().numpy() == 0).all()
    for i in (0, t.n // 2, t.n - 1):
        assert np.array_equal(d_dst[i].cpu().numpy(), t.images[i]), i
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize(dev)
    us = float(np.median([d for n, d in _cuda_events(prof) if "k_block_build" in n]))
    rd = int(t.rows) * (t.t_len + 12) + 8 * (t.n + 1)
    wr = t.n * CRYO_BLCKSZ
    del d_dst
    torch.cuda.empty_cache()
    return {"kernel_us": us, "alg_read_bytes": rd, "alg_write_bytes": wr, "alg_TBps": (rd + wr) / (us * 1e-6) / 1e12,
            "share_of_datasheet_hbm": (rd + wr) / (us * 1e-6) / 1e12 / HBM_DATASHEET_TBPS,
            "datasheet_hbm_TBps": HBM_DATASHEET_TBPS, "blocks": t.n}


def call_split(gpu, L, t, method, level, path, per_call=64):
    """Where the calls of one table flush spend their time, per call: device time of each kind of work (profiler) and
    the wall time it sits in"""
    from torch.profiler import ProfilerActivity, profile
    flush_table(gpu, L, t, path, method, level, per_call)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sec = flush_table(gpu, L, t, path, method, level, per_call)[0]
    ncalls = (t.n + per_call - 1) // per_call
    cats = {}
    for name, us in _cuda_events(prof):
        low = name.lower()
        key = ("h2d" if "htod" in low else "d2h" if "dtoh" in low else "build" if "k_block_build" in name else
               "encoder" if "encode" in low else "page_split" if "k_pages_split" in name else
               "memset" if "memset" in low else "other_kernels")
        cats[key] = cats.get(key, 0.0) + us
    per = {k: v / ncalls / 1e3 for k, v in cats.items()}
    wall = sec / ncalls * 1e3
    return {"per_call_ms": {**per, "wall_profiled": wall, "host_and_waits": wall - sum(per.values())},
            "calls": ncalls, "note": "device times are per call sums from torch.profiler; the profiled run is slower "
                                     "than an unprofiled one; host_and_waits = wall - device sums (alloc and page_ptr "
                                     "callbacks, page copies into the relation, synchronisations)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--s-rows", type=int, default=1_000_000)
    ap.add_argument("--m-rows", type=int, default=200_000)
    ap.add_argument("--d-rows", type=int, default=200_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    gpu = CryoGPU(0)
    L = batch_lib()
    result = {"card": card(), "reps": a.reps, "tables": {}}
    for name, kind, payload, rows in (("S_hex", "S", "hex", a.s_rows), ("M_lowcard", "M", "lowcard", a.m_rows),
                                      ("D_hex", "D", "hex", a.d_rows)):
        t = Table(gpu, kind, payload, rows)
        tab = {"blocks": t.n, "rows": rows, "tuple_bytes": int(rows * t.t_len),
               "build_kernel": build_kernel(gpu, t, max(a.reps, 10)), "codecs": {}}
        for label, method, level in (("zstd-1", 1, 1), ("lz4-1", 0, 1)):
            c = {f"{k}_blocks_per_call": compare_paths(gpu, L, t, method, level, k, a.reps) for k in (64, 512)}
            c["reference_all_cores"] = reference(t, method, level, a.reps)
            c["writer_end_to_end"] = writer_end_to_end(gpu, L, t, method, level)
            c["call_split_64"] = {p: call_split(gpu, L, t, method, level, p) for p in ("images", "tuples")}
            tab["codecs"][label] = c
            print(name, label, json.dumps({k: {p: round(c[k][p]["seconds"] * 1e3, 2) for p in ("images", "tuples")}
                                           for k in ("64_blocks_per_call", "512_blocks_per_call")}),
                  "reference", round(c["reference_all_cores"]["seconds"] * 1e3, 2), "ms", flush=True)
        result["tables"][name] = tab
        t.free(gpu)
    gpu.close()
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
