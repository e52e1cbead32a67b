"""Batched tuple fetch on a B200: k random TIDs out of a compressed relation, three ways.

  pages_tuples   cryogpu_decompress_pages_tuples_host: page chains in, the selected tuples out (one call)
  read_data      cryo_batch_read_data over the distinct blocks (enough cache slots), then the tuples picked out of
                 the decoded blocks on the host
  reference      the reference's codec (oracle.ref: compression.c on liblz4 / libzstd) on all cores for the distinct
                 blocks, then cryo_storage_fetch (storage.c:55-68, restated in numpy) per TID

For each: device calls, bytes over the bus each way, wall time (median of --reps after a warm-up), tuples/s.  Also the
device time of k_tuple_gather alone (torch.profiler, cryogpu_tuples_device on blocks already in HBM) and its
algorithmic bytes (read 8 + 8 * ntuples per block + the selected tuples; write MAXALIGN(len) + 12 per entry) over
that time.  Tables: the 1M-row S/hex table and an M/lowcard table.  Prints one JSON document (and writes --out).

    python tools/bench_tuple_fetch.py --out /tmp/r03_tuple_fetch.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import pages as opg, ref  # noqa: E402
from pg_cryogen_b200 import CRYO_BLCKSZ, CryoGPU, blockgen as bg  # noqa: E402
import tuple_oracle  # noqa: E402

PAGE = 8192


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:                                  # the numbers still stand; say what is missing
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def build_table(kind, payload, rows, method, level):
    blocks = bg.make_table_blocks(rows, kind, payload)
    comp = ref.compress(method, level, blocks, nthreads=os.cpu_count() or 1)[0]
    npages = sum(opg.pages_needed(c.size) for c in comp)
    rel = np.zeros((npages + 1, PAGE), dtype=np.uint8)      # page 0: the metapage
    chains, at = [], 1
    for c in comp:
        ch = list(range(at, at + opg.pages_needed(c.size)))
        opg.split(rel, ch, c, method, 100)
        chains.append(ch)
        at += len(ch)
    ntup = np.array([int(b[0:4].view(np.uint32)[0] - 8) // 8 for b in blocks], dtype=np.int64)
    return blocks, comp, rel, chains, ntup


def median_time(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def make_request(rng, ntup, k, lossy):
    """TIDs as (distinct block indices, per block the positions in request order)"""
    if lossy:
        blk = np.sort(rng.choice(len(ntup), size=min(k, len(ntup)), replace=False))
        return blk, [[0] for _ in blk], int(ntup[blk].sum())
    b = rng.integers(0, len(ntup), size=k)
    p = (rng.integers(0, 1 << 30, size=k) % ntup[b]) + 1
    order = np.argsort(b, kind="stable")
    b, p = b[order], p[order]
    blk, start = np.unique(b, return_index=True)
    sel = [list(map(int, s)) for s in np.split(p, start[1:])]
    return blk, sel, k


def run_pages_tuples(gpu, rel, chains, blk, sel, reps):
    ch = [chains[int(i)] for i in blk]
    first = gpu.decompress_pages_tuples_host(rel, ch, sel)
    dcap, tcap = first[5]
    t = median_time(lambda: gpu.decompress_pages_tuples_host(rel, ch, sel, data_cap=dcap, tup_cap=tcap), reps)
    h2d, d2h = gpu.last_transfer_bytes()
    return {"calls": 1, "h2d": h2d, "d2h": d2h, "seconds": t, "need_bytes": dcap, "entries": tcap}


def run_read_data(gpu, rel, blk, sel, blocks_first, reps):
    """cryo_batch_read_data over the distinct blocks of an in-memory relation holding the same pages"""
    from test_gpu_batch import RelOps
    L = C.CDLL(os.path.join(ROOT, "pg_cryogen_b200", "libcryo_batch.so"))
    L.cryo_memrel_create.restype = C.c_void_p
    L.cryo_memrel_create.argtypes = [C.c_uint32]
    L.cryo_memrel_ops.restype = RelOps
    L.cryo_memrel_ops.argtypes = [C.c_void_p]
    L.cryo_memrel_pages.restype = C.POINTER(C.c_uint8)
    L.cryo_memrel_pages.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    L.cryo_memrel_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_cache_create.restype = C.c_void_p
    L.cryo_batch_cache_create.argtypes = [C.c_void_p, C.c_int]
    L.cryo_batch_cache_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_cache_invalidate.argtypes = [C.c_void_p]
    L.cryo_batch_cache_stats.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 3
    L.cryo_batch_read_data.argtypes = [C.c_void_p, C.POINTER(RelOps), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.cryo_batch_get_data.restype = C.POINTER(C.c_uint8)
    L.cryo_batch_get_data.argtypes = [C.c_void_p, C.c_int]
    mr = L.cryo_memrel_create(rel.shape[0])
    ops = L.cryo_memrel_ops(mr)
    extend = C.CFUNCTYPE(C.c_uint32, C.c_void_p)(ops.extend)
    for _ in range(rel.shape[0] - 1):
        extend(ops.rel)
    nb = C.c_uint32(0)
    np.ctypeslib.as_array(L.cryo_memrel_pages(mr, C.byref(nb)), shape=(rel.shape[0], PAGE))[:] = rel
    nblk = len(blk)
    cache = L.cryo_batch_cache_create(gpu.handle, nblk)
    ask = np.array([blocks_first[int(i)] for i in blk], dtype=np.uint32)
    ent = np.zeros(nblk, dtype=np.int32)
    errs = np.zeros(nblk, dtype=np.int32)
    state = {}

    def device():
        L.cryo_batch_cache_invalidate(cache)
        assert L.cryo_batch_read_data(cache, C.byref(ops), ask.ctypes.data, nblk, ent.ctypes.data, errs.ctypes.data) == 0
        state["xfer"] = gpu.last_transfer_bytes()

    def fetch():                                            # cryo_storage_fetch per TID, over the cached blocks
        out = []
        for j in range(nblk):
            d = np.ctypeslib.as_array(L.cryo_batch_get_data(cache, int(ent[j])), shape=(CRYO_BLCKSZ,))
            items = d[: 8 + 8 * 300].view(np.uint32)
            for p in sel[j]:
                for q in (range(1, (int(items[0]) - 8) // 8 + 1) if p == 0 else (p,)):
                    o, n = int(items[2 * q]), int(items[2 * q + 1])
                    out.append(d[o: o + n].tobytes())
        return out

    t_dev = median_time(device, reps)
    assert (errs == 0).all()
    t_host = median_time(fetch, reps)
    h2d, d2h = state["xfer"]
    L.cryo_batch_cache_destroy(cache)
    L.cryo_memrel_destroy(mr)
    return {"calls": 1, "h2d": h2d, "d2h": d2h, "seconds": t_dev + t_host, "device_call_seconds": t_dev,
            "host_fetch_seconds": t_host, "pinned_slot_bytes": nblk * CRYO_BLCKSZ}


def run_reference(comp, method, blk, sel, reps):
    chunks = [comp[int(i)] for i in blk]
    buf, offs, sizes = ref.pack(chunks)
    out = np.zeros((len(chunks), CRYO_BLCKSZ), dtype=np.uint8)

    def go():
        ref.decompress([method] * len(chunks), buf, offs, sizes, nthreads=os.cpu_count() or 1, out=out)
        got = []
        for j in range(len(chunks)):
            items = out[j, : 8 + 8 * 300].view(np.uint32)
            for p in sel[j]:
                for q in (range(1, (int(items[0]) - 8) // 8 + 1) if p == 0 else (p,)):
                    o, n = int(items[2 * q]), int(items[2 * q + 1])
                    got.append(out[j, o: o + n].tobytes())
        return got

    return {"calls": 0, "h2d": 0, "d2h": 0, "seconds": median_time(go, reps), "threads": os.cpu_count(),
            "codec": ref.describe()}


def gather_kernel(gpu, blocks, blk, sel, reps):
    """k_tuple_gather's device time (torch.profiler) for cryogpu_tuples_device on the decoded blocks in HBM"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from pg_cryogen_b200.codec import _sel_arrays
    dev = torch.device("cuda", gpu.device)
    sub = blocks[blk]
    want = tuple_oracle.block_tuples(sub, sel, fill=0)
    nbytes, nent = want[5]
    n = len(blk)
    off, pos = _sel_arrays(sel, n)
    d_blk = torch.from_numpy(sub).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    d_pos = torch.from_numpy(pos.view(np.int32)).to(dev)
    d_data = torch.zeros(max(nbytes, 16), dtype=torch.uint8, device=dev)
    d_to = torch.zeros(max(nent, 1), dtype=torch.int64, device=dev)
    d_tl = torch.zeros(max(nent, 1), dtype=torch.int32, device=dev)
    d_bf = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    d_st = torch.zeros(n, dtype=torch.int32, device=dev)
    d_need = torch.zeros(2, dtype=torch.int64, device=dev)
    s = torch.cuda.current_stream(dev).cuda_stream

    def call():
        gpu.tuples_device(d_blk, CRYO_BLCKSZ, n, None, d_off, d_pos, d_data, nbytes, d_to, d_tl, nent, d_bf, d_st, d_need,
                          stream=s)
    call()
    torch.cuda.synchronize(dev)
    assert np.array_equal(d_data.cpu().numpy()[:nbytes], want[0]), "device output differs from the restatement"
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize(dev)
    times = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "k_tuple_" in ev.name:
            key = ev.name.split("(")[0].split()[-1]
            times.setdefault(key, []).append(ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time)
    us = {k: float(np.median(v)) for k, v in times.items()}
    ntup = np.array([int(b[0:4].view(np.uint32)[0] - 8) // 8 for b in sub])
    alg_read = int(8 * n + 8 * ntup.sum() + want[2].sum())
    alg_write = int(nbytes + 12 * nent)
    g = next((v for k, v in us.items() if "gather" in k), None)
    return {"kernel_us": us, "alg_read_bytes": alg_read, "alg_write_bytes": alg_write,
            "gather_alg_GBps": None if not g else (alg_read + alg_write) / (g * 1e-6) / 1e9}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--s-rows", type=int, default=1_000_000)
    ap.add_argument("--m-rows", type=int, default=200_000)
    ap.add_argument("--method", type=int, default=1)
    ap.add_argument("--level", type=int, default=1)
    ap.add_argument("--ks", default="1000,10000,100000")
    ap.add_argument("--lossy-blocks", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    gpu = CryoGPU(0)
    result = {"card": card(), "method": a.method, "level": a.level, "reps": a.reps, "tables": {}}
    rng = np.random.default_rng(1)
    for name, kind, payload, rows in (("S_hex", "S", "hex", a.s_rows), ("M_lowcard", "M", "lowcard", a.m_rows)):
        blocks, comp, rel, chains, ntup = build_table(kind, payload, rows, a.method, a.level)
        firsts = [ch[0] for ch in chains]
        cases = [(f"k={k}", k, False) for k in map(int, a.ks.split(","))] + \
                [(f"lossy_{a.lossy_blocks}_blocks", a.lossy_blocks, True)]
        tab = {"blocks": len(blocks), "rows": rows, "csize_total": int(sum(c.size for c in comp)), "cases": {}}
        for label, k, lossy in cases:
            blk, sel, ntuples = make_request(rng, ntup, k, lossy)
            case = {"tids": k if not lossy else f"{len(blk)} lossy pages", "tuples": ntuples, "distinct_blocks": len(blk)}
            for way, fn in (("pages_tuples", lambda: run_pages_tuples(gpu, rel, chains, blk, sel, a.reps)),
                            ("read_data", lambda: run_read_data(gpu, rel, blk, sel, firsts, a.reps)),
                            ("reference", lambda: run_reference(comp, a.method, blk, sel, a.reps))):
                r = fn()
                r["tuples_per_s"] = ntuples / r["seconds"]
                case[way] = r
            case["gather"] = gather_kernel(gpu, blocks, blk, sel, max(a.reps, 10))
            tab["cases"][label] = case
            print(name, label, json.dumps({w: round(case[w]["seconds"] * 1e3, 3) for w in
                                           ("pages_tuples", "read_data", "reference")}), "ms", flush=True)
        result["tables"][name] = tab
    gpu.close()
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
