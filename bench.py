#!/usr/bin/env python
"""bench.py -- benchmarks of the B200 block codec for pg_cryogen.

Default run = the headline (BASELINE.json configs[1], SURVEY.md 8(d) "Config 2"): the cryo
blocks of a synthetic 1M-row heap-tuple table (S blocks: 290 rows of 61 bytes per 1 MiB block,
3 449 blocks, 3.37 GiB of plaintext), compressed with zstd level 1 by the reference's library,
batch-decompressed on one B200 (the seq-scan read path, cache.c:178).  One "step" = one batched
decompression of every block of the table.

  value      uncompressed GB/s with inputs resident in HBM (CUDA events on the launch stream)
  e2e        the same metric through the host-buffer C ABI call (cryogpu_decompress_host):
             pinned host buffers, H2D + kernels + D2H inside the timed region
  roofline   algorithmic bytes (csize_i + 1 MiB per block) / kernel time vs measured HBM peak
  cpu_baseline   the reference's own compression.c (oracle/_ref) on the box's host cores
  secondary  the rest of BASELINE.json's metric on the same GPU: {lz4, zstd-1} x {decompress,
             compress} x block kinds, each with GB/s, roofline fraction, the reference's CPU rate
             on the same blocks (1 thread and all cores) and, for compression, the size ratio
             against the reference (N = 1 only; --no-secondary skips it)

N > 1 (torchrun, one rank per GPU): every rank decompresses its own table of the same
shape (weak scaling, no collective on the data path; SURVEY.md 8(e)).

Other configurations of BASELINE.json (each prints one JSON line of the same shape):
  --config 3   lz4_acceleration sweep on 64 KiB blocks (COPY flush path), ratio vs the reference
  --config 4   zstd levels -5..3, compress + decompress of ~10 GB sharded by block range over
               the ranks (strong scaling)
  --config 5   small batches (1..256 blocks) through the device call: latency and GB/s beside
               the reference on one host thread and on all of them

`--impl reference` times the reference's CPU implementation on the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# hardware work queues for the streams of the process (default 8): the pipeline's three streams must not share one
# (cryogpu_init sets this too, but torch creates the CUDA context first here)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

CRYO_BLCKSZ = 1 << 20
COMP_LZ4, COMP_ZSTD = 0, 1
NROWS = 1_000_000
KIND, PAYLOAD = "S", "hex"
METHOD, LEVEL = COMP_ZSTD, 1
METRIC = "decompress_GBps_zstd1_1Mrow_table"
# kernels of ours per headline step: method check; LZ4 warp decoder, CTA decoder (both exit: no LZ4
# blocks); the pipeline's parse, Huffman tables, literals, FSE tables, sequence walk x2 size classes,
# raw/RLE blocks (early pass, late pass + the executor's long runs), warp executor, CTA executor
# (exits: nothing routed), the check of what the raw/RLE stage published; the fallback decoder (exits)
LAUNCHES_PER_STEP = 15
SECONDARY_KINDS = (("S", "hex"), ("S", "lowcard"), ("M", "hex"), ("M", "lowcard"), ("D", "hex"), ("D", "lowcard"))


def workload_string(rows: int, nblk: int) -> str:
    return (f"{rows}-row S/hex table ({nblk} cryo blocks of 1 MiB per GPU), zstd level 1 frames written by "
            "libzstd 1.5.5, batched decompress")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic():
    """dram bytes per step (all kernels of the zstd pipeline) from the committed ncu capture, or None."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("zstd_pipeline_dram_bytes_per_step")
        except Exception:
            return None
    return None


# ---- digests: every block of a batch is checked, not a sample --------------------------------

_W = None


def _weights():
    global _W
    if _W is None:
        _W = (np.arange(CRYO_BLCKSZ // 8, dtype=np.int64) * 2 + 1) * np.int64(-7046029254386353131)
    return _W


def digest_np(blocks: np.ndarray) -> np.ndarray:
    """[n, 1 MiB] uint8 -> [n, 2] int64: the wrapping sum of the block's 64-bit words and a sum weighted by
    odd multipliers of the word index (so moved or swapped words change it)."""
    v = np.ascontiguousarray(blocks).reshape(-1, CRYO_BLCKSZ).view(np.int64)
    with np.errstate(over="ignore"):
        return np.stack([v.sum(axis=1), (v * _weights()).sum(axis=1)], axis=1)


def digest_torch(d_blocks):
    import torch
    v = d_blocks.view(torch.int64)
    w = torch.from_numpy(_weights()).to(d_blocks.device)
    out = torch.empty((v.shape[0], 2), dtype=torch.int64, device=d_blocks.device)
    for lo in range(0, v.shape[0], 256):            # bounded temporaries
        x = v[lo:lo + 256]
        out[lo:lo + 256, 0] = x.sum(dim=1)
        out[lo:lo + 256, 1] = (x * w).sum(dim=1)
    return out


class ClockSampler:
    """nvidia-smi clocks and throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def keep_sampling(sampler, dev, step):
    """The timed region is a few milliseconds, nvidia-smi samples every 100 ms: keep the same steps running
    (untimed) under the sampler until it has seen the clocks under this load."""
    import torch
    t_more = time.perf_counter()
    while len(sampler.rows) < 4 and time.perf_counter() - t_more < 3.0:
        for _ in range(20):
            step()
        torch.cuda.synchronize(dev)
    clocks = sampler.stop()
    clocks["note"] = "sampled every 100 ms over the timed steps and the same steps repeated after them"
    return clocks


def cpu_reference_decompress(method, chunks, threads: int, target_seconds: float):
    """The reference's compression.c (oracle/_ref) decompressing `chunks` on the host cores, repeated for
    about target_seconds.  Returns (GB/s, reps)."""
    from oracle import ref           # cpu_baseline leg: the one place bench.py touches oracle/
    buf, offs, sizes = ref.pack(chunks)
    out = np.empty((len(chunks), CRYO_BLCKSZ), dtype=np.uint8)
    methods = np.full(len(chunks), method, dtype=np.int32)
    _, ok, t1 = ref.decompress(methods, buf, offs, sizes, nthreads=threads, reps=1, out=out)
    assert ok.all()
    reps = max(1, min(200, int(target_seconds / max(t1, 1e-4))))
    _, ok, t = ref.decompress(methods, buf, offs, sizes, nthreads=threads, reps=reps, out=out)
    return len(chunks) * reps * CRYO_BLCKSZ / t / 1e9, reps


def cpu_reference_compress(method, level, blocks, threads: int, target_seconds: float):
    """-> (GB/s of input, sizes of the reference's output)"""
    from oracle import ref
    _, sizes, t1 = ref.compress(method, level, blocks, nthreads=threads, keep=False)
    reps = max(1, min(50, int(target_seconds / max(t1, 1e-4))))
    _, _, t = ref.compress(method, level, blocks, nthreads=threads, reps=reps, keep=False)
    return blocks.shape[0] * reps * CRYO_BLCKSZ / t / 1e9, sizes


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path on this box's host cores (rank 0 only), on the whole
    workload of the other arm."""
    if rank != 0:
        return
    import benchdata
    from pg_cryogen_b200 import blockgen as bg
    threads = os.cpu_count() or 1
    nblk = bg.table_block_count(args.rows, KIND)
    chunks, _ = benchdata.build_table(args.rows, KIND, PAYLOAD, METHOD, LEVEL, keep_plain=1, threads=min(threads, 16))
    from oracle import ref
    buf, offs, sizes = ref.pack(chunks)
    out = np.empty((nblk, CRYO_BLCKSZ), dtype=np.uint8)
    methods = np.full(nblk, METHOD, dtype=np.int32)
    for _ in range(max(args.warmup, 1)):
        ref.decompress(methods, buf, offs, sizes, nthreads=threads, out=out)
    times = []
    for _ in range(args.steps):
        _, ok, t = ref.decompress(methods, buf, offs, sizes, nthreads=threads, out=out)
        assert ok.all()
        times.append(t)
    ms = 1e3 * sum(times) / len(times)
    gbs = nblk * CRYO_BLCKSZ / (ms * 1e-3) / 1e9
    sample = f"all {nblk} zstd-1 S blocks per step, all {threads} host threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_string(args.rows, nblk), "blocks_per_gpu": nblk, "block_bytes": CRYO_BLCKSZ,
                   "compressed_bytes_per_gpu": int(sizes.astype(np.int64).sum())},
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "reference",
                         "sample": sample},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---- device helpers ---------------------------------------------------------------------------

class DeviceBatch:
    """Compressed blocks resident in HBM plus the outputs of the device call."""

    def __init__(self, dev, chunks, methods, block_size=CRYO_BLCKSZ):
        import torch
        from pg_cryogen_b200.codec import pack_chunks
        buf, offs, sizes = pack_chunks(chunks)
        n = len(chunks)
        self.n, self.block_size = n, block_size
        self.csize_total = int(sizes.astype(np.int64).sum())
        self.src = torch.from_numpy(buf).to(dev)
        self.off = torch.from_numpy(offs.view(np.int64)).to(dev)
        self.sz = torch.from_numpy(sizes.view(np.int32)).to(dev)
        m = np.ascontiguousarray(np.broadcast_to(np.asarray(methods, dtype=np.int32), (n,)))
        self.me = torch.from_numpy(m.copy()).to(dev)
        self.stride = (block_size + 15) & ~15
        self.dst = torch.empty((n, self.stride), dtype=torch.uint8, device=dev)
        self.osz = torch.zeros((n,), dtype=torch.int32, device=dev)
        self.st = torch.full((n,), -1, dtype=torch.int32, device=dev)
        self.stream = torch.cuda.current_stream(dev).cuda_stream

    def decode(self, gpu):
        gpu.decompress_device(self.me, self.src, self.off, self.sz, self.dst, self.stride, self.osz, self.st,
                              self.n, block_size=self.block_size, stream=self.stream)


DUMP_SEED, DUMP_SAMPLE = 20240611, 12        # 12 whole blocks as float32: 48 MiB of the at most 64 MB dumped


def dump_outputs(path: str, d_dst, d_osz, d_st) -> None:
    """What one batched decompression returned, as float .npy files under path, so that two builds can be
    compared output for output: the status and output size of every block, and the bytes of the first block,
    the last (partial) block and a fixed, seeded sample of the others."""
    import torch
    os.makedirs(path, exist_ok=True)
    nblk = d_dst.shape[0]
    rng = np.random.default_rng(DUMP_SEED)
    inner = rng.choice(np.arange(1, nblk - 1), size=min(DUMP_SAMPLE - 2, max(nblk - 2, 0)), replace=False)
    pick = np.unique(np.concatenate([[0, nblk - 1], inner]).astype(np.int64))
    blocks = d_dst[torch.from_numpy(pick).to(d_dst.device)].cpu().numpy()
    np.save(os.path.join(path, "status.npy"), d_st.cpu().numpy().astype(np.float64))
    np.save(os.path.join(path, "out_size.npy"), d_osz.cpu().numpy().astype(np.float64))
    np.save(os.path.join(path, "sample_index.npy"), pick.astype(np.float64))
    np.save(os.path.join(path, "sample_blocks.npy"), blocks.astype(np.float32))


def time_device(fn, dev, warmup: int, reps: int) -> float:
    """ms per call, CUDA events on the current (launching) stream."""
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def secondary_cells(gpu, dev, peak, uniq: int, n: int, threads: int):
    """BASELINE.json's metric beyond the headline cell: {lz4, zstd-1} x {decompress, compress} x block kinds
    on one GPU.  `uniq` different blocks per kind, tiled to n in HBM (n x 1 MiB is far above the L2)."""
    import torch
    from oracle import ref           # checker + cpu_baseline leg only
    from pg_cryogen_b200 import blockgen as bg
    from pg_cryogen_b200.codec import compress_bound
    cells = []
    tile = [i % uniq for i in range(n)]
    for kind, payload in SECONDARY_KINDS:
        blocks = bg.make_blocks(kind, payload, 1000, uniq)
        d_plain = torch.from_numpy(blocks).to(dev)
        want = digest_torch(d_plain)
        for method, level, name in ((COMP_LZ4, 1, "lz4 acceleration 1"), (COMP_ZSTD, 1, "zstd level 1")):
            comp, rsz, _ = ref.compress(method, level, blocks, nthreads=threads)
            # -- decompress: frames written by the reference's library
            batch = DeviceBatch(dev, [comp[i] for i in tile], method)
            ms = time_device(lambda: batch.decode(gpu), dev, 2, 5)
            ok = bool((batch.st == 0).all().item()) and bool((batch.osz == CRYO_BLCKSZ).all().item())
            got = digest_torch(batch.dst)
            exact = ok and bool((got == want[torch.tensor(tile, device=dev)]).all().item())
            alg = n * CRYO_BLCKSZ + batch.csize_total
            cpu_all, _ = cpu_reference_decompress(method, comp, threads, 1.0)
            cpu_one, _ = cpu_reference_decompress(method, comp[: max(4, uniq // 8)], 1, 0.5)
            cells.append({"op": "decompress", "codec": name, "blocks": f"{kind}/{payload}", "n_blocks": n,
                          "unique_blocks": uniq, "ms": ms, "value": n * CRYO_BLCKSZ / ms / 1e6, "unit": "GB/s",
                          "roofline_frac": alg / ms / 1e6 / peak, "algorithmic_bytes": alg, "bit_exact_all_blocks": exact,
                          "cpu_reference": {"all_cores": cpu_all, "one_thread": cpu_one, "cores": threads, "unit": "GB/s"}})
            del batch
            # -- compress: the GPU's blocks must be read back by the reference's decompressor
            bound = compress_bound(method)
            stride = (bound + 15) & ~15
            d_src = d_plain[torch.tensor(tile, device=dev)].contiguous()
            d_dst = torch.zeros((n, stride), dtype=torch.uint8, device=dev)
            d_sz = torch.zeros((n,), dtype=torch.int32, device=dev)
            d_st = torch.full((n,), -1, dtype=torch.int32, device=dev)
            stream = torch.cuda.current_stream(dev).cuda_stream

            def enc():
                gpu.compress_device(method, level, d_src, CRYO_BLCKSZ, d_dst, stride, stride, d_sz, d_st, n, stream=stream)
            ms = time_device(enc, dev, 1, 3)
            okc = bool((d_st == 0).all().item())
            gsz = d_sz[:uniq].cpu().numpy().astype(np.int64)
            out = d_dst[:uniq].cpu().numpy()
            gcomp = [out[i, : gsz[i]].copy() for i in range(uniq)]
            back, okd, _ = ref.decompress([method] * uniq, *ref.pack(gcomp), nthreads=threads)
            roundtrip = okc and bool(okd.all()) and np.array_equal(back, blocks)
            cpu_call, _ = cpu_reference_compress(method, level, blocks, threads, 1.0)
            cpu_cone, _ = cpu_reference_compress(method, level, blocks[: max(4, uniq // 8)], 1, 0.5)
            alg = n * CRYO_BLCKSZ + int(gsz.sum()) * (n // uniq)
            cells.append({"op": "compress", "codec": name, "blocks": f"{kind}/{payload}", "n_blocks": n,
                          "unique_blocks": uniq, "ms": ms, "value": n * CRYO_BLCKSZ / ms / 1e6, "unit": "GB/s of input",
                          "roofline_frac": alg / ms / 1e6 / peak, "algorithmic_bytes": alg,
                          "roundtrip_through_reference_decompressor": roundtrip,
                          "ratio_vs_reference": {"mean": float(gsz.sum() / rsz.astype(np.int64).sum()),
                                                 "worst_block": float(np.max(gsz / rsz.astype(np.float64)))},
                          "cpu_reference": {"all_cores": cpu_call, "one_thread": cpu_cone, "cores": threads,
                                            "unit": "GB/s of input"}})
            del d_src, d_dst
        del d_plain
    return cells


def next_row_cells(gpu, chunks, want, threads):
    """The rows SURVEY.md 8(f) marks "next", measured on the headline table through their host entry points:
    f-4 count pushdown (cryogpu_decompress_count_host) and f-1 decompress from page chains
    (cryogpu_decompress_pages_host, pages laid out by the restatement of the reference's split)."""
    from oracle import pages as opg, ref          # checker / input preparation only
    cells = []
    n = len(chunks)
    methods = np.full(n, METHOD, dtype=np.int32)
    # ---- f-4: select count(*) pushed down: compressed blocks in, 24 bytes per block out
    nt, by, st = gpu.decompress_count_host(methods, chunks)
    assert (st == 0).all() and int(nt.sum()) > 0
    t0 = time.perf_counter()
    for _ in range(3):
        nt, by, st = gpu.decompress_count_host(methods, chunks)
    t = (time.perf_counter() - t0) / 3
    bi, bo = gpu.last_transfer_bytes()
    # the reference: cryo_decompress + the item walk of cryo_getnextslot, all cores (the walk is negligible beside the codec)
    cpu_all, _ = cpu_reference_decompress(METHOD, chunks[: max(64, threads * 16)], threads, 2.0)
    cpu_one, _ = cpu_reference_decompress(METHOD, chunks[:64], 1, 1.0)     # one backend = one thread
    cells.append({"row": "f-4 count pushdown", "api": "cryogpu_decompress_count_host", "blocks": n, "tuples_counted": int(nt.sum()),
                  "value": n * CRYO_BLCKSZ / t / 1e9, "unit": "GB/s of decompressed data scanned", "h2d_bytes": bi, "d2h_bytes": bo,
                  "cpu_reference_all_cores": cpu_all, "cpu_reference_one_thread": cpu_one, "cores": threads})
    # ---- f-1: the same blocks as page chains on "disk" (8 KiB pages, first page header 48 bytes, others 32)
    m = min(n, 1024)
    npages = [opg.pages_needed(len(c)) for c in chunks[:m]]
    rel = np.zeros((sum(npages) + 1, 8192), dtype=np.uint8)
    chains, at = [], 1
    for i in range(m):
        ch = list(range(at, at + npages[i]))
        opg.split(rel, ch, chunks[i], METHOD, 1)
        chains.append(ch)
        at += npages[i]
    out, osz, st, me, csz = gpu.decompress_pages_host(rel, chains)
    assert (st == 0).all() and np.array_equal(digest_np(out), want[:m]), "page-chain decode differs"
    t0 = time.perf_counter()
    for _ in range(3):
        gpu.decompress_pages_host(rel, chains)
    t = (time.perf_counter() - t0) / 3
    cells.append({"row": "f-1 decompress from page chains", "api": "cryogpu_decompress_pages_host (pageable pages in, pageable blocks out, "
                  "every byte written; includes the Python binding's per-call array setup)", "blocks": m, "pages": int(sum(npages)),
                  "value": m * CRYO_BLCKSZ / t / 1e9, "unit": "GB/s", "bit_exact_all_blocks": True,
                  "cpu_reference_all_cores": cpu_all, "cpu_reference_one_thread": cpu_one, "cores": threads})
    cells += batched_caller_cells(gpu, threads)
    return cells


def batched_caller_cells(gpu, threads):
    """f-3 / f-2 through pg_cryogen_b200/host/cryo_batch.c over its in-memory relation: COPY of S-kind tuples with
    64 blocks per flush call, then a sequential scan with a read-ahead of 64 blocks."""
    import ctypes as C
    from oracle import ref
    from pg_cryogen_b200 import blockgen as bg

    class RelOps(C.Structure):
        _fields_ = [("rel", C.c_void_p), ("nblocks", C.c_void_p), ("read_page", C.c_void_p), ("extend", C.c_void_p)]
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
    L.cryo_batch_cache_create.restype = C.c_void_p
    L.cryo_batch_cache_create.argtypes = [C.c_void_p, C.c_int]
    L.cryo_batch_cache_destroy.argtypes = [C.c_void_p]
    L.cryo_batch_cache_stats.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 3
    L.cryo_batch_scan_begin.restype = C.c_void_p
    L.cryo_batch_scan_begin.argtypes = [C.c_void_p, C.POINTER(RelOps), C.c_int]
    L.cryo_batch_scan_next.restype = C.POINTER(C.c_uint8)
    L.cryo_batch_scan_next.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
    L.cryo_batch_scan_end.argtypes = [C.c_void_p]
    nblocks, per = 512, bg.KINDS["S"][0]
    tuples = np.concatenate([bg.make_tuples("S", "hex", 5000 + b, per) for b in range(nblocks)])
    rel = L.cryo_memrel_create(nblocks * 4 + 64)
    ops = L.cryo_memrel_ops(rel)
    cells = []
    w = L.cryo_batch_writer_create(gpu.handle, C.byref(ops), METHOD, LEVEL, 64, 7)
    t0 = time.perf_counter()
    rc = L.cryo_batch_insert_many(w, tuples.ctypes.data, tuples.shape[1], tuples.shape[0])
    rc = rc or L.cryo_batch_flush(w)
    t = time.perf_counter() - t0
    assert rc == 0
    calls, blocks, pages = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    L.cryo_batch_writer_stats(w, C.byref(calls), C.byref(blocks), C.byref(pages))
    t_flush = L.cryo_batch_writer_flush_seconds(w)
    L.cryo_batch_writer_destroy(w)
    plain = np.stack([bg.pack_block(tuples[b * per:(b + 1) * per]) for b in range(min(64, nblocks))])
    cpu_c, _ = cpu_reference_compress(METHOD, LEVEL, plain, threads, 1.0)
    cpu_c1, _ = cpu_reference_compress(METHOD, LEVEL, plain[:16], 1, 0.5)
    cells.append({"row": "f-3 batched flush on COPY", "api": "cryo_batch_insert / cryo_batch_flush (host/cryo_batch.c) -> "
                  "cryogpu_compress_pages_alloc_host, 64 blocks per device call; value = the flush calls (compress, page "
                  "split, copies both ways), as the reference beside it is cryo_compress alone",
                  "blocks": int(blocks.value), "device_calls": int(calls.value), "pages_written": int(pages.value),
                  "value": blocks.value * CRYO_BLCKSZ / t_flush / 1e9, "unit": "GB/s of block data",
                  "value_with_tuple_inserts": blocks.value * CRYO_BLCKSZ / t / 1e9,
                  "cpu_reference_all_cores": cpu_c, "cpu_reference_one_thread": cpu_c1, "cores": threads})
    cache = L.cryo_batch_cache_create(gpu.handle, 128)
    for attempt in range(2):                            # the second pass is the timed one (work areas are warm)
        L.cryo_batch_cache_destroy(cache)
        cache = L.cryo_batch_cache_create(gpu.handle, 128)
        scan = L.cryo_batch_scan_begin(cache, C.byref(ops), 64)
        bno, xid, err = C.c_uint32(0), C.c_uint32(0), C.c_int(0)
        got, first = 0, None
        t0 = time.perf_counter()
        while True:
            d = L.cryo_batch_scan_next(scan, C.byref(bno), C.byref(xid), C.byref(err))
            if not d:
                break
            if first is None:
                first = np.ctypeslib.as_array(d, shape=(CRYO_BLCKSZ,)).copy()
            got += 1
        t = time.perf_counter() - t0
        L.cryo_batch_scan_end(scan)
    assert err.value == 0 and got == blocks.value and np.array_equal(first, plain[0]), (err.value, got)
    L.cryo_batch_cache_stats(cache, C.byref(calls), C.byref(blocks), C.byref(pages))
    pc = ref.compress(METHOD, LEVEL, plain, nthreads=threads)[0]
    cpu_d, _ = cpu_reference_decompress(METHOD, pc, threads, 1.0)
    cpu_d1, _ = cpu_reference_decompress(METHOD, pc[:16], 1, 0.5)
    cells.append({"row": "f-2 batched cache fill / read-ahead", "api": "cryo_batch_scan_next (host/cryo_batch.c) -> "
                  "cryogpu_decompress_pages_host, read-ahead 64 blocks per device call, every byte of every block written",
                  "blocks": got, "device_calls": int(calls.value), "value": got * CRYO_BLCKSZ / t / 1e9, "unit": "GB/s",
                  "cpu_reference_all_cores": cpu_d, "cpu_reference_one_thread": cpu_d1, "cores": threads})
    L.cryo_batch_cache_destroy(cache)
    L.cryo_memrel_destroy(rel)
    return cells


# ---- BASELINE.json configs[2]: lz4_acceleration sweep on 64 KiB blocks ---------------------------

def run_config3(args, gpu, dev, rank, world):
    import torch
    import benchdata
    from pg_cryogen_b200 import blockgen as bg
    from pg_cryogen_b200.codec import compress_bound
    bs = 64 << 10
    peak, peak_src = measured_peak()
    threads = os.cpu_count() or 1
    per_kind = 16                       # 1 MiB blocks per kind, cut into 64 KiB pieces
    pieces = np.concatenate([bg.make_blocks(k, p, 2000, per_kind).reshape(-1, bs) for k, p in SECONDARY_KINDS])
    n = pieces.shape[0]
    reps = 8                            # tiled in HBM: 8 x 1 536 pieces = 805 MB per launch
    d_src = torch.from_numpy(pieces).to(dev).repeat(reps, 1).contiguous()
    bound = compress_bound(COMP_LZ4, bs)
    stride = (bound + 15) & ~15
    d_dst = torch.zeros((n * reps, stride), dtype=torch.uint8, device=dev)
    d_sz = torch.zeros((n * reps,), dtype=torch.int32, device=dev)
    d_st = torch.full((n * reps,), -1, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    scratch = np.empty(bound + 64, dtype=np.uint8)
    rows = []
    for accel in (1, 2, 3, 5, 8, 10, 15, 20, 25, 30, 40, 50):
        def enc():
            gpu.compress_device(COMP_LZ4, accel, d_src, bs, d_dst, stride, stride, d_sz, d_st, n * reps,
                                block_size=bs, stream=stream)
        ms = time_device(enc, dev, 1, 3)
        assert bool((d_st == 0).all().item())
        gsz = d_sz[:n].cpu().numpy().astype(np.int64)
        t0 = time.perf_counter()
        rsz = np.array([benchdata.library_compress(COMP_LZ4, accel, pieces[i], scratch).size for i in range(n)], dtype=np.int64)
        t_cpu = time.perf_counter() - t0
        # conformance: a sample of the GPU's blocks back through liblz4 (the reference's decompressor for this size)
        out = d_dst[:n:97].cpu().numpy()
        lz4 = benchdata._libs()[0]
        back = np.empty(bs, dtype=np.uint8)
        for j, i in enumerate(range(0, n, 97)):
            c = np.ascontiguousarray(out[j, : gsz[i]])
            got = lz4.LZ4_decompress_safe(c.ctypes.data, back.ctypes.data, int(gsz[i]), bs)
            assert got == bs and np.array_equal(back, pieces[i]), "liblz4 cannot read the GPU's block"
        rows.append({"lz4_acceleration": accel, "gpu_GBps_in": n * reps * bs / ms / 1e6, "ms": ms,
                     "ratio_vs_reference_mean": float(gsz.sum() / rsz.sum()),
                     "ratio_vs_reference_worst_piece": float(np.max(gsz / rsz)),
                     "gpu_compression_ratio": float(n * bs / gsz.sum()), "reference_compression_ratio": float(n * bs / rsz.sum()),
                     "cpu_reference_GBps_in_1_thread": n * bs / t_cpu / 1e9,
                     "roofline_frac": (n * reps * bs + int(gsz.sum()) * reps) / ms / 1e6 / peak})
    if rank == 0:
        best = rows[0]
        print(json.dumps({
            "metric": "compress_GBps_lz4_accel_sweep_64KiB_blocks", "value": best["gpu_GBps_in"], "unit": "GB/s",
            "n_gpus": world, "steps": 3, "warmup": 1, "ms_per_step": best["ms"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"lz4_acceleration 1..50 on {n * reps} blocks of 64 KiB ({n} different pieces of S/M/D x hex/lowcard "
                                   "cryo blocks), compress; value = acceleration 1", "block_bytes": bs,
                       "l2": "805 MB read per launch, above the 126 MB L2"},
            "sweep": rows, "roofline": {"bound": "hbm", "achieved": best["roofline_frac"] * peak, "peak": peak, "unit": "GB/s",
                                        "frac": best["roofline_frac"], "traffic": None, "peak_source": peak_src},
            "gpu_launches": 12 * 4}), flush=True)


# ---- BASELINE.json configs[3]: zstd levels -5..3, ~10 GB sharded over the ranks (strong scaling) ---

def run_config4(args, gpu, dev, rank, world):
    import torch
    import torch.distributed as dist
    from oracle import ref
    from pg_cryogen_b200 import blockgen as bg, shard
    from pg_cryogen_b200.codec import compress_bound
    peak, peak_src = measured_peak()
    threads = max(1, (os.cpu_count() or 8) // world)
    total_blocks = args.blocks or 10240                 # 10 GiB of cryo blocks
    lo, hi = shard.block_range(total_blocks, rank, world)
    mine = hi - lo
    uniq = 16                                           # per kind; the job's blocks are these 96, in rotation
    pool = np.concatenate([bg.make_blocks(k, p, 3000, uniq) for k, p in SECONDARY_KINDS])
    idx = torch.tensor([(b * 37) % pool.shape[0] for b in range(lo, hi)], device=dev)
    d_pool = torch.from_numpy(pool).to(dev)
    d_src = d_pool[idx].contiguous()
    want = digest_torch(d_pool)[idx]
    bound = compress_bound(COMP_ZSTD)
    stride = (bound + 15) & ~15
    d_comp = torch.zeros((mine, stride), dtype=torch.uint8, device=dev)
    d_csz = torch.zeros((mine,), dtype=torch.int32, device=dev)
    d_cst = torch.full((mine,), -1, dtype=torch.int32, device=dev)
    d_off = (torch.arange(mine, device=dev, dtype=torch.int64) * stride)
    d_me = torch.full((mine,), COMP_ZSTD, dtype=torch.int32, device=dev)
    d_out = torch.empty((mine, CRYO_BLCKSZ), dtype=torch.uint8, device=dev)
    d_osz = torch.zeros((mine,), dtype=torch.int32, device=dev)
    d_st = torch.full((mine,), -1, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    rows = []
    for level in range(-5, 4):
        if level == 0:
            continue                                    # ZSTD_compress treats 0 as the default level 3
        def enc():
            gpu.compress_device(COMP_ZSTD, level, d_src, CRYO_BLCKSZ, d_comp, stride, stride, d_csz, d_cst, mine, stream=stream)

        def dec():
            gpu.decompress_device(d_me, d_comp.view(-1), d_off, d_csz, d_out, CRYO_BLCKSZ, d_osz, d_st, mine, stream=stream)
        enc()
        barrier()
        t_enc = shard.max_over_ranks(time_device(enc, dev, 0, 2), dev)
        assert bool((d_cst == 0).all().item())
        dec()
        barrier()
        t_dec = shard.max_over_ranks(time_device(dec, dev, 0, 2), dev)
        ok = bool((d_st == 0).all().item()) and bool((digest_torch(d_out) == want).all().item())
        assert ok, "decompress(compress(x)) != x"
        row = {"zstd_compression_level": level, "compress_GBps_in": total_blocks * CRYO_BLCKSZ / t_enc / 1e6,
               "decompress_GBps_out": total_blocks * CRYO_BLCKSZ / t_dec / 1e6, "compress_ms": t_enc, "decompress_ms": t_dec,
               "roundtrip_bit_exact_all_blocks": ok}
        if rank == 0:
            # ratio and CPU rates on the pool (the job's blocks are the pool in rotation); conformance: the reference's
            # libzstd reads the GPU's frames of the first blocks of this rank
            gsz = d_csz[: pool.shape[0]].cpu().numpy().astype(np.int64)
            order = idx[: pool.shape[0]].cpu().numpy()
            _, rsz, t_c = ref.compress(COMP_ZSTD, level, pool, nthreads=threads, keep=False)
            rsz = rsz.astype(np.int64)
            out = d_comp[:32].cpu().numpy()
            back, okd, _ = ref.decompress([COMP_ZSTD] * 32, *ref.pack([out[i, : gsz[i]] for i in range(32)]), nthreads=threads)
            assert okd.all() and np.array_equal(back, pool[order[:32]]), "libzstd cannot read the GPU's frames"
            rc, _, _ = ref.compress(COMP_ZSTD, level, pool, nthreads=threads)
            _, _, t_d = ref.decompress([COMP_ZSTD] * len(rc), *ref.pack(rc), nthreads=threads)
            row.update({"ratio_vs_reference_mean": float(gsz.sum() / rsz[order].sum()),
                        "ratio_vs_reference_worst_block": float(np.max(gsz / rsz[order])),
                        "cpu_reference_compress_GBps": pool.shape[0] * CRYO_BLCKSZ / t_c / 1e9,
                        "cpu_reference_decompress_GBps": pool.shape[0] * CRYO_BLCKSZ / t_d / 1e9, "cpu_threads": threads})
        rows.append(row)
    if rank == 0:
        l1 = [r for r in rows if r["zstd_compression_level"] == 1][0]
        alg = total_blocks * CRYO_BLCKSZ * (1 + 1.0 / max(l1.get("ratio_vs_reference_mean", 1.0), 1e-9) * 0 + 0.3)
        print(json.dumps({
            "metric": "compress+decompress_GBps_zstd_levels_-5..3_10GB", "value": l1["decompress_GBps_out"], "unit": "GB/s",
            "n_gpus": world, "steps": 2, "warmup": 1, "ms_per_step": l1["decompress_ms"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"{total_blocks} cryo blocks of 1 MiB (S/M/D x hex/lowcard in rotation, 96 different blocks), zstd "
                                   "levels -5..3: GPU compress, then GPU decompress of those frames; value = level 1 decompress; "
                                   f"block range sharded over {world} rank(s), no collective", "block_bytes": CRYO_BLCKSZ,
                       "blocks_total": total_blocks, "l2": "every launch reads and writes GBs per GPU, far above the L2",
                       "parallelism": f"block-range shards x{world}"},
            "levels": rows,
            "roofline": {"bound": "hbm", "achieved": l1["decompress_GBps_out"], "peak": peak * world, "unit": "GB/s",
                         "frac": l1["decompress_GBps_out"] / (peak * world), "traffic": None, "peak_source": peak_src,
                         "note": "output bytes only (the compressed size differs per level)"},
            "gpu_launches": 8 * 2 * 16}), flush=True)


# ---- BASELINE.json configs[4]: small batches through the device call ----------------------------

def run_config5(args, gpu, dev, rank, world):
    import torch
    from oracle import ref
    from pg_cryogen_b200 import blockgen as bg
    threads = os.cpu_count() or 1
    kinds = [("S", "hex"), ("M", "hex"), ("D", "lowcard"), ("S", "lowcard"), ("M", "lowcard"), ("D", "hex")]
    blocks = np.stack([bg.make_block(k, p, 4000 + i) for i, (k, p) in enumerate(kinds * 6)])
    z, _, _ = ref.compress(COMP_ZSTD, 1, blocks, nthreads=min(threads, 16))
    l, _, _ = ref.compress(COMP_LZ4, 1, blocks, nthreads=min(threads, 16))
    want_all = digest_np(blocks)
    rows = []
    for n in (1, 2, 4, 8, 16, 32, 64, 128, 256):
        methods = [i & 1 for i in range(n)]
        chunks = [(z if methods[i] else l)[i % len(z)] for i in range(n)]
        batch = DeviceBatch(dev, chunks, methods)
        ts = []
        for it in range(120):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            batch.decode(gpu)
            torch.cuda.synchronize(dev)
            ts.append(time.perf_counter() - t0)
        ts = np.sort(np.array(ts[20:])) * 1e6
        ok = bool((batch.st == 0).all().item())
        exact = ok and np.array_equal(digest_torch(batch.dst).cpu().numpy(), want_all[[i % len(z) for i in range(n)]])
        rb, ro, rs = ref.pack(chunks)
        ref.decompress(methods, rb, ro, rs, nthreads=1)
        cpu1 = ref.decompress(methods, rb, ro, rs, nthreads=1, reps=3)[2] / 3 * 1e6
        cpun = ref.decompress(methods, rb, ro, rs, nthreads=threads, reps=3)[2] / 3 * 1e6
        rows.append({"batch": n, "gpu_p50_us": float(ts[len(ts) // 2]), "gpu_p99_us": float(ts[int(len(ts) * 0.99)]),
                     "gpu_GBps_at_p50": n * CRYO_BLCKSZ / float(ts[len(ts) // 2]) / 1e3, "bit_exact": exact,
                     "cpu_reference_us_1_thread": cpu1, f"cpu_reference_us_{threads}_threads": cpun})
    if rank == 0:
        r256 = rows[-1]
        print(json.dumps({
            "metric": "decompress_small_batches_latency", "value": r256["gpu_GBps_at_p50"], "unit": "GB/s", "n_gpus": world,
            "steps": 100, "warmup": 20, "ms_per_step": r256["gpu_p50_us"] / 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "batches of 1..256 cryo blocks (lz4 and zstd-1 alternating; S/M/D x hex/lowcard in rotation) "
                                   "through cryogpu_decompress_device, host-timed call + synchronize; value = batch 256",
                       "block_bytes": CRYO_BLCKSZ},
            "batches": rows, "gpu_launches": 12 * 120 * len(rows)}), flush=True)


# ---- headline ------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cryogpu", choices=["cryogpu", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="2: headline (default); 3: lz4 acceleration sweep; 4: zstd levels, 10 GB, strong scaling; 5: small batches")
    ap.add_argument("--rows", type=int, default=NROWS, help="table rows (default: the 1M-row config)")
    ap.add_argument("--blocks", type=int, default=0, help="--config 4: blocks in the job (default 10240)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="headline only: write what the last timed step returned (every block's status and size, a "
                         "fixed sample of decoded blocks) to DIR/<name>.npy, from rank 0")
    args = ap.parse_args()
    if args.dump_outputs and (args.config != 2 or args.impl != "cryogpu"):
        ap.error("--dump-outputs applies to the headline (--config 2, --impl cryogpu)")
    args.warmup = max(args.warmup, 3) if args.impl == "cryogpu" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import benchdata
    from pg_cryogen_b200 import CryoGPU, blockgen as bg, shard
    from pg_cryogen_b200.codec import pack_chunks

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libcryogpu has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    host_threads = max(1, (os.cpu_count() or 8) // max(world, 1))
    # host threads of the library's result placement (sparse return): this rank's share of cores
    os.environ.setdefault("CRYOGPU_HOST_THREADS", str(max(1, min(16, host_threads))))
    gpu = CryoGPU(local_rank)

    if args.config != 2:
        {3: run_config3, 4: run_config4, 5: run_config5}[args.config](args, gpu, dev, rank, world)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- workload: this rank's table (weak scaling: same shape, different block seeds) ----
    nblk = bg.table_block_count(args.rows, KIND)
    chunks, plain = benchdata.build_table(args.rows, KIND, PAYLOAD, METHOD, LEVEL, keep_plain=nblk,
                                          threads=min(host_threads, 16),
                                          block_seed_offset=shard.rank_block_seed_offset(rank, nblk))
    want = digest_np(plain)                             # of EVERY block of the table
    plain_head = plain[:8].copy()
    del plain
    buf, offs, sizes = pack_chunks(chunks)
    csize_total = int(sizes.astype(np.int64).sum())
    d_src = torch.from_numpy(buf).to(dev)
    d_off = torch.from_numpy(offs.view(np.int64)).to(dev)
    d_sz = torch.from_numpy(sizes.view(np.int32)).to(dev)
    d_me = torch.full((nblk,), METHOD, dtype=torch.int32, device=dev)
    d_dst = torch.empty((nblk, CRYO_BLCKSZ), dtype=torch.uint8, device=dev)
    d_osz = torch.zeros((nblk,), dtype=torch.int32, device=dev)
    d_st = torch.full((nblk,), -1, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def step():
        gpu.decompress_device(d_me, d_src, d_off, d_sz, d_dst, CRYO_BLCKSZ, d_osz, d_st, nblk,
                              stream=stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
    barrier()
    # correctness gate over all blocks: a wrong result is not a benchmark result
    assert bool((d_st == 0).all().item()), "decode status != 0"
    assert bool((d_osz == CRYO_BLCKSZ).all().item()), "decoded size != 1 MiB"
    assert np.array_equal(digest_torch(d_dst).cpu().numpy(), want), "decoded bytes differ (digest of every block)"
    assert np.array_equal(d_dst[:8].cpu().numpy(), plain_head), "decoded bytes differ"

    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for k in range(args.steps):
        step()
        ev[k + 1].record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_dst, d_osz, d_st)
    clocks = keep_sampling(sampler, dev, step)
    total_ms = ev[0].elapsed_time(ev[-1])
    step_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    total_ms = shard.max_over_ranks(total_ms, dev)          # slowest rank, on-device events
    ms_per_step = total_ms / args.steps
    value = shard.whole_job_rate(nblk * CRYO_BLCKSZ, world, ms_per_step * 1e-3) / 1e9
    assert np.array_equal(digest_torch(d_dst).cpu().numpy(), want), "decoded bytes differ after the timed steps"

    # ---- roofline of the step: one batched decompression = the launches of the zstd pipeline
    #      (zstd_decode_p.cuh: parse, Huffman tables, literal streams, FSE tables, sequence walk
    #      x2 size classes, raw/RLE blocks, executor) plus launches that exit at once.  The
    #      algorithmic bytes are the step's, so the duration is the step's too (CUDA events on the
    #      launching stream; the side streams are joined into it before the step ends). ----
    peak, peak_src = measured_peak()
    kern_ms = statistics.mean(step_ms)
    alg_bytes = nblk * CRYO_BLCKSZ + csize_total
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    frames, fallback = gpu.zstd_pipeline_stats()
    assert frames == nblk and fallback == 0, "the zstd pipeline handed frames to the fallback decoder"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": recorded_traffic(), "peak_source": peak_src,
                "frac_of_nominal_8TBps": achieved / 8000.0,
                "kernel": "zstd pipeline (k_zp_parse, k_zp_huftab, k_zp_literals, k_zp_fsetab, "
                          "k_zp_sequences_small/large, k_zp_prefill_early, k_zp_prefill, k_zp_execute); by "
                          "device time k_zp_execute and k_zp_prefill dominate (profiles/)",
                "algorithmic_bytes_per_launch": alg_bytes,
                "frames_decoded_by_fallback_kernel": fallback}

    # ---- e2e: host buffers through the C ABI, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        import ctypes as C
        lib = gpu.lib
        in_bytes = int(buf.size)
        h_in = lib.cryogpu_host_alloc(in_bytes)
        if not h_in:
            raise SystemExit("pinned allocation failed")
        C.memmove(h_in, buf.ctypes.data, in_bytes)
        srcp = (C.c_void_p * nblk)(*[h_in + int(o) for o in offs])
        methods = np.full(nblk, METHOD, dtype=np.int32)
        osz = np.zeros(nblk, dtype=np.uint32)
        st = np.full(nblk, -1, dtype=np.int32)
        e2e_steps = max(1, min(args.steps, 5))

        def run_e2e(out_base, unmap):
            """(GB/s whole job, h2d, d2h) into the blocks at out_base"""
            dstp = (C.c_void_p * nblk)(*[out_base + i * CRYO_BLCKSZ for i in range(nblk)])
            lib.cryogpu_set_zero_by_unmap(gpu.handle, 1 if unmap else 0)

            def host_step():
                rc = lib.cryogpu_decompress_host(gpu.handle, nblk, methods.ctypes.data, srcp,
                                                 sizes.ctypes.data, dstp, CRYO_BLCKSZ,
                                                 osz.ctypes.data, st.ctypes.data)
                if rc != 0:
                    raise SystemExit("cryogpu_decompress_host: " + lib.cryogpu_last_error().decode())
            st[:] = -1
            host_step()
            assert (st == 0).all()
            got = np.ctypeslib.as_array(C.cast(out_base, C.POINTER(C.c_uint8)), shape=(nblk, CRYO_BLCKSZ))
            assert np.array_equal(digest_np(got), want), "e2e bytes differ (digest of every block)"
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                host_step()
            torch.cuda.synchronize(dev)
            t = shard.max_over_ranks((time.perf_counter() - t0) / e2e_steps, dev)
            assert np.array_equal(digest_np(got), want), "e2e bytes differ after the timed steps"
            bi, bo = gpu.last_transfer_bytes()          # counted by the library from what it copied
            lib.cryogpu_set_zero_by_unmap(gpu.handle, 0)
            return shard.whole_job_rate(nblk * CRYO_BLCKSZ, world, t) / 1e9, bi, bo

        # (1) the caller's blocks are private anonymous memory, as the reference's per-backend cache is (cache.c:49):
        #     zero runs are returned to the kernel (cryogpu_set_zero_by_unmap), non-zero pages are copied in
        out_np = np.empty(nblk * CRYO_BLCKSZ + 4096, dtype=np.uint8)
        v1, bi, bo = run_e2e(out_np.ctypes.data, True)
        # (2) pinned destination, every byte of every block written by the library (streaming stores)
        h_out = lib.cryogpu_host_alloc(nblk * CRYO_BLCKSZ)
        if not h_out:
            raise SystemExit("pinned allocation failed")
        v2, _, _ = run_e2e(h_out, False)
        e2e = {"value": v1, "unit": "GB/s", "h2d_bytes_per_step": bi, "d2h_bytes_per_step": bo, "steps": e2e_steps,
               "api": "cryogpu_decompress_host: compressed blocks in pinned host memory, destination blocks in private "
                      "anonymous host memory (what the reference's cache is, cache.c:49).  Only the non-zero 4 KiB pages of "
                      "each decoded block cross the bus; the library copies them into the caller's block and gives the whole "
                      "OS pages of the zero runs back to the kernel (cryogpu_set_zero_by_unmap: they read as zeros, on "
                      "demand).  Every block is read back and checked (digest) before and after the timed steps.",
               "value_every_byte_written": v2,
               "every_byte_written": "the same call into a pinned destination: the library writes the zero runs itself with "
                                     "%s host threads (streaming stores); host-DRAM-bound" % os.environ["CRYOGPU_HOST_THREADS"]}
        lib.cryogpu_host_free(h_in)
        lib.cryogpu_host_free(h_out)
        del out_np

    # ---- CPU baseline beside it: the reference's compression.c on this box's cores ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import ref
        threads = os.cpu_count() or 1
        sample = chunks[: min(len(chunks), max(64, threads * 16))]
        gbs_all, reps = cpu_reference_decompress(METHOD, sample, threads, 10.0)
        gbs_one, _ = cpu_reference_decompress(METHOD, sample, 1, 4.0)
        cpu = {"value": gbs_all, "unit": "GB/s", "cores": threads, "kind": "reference",
               "sample": f"{len(sample)} of the {nblk} blocks x {reps} passes through {ref.describe()}, "
                         f"{threads} threads",
               "value_1_thread": gbs_one}

    # ---- the rest of the metric: lz4 and zstd-1, both directions, every block kind ----
    secondary = next_rows = None
    if rank == 0 and world == 1 and not args.no_secondary:
        del d_dst, d_src
        torch.cuda.empty_cache()
        secondary = secondary_cells(gpu, dev, peak, uniq=32, n=512, threads=os.cpu_count() or 1)
        next_rows = next_row_cells(gpu, chunks, want, os.cpu_count() or 1)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_string(args.rows, nblk),
                       "blocks_per_gpu": nblk, "block_bytes": CRYO_BLCKSZ,
                       "compressed_bytes_per_gpu": csize_total,
                       "l2": "each step writes %.2f GB per GPU, far above the 126 MB L2"
                             % (nblk * CRYO_BLCKSZ / 1e9),
                       "parallelism": f"block-range shards x{world}, no collective",
                       "gate": "status, size and a 128-bit digest of every decoded block, before and after the timed steps"},
            "ms_per_step_min_median_max": [min(step_ms), statistics.median(step_ms), max(step_ms)],
            "clocks": clocks, "e2e": e2e, "gpu_launches": LAUNCHES_PER_STEP * args.steps, "roofline": roofline,
            "cpu_baseline": cpu, "secondary": secondary, "next_rows": next_rows,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
