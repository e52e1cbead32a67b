"""ctypes binding of libcryogpu.so (include/cryogpu.h).

Mirrors the reference's codec boundary (compression.h:7-24): methods COMP_LZ4 /
COMP_ZSTD, compress one 1 MiB cryo block, decompress into a 1 MiB buffer -- but
batched, because a GPU wants many independent blocks per launch.  There is no
fallback: if libcryogpu.so is missing or no B200 is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

COMP_LZ4, COMP_ZSTD = 0, 1              # compression.h:7-11
CRYO_BLCKSZ = 1 << 20                   # storage.h:18

STATUS_NAMES = {0: "ok", 1: "input", 2: "output", 3: "offset", 4: "format", 5: "size",
                6: "method", 7: "unsupported"}

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


class CryoGPUError(RuntimeError):
    """Call-level failure of libcryogpu (the C shim turns these into elog(ERROR))."""


def lib_path() -> str:
    """libcryogpu.so beside this file; CRYOGPU_LIB names another build of it (A/B runs of development variants)."""
    return os.environ.get("CRYOGPU_LIB") or os.path.join(_HERE, "libcryogpu.so")


_PROTOS = {
    "cryogpu_version": (C.c_int, []),
    "cryogpu_last_error": (C.c_char_p, []),
    "cryogpu_status_string": (C.c_char_p, [C.c_int]),
    "cryogpu_device_count": (C.c_int, []),
    "cryogpu_init": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "cryogpu_shutdown": (None, [C.c_void_p]),
    "cryogpu_device": (C.c_int, [C.c_void_p]),
    "cryogpu_compress_bound": (C.c_uint64, [C.c_int, C.c_uint64]),
    "cryogpu_host_alloc": (C.c_void_p, [C.c_size_t]),
    "cryogpu_host_free": (None, [C.c_void_p]),
    "cryogpu_decompress_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                            C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_compress_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p,
                                          C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64,
                                          C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_set_zero_by_unmap": (C.c_int, [C.c_void_p, C.c_int]),
    "cryogpu_last_transfer_bytes": (None, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "cryogpu_zstd_pipeline_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "cryogpu_lz4_route_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "cryogpu_decompress_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                          C.c_void_p]),
    "cryogpu_compress_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p,
                                        C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p,
                                        C.c_void_p]),
    "cryogpu_pages_needed": (C.c_uint32, [C.c_uint64]),
    "cryogpu_decompress_pages_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64, C.c_uint32,
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_compress_pages_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_uint64,
                                                C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_decompress_pages_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p]),
    "cryogpu_compress_pages_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_uint32,
                                              C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p]),
    "cryogpu_compress_pages_alloc_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_uint32,
                                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_build_blocks_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "cryogpu_compress_tuples_pages_alloc_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_uint64,
                                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                                           C.c_void_p, C.c_void_p]),
    "cryogpu_tuple_stats_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_decompress_count_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                                C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_tuples_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_decompress_tuples_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                                 C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cryogpu_decompress_pages_tuples_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                                       C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                                       C.c_void_p, C.c_void_p]),
    "cryogpu_decompress_host_multi": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                                C.c_void_p, C.c_void_p]),
    "cryogpu_compress_host_multi": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_int,
                                              C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32,
                                              C.c_void_p, C.c_void_p]),
}


def exported_symbols() -> list[str]:
    """Every symbol include/cryogpu.h declares."""
    return sorted(_PROTOS)


def load_library():
    """dlopen libcryogpu.so and bind the C ABI.  Raises if the library is not built."""
    global _lib
    if _lib is None:
        p = lib_path()
        if not os.path.exists(p):
            raise CryoGPUError(f"{p} is not built (run `python -c 'import __graft_entry__ as g; "
                               "g.build()'`); there is no CPU fallback")
        L = C.CDLL(p)
        for name, (res, args) in _PROTOS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def compress_bound(method: int, block_size: int = CRYO_BLCKSZ) -> int:
    return int(load_library().cryogpu_compress_bound(method, block_size))


def _stream(s):
    """cudaStream_t handle for the C ABI: None -> the context's own stream; torch's default
    stream has handle 0, which the C ABI spells cudaStreamLegacy (1)."""
    if s is None:
        return None
    return 1 if int(s) == 0 else int(s)


def _ptr(t):
    """data pointer of a torch tensor / numpy array / int"""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


class CryoGPU:
    """One libcryogpu context (one GPU)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.cryogpu_init(device, C.byref(h))
        if rc != 0:
            raise CryoGPUError(f"cryogpu_init({device}) = {rc}: {self.lib.cryogpu_last_error().decode()}")
        self.handle = h
        self.device = device

    def last_transfer_bytes(self) -> tuple[int, int]:
        """(host->device, device->host) bytes of the last decompress_host call."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        self.lib.cryogpu_last_transfer_bytes(self.handle, C.byref(a), C.byref(b))
        return int(a.value), int(b.value)

    def zstd_pipeline_stats(self) -> tuple[int, int]:
        """(zstd frames given to the phase-split pipeline, frames it handed to the fallback decoder)
        of the last decompress_device call."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        rc = self.lib.cryogpu_zstd_pipeline_stats(self.handle, C.byref(a), C.byref(b))
        if rc != 0:
            raise CryoGPUError("cryogpu_zstd_pipeline_stats: " + self.lib.cryogpu_last_error().decode())
        return int(a.value), int(b.value)

    def lz4_route_stats(self) -> tuple[int, int]:
        """(blocks of the last routed decompress_device call, blocks the router gave to the CTA-per-block decoder)."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        rc = self.lib.cryogpu_lz4_route_stats(self.handle, C.byref(a), C.byref(b))
        if rc != 0:
            raise CryoGPUError("cryogpu_lz4_route_stats: " + self.lib.cryogpu_last_error().decode())
        return int(a.value), int(b.value)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.cryogpu_shutdown(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise CryoGPUError(f"{what} = {rc}: {self.lib.cryogpu_last_error().decode()}")

    # ---- device-resident batches (torch CUDA tensors or raw device pointers) ----

    def decompress_device(self, methods, src, src_off, src_size, dst, dst_stride, out_size, status,
                          n: int, block_size: int = CRYO_BLCKSZ, stream: int | None = None):
        self._check(self.lib.cryogpu_decompress_device(
            self.handle, n, _ptr(methods), _ptr(src), _ptr(src_off), _ptr(src_size), _ptr(dst),
            dst_stride, block_size, _ptr(out_size), _ptr(status), _stream(stream)),
            "cryogpu_decompress_device")

    def compress_device(self, method: int, level_or_accel: int, src, src_stride, dst, dst_stride,
                        dst_cap, dst_size, status, n: int, block_size: int = CRYO_BLCKSZ,
                        stream: int | None = None):
        self._check(self.lib.cryogpu_compress_device(
            self.handle, n, method, level_or_accel, _ptr(src), src_stride, block_size, _ptr(dst),
            dst_stride, dst_cap, _ptr(dst_size), _ptr(status), _stream(stream)),
            "cryogpu_compress_device")

    # ---- host batches (numpy) ----

    def decompress_host(self, methods, chunks, block_size: int = CRYO_BLCKSZ, out: np.ndarray | None = None):
        """chunks: list of uint8 arrays.  Returns (out [n, block_size], out_size, status)."""
        n = len(chunks)
        chunks = [np.ascontiguousarray(c, dtype=np.uint8) for c in chunks]
        methods = np.ascontiguousarray(np.broadcast_to(np.asarray(methods, dtype=np.int32), (n,)))
        sizes = np.array([c.size for c in chunks], dtype=np.uint32)
        if out is None:
            out = np.zeros((n, block_size), dtype=np.uint8)
        srcp = (C.c_void_p * n)(*[c.ctypes.data for c in chunks])
        dstp = (C.c_void_p * n)(*[out[i].ctypes.data for i in range(n)])
        osz = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        self._check(self.lib.cryogpu_decompress_host(
            self.handle, n, methods.ctypes.data, srcp, sizes.ctypes.data, dstp, block_size,
            osz.ctypes.data, st.ctypes.data), "cryogpu_decompress_host")
        return out, osz, st

    def compress_host(self, method: int, level_or_accel: int, blocks: np.ndarray,
                      block_size: int = CRYO_BLCKSZ):
        """blocks: [n, block_size] uint8.  Returns (list of compressed arrays, status)."""
        blocks = np.ascontiguousarray(blocks, dtype=np.uint8).reshape(-1, block_size)
        n = blocks.shape[0]
        bound = compress_bound(method, block_size)
        dst = np.zeros((n, bound), dtype=np.uint8)
        srcp = (C.c_void_p * n)(*[blocks[i].ctypes.data for i in range(n)])
        dstp = (C.c_void_p * n)(*[dst[i].ctypes.data for i in range(n)])
        sz = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        self._check(self.lib.cryogpu_compress_host(
            self.handle, n, method, level_or_accel, srcp, block_size, dstp, bound,
            sz.ctypes.data, st.ctypes.data), "cryogpu_compress_host")
        return [dst[i, : sz[i]].copy() for i in range(n)], st


    def decompress_count_host(self, methods, chunks, block_size: int = CRYO_BLCKSZ):
        """Count pushdown: (ntuples, tuple_bytes, status) per block; the decoded blocks stay in HBM."""
        n = len(chunks)
        chunks = [np.ascontiguousarray(c, dtype=np.uint8) for c in chunks]
        methods = np.ascontiguousarray(np.broadcast_to(np.asarray(methods, dtype=np.int32), (n,)))
        sizes = np.array([c.size for c in chunks], dtype=np.uint32)
        srcp = (C.c_void_p * n)(*[c.ctypes.data for c in chunks])
        nt = np.zeros(n, dtype=np.uint32)
        by = np.zeros(n, dtype=np.uint64)
        st = np.full(n, -1, dtype=np.int32)
        self._check(self.lib.cryogpu_decompress_count_host(
            self.handle, n, methods.ctypes.data, srcp, sizes.ctypes.data, block_size, nt.ctypes.data,
            by.ctypes.data, st.ctypes.data), "cryogpu_decompress_count_host")
        return nt, by, st

    # ---- page chains (storage.h:49-67; cache.c:151-176, pg_cryogen.c:761-805) ----

    def decompress_pages_host(self, relation: np.ndarray, chains, block_size: int = CRYO_BLCKSZ):
        """relation: [npages, 8192] uint8, indexed by block number; chains: per cryo block the list of
        block numbers of its pages, first page first (what the reader found following `next`).
        Returns (out [n, block_size], out_size, status, methods, comp_size)."""
        n = len(chains)
        flat = [b for ch in chains for b in ch]
        coff = np.zeros(n + 1, dtype=np.uint32)
        coff[1:] = np.cumsum([len(ch) for ch in chains])
        blk = np.asarray(flat, dtype=np.uint32)
        pagep = (C.c_void_p * max(len(flat), 1))(*[relation[b].ctypes.data for b in flat])
        out = np.zeros((n, block_size), dtype=np.uint8)
        dstp = (C.c_void_p * n)(*[out[i].ctypes.data for i in range(n)])
        osz = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        me = np.full(n, -1, dtype=np.int32)
        csz = np.zeros(n, dtype=np.uint32)
        self._check(self.lib.cryogpu_decompress_pages_host(
            self.handle, n, pagep, blk.ctypes.data, coff.ctypes.data, dstp, block_size, osz.ctypes.data,
            st.ctypes.data, me.ctypes.data, csz.ctypes.data), "cryogpu_decompress_pages_host")
        return out, osz, st, me, csz

    def compress_pages_host(self, method: int, level_or_accel: int, blocks: np.ndarray, relation: np.ndarray,
                            blknos: np.ndarray, created_xid: int, block_size: int = CRYO_BLCKSZ):
        """blocks: [n, block_size]; blknos: [n, cap_pages] block numbers reserved per block; the pages
        are written into relation[blkno].  Returns (npages, comp_size, status)."""
        blocks = np.ascontiguousarray(blocks, dtype=np.uint8).reshape(-1, block_size)
        n = blocks.shape[0]
        blknos = np.ascontiguousarray(blknos, dtype=np.uint32).reshape(n, -1)
        cap = blknos.shape[1]
        srcp = (C.c_void_p * n)(*[blocks[i].ctypes.data for i in range(n)])
        outp = (C.c_void_p * (n * cap))(*[relation[int(b)].ctypes.data for b in blknos.reshape(-1)])
        npg = np.zeros(n, dtype=np.uint32)
        csz = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        self._check(self.lib.cryogpu_compress_pages_host(
            self.handle, n, method, level_or_accel, srcp, block_size, blknos.ctypes.data, cap, created_xid, outp,
            npg.ctypes.data, csz.ctypes.data, st.ctypes.data), "cryogpu_compress_pages_host")
        return npg, csz, st


    # ---- batched tuple fetch (cryo_storage_fetch, storage.c:55-68, for many TIDs at once) ----

    def tuples_device(self, blocks, stride, n: int, block_status, sel_off, sel_pos, data, data_cap: int, tup_off, tup_len,
                      tup_cap: int, block_first, status, need, block_size: int = CRYO_BLCKSZ, stream: int | None = None):
        """Decoded blocks in HBM -> packed tuples (torch CUDA tensors or device pointers); only enqueues."""
        self._check(self.lib.cryogpu_tuples_device(
            self.handle, n, _ptr(blocks), stride, block_size, _ptr(block_status), _ptr(sel_off), _ptr(sel_pos), _ptr(data),
            data_cap, _ptr(tup_off), _ptr(tup_len), tup_cap, _ptr(block_first), _ptr(status), _ptr(need),
            _stream(stream)), "cryogpu_tuples_device")

    def _tuples_host(self, call, what, n, sel, data_cap, tup_cap):
        """Runs call(sel_off, sel_pos, data, data_cap, tup_off, tup_len, tup_cap, block_first, status, need); with a
        capacity of None it first asks for what the batch needs (a call with no room), then fetches."""
        sel_off, sel_pos = _sel_arrays(sel, n)
        bf = np.zeros(n + 1, dtype=np.uint64)
        st = np.full(n, -1, dtype=np.int32)
        need = np.zeros(2, dtype=np.uint64)
        if data_cap is None or tup_cap is None:
            self._check(call(_ptr(sel_off), _ptr(sel_pos), None, 0, None, None, 0, bf.ctypes.data, st.ctypes.data,
                             need.ctypes.data), what)
            data_cap = int(need[0]) if data_cap is None else data_cap
            tup_cap = int(need[1]) if tup_cap is None else tup_cap
        data = np.zeros(max(data_cap, 1), dtype=np.uint8)
        to = np.zeros(max(tup_cap, 1), dtype=np.uint64)
        tl = np.zeros(max(tup_cap, 1), dtype=np.uint32)
        self._check(call(_ptr(sel_off), _ptr(sel_pos), data.ctypes.data, data_cap, to.ctypes.data, tl.ctypes.data, tup_cap,
                         bf.ctypes.data, st.ctypes.data, need.ctypes.data), what)
        return data[:data_cap], to[:tup_cap], tl[:tup_cap], bf, st, (int(need[0]), int(need[1]))

    def decompress_tuples_host(self, methods, chunks, sel=None, block_size: int = CRYO_BLCKSZ, data_cap: int | None = None,
                               tup_cap: int | None = None):
        """Compressed blocks in, tuples out.  sel: None (every item) or per block a list of positions (0 = every item).
        Returns (data, tup_off, tup_len, block_first, status, (bytes, entries) needed)."""
        n = len(chunks)
        chunks = [np.ascontiguousarray(c, dtype=np.uint8) for c in chunks]
        methods = np.ascontiguousarray(np.broadcast_to(np.asarray(methods, dtype=np.int32), (n,)))
        sizes = np.array([c.size for c in chunks], dtype=np.uint32)
        srcp = (C.c_void_p * max(n, 1))(*[c.ctypes.data for c in chunks])

        def call(*a):
            return self.lib.cryogpu_decompress_tuples_host(self.handle, n, methods.ctypes.data, srcp, sizes.ctypes.data,
                                                           block_size, *a)
        return self._tuples_host(call, "cryogpu_decompress_tuples_host", n, sel, data_cap, tup_cap)

    def decompress_pages_tuples_host(self, relation: np.ndarray, chains, sel=None, block_size: int = CRYO_BLCKSZ,
                                     data_cap: int | None = None, tup_cap: int | None = None):
        """Page chains (as decompress_pages_host takes them) in, tuples out.  Returns (data, tup_off, tup_len,
        block_first, status, need, methods, comp_size)."""
        n = len(chains)
        flat = [b for ch in chains for b in ch]
        coff = np.zeros(n + 1, dtype=np.uint32)
        coff[1:] = np.cumsum([len(ch) for ch in chains])
        blk = np.asarray(flat + [0], dtype=np.uint32)
        pagep = (C.c_void_p * max(len(flat), 1))(*[relation[b].ctypes.data for b in flat])
        me = np.full(n, -1, dtype=np.int32)
        csz = np.zeros(n, dtype=np.uint32)

        def call(so, sp, data, dcap, to, tl, tcap, bf, st, need):
            return self.lib.cryogpu_decompress_pages_tuples_host(self.handle, n, pagep, blk.ctypes.data, coff.ctypes.data,
                                                                 block_size, so, sp, data, dcap, to, tl, tcap, bf, st,
                                                                 me.ctypes.data, csz.ctypes.data, need)
        return self._tuples_host(call, "cryogpu_decompress_pages_tuples_host", n, sel, data_cap, tup_cap) + (me, csz)

    # ---- cryo blocks from packed tuples (the write-side mirror of the tuple fetch) ----

    def build_blocks_device(self, data, data_size: int, tup_off, tup_len, block_first, n: int, dst, dst_stride: int, status,
                            block_size: int = CRYO_BLCKSZ, stream: int | None = None):
        """Packed tuples in HBM -> cryo blocks at dst + i * dst_stride (torch CUDA tensors or device pointers); only
        enqueues."""
        self._check(self.lib.cryogpu_build_blocks_device(
            self.handle, n, _ptr(data), data_size, _ptr(tup_off), _ptr(tup_len), _ptr(block_first), block_size, _ptr(dst),
            dst_stride, _ptr(status), _stream(stream)), "cryogpu_build_blocks_device")

    def compress_tuples_pages_host(self, method: int, level_or_accel: int, data: np.ndarray, tup_off: np.ndarray,
                                   tup_len: np.ndarray, block_first: np.ndarray, relation: np.ndarray, first_blkno,
                                   next_blkno: int, created_xid: int, block_size: int = CRYO_BLCKSZ):
        """The COPY flush from packed tuples into relation [npages, 8192] (indexed by block number): block i's first
        page is first_blkno[i], further pages are handed out from next_blkno on.  Returns (npages, comp_size, status,
        the block numbers handed out in order)."""
        n = block_first.size - 1
        data = np.ascontiguousarray(data, dtype=np.uint8)
        to = np.ascontiguousarray(tup_off, dtype=np.uint64)
        tl = np.ascontiguousarray(tup_len, dtype=np.uint32)
        bf = np.ascontiguousarray(block_first, dtype=np.uint64)
        first = np.ascontiguousarray(first_blkno, dtype=np.uint32)
        alloc, page_ptr, handed = page_callbacks(relation, next_blkno)
        npg = np.zeros(max(n, 1), dtype=np.uint32)
        csz = np.zeros(max(n, 1), dtype=np.uint32)
        st = np.full(max(n, 1), -1, dtype=np.int32)
        self._check(self.lib.cryogpu_compress_tuples_pages_alloc_host(
            self.handle, n, method, level_or_accel, data.ctypes.data, data.size, to.ctypes.data, tl.ctypes.data,
            bf.ctypes.data, block_size, first.ctypes.data, alloc, page_ptr, None, created_xid, npg.ctypes.data,
            csz.ctypes.data, st.ctypes.data), "cryogpu_compress_tuples_pages_alloc_host")
        return npg[:n], csz[:n], st[:n], handed


ALLOC_PAGE_FN = C.CFUNCTYPE(C.c_uint32, C.c_void_p)
PAGE_PTR_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_uint32)


def page_callbacks(relation: np.ndarray, next_blkno: int):
    """(alloc, page_ptr, handed) for the *_pages_alloc_host calls over relation [npages, 8192]: alloc hands out
    next_blkno, next_blkno + 1, ... and records them in the list `handed`; page_ptr(b) is relation[b]."""
    handed = []

    def alloc(_arg):
        handed.append(next_blkno + len(handed))
        return handed[-1]

    def page_ptr(_arg, b):
        return relation[b].ctypes.data if b < relation.shape[0] else None
    return ALLOC_PAGE_FN(alloc), PAGE_PTR_FN(page_ptr), handed


def _sel_arrays(sel, n: int):
    """Per-block position lists (None: every item) -> (sel_off uint64 [n + 1], sel_pos uint32) or (None, None)."""
    if sel is None:
        return None, None
    assert len(sel) == n
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for s in sel])
    return off, np.array([p for s in sel for p in s] + [0], dtype=np.uint32)


def pages_needed(compressed_size: int) -> int:
    """cryo_pages_needed, pg_cryogen.c:692-704"""
    return int(load_library().cryogpu_pages_needed(compressed_size))


def pack_chunks(chunks, align: int = 16):
    """Concatenate compressed blocks with `align`-byte aligned starts.
    Returns (buffer uint8, offsets uint64, sizes uint32); the buffer is padded to 16 bytes."""
    sizes = np.array([len(c) for c in chunks], dtype=np.uint32)
    padded = (sizes.astype(np.uint64) + np.uint64(align - 1)) & ~np.uint64(align - 1)
    offs = np.zeros(len(chunks), dtype=np.uint64)
    if len(chunks) > 1:
        offs[1:] = np.cumsum(padded)[:-1]
    total = int(padded.sum()) if len(chunks) else 0
    buf = np.zeros(max(total, 16) + 16, dtype=np.uint8)
    for i, c in enumerate(chunks):
        o = int(offs[i])
        buf[o:o + len(c)] = np.frombuffer(bytes(c), dtype=np.uint8) if not isinstance(c, np.ndarray) else c
    return buf, offs, sizes
