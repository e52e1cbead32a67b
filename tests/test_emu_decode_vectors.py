"""The crafted vectors and the mutation corpus of tests/decode_vectors.py through the emulated decoder bodies (CPU, not
gpu): the warp decoders (emu_lz4w_decode, emu_zstdw_decode), the CTA decoders (libcryoemu_cx64.so) and the phase-split
pipeline (emu_zstdp_decode_multi).  Each must give the plain-C restatement's verdict and bytes.  A stream reaches the
device tests (tests/test_gpu_decode_contract.py) only after these bodies handle it cleanly."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import decode_vectors as dv
from pg_cryogen_b200 import COMP_LZ4

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def bodies():
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "emu")])
    W = C.CDLL(os.path.join(HERE, "emu", "libcryoemu.so"))
    X = C.CDLL(os.path.join(HERE, "emu", "libcryoemu_cx64.so"))
    sig = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint, C.POINTER(C.c_uint32)]
    for f in (W.emu_lz4w_decode, W.emu_zstdw_decode, X.emu_lz4c_decode):
        f.argtypes, f.restype = sig, C.c_int
    X.emu_zstdc_decode.argtypes, X.emu_zstdc_decode.restype = sig + [C.POINTER(C.c_uint32)], C.c_int
    W.emu_zstdp_decode_multi.restype = C.c_int

    def one(body, method, stream, cap, shift):
        s = np.ascontiguousarray(stream, dtype=np.uint8)
        out, sz = np.zeros(max(cap, 16), dtype=np.uint8), C.c_uint32(0)
        src = s.ctypes.data if s.size else None
        if body == "warp":
            fn = W.emu_lz4w_decode if method == COMP_LZ4 else W.emu_zstdw_decode
            st = fn(src, s.size, out.ctypes.data, cap, shift, C.byref(sz))
        elif method == COMP_LZ4:
            st = X.emu_lz4c_decode(src, s.size, out.ctypes.data, cap, shift, C.byref(sz))
        else:
            st = X.emu_zstdc_decode(src, s.size, out.ctypes.data, cap, shift, C.byref(sz), C.byref(C.c_uint32(0)))
        return st, sz.value, out[:cap]
    return one, W


def _pipeline(W, frames, cap, shift):
    import test_emu_kernels as tk
    return tk._run_pipeline(W, frames, cap=cap, shift=shift)[:3]


def _check(tag, want, st, sz, out, cap):
    assert st not in (-100, -101), (tag, "emulator check", st)
    assert dv.accepts(want, cap, st, sz, out), (tag, st, sz, None if want is None else want.size)


def _run_all(bodies, items, cap):
    """items: (method, stream, want, tag) through the warp and CTA bodies one by one, the zstd ones through the pipeline
    in batches of nine (odd, so the emulated stages split their groups three ways)"""
    one, W = bodies
    for k, (m, s, w, t) in enumerate(items):
        for body in ("warp", "cta"):
            _check(f"{t} {body}", w, *one(body, m, s, cap, k % 16), cap)
    z = [it for it in items if it[0] != COMP_LZ4]
    for b in range(0, len(z), 9):
        batch = z[b:b + 9]
        st, osz, outs = _pipeline(W, [it[1] for it in batch], cap, b % 16)
        for (m, s, w, t), a, c, o in zip(batch, st, osz, outs):
            _check(f"{t} pipeline", w, a, c, o, cap)


@pytest.mark.parametrize("n", [255, 65791, 300017])
def test_emulated_bodies_on_crafted_vectors(bodies, oracle_port, n):
    items = []
    for v in dv.vectors(n):
        want = dv.verdict(v.method, v.stream, n)
        if v.plain is not None:
            assert want is not None and np.array_equal(want, v.plain), v.name
        items.append((v.method, v.stream, want, v.name))
    # the content checksum is skipped, not verified (DESIGN.md section 1): a wrong one is accepted
    body = [dv.raw(bytes(range(16)))] + dv._fill_rle(16, n)
    bad, plan = dv.zstd_frame(body, checksum="bad")
    items.append((1, bad, dv._u8(plan), "zstd-checksum-bad"))
    _run_all(bodies, items, n)


def test_emulated_bodies_on_the_mutation_corpus(bodies, oracle_port):
    cap = dv.CORPUS_CAP
    items = [(m, s, b if b is not None else dv.verdict(m, s, cap), t) for m, s, b, t in dv.corpus()]
    for m, s, b, t in dv.corpus():
        if b is not None:
            assert np.array_equal(dv.verdict(m, s, cap), b), t
    _run_all(bodies, items, cap)
