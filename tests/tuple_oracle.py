"""ctypes binding of the batched tuple fetch's restatement in tests/tuple_oracle.c (TEST INFRASTRUCTURE ONLY), and the
builder of the test libraries that go with it (the restatement, the kernel bodies under the SIMT emulator).  They are
compiled on first use into a private temporary directory, so a read-only tree works."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_CXXFLAGS = ["-O1", "-g", "-std=c++17", "-fPIC", "-Wall", "-Wno-unused-function", "-Wno-unused-variable",
                "-Wno-sign-compare", "-Wno-unknown-pragmas", "-Wno-comment"]     # tests/emu/Makefile's flags
_dir = None
_libs = {}


def build(name: str, cmd: list[str]) -> C.CDLL:
    """compile (once per process) with cmd + [-o <lib>] and load it"""
    global _dir
    if name not in _libs:
        if _dir is None:
            _dir = tempfile.mkdtemp(prefix="cryo_tuples_")
            atexit.register(shutil.rmtree, _dir, True)
        out = os.path.join(_dir, name)
        subprocess.check_call(cmd + ["-o", out])
        _libs[name] = C.CDLL(out)
    return _libs[name]


def _lib():
    return build("libtupleoracle.so", ["gcc", "-O2", "-fPIC", "-Wall", "-std=c11", "-shared",
                                       os.path.join(HERE, "tuple_oracle.c")])


def emu_lib():
    """tests/emu/emu_tuples.cpp: the tuple-fetch kernel bodies under cuda_emu.h"""
    return build("libcryoemu_tuples.so", ["g++", *EMU_CXXFLAGS, "-I" + os.path.join(HERE, "emu"), "-shared",
                                          os.path.join(HERE, "emu", "emu_tuples.cpp")])


def sel_arrays(sel, n: int):
    """Per-block position lists (None = every item of every block) -> (sel_off uint64 [n + 1], sel_pos uint32)."""
    if sel is None:
        return None, None
    assert len(sel) == n
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for s in sel])
    pos = np.array([p for s in sel for p in s] + [0], dtype=np.uint32)
    return off, pos


def block_tuples(blocks: np.ndarray, sel=None, block_status=None, data_cap: int | None = None,
                 tup_cap: int | None = None, block_size: int | None = None, fill: int = 0):
    """The batched tuple fetch over decoded blocks [n, stride] (cryo_oracle_block_tuples).  sel: None (every item) or
    per block a list of positions (0 = every item).  Caps None: what the batch needs.  Returns (data, tup_off,
    tup_len, block_first, status, need); data / tup_off / tup_len hold `fill` where nothing was written."""
    L = _lib()
    blocks = np.ascontiguousarray(blocks, dtype=np.uint8)
    n, stride = blocks.shape
    bs = stride if block_size is None else block_size
    off, pos = sel_arrays(sel, n)
    bst = None if block_status is None else np.ascontiguousarray(block_status, dtype=np.int32)
    bf = np.zeros(n + 1, dtype=np.uint64)
    st = np.zeros(n, dtype=np.int32)
    need = np.zeros(2, dtype=np.uint64)

    def call(dcap, tcap):
        data = np.full(max(dcap, 1), fill, dtype=np.uint8)
        to = np.full(max(tcap, 1), fill * 0x0101010101010101, dtype=np.uint64)
        tl = np.full(max(tcap, 1), fill * 0x01010101, dtype=np.uint32)
        L.cryo_oracle_block_tuples(C.c_void_p(blocks.ctypes.data), C.c_uint64(stride), C.c_uint32(n), C.c_uint32(bs),
                                   None if bst is None else C.c_void_p(bst.ctypes.data),
                                   None if off is None else C.c_void_p(off.ctypes.data),
                                   None if pos is None else C.c_void_p(pos.ctypes.data),
                                   C.c_void_p(data.ctypes.data), C.c_uint64(dcap), C.c_void_p(to.ctypes.data),
                                   C.c_void_p(tl.ctypes.data), C.c_uint64(tcap), C.c_void_p(bf.ctypes.data),
                                   C.c_void_p(st.ctypes.data), C.c_void_p(need.ctypes.data))
        return data[:dcap], to[:tcap], tl[:tcap]

    if data_cap is None or tup_cap is None:
        call(0, 0)
        data_cap = int(need[0]) if data_cap is None else data_cap
        tup_cap = int(need[1]) if tup_cap is None else tup_cap
    data, to, tl = call(data_cap, tup_cap)
    return data, to, tl, bf.copy(), st.copy(), (int(need[0]), int(need[1]))
