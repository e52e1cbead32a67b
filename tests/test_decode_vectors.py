"""The stream writers of tests/decode_vectors.py (CPU): every vector gives its planned bytes through liblz4 / libzstd at
capacity = its size and through the plain-C restatement; every rule-breaking one gets the same verdict from both."""
import numpy as np
import pytest

import decode_vectors as dv
import encode_check as ec
from oracle import port
from pg_cryogen_b200 import COMP_LZ4

SIZES = [255, 65791, 300017]


def _lib(method, stream, cap):
    """liblz4's LZ4_decompress_safe / libzstd's ZSTD_decompress at capacity cap: (bytes or negative, out)"""
    lz4, zs = ec._syslibs()
    c = np.ascontiguousarray(stream, dtype=np.uint8)
    out = np.zeros(max(cap, 1), dtype=np.uint8)
    if method == COMP_LZ4:
        return int(lz4.LZ4_decompress_safe(c.ctypes.data, out.ctypes.data, c.size, cap)), out
    r = zs.ZSTD_decompress(out.ctypes.data, cap, c.ctypes.data, c.size)
    return (-1 if zs.ZSTD_isError(r) else int(r)), out


@pytest.mark.parametrize("n", SIZES)
def test_vectors_give_their_planned_bytes(oracle_port, n):
    vs = dv.vectors(n)
    assert len({v.name for v in vs}) == len(vs)
    for v in vs:
        lib_n, lib_out = _lib(v.method, v.stream, n)
        got, out = dv.restate(v.method, v.stream, n)
        if v.name == "zstd-window-28":
            # stricter than libzstd 1.5.5, whose one-shot ZSTD_decompress takes windows up to 2^31 (its streaming
            # decoder's default limit is 2^27): DESIGN.md section 1
            assert lib_n == n and got < 0, (lib_n, got)
            continue
        if v.plain is None:
            assert (lib_n == n) == (got == n) == False, (v.name, lib_n, got)       # noqa: E712
            w = dv.verdict(v.method, v.stream, n)
            assert w is None or w.size != n, v.name
            continue
        assert v.plain.size == n, v.name
        assert lib_n == n and np.array_equal(lib_out[:n], v.plain), (v.name, lib_n)
        assert got == n and np.array_equal(out[:n], v.plain), (v.name, got)


def test_vectors_cover_what_they_are_named_for(oracle_port):
    """The structure the routes depend on: sequence counts, block counts, FCS widths, the run lengths."""
    vs = {v.name: v for v in dv.vectors(300017)}
    for k in (3071, 3072, 3073):
        assert ec.lz4_walk(vs[f"lz4-seqs-{k}"].stream, 300017) == k
    for k in (8191, 8192, 8193):
        assert port.zstd_decode(vs[f"zstd-seqs-{k}"].stream, 300017, stats=True)[2]["sequences"] == k
    for nb in (16, 17):
        st = port.zstd_decode(vs[f"zstd-{nb}-blocks"].stream, 300017, stats=True)[2]
        assert st["blocks_raw"] + st["blocks_rle"] + st["blocks_compressed"] == nb
    st = port.zstd_decode(vs["zstd-dense"].stream, 300017, stats=True)[2]
    assert st["sequences"] > 300017 // 8 + 64 and st["mode_rle"] > 0
    seqs = port.zstd_decode(vs["zstd-runs-32767-32768-32769"].stream, 300017, trace=True)[2]
    assert [ml for _, ml, _ in seqs] == [32767, 32768, 32769]
    runs = port.zstd_decode(vs["zstd-three-long-runs"].stream, 300017, trace=True)[2]
    assert sum(1 for _, ml, off in runs if off == 1 and ml >= dv.ZP_JOB_MIN) == 3
    offs = {off for _, _, off in port.lz4_decode(vs["lz4-offset-65535"].stream, 300017, trace=True)[2]}
    assert 65535 in offs
    fh = {w: vs[f"zstd-fcs-{w}"].stream[4] >> 6 for w in (4, 8)}
    assert fh == {4: 2, 8: 3}
    small = {v.name for v in dv.vectors(255)} | {v.name for v in dv.vectors(65791)}
    assert {"zstd-fcs-1", "zstd-fcs-2"} <= small


def test_checksum_vectors(oracle_port):
    """A correct content checksum passes everywhere; a wrong one is rejected by libzstd and the restatement (the
    library's decoders skip it: DESIGN.md section 1, pinned by the emulator and device tests)."""
    body = [dv.raw(b"0123456789abcdef"), dv.seqs(b"q", [(1, 300, 7)])]
    good, plan = dv.zstd_frame(body, checksum="good")
    bad, _ = dv.zstd_frame(body, checksum="bad")
    n = len(plan)
    assert _lib(1, good, n)[0] == n and dv.restate(1, good, n)[0] == n
    assert _lib(1, bad, n)[0] < 0 and dv.restate(1, bad, n)[0] < 0
