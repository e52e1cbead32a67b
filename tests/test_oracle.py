"""The oracle is pinned before it is trusted (not gpu):

* oracle/_ref (the reference's own compression.c on liblz4/libzstd) round-trips and
  reproduces the committed golden streams byte for byte;
* oracle/cryo_oracle.c (our plain-C restatement of the two formats) decodes every
  golden stream, every block kind x payload x level, and the hand-crafted conformance
  frames to exactly what the reference produces, and agrees with the reference's
  verdict on malformed inputs.
"""
import hashlib

import numpy as np
import pytest

from pg_cryogen_b200 import blockgen as bg

import golden_util
from zstd_vectors import conformance_frames

MiB = 1 << 20


def test_reference_library_versions_are_the_pinned_ones(oracle_ref):
    assert oracle_ref.versions() == (10904, 10505)       # liblz4 1.9.4, libzstd 1.5.5
    if oracle_ref.available():                            # the reference's own GUC table (oracle/_ref)
        assert oracle_ref.guc_defaults() == (1, 1, 1)     # compression.c:16-18
    assert oracle_ref.compress_bound(0) == 1052704        # LZ4_compressBound(1 MiB)
    assert oracle_ref.compress_bound(1) == 1052672        # ZSTD_compressBound(1 MiB)


def test_golden_streams_are_what_the_reference_writes(oracle_ref):
    for name, method, level, stream, sha in golden_util.load():
        blk = golden_util.plaintext(name)
        assert hashlib.sha256(blk.tobytes()).digest() == sha, name
        comp, _, _ = oracle_ref.compress(method, level, blk)
        assert np.array_equal(comp[0], stream), name
        out, ok = oracle_ref.decompress_one(method, stream)
        assert ok and np.array_equal(out, blk), name


def test_compressed_sizes_are_what_the_reference_wrote(oracle_ref):
    """Total compressed bytes of blocks 1000..1031 of each benchmark kind at lz4 acceleration 1 and zstd level 1,
    as the reference wrote them in a recorded benchmark run (tests/golden/reference_outputs.json)."""
    want = golden_util.reference_outputs()["compressed_bytes_blocks_1000_to_1031"]
    assert len(want) == 12
    for key, total in want.items():
        kind, payload, codec = key.split("_")
        blocks = bg.make_blocks(kind, payload, 1000, 32)
        _, sizes, _ = oracle_ref.compress(0 if codec == "lz4a1" else 1, 1, blocks, nthreads=8, keep=False)
        assert int(sizes.astype(np.int64).sum()) == total, key


def test_port_decodes_golden_streams(oracle_port):
    for name, method, level, stream, sha in golden_util.load():
        dec = oracle_port.lz4_decode if method == 0 else oracle_port.zstd_decode
        n, out = dec(stream)[:2]
        assert n == MiB, name
        assert hashlib.sha256(out.tobytes()).digest() == sha, name


@pytest.mark.parametrize("kind", ["S", "M", "D"])
def test_port_matches_reference_on_every_kind_payload_level(oracle_ref, oracle_port, kind):
    for payload in bg.PAYLOADS:
        blk = bg.make_block(kind, payload, 13)
        for accel in (0, 1, 2, 5, 10, 25, 50):
            c = oracle_ref.compress(0, accel, blk)[0][0]
            n, out = oracle_port.lz4_decode(c)[:2]
            assert n == MiB and np.array_equal(out, blk), (kind, payload, accel)
        for level in (-5, -4, -3, -2, -1, 0, 1, 2, 3, 4, 7, 12, 19, 22):
            c = oracle_ref.compress(1, level, blk)[0][0]
            n, out = oracle_port.zstd_decode(c)[:2]
            assert n == MiB and np.array_equal(out, blk), (kind, payload, level)


def test_port_format_census_matches_survey(oracle_ref, oracle_port):
    """SURVEY.md C.2/C.3: what the streams of a sparse block look like."""
    blk = bg.make_block("S", "hex", 7)
    st = oracle_port.zstd_decode(oracle_ref.compress(1, 1, blk)[0][0], stats=True)[2]
    assert st["blocks_rle"] == 6 and st["blocks_compressed"] == 2 and st["window_size"] == 512 << 10
    assert st["lit_huf4"] == 2 and st["mode_fse"] == 6
    st = oracle_port.zstd_decode(oracle_ref.compress(1, 3, blk)[0][0], stats=True)[2]
    assert st["single_segment"] == 1
    st = oracle_port.lz4_decode(oracle_ref.compress(0, 1, blk)[0][0], stats=True)[2]
    assert st["longest_match"] > 1_000_000 and st["overlap_match_bytes"] > 1_000_000


def test_port_decodes_conformance_vectors_like_the_reference(oracle_ref, oracle_port):
    for name, frame, expect in conformance_frames():
        out, ok = oracle_ref.decompress_one(1, frame)
        assert ok and bytes(out[: len(expect)]) == expect, name
        n, pout = oracle_port.zstd_decode(frame)[:2]
        assert n == len(expect) and bytes(pout[: len(expect)]) == expect, name


def _malformed_lz4(c):
    far = np.array([0x10, 65, 5, 0, 0x50, 97, 98, 99, 100, 101], dtype=np.uint8)
    return [("valid", c), ("truncated-100", c[:-100]), ("truncated-1", c[:-1]),
            ("trailing", np.concatenate([c, np.array([1, 2, 3], dtype=np.uint8)])),
            ("offset-before-start", far), ("one-byte", c[:1]), ("empty", c[:0]),
            ("short-valid", np.array([0x50, 1, 2, 3, 4, 5], dtype=np.uint8))]


def _malformed_zstd(c):
    bad_magic = c.copy()
    bad_magic[0] ^= 0xFF
    reserved = c.copy()
    reserved[9] |= 0x06
    wrong_fcs = c.copy()
    wrong_fcs[6] ^= 0x01
    return [("valid", c), ("truncated-100", c[:-100]), ("truncated-1", c[:-1]),
            ("trailing", np.concatenate([c, np.array([1, 2, 3], dtype=np.uint8)])),
            ("bad-magic", bad_magic), ("reserved-block-type", reserved),
            ("wrong-content-size", wrong_fcs), ("empty", c[:0]), ("header-only", c[:8])]


def test_port_agrees_with_reference_verdict_on_malformed_input(oracle_ref, oracle_port):
    blk = bg.make_block("S", "hex", 5)
    for method, cases, dec in (
            (0, _malformed_lz4(oracle_ref.compress(0, 1, blk)[0][0]), oracle_port.lz4_decode),
            (1, _malformed_zstd(oracle_ref.compress(1, 1, blk)[0][0]), oracle_port.zstd_decode)):
        for name, stream in cases:
            _, ref_ok = oracle_ref.decompress_one(method, stream)
            n = dec(stream)[0]
            assert (n >= 0) == ref_ok, (method, name, n, ref_ok)


def test_port_rejects_output_capacity_one_short(oracle_ref, oracle_port):
    blk = bg.make_block("M", "hex", 2)
    assert oracle_port.lz4_decode(oracle_ref.compress(0, 1, blk)[0][0], cap=MiB - 1)[0] < 0
    assert oracle_port.zstd_decode(oracle_ref.compress(1, 1, blk)[0][0], cap=MiB - 1)[0] < 0


def test_xxh64_known_answers(oracle_port):
    assert oracle_port.xxh64(b"") == 0xEF46DB3751D8E999
    assert oracle_port.xxh64(b"a") == 0xD24EC4F1A98C6E5B
    assert oracle_port.xxh64(b"abc") == 0x44BC2CF5AD770999


def test_port_is_never_looser_than_the_reference_on_corrupted_frames(oracle_ref, oracle_port):
    """Single-byte corruptions of zstd frames (DESIGN.md, known deviations): libzstd 1.5.5's fast Huffman path
    accepts some frames whose literal streams do not end exactly where they should and returns garbage; the
    port -- and every GPU decoder, which is pinned to it -- rejects them.  The asymmetry is pinned on purpose:
    the port may reject what the reference accepts, never the other way round, and where both accept the
    bytes are the same."""
    rng = np.random.default_rng(17)
    blk = bg.make_block("D", "lowcard", 3)
    z = oracle_ref.compress(1, 1, blk)[0][0]
    stricter = same = 0
    for k in range(150):
        m = z.copy()
        pos = int(rng.integers(0, m.size))
        m[pos] ^= int(rng.integers(1, 256))
        want, ok = oracle_ref.decompress_one(1, m)
        got_n, got = oracle_port.zstd_decode(m)
        if got_n >= 0:
            assert ok, (k, pos, "the port accepted a frame the reference rejects")
            assert got_n == want.size and np.array_equal(got[:got_n], want), (k, pos)
            same += 1
        elif ok:
            stricter += 1
    assert same + stricter > 0
    assert stricter <= 75, stricter         # the deviation stays a minority of the corruptions (39 of 150 when measured)
