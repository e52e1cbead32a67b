"""Stream writers for the decoders' tests (TEST INFRASTRUCTURE ONLY): LZ4 blocks and zstd frames that liblz4 and libzstd
never emit, with the sequence structure set exactly, and the seeded vectors built from them.

lz4_block writes sequences as given and does not enforce the end-of-block rules, so it also writes the rule-breaking
blocks the verdict tests need.  zstd_frame writes Raw, RLE and Compressed blocks; a Compressed block has Raw or RLE
literals and RLE-mode sequence tables: every sequence of a block shares its LL / ML / OF code, and the extra bits still
vary per sequence (as vector 7 of tests/zstd_vectors.py).  Both writers also return the planned bytes, computed here
from the sequences, so that liblz4 / libzstd and the plain-C restatement are checked against a plan, not each other.

Every vector fills exactly the capacity it is built for, so that one batch of them shares one block size, and is
tagged with the route it targets:
  lz4-warp / lz4-cta:  at most / more than LZ4W_BUDGET = 3 072 sequences (what a large batch does with the block);
  zp / zp-cx:          the pipeline's warp or CTA executor (ZP_CX_SEQS = 8 192 sequences) in a large batch;
  zp-fallback:         a frame stage 1 declines (17 blocks, a window above 2^27);
  dense:               more sequences than the pool's per-frame share (cap / 8 + 64): placement depends on the batch;
  any:                 no route of its own.
plain is None for a rule-breaking vector: its verdict is the restatement's (see verdict())."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from oracle import port
from pg_cryogen_b200 import COMP_LZ4, COMP_ZSTD
from zstd_vectors import _block_header, _frame

ZS_BLOCK = 128 << 10
LZ4_BUDGET = 3072             # lz4_decode_w.cuh hands a block on after this many sequences (cryogpu.cu LZ4W_BUDGET)
ZP_CX_SEQS = 8192             # zstd_decode_p.cuh: frames with at least this many sequences go to the CTA executor
ZP_MAXB = 16                  # zstd blocks per frame the pipeline takes
ZP_JOB_MIN = 32768            # an offset-1 match this long is a job for the raw / RLE stage (ZP_JOBS = 2 per frame)


@dataclass
class Vector:
    name: str
    method: int
    stream: np.ndarray
    cap: int
    plain: np.ndarray | None          # the planned bytes; None: the stream breaks a rule
    route: str


def _u8(b) -> np.ndarray:
    return np.frombuffer(bytes(b), dtype=np.uint8).copy()


def _copy(out: bytearray, off: int, ml: int) -> None:
    """the match as the formats define it: byte by byte, so an offset below the length repeats the last off bytes"""
    start = len(out) - off
    if off >= ml:
        out += out[start:start + ml]
    else:
        pat = bytes(out[start:])
        out += (pat * (ml // off + 1))[:ml]


# ---- LZ4 -----------------------------------------------------------------------------------------------------------

def _lz4_len(v: int) -> bytes:
    out = bytearray()
    while v >= 255:
        out.append(255)
        v -= 255
    out.append(v)
    return bytes(out)


def lz4_block(seqs, last_literals) -> tuple[np.ndarray, bytes]:
    """seqs: (literals, match_len >= 4, offset) per sequence; then a literals-only closing sequence.  Returns
    (stream, planned bytes, or None when an offset reaches before the block's start)."""
    s, out, broken = bytearray(), bytearray(), False
    for lits, ml, off in seqs:
        ll, m = len(lits), ml - 4
        s.append((min(ll, 15) << 4) | min(m, 15))
        if ll >= 15:
            s += _lz4_len(ll - 15)
        s += lits
        s += bytes([off & 255, off >> 8])
        if m >= 15:
            s += _lz4_len(m - 15)
        out += lits
        if not 0 < off <= len(out):
            broken = True
            continue
        _copy(out, off, ml)
    ll = len(last_literals)
    s.append(min(ll, 15) << 4)
    if ll >= 15:
        s += _lz4_len(ll - 15)
    s += last_literals
    out += last_literals
    return _u8(s), None if broken else bytes(out)


def _lz4_out_len(seqs) -> int:
    return sum(len(lit) + ml for lit, ml, _ in seqs)


def _lz4_close(seqs, n: int, tail: bytes):
    """a match of offset 1 that fills up to n - len(tail), then the closing literal run tail"""
    fill = n - len(tail) - _lz4_out_len(seqs)
    assert fill >= 4, fill
    return lz4_block(seqs + [(b"", fill, 1)], tail)


def _lz4_vec(name, n, route, built, valid=True):
    stream, plan = built
    if valid:
        assert plan is not None and len(plan) == n, (name, plan and len(plan), n)
    return Vector(name, COMP_LZ4, stream, n, _u8(plan) if valid else None, route)


def lz4_vectors(n: int, seed: int = 1) -> list[Vector]:
    """The LZ4 vectors that fit a capacity of n bytes"""
    rng = np.random.default_rng([seed, n, 4])
    rb = lambda k: bytes(rng.integers(0, 256, size=k, dtype=np.uint8))      # noqa: E731
    tail = rb(5)
    out = []
    # sequence counts around the warp decoder's budget (tokens, the closing one included); match lengths vary
    for k in (LZ4_BUDGET - 1, LZ4_BUDGET, LZ4_BUDGET + 1):
        seqs = [(rb(16), 4, 16)] + [(rb(1), 4 + int(rng.integers(0, 15)), int(rng.integers(1, 9))) for _ in range(k - 3)]
        if _lz4_out_len(seqs) + 9 <= n:
            out.append(_lz4_vec(f"lz4-seqs-{k}", n, "lz4-cta" if k > LZ4_BUDGET else "lz4-warp", _lz4_close(seqs, n, tail)))
    # overlapping copies: offsets 1-15, lengths across 16, 32 and the warp decoder's 2 KiB ring
    seqs = [(rb(int(rng.integers(1, 4))), ml, off) for off in range(1, 16)
            for ml in (15, 16, 17, 31, 32, 33, 2047, 2048, 2049)]
    if _lz4_out_len(seqs) + 9 <= n:
        out.append(_lz4_vec("lz4-overlap", n, "lz4-warp", _lz4_close(seqs, n, tail)))
    # literal and match lengths at the edges of the token nibble and of the 255-byte extensions
    edges = (14, 15, 16, 15 + 254, 15 + 255, 15 + 256, 15 + 509, 15 + 510, 15 + 511)
    seqs = [(rb(64), 4, 64)] + [(rb(ll), 4 + m, int(rng.integers(1, 64))) for ll in edges for m in (0, 14, 15, 16, 269, 270, 525)]
    if _lz4_out_len(seqs) + 9 <= n:
        out.append(_lz4_vec("lz4-lengths", n, "lz4-warp", _lz4_close(seqs, n, tail)))
    # the farthest offset, from a literal run long enough for it
    seqs = [(rb(65600), 300, 65535), (rb(3), 20, 65535), (rb(1), 70, 65000)]
    if _lz4_out_len(seqs) + 9 <= n:
        out.append(_lz4_vec("lz4-offset-65535", n, "lz4-warp", _lz4_close(seqs, n, tail)))
    base = [(rb(40), 100, 7)]
    if n >= 200:
        # the last match ends exactly 5 bytes before the capacity, closing literal run of exactly 5 (already above);
        # alone: a block of one long match
        out.append(_lz4_vec("lz4-close-5", n, "lz4-warp", _lz4_close(base, n, tail)))
        # rule-breaking: a match up to the capacity (no closing literals), one into the last 5 bytes, a match that
        # starts after n - 12, an offset before the start, a block one byte short of the capacity
        fill = n - _lz4_out_len(base)
        out.append(_lz4_vec("lz4-match-to-cap", n, "any", lz4_block(base + [(b"", fill, 1)], b""), False))
        out.append(_lz4_vec("lz4-close-4", n, "any", _lz4_close(base, n, tail[:4]), False))
        late = base + [(b"", n - 11 - _lz4_out_len(base), 1), (rb(1), 4, 1)]
        out.append(_lz4_vec("lz4-late-match", n, "any", lz4_block(late, rb(6)), False))
        out.append(_lz4_vec("lz4-offset-before-start", n, "any", _lz4_close([(rb(10), 20, 11)], n, tail), False))
        out.append(_lz4_vec("lz4-one-short", n, "any", _lz4_close(base, n - 1, tail), False))
    return out


# ---- zstd ----------------------------------------------------------------------------------------------------------

_LL = [(i, 0) for i in range(16)] + [(16, 1), (18, 1), (20, 1), (22, 1), (24, 2), (28, 2), (32, 3), (40, 3), (48, 4),
                                     (64, 6), (128, 7), (256, 8), (512, 9), (1024, 10), (2048, 11), (4096, 12),
                                     (8192, 13), (16384, 14), (32768, 15), (65536, 16)]
_ML = [(i + 3, 0) for i in range(32)] + [(35, 1), (37, 1), (39, 1), (41, 1), (43, 2), (47, 2), (51, 3), (59, 3), (67, 4),
                                         (83, 4), (99, 5), (131, 7), (259, 8), (515, 9), (1027, 10), (2051, 11),
                                         (4099, 12), (8195, 13), (16387, 14), (32771, 15), (65539, 16)]


def _code(table, v):
    for c in range(len(table) - 1, -1, -1):
        if table[c][0] <= v:
            base, bits = table[c]
            assert v - base < 1 << bits, v
            return c, bits, v - base
    raise ValueError(v)


def _of_code(ov):
    c = ov.bit_length() - 1
    return c, c, ov - (1 << c)


def raw(data) -> tuple:
    return ("raw", bytes(data))


def rle(byte: int, count: int) -> tuple:
    return ("rle", byte, count)


def seqs(lits, sequences, lit_mode="raw") -> tuple:
    """A Compressed block: literals (Raw, or RLE when lit_mode is "rle": then all one byte) and sequences
    (literal_len, match_len, offset_value) sharing their codes; offset_value is the format's: 1-3 repeat codes,
    otherwise offset + 3."""
    return ("seq", bytes(lits), list(sequences), lit_mode)


def _lit_header(lt: int, size: int) -> bytes:
    if size < 32:
        return bytes([lt | (size << 3)])
    if size < 4096:
        return bytes([lt | (1 << 2) | ((size & 15) << 4), size >> 4])
    assert size < 1 << 20
    return bytes([lt | (3 << 2) | ((size & 15) << 4), (size >> 4) & 255, size >> 12])


def _seq_body(lits: bytes, sq, lit_mode: str) -> bytes:
    if lit_mode == "rle":
        assert len(set(lits)) <= 1
        body = bytearray(_lit_header(1, len(lits)) + (lits[:1] or b"\0"))
    else:
        body = bytearray(_lit_header(0, len(lits)) + lits)
    nb = len(sq)
    if nb < 128:
        body.append(nb)
    elif nb < 0x7F00:
        body += bytes([(nb >> 8) + 128, nb & 255])
    else:
        body += bytes([255, (nb - 0x7F00) & 255, (nb - 0x7F00) >> 8])
    if nb == 0:
        return bytes(body)
    codes, bits = set(), ["1"]
    for ll, ml, ov in sq:
        lc, lb, lx = _code(_LL, ll)
        mc, mb, mx = _code(_ML, ml)
        oc, ob, ox = _of_code(ov)
        codes.add((lc, oc, mc))
        # read order of the decoder: offset, match length, literal length extra bits (the RLE tables read no state bits)
        for x, b in ((ox, ob), (mx, mb), (lx, lb)):
            if b:
                bits.append(format(x, f"0{b}b"))
    assert len(codes) == 1, "RLE-mode tables: one code each per block"
    lc, oc, mc = codes.pop()
    body += bytes([(1 << 6) | (1 << 4) | (1 << 2), lc, oc, mc])
    v = int("".join(bits), 2)
    body += v.to_bytes((v.bit_length() + 7) // 8, "little")
    return bytes(body)


def _run_seqs(out: bytearray, rep: list, lits: bytes, sq) -> bool:
    """executes one block's sequences with the format's repeat-offset rules; False when an offset reaches before
    the frame's first byte"""
    lp = 0
    for ll, ml, ov in sq:
        out += lits[lp:lp + ll]
        lp += ll
        if ov > 3:
            off = ov - 3
            rep[:] = [off, rep[0], rep[1]]
        else:
            idx = ov if ll == 0 else ov - 1
            if idx == 0:
                off = rep[0]
            elif idx == 3:
                off = rep[0] - 1
                rep[:] = [off, rep[0], rep[1]]
            elif idx == 1:
                off = rep[1]
                rep[:] = [off, rep[0], rep[2]]
            else:
                off = rep[2]
                rep[:] = [off, rep[0], rep[1]]
        if off < 1 or off > len(out):
            return False
        _copy(out, off, ml)
    out += lits[lp:]
    return True


def zstd_frame(blocks, content_size="auto", fcs_bytes=None, window_log=None, checksum=None, last=True):
    """Writes a frame of the given blocks (raw(), rle(), seqs()).  content_size: the size written in the header
    ("auto": the planned size; None: no content size, which needs window_log).  fcs_bytes: its width (default the
    narrowest).  checksum: None, "good" or "bad".  last: set the last-block flag on the last block.  Returns (frame,
    planned bytes or None when an offset reaches before the frame)."""
    out, rep, ok, parts = bytearray(), [1, 4, 8], True, []
    for k, b in enumerate(blocks):
        end = last and k == len(blocks) - 1
        if b[0] == "raw":
            parts.append(_block_header(end, 0, len(b[1])) + b[1])
            out += b[1]
        elif b[0] == "rle":
            parts.append(_block_header(end, 1, b[2]) + bytes([b[1]]))
            out += bytes([b[1]]) * b[2]
        else:
            body = _seq_body(b[1], b[2], b[3])
            parts.append(_block_header(end, 2, len(body)) + body)
            ok = _run_seqs(out, rep, b[1], b[2]) and ok
    size = len(out) if content_size == "auto" else content_size
    if size is None:
        assert window_log is not None
        fcs_bytes = 0
    elif fcs_bytes is None:
        fcs_bytes = 1 if size < 256 and window_log is None else 2 if 256 <= size < 65792 else 4 if size < 1 << 32 else 8
    ck = None
    if checksum is not None:
        ck = (port.xxh64(bytes(out)) & 0xFFFFFFFF).to_bytes(4, "little")
        if checksum == "bad":
            ck = bytes([ck[0] ^ 1]) + ck[1:]
    return _u8(_frame(size or 0, parts, fcs_bytes=fcs_bytes, window_log=window_log, checksum=ck)), \
        (bytes(out) if ok else None)


def _fill_rle(have: int, n: int, nblocks: int | None = None, byte: int = 0x3C) -> list:
    """RLE blocks that take the frame from `have` to n bytes: as few as fit, or exactly nblocks"""
    rem = n - have
    k = nblocks if nblocks is not None else max(1, -(-rem // ZS_BLOCK))
    assert 0 < rem <= k * ZS_BLOCK and rem >= k, (rem, k)
    sizes = [rem // k + (1 if i < rem % k else 0) for i in range(k)]
    return [rle(byte + i, s) for i, s in enumerate(sizes)]


def _planned(blocks) -> int:
    return len(zstd_frame(blocks)[1])


def dense_frame(n: int, seed: int = 0) -> tuple[np.ndarray, bytes]:
    """A frame of n bytes with about n / 3 sequences: ML = 3 and LL = 0 with a repeat offset (offset value 1 with no
    literals: the second repeat offset, so the match distance alternates 4, 1, 4, ...), 43 690 to a 128 KiB block and
    about 349 000 to a MiB -- far more than the pipeline's pool holds per frame (cap / 8 + 64)."""
    rng = np.random.default_rng([seed, n, 3])
    head = bytes(rng.integers(0, 256, size=16, dtype=np.uint8))
    blocks, have = [raw(head)], 16
    while have < n:
        m = min(ZS_BLOCK, n - have)
        k, t = m // 3, m % 3
        blocks.append(seqs(bytes(rng.integers(0, 256, size=t, dtype=np.uint8)), [(0, 3, 1)] * k))
        have += m
    return zstd_frame(blocks)


def _zvec(name, n, route, built, valid=True):
    frame, plan = built
    if valid:
        assert plan is not None and len(plan) == n, (name, None if plan is None else len(plan), n)
    return Vector(name, COMP_ZSTD, frame, n, _u8(plan) if valid else None, route)


def zstd_vectors(n: int, seed: int = 1) -> list[Vector]:
    """The zstd vectors that fit a capacity of n bytes"""
    rng = np.random.default_rng([seed, n, 5])
    rb = lambda k: bytes(rng.integers(0, 256, size=k, dtype=np.uint8))      # noqa: E731
    out = []
    head = raw(rb(16))
    # sequence counts around ZP_CX_SEQS: LL 0, ML 4, offsets 5-12 from the extra bits of one offset code
    for k in (ZP_CX_SEQS - 1, ZP_CX_SEQS, ZP_CX_SEQS + 1):
        blk = [head, seqs(b"", [(0, 4, 8 + int(rng.integers(0, 8))) for _ in range(k)])]
        if _planned(blk) < n:
            out.append(_zvec(f"zstd-seqs-{k}", n, "zp-cx" if k >= ZP_CX_SEQS else "zp",
                             zstd_frame(blk + _fill_rle(_planned(blk), n))))
    # overlapping copies: offsets 1-15 (one frame per offset code), lengths across 16, 32 and 2 KiB, Raw and RLE literals
    for lo, hi in ((1, 4), (5, 12), (13, 15)):
        blk = [head]
        for j, mls in enumerate(((15,), (16,), (17,), (31,), (32,), (33,), (2047, 2048, 2049))):
            lit = bytes([97 + j]) * (len(mls) * (hi - lo + 1)) if j % 2 else rb(len(mls) * (hi - lo + 1))
            blk.append(seqs(lit, [(1, ml, off + 3) for off in range(lo, hi + 1) for ml in mls], "rle" if j % 2 else "raw"))
        if _planned(blk) < n and len(blk) < ZP_MAXB:
            out.append(_zvec(f"zstd-overlap-{lo}-{hi}", n, "zp", zstd_frame(blk + _fill_rle(_planned(blk), n))))
    # matches reaching back into earlier blocks: a Raw block, an RLE block, then copies from both, as far as 65 532 back
    blk = [raw(rb(50000)), rle(0x41, 20000),
           seqs(rb(8), [(2, 43 + int(rng.integers(0, 4)), 32768 + int(rng.integers(0, 32768))) for _ in range(4)]),
           seqs(rb(2), [(1, 100, 20000 + 3), (1, 120, 20150 + 3)]), seqs(rb(2), [(1, 70, 60000 + 3), (1, 80, 65000 + 3)])]
    if _planned(blk) < n:
        out.append(_zvec("zstd-back-into-earlier-blocks", n, "zp", zstd_frame(blk + _fill_rle(_planned(blk), n))))
    # long runs at the size of a job for the raw / RLE stage, and three of them in one frame (two are jobs)
    blk = [head, seqs(b"zzz", [(1, 32767, 4), (1, 32768, 4), (1, 32769, 4)], "rle")]
    if _planned(blk) < n:
        out.append(_zvec("zstd-runs-32767-32768-32769", n, "zp", zstd_frame(blk + _fill_rle(_planned(blk), n))))
    blk = [head, seqs(rb(2), [(1, 40000, 4), (1, 40001, 4)]), seqs(rb(1), [(1, 50000, 4)])]
    if _planned(blk) < n:
        out.append(_zvec("zstd-three-long-runs", n, "zp", zstd_frame(blk + _fill_rle(_planned(blk), n))))
    # 16 and 17 blocks
    for nb in (ZP_MAXB, ZP_MAXB + 1):
        fill_k = max(1, -(-max(n - 2000, 1) // ZS_BLOCK))
        small = []
        for j in range(nb - fill_k):
            small.append([raw(rb(30)), rle(0x20 + j, 50), seqs(rb(6), [(2, 20, 4 + 10), (2, 20, 4 + 8)])][j % 3]
                         if j else head)
        if nb - fill_k >= 1 and n - _planned(small) >= fill_k:
            try:
                blk = small + _fill_rle(_planned(small), n, fill_k)
            except AssertionError:
                continue
            out.append(_zvec(f"zstd-{nb}-blocks", n, "zp" if nb <= ZP_MAXB else "zp-fallback", zstd_frame(blk)))
    body = [head, seqs(rb(5), [(1, 67, 8), (1, 70, 9)])]
    if _planned(body) < n:
        body = body + _fill_rle(_planned(body), n)
        # window descriptors: 2^27 is the largest ZSTD_decompress takes by default, 2^28 is rejected
        out.append(_zvec("zstd-window-27", n, "zp", zstd_frame(body, window_log=27)))
        out.append(_zvec("zstd-window-28", n, "zp-fallback", zstd_frame(body, window_log=28), False))
        out.append(_zvec("zstd-no-content-size", n, "zp", zstd_frame(body, content_size=None, window_log=20)))
        out.append(_zvec("zstd-checksum", n, "zp", zstd_frame(body, checksum="good")))
        for w in (1, 2, 4, 8):
            if w == 1 and n >= 256 or w == 2 and not 256 <= n < 65792:
                continue
            out.append(_zvec(f"zstd-fcs-{w}", n, "zp", zstd_frame(body, fcs_bytes=w)))
        # rule-breaking: content size one short of the blocks, blocks one short of the capacity, no last block,
        # a byte after the frame, an offset before the frame's start
        out.append(_zvec("zstd-fcs-short", n, "any", zstd_frame(body, content_size=n - 1), False))
        out.append(_zvec("zstd-one-short", n, "any", zstd_frame(body[:-1] + _fill_rle(_planned(body[:-1]), n - 1)), False))
        out.append(_zvec("zstd-no-last-block", n, "any", zstd_frame(body, last=False), False))
        f, _ = zstd_frame(body)
        out.append(Vector("zstd-trailing-byte", COMP_ZSTD, np.concatenate([f, _u8(b"\0")]), n, None, "any"))
        far = [raw(rb(16)), seqs(rb(2), [(1, 8, 30 + 3)])]
        out.append(_zvec("zstd-offset-before-start", n, "any", zstd_frame(far + _fill_rle(18, n)), False))
    # the match that ends exactly at the capacity (legal in zstd)
    tail = [head] + (_fill_rle(16, n - 500) if n - 516 > 0 else [])
    have = _planned(tail)
    if n - have >= 10:
        out.append(_zvec("zstd-match-to-cap", n, "zp",
                         zstd_frame(tail + [seqs(rb(2), [(2, n - have - 2, 7 + 3)])])))
    if n >= 64:
        out.append(_zvec("zstd-dense", n, "dense", dense_frame(n, seed)))
    return out


def vectors(n: int, seed: int = 1) -> list[Vector]:
    return lz4_vectors(n, seed) + zstd_vectors(n, seed)


# ---- verdicts and mutations ----------------------------------------------------------------------------------------

def restate(method: int, stream, cap: int) -> tuple[int, np.ndarray]:
    """the plain-C restatement: (bytes written or negative, out[cap])"""
    fn = port.lz4_decode if method == COMP_LZ4 else port.zstd_decode
    return fn(np.ascontiguousarray(stream, dtype=np.uint8), cap=cap)[:2]


def verdict(method: int, stream, cap: int) -> np.ndarray | None:
    """What a decoder of the library must do with the stream at capacity cap: the restatement's bytes, or None for a
    rejection.  A stream that fills less than the capacity may be rejected or give those bytes with out_size set to
    their count (see accepts()).  (A zstd content checksum is skipped, not verified: DESIGN.md section 1.)"""
    got, out = restate(method, stream, cap)
    return out[:got].copy() if got >= 0 else None


def accepts(want, cap: int, status: int, out_size: int, out) -> bool:
    """Whether a decoder's (status, out_size, bytes) is the verdict want (verdict()) at capacity cap"""
    if want is None:
        return status != 0
    if status != 0:
        return want.size != cap
    return out_size == want.size and np.array_equal(out[:want.size], want)


def mutate(rng, stream: np.ndarray) -> tuple[np.ndarray, str]:
    """One of tools/emu_fuzz.py's mutations: flipped bytes, a flipped header bit, a cut, appended bytes"""
    m = stream.copy()
    how = int(rng.integers(0, 4))
    if how == 0 and m.size:
        for _ in range(int(rng.integers(1, 4))):
            m[int(rng.integers(0, m.size))] ^= int(rng.integers(1, 256))
        return m, "flip"
    if how == 1 and m.size:
        m[int(rng.integers(0, min(m.size, 24)))] ^= 1 << int(rng.integers(0, 8))
        return m, "header"
    if how == 2:
        return m[: int(rng.integers(0, max(m.size, 1)))].copy(), "cut"
    return np.concatenate([m, rng.integers(0, 256, size=int(rng.integers(1, 9)), dtype=np.uint8)]), "append"


# ---- streams of the system libraries, and the mutation corpus ------------------------------------------------------

_clibs = None


def _compressors():
    global _clibs
    if _clibs is None:
        import ctypes as C
        lz4, zs = C.CDLL("liblz4.so.1"), C.CDLL("libzstd.so.1")
        for f in (lz4.LZ4_compress_fast, lz4.LZ4_compress_HC):
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
            f.restype = C.c_int
        zs.ZSTD_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int]
        zs.ZSTD_compress.restype = C.c_size_t
        zs.ZSTD_isError.argtypes = [C.c_size_t]
        _clibs = lz4, zs
    return _clibs


LZ4_PRODUCERS = [("lz4", 1), ("lz4", 9), ("lz4", 65537), ("lz4hc", 9)]
ZSTD_PRODUCERS = [("zstd", -5), ("zstd", 1), ("zstd", 3), ("zstd", 9), ("zstd", 19), ("zstd", 22)]


def produce(producer: tuple, block: np.ndarray) -> tuple[int, np.ndarray]:
    """(method, stream) of liblz4 (LZ4_compress_fast at an acceleration, LZ4_compress_HC at a level) or libzstd
    (ZSTD_compress at a level)"""
    lz4, zs = _compressors()
    kind, arg = producer
    b = np.ascontiguousarray(block, dtype=np.uint8)
    out = np.zeros(b.size + b.size // 128 + 4096, dtype=np.uint8)
    if kind == "zstd":
        got = zs.ZSTD_compress(out.ctypes.data, out.size, b.ctypes.data, b.size, arg)
        assert not zs.ZSTD_isError(got)
        return COMP_ZSTD, out[:got].copy()
    fn = lz4.LZ4_compress_fast if kind == "lz4" else lz4.LZ4_compress_HC
    got = fn(b.ctypes.data, out.ctypes.data, b.size, out.size, arg)
    assert got > 0
    return COMP_LZ4, out[:got].copy()


CORPUS_CAP = 160 * 1024


def corpus(cap: int = CORPUS_CAP, seed: int = 7) -> list[tuple[int, np.ndarray, np.ndarray | None, str]]:
    """A fixed seeded corpus at capacity cap: streams of liblz4 and libzstd over the layouts of tools/emu_fuzz.py (long
    one-byte runs, random bytes, text, copies from anywhere earlier), the crafted vectors that fit, and about a third of
    them mutated (mutate()).  Per stream: (method, stream, the intact block or None when mutated, tag)."""
    import encode_check as ec
    rng = np.random.default_rng([seed, cap])
    base = []
    for i, kind in enumerate(["copies", "text", "sparse", "run-00", "random", "tile65537", "copies", "sparse"]):
        blk = ec.layout(kind, cap, seed + i)
        for p in (LZ4_PRODUCERS[i % 4], ZSTD_PRODUCERS[i % 4], ZSTD_PRODUCERS[(i + 1) % 3]):
            m, s = produce(p, blk)
            base.append((m, s, blk, f"{kind}/{p[0]}{p[1]}"))
    for v in vectors(cap, seed):
        # (not the checksum frame: a mutation there is the documented deviation, which has tests of its own)
        if v.plain is not None and v.route != "dense" and v.name != "zstd-checksum":
            base.append((v.method, v.stream, v.plain, v.name))
    out = []
    for k, (m, s, blk, tag) in enumerate(base):
        out.append((m, s, blk, tag))
        if k % 2 == 0:
            ms, how = mutate(rng, s)
            out.append((m, ms, None, f"{tag}/{how}"))
    return out
