"""Hand-crafted zstd conformance frames for format branches ZSTD_compress never emits
(SURVEY.md appendix B): RLE literals, direct (4-bit) Huffman weights, single-stream
Huffman literals, Raw/RLE blocks in a single-segment frame, RLE sequence tables.
Each is (name, frame bytes as uint8 array, expected output bytes)."""
import numpy as np


def _frame(content_len, blocks, fcs_bytes=1, window_log=None, checksum=None):
    """A frame around the given blocks.  window_log None: single segment with a content size of fcs_bytes (1, 2, 4
    or 8) bytes; otherwise a window descriptor of that log and a content size of fcs_bytes (0: none, 2, 4 or 8).
    checksum: the 4 bytes written after the last block (sets the checksum flag)."""
    if window_log is None:
        flag = {1: 0, 2: 1, 4: 2, 8: 3}[fcs_bytes]
        fhd, wd = 0x20 | (flag << 6), b""
    else:
        flag = {0: 0, 2: 1, 4: 2, 8: 3}[fcs_bytes]
        fhd, wd = flag << 6, bytes([(window_log - 10) << 3])
    if checksum is not None:
        fhd |= 0x04
    v = content_len - 256 if fcs_bytes == 2 else content_len
    assert 0 <= v < 1 << (8 * fcs_bytes) or fcs_bytes == 0
    return (bytes([0x28, 0xB5, 0x2F, 0xFD, fhd]) + wd + v.to_bytes(fcs_bytes, "little") + b"".join(blocks) +
            (bytes(checksum) if checksum is not None else b""))


def _block_header(last, btype, size):
    """btype 0 Raw, 1 RLE, 2 Compressed; size: the bytes of a Raw or Compressed block, the count of an RLE one"""
    v = (1 if last else 0) | (btype << 1) | (size << 3)
    return bytes([v & 0xFF, (v >> 8) & 0xFF, (v >> 16) & 0xFF])


def _huffman_bits(codes, message):
    """backward bitstream: codes in message order, end-marker bit above them"""
    s = "".join(codes[m] for m in message)
    val = int("1" + s[::-1][::-1], 2) if False else None
    # first symbol is read first = most significant bits below the marker
    val = int("1" + s, 2)
    n = (val.bit_length() + 7) // 8
    return val.to_bytes(n, "little")


def conformance_frames():
    out = []
    # 1. raw block
    out.append(("raw-block", _frame(5, [_block_header(True, 0, 5) + b"hello"]), b"hello"))
    # 2. rle block
    out.append(("rle-block", _frame(200, [_block_header(True, 1, 200) + b"z"]), b"z" * 200))
    # 3. compressed block, RLE literals, zero sequences
    n = 20
    body = bytes([1 | (n << 3), ord("q")]) + b"\x00"
    out.append(("rle-literals", _frame(n, [_block_header(True, 2, len(body)) + body]), b"q" * n))
    # 4. compressed block, raw literals, zero sequences
    body = bytes([0 | (7 << 3)]) + b"literal" + b"\x00"
    out.append(("raw-literals", _frame(7, [_block_header(True, 2, len(body)) + body]), b"literal"))
    # 5. direct-weight Huffman, single stream: symbols 0,1,2 with weights 2,1,(1)
    codes = {0: "1", 1: "00", 2: "01"}
    msg = [0, 1, 2, 0, 0, 2, 1, 0, 0, 0, 1, 2, 2, 0, 1, 0, 0, 0, 2, 0]
    stream = _huffman_bits(codes, msg)
    tree = bytes([0x81, 0x21])
    regen, csize = len(msg), len(tree) + len(stream)
    hdr = 2 | (0 << 2) | (regen << 4) | (csize << 14)
    body = bytes([hdr & 0xFF, (hdr >> 8) & 0xFF, (hdr >> 16) & 0xFF]) + tree + stream + b"\x00"
    out.append(("huffman-direct-weights-1stream",
                _frame(regen, [_block_header(True, 2, len(body)) + body]), bytes(msg)))
    # 6. several blocks: raw + rle + raw, not-last flags
    blocks = [_block_header(False, 0, 3) + b"abc", _block_header(False, 1, 10) + b"-",
              _block_header(True, 0, 2) + b"xy"]
    out.append(("multi-block", _frame(15, blocks), b"abc" + b"-" * 10 + b"xy"))
    # 7. one sequence with predefined tables: literals "abcd", match len 8 offset 4
    #    LL=4 (code 4), ML=8 (code 5), offset value 4+3=7 -> code 2, extra bits 3 (2 bits)
    #    states: predefined tables; simplest is RLE mode for all three tables
    #    modes byte: LL RLE(1)<<6 | OF RLE(1)<<4 | ML RLE(1)<<2 ; symbols 4, 2, 5
    #    bitstream: initial states take 0 bits each (RLE tables have log 0);
    #    offset extra: 2 bits = 0b11 ; ML, LL have 0 extra bits.
    #    backward stream bytes: value = marker(1) followed by '11' -> 0b111 = 0x07
    body = bytes([0 | (4 << 3)]) + b"abcd" + bytes([1, (1 << 6) | (1 << 4) | (1 << 2), 4, 2, 5, 0x07])
    out.append(("rle-sequence-tables", _frame(12, [_block_header(True, 2, len(body)) + body]),
                b"abcd" + b"abcd" * 2))
    return [(n, np.frombuffer(f, dtype=np.uint8).copy(), e) for n, f, e in out]
