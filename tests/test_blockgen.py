"""blockgen restates storage.c:15-50; check it byte for byte against the reference's
own cryo_init_page / cryo_storage_insert (SHA-256 of the blocks it built, stored in
tests/golden and checked through oracle/_ref where present)."""
import hashlib

import numpy as np
import pytest

from pg_cryogen_b200 import blockgen as bg

from golden_util import reference_block_sha256


def _sha(blk) -> str:
    return hashlib.sha256(blk.tobytes()).hexdigest()


@pytest.mark.parametrize("kind", ["S", "M", "D"])
@pytest.mark.parametrize("payload", bg.PAYLOADS)
def test_pack_block_matches_reference_storage(oracle_ref, kind, payload):
    t = bg.make_tuples(kind, payload, 5)
    assert _sha(bg.pack_block(t)) == reference_block_sha256(oracle_ref, f"{kind}_{payload}_5", t)


def test_ragged_tuples_and_partial_last_block(oracle_ref):
    tuples = [bytes([i % 251]) * (25 + 7 * i) for i in range(100)]
    assert _sha(bg.pack_block(tuples)) == reference_block_sha256(oracle_ref, "ragged_100", tuples)
    t = bg.make_tuples("S", "hex", 3448, ntuples=80)     # last block of the 1M-row table
    assert _sha(bg.pack_block(t)) == reference_block_sha256(oracle_ref, "S_hex_3448_80", t)
    assert _sha(bg.pack_block(np.zeros((0, 61), np.uint8))) == reference_block_sha256(oracle_ref, "empty", [])


def test_tuple_limits_follow_storage_c(oracle_ref):
    """storage.c:32-33: at most 290 tuples; a tuple must fit between lower and upper."""
    t = bg.make_tuples("S", "hex", 0)
    assert t.shape[0] == 290
    with pytest.raises(ValueError):
        bg.pack_block(np.zeros((291, 61), np.uint8))
    if oracle_ref.available():
        with pytest.raises(ValueError):
            oracle_ref.build_block([bytes(61)] * 291)
    with pytest.raises(ValueError):
        bg.pack_block(np.zeros((290, 3624), np.uint8))
    hdr = bg.pack_block(t)[:8].view(np.uint32)
    assert hdr[0] == 8 + 8 * 290 and hdr[1] == (1 << 20) - 290 * 64


def test_table_shape_of_the_headline_config():
    assert bg.table_block_count(1_000_000, "S") == 3449
    blk = bg.make_table_blocks(1_000_000, "S", "hex", first_block=3448, count=1)[0]
    assert blk[:4].view(np.uint32)[0] == 8 + 8 * 80     # 1M - 3448*290 = 80 rows


def test_blocks_are_deterministic_and_independent():
    a = bg.make_block("M", "lowcard", 17)
    b = bg.make_blocks("M", "lowcard", 16, 3)[1]
    assert np.array_equal(a, b)
    assert not np.array_equal(a, bg.make_block("M", "lowcard", 18))
