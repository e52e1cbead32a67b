"""The page chain around the codec (SURVEY.md 8 f-1, a10), CPU part: the restatement of the reference's
split (pg_cryogen.c:689-805) and gather (cache.c:100-176) in oracle/cryo_pages.c, pinned against the
reference's own storage.h as compiled into oracle/_ref, and against its stored outputs (tests/golden)."""
import ctypes as C

import numpy as np

from oracle import pages as opg
from pg_cryogen_b200 import blockgen as bg

import golden_util

PAGE = 8192


def test_page_header_layout_is_the_references(oracle_ref):
    """sizeof / offsetof from the reference's storage.h (stored; compiled in oracle/_ref where present) = the
    restatement's."""
    want = golden_util.reference_outputs()["layout"]
    if oracle_ref.available():
        got = (C.c_uint32 * 12)()
        oracle_ref.lib().oref_page_layout(got)
        assert list(got) == want
    assert want == opg.layout()
    assert want[:2] == [32, 48]                 # SURVEY.md A.1: payload offsets 32 / 48


def test_pages_needed_edges():
    # pg_cryogen.c:692-704: first page holds 8192 - 48, the others 8192 - 32
    for size, want in ((1, 1), (8144, 1), (8145, 2), (8144 + 8160, 2), (8144 + 8160 + 1, 3), (1 << 20, 129),
                       ((1 << 20) + 4112, 130)):
        assert opg.pages_needed(size) == want, size


def test_split_then_gather_roundtrip_and_errors(oracle_ref):
    rng = np.random.default_rng(3)
    rel = np.zeros((400, PAGE), dtype=np.uint8)
    blocks = [bg.make_block("S", "hex", 1), bg.make_block("M", "hex", 2), bg.make_block("D", "random", 3)]
    comp = [oracle_ref.compress(i & 1, 1, b)[0][0] for i, b in enumerate(blocks)]
    free = list(rng.permutation(np.arange(1, 400)))         # block 0 is the metapage; chains are NOT adjacent
    chains = []
    for i, c in enumerate(comp):
        need = opg.pages_needed(c.size)
        ch = [int(free.pop()) for _ in range(need)]
        assert opg.split(rel, ch, c, i & 1, 1000 + i) == need
        chains.append(ch)
    for i, c in enumerate(comp):
        err, method, size, got, chain = opg.gather(rel, chains[i][0])
        assert err == opg.ERR_SUCCESS and method == (i & 1) and size == c.size and chain == chains[i]
        assert np.array_equal(got, c)
        back, ok = oracle_ref.decompress_one(method, got)
        assert ok and np.array_equal(back, blocks[i])
    # cache.c:115-129
    assert opg.gather(rel, int(free[0]))[0] == opg.ERR_EMPTY_BLOCK
    assert opg.gather(rel, chains[1][1])[0] == opg.ERR_WRONG_STARTING_BLOCK
    # a chain cut short: fewer bytes than compressed_size come back (the reference then fails in cryo_decompress)
    rel2 = rel.copy()
    rel2[chains[2][3], 28:32] = 0xFF
    err, method, size, got, chain = opg.gather(rel2, chains[2][0])
    assert err == opg.ERR_SUCCESS and got.size < size and len(chain) == 4


def test_tuple_walk_restatement_equals_the_references(oracle_ref):
    """cryo_oracle_block_tuple_stats against the loop of cryo_getnextslot around the reference's own
    cryo_storage_fetch (oref_block_walk in oracle/_ref where present; its stored results)."""
    stored = golden_util.reference_outputs()["tuple_walk"]
    for kind, pl, seed in (("S", "hex", 1), ("M", "lowcard", 2), ("D", "hex", 3), ("D", "random", 4)):
        b = bg.make_block(kind, pl, seed)
        want = tuple(stored[f"{kind}_{pl}_{seed}"])
        if oracle_ref.available():
            n, by = C.c_uint32(0), C.c_uint64(0)
            oracle_ref.lib().oref_block_walk(C.c_void_p(b.ctypes.data), C.byref(n), C.byref(by))
            assert (n.value, by.value) == want, (kind, pl)
        assert opg.block_tuple_stats(b) == (*want, 1), (kind, pl)
    empty = np.zeros(1 << 20, dtype=np.uint8)
    if oracle_ref.available():
        oracle_ref.lib().oref_init_page(C.c_void_p(empty.ctypes.data))
    else:
        empty[:8] = np.array([8, 1 << 20], dtype=np.uint32).view(np.uint8)      # cryo_init_page: lower, upper
    assert opg.block_tuple_stats(empty) == (0, 0, 1)
    bad = bg.make_block("S", "hex", 5).copy()
    bad[8 + 8 * 7: 8 + 8 * 7 + 4] = 0xFF                # item 8 points outside the block
    assert opg.block_tuple_stats(bad)[2] == 0
