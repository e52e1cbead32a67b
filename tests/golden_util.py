"""Load tests/golden/reference_streams.npz -> list of (name, method, level, stream, sha256)."""
import os

import numpy as np

from pg_cryogen_b200 import blockgen as bg

HERE = os.path.dirname(os.path.abspath(__file__))

# how to rebuild the plaintext of each fixture (must match tests/golden/make_golden.py)
PLAINTEXT = {
    "regr_rows_1_290": lambda: bg.regression_block(1, 290),
    "regr_rows_291_500": lambda: bg.regression_block(291, 500),
    "regr_rows_501_790": lambda: bg.regression_block(501, 790),
    "regr_rows_791_1000": lambda: bg.regression_block(791, 1000),
    "S_hex_b7": lambda: bg.make_block("S", "hex", 7),
    "S_lowcard_b7": lambda: bg.make_block("S", "lowcard", 7),
    "M_lowcard_b7": lambda: bg.make_block("M", "lowcard", 7),
    "D_lowcard_b7": lambda: bg.make_block("D", "lowcard", 7),
}


def load():
    z = np.load(os.path.join(HERE, "golden", "reference_streams.npz"))
    names = sorted(k[: -len("__stream")] for k in z.files if k.endswith("__stream"))
    out = []
    for n in names:
        method, level = (int(v) for v in z[n + "__method"])
        out.append((n, method, level, z[n + "__stream"], bytes(z[n + "__sha256"])))
    return out


def plaintext(name: str) -> np.ndarray:
    key = name.rsplit("_", 1)[0]
    return PLAINTEXT[key]()


def reference_outputs() -> dict:
    """tests/golden/reference_outputs.json: what the reference's storage.c, storage.h and compression.c produced
    (page layout, tuple walks, SHA-256 of built blocks, compressed sizes); README.md there says where from."""
    import json
    with open(os.path.join(HERE, "golden", "reference_outputs.json")) as f:
        return json.load(f)


def reference_block_sha256(oracle_ref, key: str, tuples) -> str:
    """SHA-256 of the block the reference's storage.c builds from `tuples`: checked against the stored value
    through oracle/_ref where it is present; the stored value is returned either way."""
    import hashlib
    want = reference_outputs()["block_sha256"][key]
    if oracle_ref.available():
        got = oracle_ref.build_block([bytes(t) for t in tuples])
        assert hashlib.sha256(got.tobytes()).hexdigest() == want, key
    return want
