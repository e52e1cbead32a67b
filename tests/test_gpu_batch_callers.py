"""-m gpu: the batched callers of pg_cryogen_b200/host/cryo_batch.c (block cache, read-ahead scan, TID fetch, COPY
writer) through libcryo_batch.so on the device: the scenarios of tests/batch_scenarios.py that tests/test_batch_callers.py
runs on the CPU stand-in, checked against the same model of the reference's callers (tests/caller_model.py), the
restated gather and the reference's codec."""
import ctypes as C
import os

import pytest

import batch_scenarios as sc

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def dev(gpu):
    return sc.Backend(sc.bind(C.CDLL(os.path.join(HERE, "..", "pg_cryogen_b200", "libcryo_batch.so"))), gpu.handle)


def test_repeated_blocks_in_one_call(dev):
    sc.repeat_case(dev)


@pytest.mark.parametrize("nslots", [1, 3, 16])
def test_cache_sequences(dev, nslots):
    model = sc.run_cache(dev, nslots, seed=11)
    assert model.hits and model.blocks


@pytest.mark.parametrize("nslots,readahead", [(4, 1), (4, 2), (4, 4), (4, 9), (1, 1), (16, 21)])
def test_scan(dev, nslots, readahead):
    sc.run_scan(dev, nslots, readahead)


@pytest.mark.parametrize("method", [0, 1])
@pytest.mark.parametrize("batch,big", [(1, 5), (3, 5), (129, 131)])
def test_writer(dev, method, batch, big):
    sc.run_writer(dev, method, batch, big)


def test_fetch_tuples(dev):
    sc.run_fetch(dev, seed=5)
