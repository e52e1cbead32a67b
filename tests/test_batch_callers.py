"""The batched callers of pg_cryogen_b200/host/cryo_batch.c (block cache, read-ahead scan, TID fetch, COPY writer) on
the CPU: a private copy of cryo_batch.c built against tests/cryogpu_stub.c, the stand-in of the five libcryogpu calls
it makes.  The scenarios (tests/batch_scenarios.py) are the ones tests/test_gpu_batch_callers.py runs on the device;
both must agree with the model of the reference's callers in tests/caller_model.py."""
import pytest

import batch_scenarios as sc


@pytest.fixture(scope="module")
def stub():
    return sc.Backend(sc.stub_library(), None)


def test_repeated_blocks_in_one_call(stub):
    sc.repeat_case(stub)


@pytest.mark.parametrize("nslots", [1, 3, 16])
def test_cache_sequences(stub, nslots):
    model = sc.run_cache(stub, nslots, seed=11)
    assert model.hits and model.blocks


@pytest.mark.parametrize("nslots,readahead", [(4, 1), (4, 2), (4, 4), (4, 9), (1, 1), (16, 21)])
def test_scan(stub, nslots, readahead):
    sc.run_scan(stub, nslots, readahead)


@pytest.mark.parametrize("method", [0, 1])
@pytest.mark.parametrize("batch,big", [(1, 5), (3, 5), (129, 131)])
def test_writer(stub, method, batch, big):
    sc.run_writer(stub, method, batch, big)


def test_fetch_tuples(stub):
    sc.run_fetch(stub, seed=5)
