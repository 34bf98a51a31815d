"""Host-side error paths: a device allocation that fails is reported as a CUDA error (-2) and leaves nothing behind that fails
later calls on the same engine or store from the same host thread."""
import numpy as np
import pytest

import corpus

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def trip(octx):
    n = 6
    return corpus.gen_valid(octx, n, seed=b"host-errors", threads=4), corpus.trip_streams(b"host-errors", n)


def test_failed_allocation_leaves_the_engine_usable(act, engine, octx, trip):
    base, streams = trip
    lib = act.load_library()
    small = np.zeros(256, np.uint8)
    # 2^40 requests: the first staging buffer would take 64 TB, so cudaMalloc fails before any host byte is read
    rc = lib.act_batch_request(engine._h, 2 ** 40, small.ctypes.data, small.ctypes.data, small.ctypes.data)
    with pytest.raises(act.ActError, match=r"failed \(-2\): cudaMalloc"):
        act._check(rc, "act_batch_request")
    assert rc == -2
    assert (engine.batch_request(streams["pre"], streams["req_rnd"]) == base["req"]).all()
    ref, nul, st = engine.batch_verify_spend_and_refund(base["proofs"], base["rnd"])
    o_ref, o_nul, o_st, _ = octx.batch_refund(base["proofs"], base["rnd"], threads=4)
    assert st.tolist() == o_st.tolist() and (st == 0).all()
    assert (ref == o_ref).all() and (nul == o_nul).all()


def test_failed_allocation_leaves_later_stores_usable(act):
    with pytest.raises(act.ActError, match=r"failed \(-2\): cudaMalloc"):
        act.NullifierStore(device=0, capacity=2 ** 45)           # a 2 PB table
    keys = np.random.RandomState(3).randint(0, 256, size=(64, 32)).astype(np.uint8)
    keys[:, 31] &= 0x0f                                          # reduced mod l
    keys[32:] = keys[:32]
    with act.NullifierStore(device=0, capacity=1024) as store:
        assert store.screen(np.zeros(64, np.uint8), keys).tolist() == [0] * 32 + [3] * 32
        assert store.size == 32
