"""Issuer key slots without a GPU: the keyed head stage of the device code, compiled for the host (tests/hostsim_keys), against the
oracle's cross-key refund; and the new C entry points refuse to run without a device or with NULL."""
import numpy as np
import pytest

import corpus
import hostsim_keys_lib as HK
import oracle_keys_lib as OK

PB = corpus.PROOF_BYTES


@pytest.fixture(scope="module")
def keys():
    """three issuer keys over the test Params: oracle and host-simulation contexts of each"""
    octxs = [corpus.make_ctx(corpus.TEST_PARAMS, key_seed=b"act-b200-key-%d" % k) for k in range(3)]
    return octxs, [HK.Ctx(c.h, c.x, c.w) for c in octxs]


def test_oracle_cross_refund_with_one_key_is_the_oracle_refund(keys):
    octxs, _ = keys
    base = corpus.gen_valid(octxs[0], 12, seed=b"keys-same", threads=8)
    proofs, rnd, _, _ = corpus.mutate_proofs(octxs[0], base)
    ref, nul, st, _ = octxs[0].batch_refund(proofs, rnd, threads=8)
    ref2, nul2, st2 = OK.batch_refund_keyed({0: octxs[0]}, octxs[0], proofs, np.zeros(12, np.uint8), rnd)
    assert (st2 == st).all() and (ref2 == ref).all() and (nul2 == nul).all()
    assert (st == 0).sum() >= 3


def test_hostsim_keyed_refund_matches_the_oracle(keys):
    """Proofs under three keys in slots 0, 3 and 7 (slot 3 selected): right ids, wrong-slot ids, empty-slot ids, ids >= 16,
    bad points and an identity A'."""
    octxs, hctxs = keys
    slot_of = {0: 0, 1: 3, 2: 7}
    o_slots = {slot_of[k]: octxs[k] for k in range(3)}
    h_slots = {slot_of[k]: hctxs[k] for k in range(3)}
    proofs, rnd, ids = [], [], []
    for k in range(3):
        base = corpus.gen_valid(octxs[k], 12, seed=b"keys-mixed-%d" % k, threads=8)
        pf, r, _, _ = corpus.mutate_proofs(octxs[k], base)   # kinds 0..11: valid, failed checks, identity A', bad points, ...
        pf = pf.reshape(12, PB); r = r.reshape(12, 128)
        for i in range(12):
            proofs.append(pf[i]); rnd.append(r[i])
            ids.append(slot_of[k])
        for i, wrong in ((0, slot_of[(k + 1) % 3]), (6, 5), (0, 16), (6, 255), (3, 9), (5, 200)):
            proofs.append(pf[i]); rnd.append(r[i]); ids.append(wrong)   # another key's slot, empty slots, ids past the table
    proofs = np.concatenate(proofs); rnd = np.concatenate(rnd); ids = np.array(ids, np.uint8)
    o_ref, o_nul, o_st = OK.batch_refund_keyed(o_slots, o_slots[3], proofs, ids, rnd)
    ref, nul, st = HK.refund_keyed(h_slots[3], h_slots, proofs, ids, rnd)
    assert (st == o_st).all(), (st, o_st)
    assert (ref == o_ref).all() and (nul == o_nul).all()
    seen = set(o_st.tolist())
    assert {0, 6, 7, 0x81} <= seen, seen
    # accepted refunds verify under the selected key's W; proofs of key 0 under slot 0 were accepted
    com = proofs.reshape(-1, PB)[:, 4 * 32:132 * 32].reshape(-1)
    ok = o_st == 0
    chk = h_slots[3].refund_check(com.reshape(-1, 4096)[ok].reshape(-1), ref.reshape(-1, 128)[ok].reshape(-1))
    assert (chk == 0).all()
    assert o_st[0] == 0 and o_st[18] == 0 and o_st[36] == 0


def test_key_entry_points_fail_without_a_device_or_with_null(act):
    lib = act.load_library()
    one = np.zeros(64, np.uint8)
    p = one.ctypes.data
    assert lib.act_engine_set_key(None, 1, p, p) != 0
    assert lib.act_engine_clear_key(None, 1) != 0
    assert lib.act_engine_select_key(None, 0) != 0
    assert lib.act_engine_selected_key(None) == -1
    assert lib.act_engine_key_slots(None) == 0
    assert lib.act_batch_verify_spend_and_refund_keyed_dev(None, 1, p, p, p, p, p, p, None) != 0
    assert lib.act_batch_verify_spend_and_refund_keyed(None, 1, p, p, p, None, p, p, p) != 0
    assert lib.act_batch_spend_verify_keyed(None, 1, p, p, p, p, p) != 0
    if act.device_count() == 0:
        with pytest.raises(act.ActError):
            act.Engine(act.Params(bytes(96)), act.PrivateKey(bytes(32), bytes(32)))
