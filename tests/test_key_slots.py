"""Issuer key slots on the GPU (act_engine_set_key / _select_key / _clear_key, act_batch_verify_spend_and_refund_keyed[_dev],
act_batch_spend_verify_keyed).

Oracle: the CPU oracle's cross-key refund (tests/oracle_keys: verify under the key the proof names, sign under the selected key),
the oracle's own calls for everything unkeyed, and a Python NullifierDb per store."""
import os
import struct
import subprocess

import numpy as np
import pytest

import corpus
import oracle_keys_lib as OK
import oracle_lib as O

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
CPP = os.path.join(HERE, "cpp")
PB = corpus.PROOF_BYTES
SLOTS = (0, 3, 7)   # where the three test keys live


@pytest.fixture(scope="module")
def keys():
    """oracle contexts of three issuer keys over the test Params, by slot"""
    return {s: corpus.make_ctx(corpus.TEST_PARAMS, key_seed=b"act-b200-key-%d" % i) for i, s in enumerate(SLOTS)}


@pytest.fixture(scope="module")
def corpora(keys):
    """per slot: adversarial spend corpus (valid proofs, failed checks, identity A', bad points, replays) under that slot's key"""
    out = {}
    for s, ctx in keys.items():
        base = corpus.gen_valid(ctx, 24, seed=b"key-slots-%d" % s, threads=16)
        proofs, rnd, _, _ = corpus.mutate_proofs(ctx, base)
        out[s] = dict(base=base, proofs=proofs.reshape(-1, PB), rnd=rnd.reshape(-1, 128))
    return out


def _key(act, ctx):
    return act.PrivateKey(ctx.x, ctx.w)


def _engine(act, keys, slots=SLOTS, **kw):
    eng = act.Engine(act.Params(keys[0].h), _key(act, keys[0]), **kw)
    for s in slots:
        if s != 0:
            eng.set_key(s, _key(act, keys[s]))
    return eng


def _mixed(corpora, extra_ids=True):
    """a batch over the three keys with the right ids, plus wrong-slot, empty-slot and out-of-range ids"""
    pf, rnd, ids = [], [], []
    for s in SLOTS:
        c = corpora[s]
        for i in range(len(c["proofs"])):
            pf.append(c["proofs"][i]); rnd.append(c["rnd"][i]); ids.append(s)
        if extra_ids:
            for i, wrong in ((0, SLOTS[(SLOTS.index(s) + 1) % 3]), (12, 5), (0, 16), (12, 255), (24 % len(c["proofs"]), 1)):
                pf.append(c["proofs"][i]); rnd.append(c["rnd"][i]); ids.append(wrong)
    order = np.random.RandomState(5).permutation(len(ids))
    return (np.stack(pf)[order].reshape(-1), np.stack(rnd)[order].reshape(-1), np.array(ids, np.uint8)[order])


def _com(proofs):
    return proofs.reshape(-1, PB)[:, 4 * 32:132 * 32].reshape(-1)


# ---- slot management ------------------------------------------------------------------------------------------------------------
def test_slot_management(act, keys, corpora):
    with _engine(act, keys, slots=(0,)) as eng:
        assert eng.key_slots == [0] and eng.selected_key == 0
        bad = act.PrivateKey(keys[3].x, keys[7].w)
        with pytest.raises(act.ActError, match="not the public key"):
            eng.set_key(3, bad)
        assert eng.key_slots == [0]
        eng.set_key(3, _key(act, keys[7]))
        with pytest.raises(act.ActError):
            eng.set_key(3, bad)               # a failed replacement leaves the key that was there
        with pytest.raises(act.ActError):
            eng.set_key(16, _key(act, keys[3]))
        with pytest.raises(act.ActError, match="holds no key"):
            eng.select_key(5)
        with pytest.raises(act.ActError, match="selected"):
            eng.clear_key(0)
        assert eng.key_slots == [0, 3]
        c7 = corpora[7]
        n = len(c7["proofs"])
        ids = np.full(n, 3, np.uint8)
        o_ref, o_nul, o_st = OK.batch_refund_keyed({3: keys[7]}, keys[0], c7["proofs"], ids, c7["rnd"])
        ref, nul, st = eng.batch_verify_spend_and_refund_keyed(c7["proofs"], ids, c7["rnd"])
        assert (st == o_st).all() and (ref == o_ref).all() and (nul == o_nul).all()
        assert (st == 0).sum() >= 5
        # replacing the key: slot 3 now holds key 3, so the proofs of key 7 named by slot 3 fail, and key 3's pass
        eng.set_key(3, _key(act, keys[3]))
        _, _, st2 = eng.batch_verify_spend_and_refund_keyed(c7["proofs"], ids, c7["rnd"])
        assert ((st2 == 7) | (st == st2)).all() and (st2[st == 0] == 7).all()
        c3 = corpora[3]
        o_ref, o_nul, o_st = OK.batch_refund_keyed({3: keys[3]}, keys[0], c3["proofs"], ids, c3["rnd"])
        ref, nul, st = eng.batch_verify_spend_and_refund_keyed(c3["proofs"], ids, c3["rnd"])
        assert (st == o_st).all() and (ref == o_ref).all() and (nul == o_nul).all()
        # a cleared slot rejects its proofs with 7, like an empty one
        eng.clear_key(3)
        assert eng.key_slots == [0]
        o_ref, o_nul, o_st = OK.batch_refund_keyed({}, keys[0], c3["proofs"], ids, c3["rnd"])
        ref, nul, st = eng.batch_verify_spend_and_refund_keyed(c3["proofs"], ids, c3["rnd"])
        assert (st == o_st).all() and (ref == o_ref).all() and (nul == o_nul).all()
        assert set(st.tolist()) <= {6, 7, 0x81} and (st == 7).sum() >= 12
        with pytest.raises(act.ActError, match="holds no key"):
            eng.clear_key(3)


# ---- unchanged default --------------------------------------------------------------------------------------------------------------
def test_unkeyed_calls_ignore_extra_slots(act, keys, corpora):
    """keys in slots 3 and 7 with slot 0 selected: every unkeyed call returns the bytes of an engine without them"""
    c = corpora[0]
    base = c["base"]
    pf, rnd = c["proofs"].reshape(-1), c["rnd"].reshape(-1)
    with _engine(act, keys, slots=(0,)) as plain, _engine(act, keys) as slotted:
        for eng in (plain, slotted):
            eng.set_spend_chunk(16)
        outs = []
        for eng in (plain, slotted):
            ref, nul, st = eng.batch_verify_spend_and_refund(pf, rnd)
            resp, ist = eng.batch_issue(base["req"], base["cs"], base["rnd"])
            chk = eng.batch_issuance_check(base["req"].reshape(-1, 128)[:, :32].reshape(-1), resp)
            rchk = eng.batch_refund_check(_com(pf), ref)
            nul2, st2, kp = eng.batch_spend_verify(pf)
            sref, snul, sst = eng.batch_verify_spend_and_refund_screened(pf, rnd)
            outs.append([ref, nul, st, resp, ist, chk, rchk, nul2, st2, kp, sref, snul, sst])
        for a, b in zip(*outs):
            assert (a == b).all()
        o_ref, o_nul, o_st, _ = keys[0].batch_refund(pf, rnd, threads=16)
        assert (outs[1][2] == o_st).all() and (outs[1][0] == o_ref).all()


# ---- mixed batch ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("selected", [0, 3])
def test_mixed_batch_matches_the_cross_key_oracle(act, keys, corpora, selected):
    pf, rnd, ids = _mixed(corpora)
    with _engine(act, keys) as eng:
        eng.select_key(selected)
        assert eng.selected_key == selected
        eng.set_spend_chunk(32)
        ref, nul, st = eng.batch_verify_spend_and_refund_keyed(pf, ids, rnd)
        o_ref, o_nul, o_st = OK.batch_refund_keyed(keys, keys[selected], pf, ids, rnd)
        assert (st == o_st).all(), np.flatnonzero(st != o_st)
        assert (ref == o_ref).all() and (nul == o_nul).all()
        assert {0, 6, 7, 0x81} <= set(st.tolist())
        ok = st == 0
        com = _com(pf).reshape(-1, 4096)[ok].reshape(-1)
        refs = ref.reshape(-1, 128)[ok].reshape(-1)
        assert (eng.batch_refund_check(com, refs) == 0).all()                     # the engine checks under the selected W
        o_chk, _ = keys[selected].batch_refund_check(com, refs, threads=16)
        assert (o_chk == 0).all()
        other = keys[SLOTS[(SLOTS.index(selected) + 1) % 3]]
        o_bad, _ = other.batch_refund_check(com, refs, threads=16)
        assert (o_bad == 4).all()                                                 # and under no other key
        # two-pass form: keyed verification, then act_batch_refund_sign under the selected key
        nul2, st2, kp = eng.batch_spend_verify_keyed(pf, ids)
        acc = np.flatnonzero(st2 == 0)
        ref2 = eng.batch_refund_sign(kp, st2, rnd.reshape(-1, 128)[acc].reshape(-1).copy())
        assert (st2 == st).all() and (nul2 == nul).all() and (ref2 == ref).all()


def test_issuance_under_a_selected_slot(act, keys, corpora):
    base = corpora[3]["base"]
    with _engine(act, keys) as eng:
        eng.select_key(3)
        resp, st = eng.batch_issue(base["req"], base["cs"], base["rnd"])
        o_resp, o_st, _ = keys[3].batch_issue(base["req"], base["cs"], base["rnd"])
        assert (st == 0).all() and (st == o_st).all() and (resp == o_resp).all()
        K = base["req"].reshape(-1, 128)[:, :32].reshape(-1).copy()
        o_chk, _ = keys[3].batch_issuance_check(K, resp, threads=16)
        assert (o_chk == 0).all() and (eng.batch_issuance_check(K, resp) == 0).all()


# ---- same-key equivalence -------------------------------------------------------------------------------------------------------------
def test_keyed_with_the_selected_slot_equals_the_unkeyed_call(act, keys, corpora):
    """every id = the selected slot: the unkeyed call's bytes, over a batch that spans the ramp and both streams; the _dev form
    equals the host form"""
    import torch
    c = corpora[3]
    reps = 220                                       # 5280 proofs: chunk 4096 -> ramp 512, 2048, then 2720
    pf = np.tile(c["proofs"], (reps, 1)).reshape(-1)
    rnd = np.tile(c["rnd"], (reps, 1)).reshape(-1)
    n = len(pf) // PB
    ids = np.full(n, 3, np.uint8)
    with _engine(act, keys) as eng:
        eng.select_key(3)
        eng.set_spend_chunk(4096)
        ref, nul, st = eng.batch_verify_spend_and_refund(pf, rnd)
        kref, knul, kst = eng.batch_verify_spend_and_refund_keyed(pf, ids, rnd)
        assert (kst == st).all() and (kref == ref).all() and (knul == nul).all()
        assert (st == 0).sum() >= n // 5
        eng.set_spend_chunk(1000)                    # _dev: chunks alternate over the two streams
        t_pf, t_rnd = torch.from_numpy(pf).cuda(), torch.from_numpy(rnd).cuda()
        t_ids = torch.from_numpy(np.concatenate([np.zeros(1, np.uint8), ids])).cuda()[1:]   # key ids need no alignment
        t_ref = torch.zeros(n * 128, dtype=torch.uint8, device="cuda"); t_nul = torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
        t_st = torch.zeros(n, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        eng.batch_verify_spend_and_refund_keyed_dev(n, t_pf.data_ptr(), t_ids.data_ptr(), t_rnd.data_ptr(), t_ref.data_ptr(), t_nul.data_ptr(),
                                                    t_st.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert (t_st.cpu().numpy() == st).all() and (t_ref.cpu().numpy() == ref).all() and (t_nul.cpu().numpy() == nul).all()


# ---- stores ------------------------------------------------------------------------------------------------------------------------------
def _db_loop(st, nul, ref, ids, dbs, store_of):
    """NullifierDb per store in slice order over accepted proofs; store_of: slot -> db name"""
    st = st.copy(); ref = ref.reshape(len(st), -1).copy()
    for i in range(len(st)):
        if st[i] == 0:
            db = dbs[store_of[int(ids[i])]]
            k = bytes(nul[32 * i:32 * i + 32])
            if k in db:
                st[i] = 3; ref[i] = 0
            else:
                db.add(k)
    return st, ref.reshape(-1)


def _members(store):
    return {bytes(r) for r in store.export().reshape(-1, 32)}


def test_stores_per_key_match_a_nullifier_db_per_store(act, keys, corpora):
    """slots 0 and 3 share a store, slot 7 has its own: replays within a store are flagged in slice order (also across the two
    slots that share it), over several batches"""
    pf, rnd, ids = _mixed(corpora)
    n = len(ids)
    with _engine(act, keys) as eng, act.NullifierStore(0, 64) as a, act.NullifierStore(0, 64) as b:
        eng.set_spend_chunk(40)
        store_of = {0: "a", 3: "a", 7: "b"}
        dbs = {"a": set(), "b": set()}
        stores = {0: a, 3: a, 7: b}
        order = np.random.RandomState(9)
        for batch in range(4):
            sel = order.permutation(n)[: n // 2] if batch < 3 else np.arange(n)   # the last batch replays everything
            p = pf.reshape(n, PB)[sel].reshape(-1); r = rnd.reshape(n, 128)[sel].reshape(-1); k = ids[sel].copy()
            if batch == 1:   # the same proof under slot 0 at two indices: a replay inside the batch
                p = np.concatenate([p, p[:PB]]); r = np.concatenate([r, r[:128]]); k = np.concatenate([k, k[:1]])
            ref0, nul0, st0 = eng.batch_verify_spend_and_refund_keyed(p, k, r)
            exp_st, exp_ref = _db_loop(st0, nul0, ref0, k, dbs, store_of)
            ref, nul, st = eng.batch_verify_spend_and_refund_keyed(p, k, r, stores=stores)
            assert (st == exp_st).all() and (ref == exp_ref).all() and (nul == nul0).all()
            assert _members(a) == dbs["a"] and _members(b) == dbs["b"]
        assert (st == 3).sum() > 0 and a.size > 0 and b.size > 0


def test_the_same_nullifier_under_two_keys_is_two_credentials(act, keys):
    """one r|k issued under key 0 and under key 3: two proofs with one nullifier; with a store per key neither is a replay"""
    rs = np.random.RandomState(3)
    pre = O.sc_reduce32(rs.bytes(32)) + O.sc_reduce32(rs.bytes(32))       # r | k
    c = (1000).to_bytes(32, "little"); s = (10).to_bytes(32, "little")
    proofs = []
    for slot in (0, 3):
        ctx = keys[slot]
        req = ctx.request(pre, rs.bytes(128))
        st, resp = ctx.issue(req, c, rs.bytes(128))
        assert st == 0
        token = resp[:64] + pre[32:64] + pre[:32] + c
        proof, _ = ctx.prove_spend(token, s, rs.bytes(O.RND_PROVE))
        proofs.append(proof)
    pf = np.frombuffer(b"".join(proofs), np.uint8).copy()
    rnd = np.frombuffer(rs.bytes(256), np.uint8).copy()
    ids = np.array([0, 3], np.uint8)
    with _engine(act, keys) as eng, act.NullifierStore(0, 64) as a, act.NullifierStore(0, 64) as b, act.NullifierStore(0, 64) as w:
        ref, nul, st = eng.batch_verify_spend_and_refund_keyed(pf, ids, rnd, stores={0: a, 3: b, 7: w})
        assert (st == 0).all() and nul[:32].tobytes() == nul[32:].tobytes()
        assert a.size == 1 and b.size == 1 and w.size == 0
        # the same two proofs with one store for both keys: the second is a replay
        with act.NullifierStore(0, 64) as one:
            _, _, st = eng.batch_verify_spend_and_refund_keyed(pf, ids, rnd, stores=[one] * 16)
            assert st.tolist() == [0, 3]


def test_a_slot_without_a_store_fails_the_call_and_changes_no_store(act, keys, corpora):
    pf, rnd, ids = _mixed(corpora)
    with _engine(act, keys) as eng, act.NullifierStore(0, 64) as a, act.NullifierStore(0, 64) as b:
        eng.batch_verify_spend_and_refund_keyed(pf, ids, rnd, stores={0: a, 3: a, 7: b})
        before = (_members(a), _members(b))
        assert before[0] and before[1]
        with pytest.raises(act.ActError, match="slot 7 holds a key but has no store"):
            eng.batch_verify_spend_and_refund_keyed(pf, ids, rnd, stores={0: a, 3: b})
        assert (_members(a), _members(b)) == before
        # a store for an empty slot is not needed, and slots without a key need none
        eng.clear_key(7)
        _, _, st = eng.batch_verify_spend_and_refund_keyed(pf, ids, rnd, stores={0: a, 3: b})
        assert set(st[ids == 7].tolist()) <= {6, 7, 0x81} and (st[ids == 7] == 7).sum() > len(st[ids == 7]) // 2
        assert _members(a) == before[0]


def test_a_failed_store_screen_leaves_the_store_unchanged(act):
    """the prepare/commit split of the screen: a non-reduced key fails the call before anything is inserted"""
    rs = np.random.RandomState(1)
    keys = rs.randint(0, 256, size=(64, 32)).astype(np.uint8); keys[:, 31] &= 0x0F
    with act.NullifierStore(0, 16) as s:
        s.screen(np.zeros(32, np.uint8), keys[:32].reshape(-1), record=True)
        before = _members(s)
        bad = keys[32:].copy(); bad[7, 31] = 0xFF
        with pytest.raises(act.ActError, match="not reduced"):
            s.screen(np.zeros(32, np.uint8), bad.reshape(-1), record=True)
        assert _members(s) == before and s.size == 32


# ---- multi-device handle -------------------------------------------------------------------------------------------------------------------
def test_multi_device_handle_equals_the_single_device_engine(act, keys, corpora):
    devs = [0, 1] if act.device_count() >= 2 else [0, 0]
    pf, rnd, ids = _mixed(corpora)
    with _engine(act, keys) as one, _engine(act, keys, devices=devs) as multi:
        for eng in (one, multi):
            eng.select_key(7)
            assert eng.selected_key == 7 and eng.key_slots == list(SLOTS)
        r1 = one.batch_verify_spend_and_refund_keyed(pf, ids, rnd)
        r2 = multi.batch_verify_spend_and_refund_keyed(pf, ids, rnd)
        for a, b in zip(r1, r2):
            assert (a == b).all()
        v1, v2 = one.batch_spend_verify_keyed(pf, ids), multi.batch_spend_verify_keyed(pf, ids)
        for a, b in zip(v1, v2):
            assert (a == b).all()
        with act.NullifierStore(0, 64) as a1, act.NullifierStore(0, 64) as b1, act.NullifierStore(devs[0], 64) as a2, act.NullifierStore(devs[0], 64) as b2:
            s1 = one.batch_verify_spend_and_refund_keyed(pf, ids, rnd, stores={0: a1, 3: b1, 7: b1})
            s2 = multi.batch_verify_spend_and_refund_keyed(pf, ids, rnd, stores={0: a2, 3: b2, 7: b2})
            for a, b in zip(s1, s2):
                assert (a == b).all()
            assert _members(a1) == _members(a2) and _members(b1) == _members(b2)
        multi.clear_key(3)
        assert multi.key_slots == [0, 7]


# ---- C++ host layer -----------------------------------------------------------------------------------------------------------------------
def test_cpp_keyed_overload_equals_a_loop_of_oracle_calls_over_one_rng(act, keys, corpora, tmp_path):
    subprocess.check_call(["make", "-C", CPP, "-f", "keys_hpp_check.mk", "-s"])
    pf, _, ids = _mixed(corpora, extra_ids=False)
    n = len(ids)
    stream = np.frombuffer(corpus.xof(b"keys-cpp-rng", 128 * 2 * n), np.uint8)
    selected = 3
    fx = bytearray(keys[0].h)
    fx += struct.pack("<I", 3)
    for s in SLOTS:
        fx += struct.pack("<I", s) + keys[s].x + keys[s].w
    fx += struct.pack("<I", selected) + struct.pack("<I", n) + pf.tobytes() + ids.tobytes()
    fx += struct.pack("<I", len(stream)) + stream.tobytes()
    (tmp_path / "fx.bin").write_bytes(bytes(fx))
    subprocess.check_call([os.path.join(CPP, "keys_hpp_check"), str(tmp_path / "fx.bin"), str(tmp_path / "out.bin")])
    out = (tmp_path / "out.bin").read_bytes()
    # the loop: per proof, verify under its key, check the store of its slot (0 and 3 share one), draw 128 bytes, refund, record
    dbs = {0: set(), 3: None, 7: set()}
    dbs[3] = dbs[0]
    pos, o = 0, 0
    pfa = pf.reshape(n, PB)
    for _ in range(2):
        exp_st, exp_nul, exp_ref = [], [], []
        for i in range(n):
            st, _, nul = OK.refund_keyed(keys[int(ids[i])], keys[selected], pfa[i].tobytes(), bytes(128))
            ref = bytes(128)
            if st == 0:
                if nul in dbs[int(ids[i])]:
                    st = 3
                else:
                    st, ref, nul = OK.refund_keyed(keys[int(ids[i])], keys[selected], pfa[i].tobytes(), stream[pos:pos + 128].tobytes())
                    pos += 128
                    dbs[int(ids[i])].add(nul)
            exp_st.append(st); exp_nul.append(nul); exp_ref.append(ref)
        assert list(out[o:o + n]) == exp_st; o += n
        assert out[o:o + 32 * n] == b"".join(exp_nul); o += 32 * n
        assert out[o:o + 128 * n] == b"".join(exp_ref); o += 128 * n
        assert struct.unpack_from("<I", out, o)[0] == pos; o += 4
    assert struct.unpack_from("<2I", out, o) == (len(dbs[0]), len(dbs[7]))
