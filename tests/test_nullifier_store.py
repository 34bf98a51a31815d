"""Device-resident nullifier store (act_nullifier_store_*, act_batch_verify_spend_and_refund_recorded).

Oracle: the store must behave exactly like act_flag_replays(..., seen = store contents) followed by
store |= {nullifier[i] : out[i] == 0}, i.e. the reference's NullifierDb (src/tests.rs:28-50) applied in slice order and kept
between batches -- checked here against a Python set, the CPU oracle's refund() and the existing screened call."""
import importlib
import os
import struct
import subprocess

import numpy as np
import pytest

import corpus

HERE = os.path.dirname(os.path.abspath(__file__))
CPP = os.path.join(HERE, "cpp")
EXE = os.path.join(CPP, "store_hpp_check")
PB = corpus.PROOF_BYTES
ELL = corpus.ELL


def _multi_devices(act):
    return [0, 1] if act.device_count() >= 2 else [0, 0]


def _keyset(a):
    return {bytes(r) for r in np.asarray(a, np.uint8).reshape(-1, 32)}


def _random_reduced(rs, n):
    k = rs.randint(0, 256, size=(n, 32)).astype(np.uint8)
    k[:, 31] &= 0x0f                                    # < 2^252 < l
    return k


def _db_loop(st, nul, ref, db):
    """NullifierDb in slice order over ACCEPTED proofs: a nullifier already in db (or earlier in the slice) -> 3, no refund."""
    st = st.copy(); ref = ref.reshape(len(st), -1).copy()
    for i in range(len(st)):
        if st[i] == 0:
            k = bytes(nul[32 * i:32 * i + 32])
            if k in db:
                st[i] = 3; ref[i] = 0
            else:
                db.add(k)
    return st, ref.reshape(-1)


# ---- CPU: the new entry points exist, build, and refuse to run without a device ----------------------------------------------
def test_store_entry_points_fail_without_a_device(act):
    if act.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(act.ActError):
        act.NullifierStore(device=0, capacity=1024)
    lib = act.load_library()
    one = np.zeros(32, np.uint8)
    assert lib.act_nullifier_store_screen(None, 1, one.ctypes.data, one.ctypes.data, one.ctypes.data, 1) != 0
    assert lib.act_nullifier_store_screen_dev(None, 1, one.ctypes.data, one.ctypes.data, one.ctypes.data, 1, None) != 0
    assert lib.act_batch_verify_spend_and_refund_recorded(None, None, 1, one.ctypes.data, one.ctypes.data, one.ctypes.data,
                                                          one.ctypes.data, one.ctypes.data) != 0
    cnt = __import__("ctypes").c_size_t(0)
    assert lib.act_nullifier_store_export(None, one.ctypes.data, 1, __import__("ctypes").byref(cnt)) != 0
    assert lib.act_nullifier_store_size(None) == 0 and lib.act_nullifier_store_device(None) == -1
    import torch
    sh = importlib.import_module("anonymous-credit-tokens_b200.sharding")
    with pytest.raises(RuntimeError):
        sh.screen_with_store(torch.zeros(4, dtype=torch.uint8), torch.zeros(128, dtype=torch.uint8), None)


def test_store_cpp_check_compiles_links_and_needs_a_device(act, tmp_path):
    assert os.path.exists(act.LIB_PATH)
    subprocess.check_call(["make", "-C", CPP, "-f", "store_hpp_check.mk", "-s"])
    r = subprocess.run([EXE], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr
    if act.device_count() == 0:
        fix = tmp_path / "f.bin"
        fix.write_bytes(bytes(160) + struct.pack("<I", 0) + struct.pack("<I", 0) + struct.pack("<I", 0))
        r = subprocess.run([EXE, str(fix), str(tmp_path / "o.bin")], capture_output=True, text=True)
        assert r.returncode == 1 and "FAILED" in r.stderr


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pool(act, octx, engine):
    """Accepted, rejected and replayed proofs, plus a second honest proof of every base token ("same token, different proof"):
    (proofs, rnd, oracle refunds, oracle nullifiers, oracle statuses)."""
    n = 48
    base = corpus.gen_valid(octx, n, seed=b"nullifier-store", threads=8)
    proofs, rnd, _, _ = corpus.mutate_proofs(octx, base)
    tokens = corpus.tokens_from(base, corpus.trip_streams(b"nullifier-store", n)["pre"])
    ones = np.frombuffer(b"".join((1).to_bytes(32, "little") for _ in range(n)), np.uint8)
    p2, _, s2 = engine.batch_prove_spend(tokens, ones, seed=corpus.xof(b"nullifier-store/second", 32))
    assert (s2 == 0).all()
    P = np.concatenate([proofs, p2]); R = np.concatenate([rnd, np.frombuffer(corpus.xof(b"nullifier-store/rnd2", 128 * n), np.uint8)])
    o_ref, o_nul, o_st, _ = octx.batch_refund(P, R, threads=8)
    u = len(o_st)
    untouched = np.arange(0, n, 12)                     # mutate_proofs leaves every 12th proof as it was
    assert (o_st[n:] == 0).all() and (o_nul.reshape(u, 32)[n + untouched] == o_nul.reshape(u, 32)[untouched]).all()
    return P, R, o_ref, o_nul, o_st


def _batch(pool, idx):
    P, R, o_ref, o_nul, o_st = pool
    u = len(o_st)
    return (P.reshape(u, -1)[idx].reshape(-1).copy(), R.reshape(u, -1)[idx].reshape(-1).copy(),
            o_ref.reshape(u, -1)[idx].reshape(-1).copy(), o_nul.reshape(u, -1)[idx].reshape(-1).copy(), o_st[idx].copy())


@pytest.mark.gpu
def test_recorded_equals_screened_with_seen(act, engine, pool):
    P, R, o_ref, o_nul, o_st = pool
    u = len(o_st)
    n = 3000
    idx = (np.arange(n) * 13 + 2) % u
    Pb, Rb, _, _, _ = _batch(pool, idx)
    acc = np.flatnonzero(o_st == 0)
    spent = np.unique(o_nul.reshape(u, 32)[acc], axis=0)[:4]          # mutate_proofs plants exact replays among the accepted
    S = np.concatenate([spent, _random_reduced(np.random.RandomState(1), 5000)])
    with act.NullifierStore(device=0, capacity=64) as store:
        assert (store.screen(np.zeros(len(S), np.uint8), S) == 0).all() and store.size == len(S)
        a = engine.batch_verify_spend_and_refund_recorded(Pb, Rb, store)
        b = engine.batch_verify_spend_and_refund_screened(Pb, Rb, seen=S.reshape(-1))
        for x, y in zip(a, b):
            assert x.tobytes() == y.tobytes()
        st, nul = a[2], a[1]
        assert (st == 3).sum() > n // 5 and (st == 0).sum() > 10
        want = _keyset(S) | {bytes(nul[32 * i:32 * i + 32]) for i in range(n) if st[i] == 0}
        got = store.export()
        assert len(got) == 32 * len(want) and _keyset(got) == want and store.size == len(want)


def _five_batches(pool):
    u = len(pool[4])
    rs = np.random.RandomState(5)
    return [rs.randint(0, u, size=m) for m in (400, 700, 64, 1000, 333)]   # heavy repetition inside and across batches


@pytest.mark.gpu
def test_several_batches_against_a_python_set(act, engine, pool):
    db = set()
    with act.NullifierStore(device=0, capacity=16) as store:
        for idx in _five_batches(pool):
            Pb, Rb, e_ref, e_nul, e_st = _batch(pool, idx)
            e_st, e_ref = _db_loop(e_st, e_nul, e_ref, db)
            ref, nul, st = engine.batch_verify_spend_and_refund_recorded(Pb, Rb, store)
            assert (st == e_st).all() and (ref == e_ref).all() and (nul == e_nul).all()
            assert store.size == len(db)
        assert _keyset(store.export()) == db
        # the second proof of a token spent in an earlier batch is a replay too
        n = len(pool[4]) // 2
        Pb, Rb, _, _, _ = _batch(pool, np.arange(n, 2 * n))
        _, _, st = engine.batch_verify_spend_and_refund_recorded(Pb, Rb, store)
        assert (st == 3).all()


@pytest.mark.gpu
def test_multi_device_handle(act, engine, octx, pool):
    params, key = act.Params(octx.h), act.PrivateKey(octx.x, octx.w)
    devs = _multi_devices(act)
    with act.Engine(params, key, devices=devs) as m, act.NullifierStore(device=0) as s1, act.NullifierStore(device=devs[0]) as sm:
        m.set_spend_chunk(256)
        for idx in _five_batches(pool):
            Pb, Rb, _, _, _ = _batch(pool, idx)
            a = engine.batch_verify_spend_and_refund_recorded(Pb, Rb, s1)
            b = m.batch_verify_spend_and_refund_recorded(Pb, Rb, sm)
            assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
        assert _keyset(s1.export()) == _keyset(sm.export())
        if act.device_count() >= 2:
            with act.NullifierStore(device=1) as other:
                with pytest.raises(act.ActError, match="replica 0"):
                    m.batch_verify_spend_and_refund_recorded(Pb, Rb, other)
                assert other.size == 0


@pytest.mark.gpu
def test_growth_and_edge_keys(act):
    rs = np.random.RandomState(7)
    N = 2_000_000
    keys = _random_reduced(rs, N)
    keys[0] = 0                                                         # the all-zero nullifier
    keys[1] = np.frombuffer((ELL - 1).to_bytes(32, "little"), np.uint8)   # the largest reduced one
    keys[2] = np.frombuffer(((1 << 64) - 1).to_bytes(32, "little"), np.uint8)  # first word all ones
    with act.NullifierStore(device=0, capacity=1024) as store:
        lo = 0
        for m in (1000, 5000, 60000, 250_000, 700_000, N):              # crosses many doublings, one of them by a lot
            hi = min(m, N)
            out = store.screen(np.zeros(hi - lo, np.uint8), keys[lo:hi])
            assert (out == 0).all()
            lo = hi
        assert store.size == N
        for a in range(0, N, 500_000):                                  # every member present, nothing recorded by a query
            assert (store.screen(np.zeros(min(500_000, N - a), np.uint8), keys[a:a + 500_000], record=False) == 3).all()
        fresh = _random_reduced(rs, 1_000_000)
        assert (store.screen(np.zeros(len(fresh), np.uint8), fresh, record=False) == 0).all()
        assert store.size == N
        exp = store.export().reshape(-1, 32)
        assert len(exp) == N
        srt = lambda a: np.sort(np.ascontiguousarray(a).view("V32").reshape(-1))
        assert (srt(exp) == srt(keys)).all()
        # newly-inserted flags with in-batch duplicates, stored keys and rejected entries
        f = fresh[:3]
        batch = np.stack([f[0], keys[0], f[0], f[1], keys[1], f[1], f[2], keys[2]])
        st = np.array([0, 0, 0, 0, 0, 0, 7, 0], np.uint8)
        assert store.screen(st, batch).tolist() == [0, 3, 3, 0, 3, 3, 7, 3]
        assert store.size == N + 2
        assert store.screen(np.zeros(1, np.uint8), f[2:3], record=False).tolist() == [0]   # status 7 was not recorded


@pytest.mark.gpu
def test_device_form_and_sharding(act):
    import torch
    sh = importlib.import_module("anonymous-credit-tokens_b200.sharding")
    rs = np.random.RandomState(9)
    n = 50_000
    nul = _random_reduced(rs, n)
    nul[rs.randint(0, n, n // 4)] = nul[rs.randint(0, n, n // 4)]
    st = (rs.rand(n) < 0.2).astype(np.uint8) * 7
    prefill = nul[rs.randint(0, n, 2000)]
    stores = [act.NullifierStore(device=0, capacity=1000) for _ in range(3)]
    try:
        for s in stores:
            s.screen(np.zeros(len(prefill), np.uint8), prefill)
        want = stores[0].screen(st, nul)
        t_st, t_nul = torch.from_numpy(st).cuda(), torch.from_numpy(nul.reshape(-1)).cuda()
        S = torch.cuda.Stream()
        S.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(S):
            out = torch.empty_like(t_st)
            q = torch.empty_like(t_st)
            stores[1].screen_dev(n, t_st.data_ptr(), t_nul.data_ptr(), q.data_ptr(), record=False, stream=S.cuda_stream)
            size0 = stores[1].size
            stores[1].screen_dev(n, t_st.data_ptr(), t_nul.data_ptr(), out.data_ptr(), record=True, stream=S.cuda_stream)
            via_sh = sh.screen_with_store(t_st, t_nul, stores[2])          # torch's current stream: S
        S.synchronize()
        assert (out.cpu().numpy() == want).all() and (q.cpu().numpy() == want).all() and (via_sh.cpu().numpy() == want).all()
        assert size0 == len(_keyset(prefill))
        assert stores[0].size == stores[1].size == stores[2].size
        # legacy default stream: the side-stream path of screen_with_store
        again = sh.screen_with_store(t_st, t_nul, stores[2], record=False)
        assert (again.cpu().numpy() == np.where(st == 0, 3, st)).all() and stores[2].size == stores[0].size
    finally:
        for s in stores:
            s.close()


def _one_rng_expected(octx, proofs, stream, seen, passes):
    """A loop of oracle refund() calls over ONE stream behind a Python set: randomness is drawn only for survivors."""
    db = _keyset(seen) if len(seen) else set()
    pos = 0
    res = []
    n = len(proofs) // PB
    for _ in range(passes):
        sts, nuls, refs = [], [], []
        for i in range(n):
            st, ref, nul = octx.refund(proofs[i * PB:(i + 1) * PB].tobytes(), stream[pos:pos + 128].tobytes())
            if st == 0 and nul in db:
                st, ref = 3, bytes(128)
            elif st == 0:
                db.add(nul); pos += 128
            else:
                nul = bytes(32)
            sts.append(st); nuls.append(nul); refs.append(ref)
        res.append((sts, b"".join(nuls), b"".join(refs), pos))
    return res, db


@pytest.mark.gpu
@pytest.mark.parametrize("multi", [False, True])
def test_one_rng_cpp_overload(act, octx, pool, tmp_path, multi):
    subprocess.check_call(["make", "-C", CPP, "-f", "store_hpp_check.mk", "-s"])
    P, R, o_ref, o_nul, o_st = pool
    u = len(o_st)
    idx = (np.arange(150) * 7 + 3) % u
    proofs = P.reshape(u, -1)[idx].reshape(-1).copy()
    seen = np.unique(o_nul.reshape(u, 32)[np.flatnonzero(o_st == 0)], axis=0)[:2].copy()
    stream = corpus.xof(b"store/one-rng", 128 * 2 * len(idx))
    fix = tmp_path / "fixture.bin"; out = tmp_path / "out.bin"
    with open(fix, "wb") as f:
        f.write(octx.h + octx.x + octx.w)
        f.write(struct.pack("<I", len(idx)) + proofs.tobytes())
        f.write(struct.pack("<I", len(seen)) + seen.tobytes())
        f.write(struct.pack("<I", len(stream)) + stream)
    cmd = [EXE, str(fix), str(out)] + ([",".join(map(str, _multi_devices(act)))] if multi else [])
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr + r.stdout
    b = open(out, "rb").read()
    n = len(idx)
    exp, db = _one_rng_expected(octx, proofs, np.frombuffer(stream, np.uint8), seen, 2)
    o = 0
    for sts, nuls, refs, pos in exp:
        assert list(b[o:o + n]) == sts; o += n
        assert b[o:o + 32 * n] == nuls; o += 32 * n
        assert b[o:o + 128 * n] == refs; o += 128 * n
        assert struct.unpack("<I", b[o:o + 4])[0] == pos; o += 4
    size, cnt = struct.unpack("<II", b[o:o + 8]); o += 8
    assert size == cnt == len(db) and _keyset(np.frombuffer(b[o:], np.uint8)) == db
    assert 0 not in exp[1][0] and 3 in exp[0][0] and 0 in exp[0][0] and exp[1][3] == exp[0][3]


@pytest.mark.gpu
def test_one_rng_python_composition(act, engine, octx, pool):
    P, R, o_ref, o_nul, o_st = pool
    u = len(o_st)
    idx = (np.arange(150) * 7 + 3) % u
    proofs = P.reshape(u, -1)[idx].reshape(-1).copy()
    seen = np.unique(o_nul.reshape(u, 32)[np.flatnonzero(o_st == 0)], axis=0)[:2].copy()
    stream = np.frombuffer(corpus.xof(b"store/one-rng-py", 128 * len(idx)), np.uint8)
    (exp,), db = _one_rng_expected(octx, proofs, stream, seen, 1)
    with act.NullifierStore(device=0) as store:
        store.screen(np.zeros(len(seen), np.uint8), seen)
        nul, st, kp = engine.batch_spend_verify(proofs)
        st = store.screen(st, nul)
        used = 128 * int((st == 0).sum())
        ref = engine.batch_refund_sign(kp, st, stream[:used])
        assert st.tolist() == exp[0] and nul.tobytes() == exp[1] and ref.tobytes() == exp[2] and used == exp[3]
        assert _keyset(store.export()) == db


@pytest.mark.gpu
def test_failed_recording_calls_leave_the_store_unchanged(act, engine):
    import torch
    rs = np.random.RandomState(11)
    keys = _random_reduced(rs, 3000)
    with act.NullifierStore(device=0, capacity=1024) as store:
        store.screen(np.zeros(1000, np.uint8), keys[:1000])
        before = _keyset(store.export())
        buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
        p = buf.data_ptr()
        n = 2000                                      # would also force growth (1000 + 2000 > 512 slots' worth)
        with pytest.raises(act.ActError, match="null buffer"):
            store.screen_dev(n, p, None, p + 4096)
        with pytest.raises(act.ActError, match="16-byte aligned"):
            store.screen_dev(n, p, p + 65536 + 8, p + 4096)
        host = np.zeros(n * 32, np.uint8)
        with pytest.raises(act.ActError, match="device memory"):
            store.screen_dev(n, p, host.ctypes.data, p + 4096)
        for bad in (ELL, (1 << 256) - 1, ELL + 5):
            ks = keys[1000:3000].copy()
            ks[1234] = np.frombuffer(bad.to_bytes(32, "little"), np.uint8)
            with pytest.raises(act.ActError, match="not reduced"):
                store.screen(np.zeros(n, np.uint8), ks)
            assert store.size == 1000 and _keyset(store.export()) == before
        # a non-reduced key that takes no part (status != 0) is not looked at
        ks[1234] = 0xff
        st = np.zeros(n, np.uint8); st[1234] = 7
        out = store.screen(st, ks)
        assert out[1234] == 7 and store.size == 1000 + n - 1
