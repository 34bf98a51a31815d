"""Issuer key slot measurements (act_batch_verify_spend_and_refund_keyed).  Prints JSON lines.

The issuer's verify + refund step at 1M valid proofs per call from pinned host memory on one GPU, host clock around the
synchronous call, legs alternated between repetitions:
  unkeyed:        act_batch_verify_spend_and_refund, proofs under the key of slot 0
  keyed_one_slot: the keyed call over the same proofs, every key id 0
  keyed_mixed:    the keyed call over proofs issued under four keys (slots 0..3, key id i % 4), selected slot 0
  keyed_stores:   keyed_mixed with a nullifier store per slot, 1e8 members in all (fresh stores per repetition)
The first two run on one proof set and the last two on a second one, generated on the device in the same buffers.

usage: python tools/key_slots_bench.py [--proofs 1048576] [--members 1e8] [--reps 3]
"""
import argparse
import importlib
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tools"))
act = importlib.import_module("anonymous-credit-tokens_b200")
from nullifier_store_bench import emit, fill, gpu_info   # noqa: E402

KEYS = 4


def bench_keys():
    import corpus
    return [corpus.make_ctx(corpus.BENCH_PARAMS, key_seed=b"key-slots-bench-%d" % k) for k in range(KEYS)]


def make_proofs(eng, n, dev, mixed, hp, hr):
    """n unique valid proofs (request -> issue -> prove_spend on the device) into the pinned buffers hp, hr.  Proof i is issued under
    slot i % KEYS when mixed, else under slot 0.  Returns the key ids."""
    gen = torch.Generator(device=dev); gen.manual_seed(2 if mixed else 1)
    rb = lambda k: torch.randint(0, 256, (k,), dtype=torch.uint8, device=dev, generator=gen)
    PB = act.PROOF_BYTES
    S = torch.cuda.Stream(device=dev)
    step = 1 << 16
    ids = np.arange(n, dtype=np.int64) % KEYS if mixed else np.zeros(n, np.int64)
    with torch.cuda.stream(S):
        for lo in range(0, n, step):
            m = min(step, n - lo)
            pre = rb(m * 64); pre.view(m, 64)[:, 31] &= 0x0f; pre.view(m, 64)[:, 63] &= 0x0f
            req = torch.empty(m * 128, dtype=torch.uint8, device=dev)
            eng.batch_request_dev(m, pre.data_ptr(), rb(m * 128).data_ptr(), req.data_ptr(), S.cuda_stream)
            cs = torch.zeros(m, 32, dtype=torch.uint8, device=dev); cs[:, 0] = 200
            resp = torch.empty(m, 160, dtype=torch.uint8, device=dev); ist = torch.empty(m, dtype=torch.uint8, device=dev)
            irnd = rb(m * 128)
            for k in range(KEYS if mixed else 1):   # the responses of slot k's proofs come from slot k's key
                eng.select_key(k)
                r = torch.empty(m, 160, dtype=torch.uint8, device=dev); s = torch.empty(m, dtype=torch.uint8, device=dev)
                eng.batch_issue_dev(m, req.data_ptr(), cs.data_ptr(), irnd.data_ptr(), r.data_ptr(), s.data_ptr(), S.cuda_stream)
                mine = torch.from_numpy(ids[lo:lo + m] == k).to(dev)
                resp[mine] = r[mine]; ist[mine] = s[mine]
            eng.select_key(0)
            tok = torch.cat([resp[:, :64], pre.view(m, 64)[:, 32:], pre.view(m, 64)[:, :32], cs], 1).contiguous()
            ch = torch.zeros(m, 32, dtype=torch.uint8, device=dev); ch[:, 0] = 7
            pf = torch.empty(m * PB, dtype=torch.uint8, device=dev); pr = torch.empty(m * 96, dtype=torch.uint8, device=dev)
            ps = torch.empty(m, dtype=torch.uint8, device=dev)
            eng.batch_prove_spend_dev(m, tok.data_ptr(), ch.data_ptr(), None, bytes(range(32)), lo + (n if mixed else 0), pf.data_ptr(), pr.data_ptr(),
                                      ps.data_ptr(), S.cuda_stream)
            hp[lo * PB:(lo + m) * PB].copy_(pf, non_blocking=True)
            hr[lo * 128:(lo + m) * 128].copy_(rb(m * 128), non_blocking=True)
            S.synchronize()
            assert bool((ps == 0).all()) and bool((ist == 0).all())
    return ids.astype(np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--proofs", type=int, default=1 << 20)
    ap.add_argument("--members", type=float, default=1e8)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("key_slots_bench: needs a CUDA device (there is no CPU path)")
    emit(leg="gpu", info=gpu_info(), count=torch.cuda.device_count())
    dev = torch.device("cuda", 0)
    n, reps, per_store = a.proofs, a.reps, int(a.members) // KEYS
    ctxs = bench_keys()
    params = act.Params(ctxs[0].h)
    lib = act.load_library()
    PB = act.PROOF_BYTES
    hp = torch.empty(n * PB, dtype=torch.uint8, pin_memory=True); hr = torch.empty(n * 128, dtype=torch.uint8, pin_memory=True)
    href = torch.empty(n * 128, dtype=torch.uint8, pin_memory=True); hnul = torch.empty(n * 32, dtype=torch.uint8, pin_memory=True)
    hst = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    gen = torch.Generator(device=dev); gen.manual_seed(5)
    S = torch.cuda.Stream(device=dev)
    with act.Engine(params, act.PrivateKey(ctxs[0].x, ctxs[0].w), device=0) as eng:
        for k in range(1, KEYS):
            eng.set_key(k, act.PrivateKey(ctxs[k].x, ctxs[k].w))

        def run(name, ids, stores=None):
            table = None
            if stores is not None:
                import ctypes as C
                table = (C.c_void_p * act.KEY_SLOTS)(*[s._h.value for s in stores])
            t = time.perf_counter()
            if ids is None:
                rc = lib.act_batch_verify_spend_and_refund(eng._h, n, hp.data_ptr(), hr.data_ptr(), href.data_ptr(), hnul.data_ptr(), hst.data_ptr())
            else:
                rc = lib.act_batch_verify_spend_and_refund_keyed(eng._h, n, hp.data_ptr(), ids.ctypes.data, hr.data_ptr(), table, href.data_ptr(),
                                                                 hnul.data_ptr(), hst.data_ptr())
            dt = time.perf_counter() - t
            assert rc == 0, lib.act_last_error().decode()
            return dt, int((hst.numpy() == 0).sum())

        for mixed in (False, True):
            t0 = time.time()
            ids = make_proofs(eng, n, dev, mixed, hp, hr)
            emit(leg="fixtures", proofs=n, keys=KEYS if mixed else 1, seconds=round(time.time() - t0, 1))
            times, accepted = {}, {}
            for r in range(reps + 1):
                if not mixed:
                    cases = [("unkeyed", lambda: run("unkeyed", None)), ("keyed_one_slot", lambda: run("keyed_one_slot", ids))]
                else:
                    stores = [act.NullifierStore(device=0, capacity=per_store + n) for _ in range(KEYS)]
                    with torch.cuda.stream(S):
                        for s in stores:
                            fill(s, per_store, gen, dev, S)
                    cases = [("keyed_mixed", lambda: run("keyed_mixed", ids)),
                             ("keyed_stores", lambda: run("keyed_stores", ids, stores + [stores[0]] * (act.KEY_SLOTS - KEYS)))]
                for name, fn in (cases if r % 2 == 0 else cases[::-1]):
                    dt, acc = fn()
                    accepted[name] = acc
                    if r:
                        times.setdefault(name, []).append(dt)
                if mixed:
                    for s in stores:
                        s.close()
            emit(leg="step", proofs=n, keys=KEYS if mixed else 1, store_members_total=per_store * KEYS if mixed else 0, accepted=accepted,
                 **{f"{k}_s": [round(x, 4) for x in v] for k, v in times.items()},
                 **{f"{k}_proofs_per_s_median": round(n / float(np.median(v))) for k, v in times.items()})


if __name__ == "__main__":
    main()
