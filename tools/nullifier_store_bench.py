"""Nullifier store measurements (act_nullifier_store_*, act_batch_verify_spend_and_refund_recorded).  Prints JSON lines.

  store: screen + record of 1M fresh keys per call (5 calls per repetition) (device buffers, CUDA events) into one store filled to 0, 1e8 and 1e9
         members; keys/s and the bytes one key moves (model below) against the HBM data-sheet bandwidth.
  step:  the issuer's step at 1M unique valid proofs per call from pinned host memory, on one GPU and on the multi-device
         handle over every GPU of the box (two replicas on GPU 0 when it has one): _recorded against a store of 1e8 members, _screened(seen=None) and
         _screened(seen=the same 1e8 keys), alternated, host clock around the synchronous call.

usage: python tools/nullifier_store_bench.py [--proofs 1048576] [--levels 0,1e8,1e9] [--seen 1e8] [--reps 3] [--skip-step]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
act = importlib.import_module("anonymous-credit-tokens_b200")

HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU
BATCH = 1 << 20


def emit(**kv):
    print(json.dumps(kv), flush=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()


def probes(alpha):
    """Expected slots touched by an unsuccessful search (= an insert) under linear probing at load alpha (Knuth)."""
    return 0.5 * (1 + 1 / (1 - alpha) ** 2)


def bytes_per_key(alpha, n):
    """Bytes one key of a screen + record call moves, counting every random slot access as one 32-byte sector:
    lookup 33 in + 1 out + 32 per probe; dedupe (replay_insert/resolve over a 4-byte table of >= 2n slots) 2 x 33 in,
    2 sectors, 1 out, the table clear; insert 33 in + 32 per probe + 32 written."""
    dd = 1024
    while dd < 2 * n:
        dd *= 2
    u = probes(alpha)
    return (34 + 32 * u) + (33 + 32) + (34 + 32) + 4 * dd / n + (33 + 32 * u + 32)


def slots_for(capacity):
    """Table slots of a store created for `capacity` members (act_nullifier_store_create: power of two >= 1024, load <= 1/2)."""
    s = 1024
    while s // 2 < capacity:
        s *= 2
    return s


def random_keys(n, gen, dev):
    k = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=gen)
    k[:, 31] &= 0x0f                     # < 2^252 < l: reduced
    return k


def fill(store, target, gen, dev, stream, chunk=1 << 25, keep_host=None):
    """Import fresh random keys until the store holds `target`; optionally keep a pinned host copy of everything imported."""
    have = store.size
    while have < target:
        m = min(chunk, target - have)
        k = random_keys(m, gen, dev)
        st = torch.zeros(m, dtype=torch.uint8, device=dev)
        store.screen_dev(m, st.data_ptr(), k.data_ptr(), st.data_ptr(), True, stream.cuda_stream)
        if keep_host is not None:
            keep_host[have * 32:(have + m) * 32].copy_(k.view(-1), non_blocking=True)
        stream.synchronize()
        have += m
    assert store.size == target, (store.size, target)


def store_leg(levels, reps, dev):
    gen = torch.Generator(device=dev); gen.manual_seed(11)
    S = torch.cuda.Stream(device=dev)
    calls = 5                # 5M keys per timed repetition: the 1e9 level still fits 2^31 slots (68.7 GB)
    capacity = int(max(levels)) + (len(levels) * (reps + 1) * calls + 4) * BATCH
    with act.NullifierStore(device=dev.index, capacity=capacity) as store:
        for level in levels:
            with torch.cuda.stream(S):
                fill(store, max(int(level), store.size), gen, dev, S)
            members = store.size
            with torch.cuda.stream(S):
                batches = [random_keys(BATCH, gen, dev) for _ in range(calls)]
                st = torch.zeros(BATCH, dtype=torch.uint8, device=dev); out = torch.empty_like(st)
                S.synchronize()
                per_rep = []
                for r in range(reps + 1):
                    size0 = store.size
                    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
                    a.record(S)
                    for k in batches:
                        store.screen_dev(BATCH, st.data_ptr(), k.data_ptr(), out.data_ptr(), True, S.cuda_stream)
                    b.record(S)
                    S.synchronize()
                    if r:
                        per_rep.append(a.elapsed_time(b) / calls)
                    # the batches are fresh only once: draw new ones for the next repetition
                    batches = [random_keys(BATCH, gen, dev) for _ in range(calls)]
                    S.synchronize()
                    assert store.size == size0 + calls * BATCH
            alpha = members / slots_for(capacity)
            ms = float(np.median(per_rep))
            bpk = bytes_per_key(alpha, BATCH)
            emit(leg="store", members=members, load_before=round(alpha, 4), load_after=round(store.size / slots_for(capacity), 4), keys_per_call=BATCH, ms_per_call_median=round(ms, 4),
                 ms_per_call_all=[round(x, 4) for x in per_rep], keys_per_s=round(BATCH / (ms / 1e3)),
                 model_bytes_per_key=round(bpk, 1), model_bytes_per_s=round(bpk * BATCH / (ms / 1e3)),
                 share_of_hbm_datasheet=round(bpk * BATCH / (ms / 1e3) / HBM_BYTES_PER_S, 4))


def make_proofs(n, dev):
    """n unique valid proofs generated on the device (request -> issue -> prove_spend), copied to pinned host memory."""
    import corpus
    ctx = corpus.make_ctx(corpus.BENCH_PARAMS)
    params, key = act.Params(ctx.h), act.PrivateKey(ctx.x, ctx.w)
    gen = torch.Generator(device=dev); gen.manual_seed(1)
    rb = lambda k: torch.randint(0, 256, (k,), dtype=torch.uint8, device=dev, generator=gen)
    PB = act.PROOF_BYTES
    hp = torch.empty(n * PB, dtype=torch.uint8, pin_memory=True)
    hr = torch.empty(n * 128, dtype=torch.uint8, pin_memory=True)
    with act.Engine(params, key, device=dev.index) as e0:
        S = torch.cuda.Stream(device=dev)
        step = 1 << 17
        with torch.cuda.stream(S):
            for lo in range(0, n, step):
                m = min(step, n - lo)
                pre = rb(m * 64); pre.view(m, 64)[:, 31] &= 0x0f; pre.view(m, 64)[:, 63] &= 0x0f
                req = torch.empty(m * 128, dtype=torch.uint8, device=dev)
                e0.batch_request_dev(m, pre.data_ptr(), rb(m * 128).data_ptr(), req.data_ptr(), S.cuda_stream)
                cs = torch.zeros(m, 32, dtype=torch.uint8, device=dev); cs[:, 0] = 200
                resp = torch.empty(m * 160, dtype=torch.uint8, device=dev); ist = torch.empty(m, dtype=torch.uint8, device=dev)
                e0.batch_issue_dev(m, req.data_ptr(), cs.data_ptr(), rb(m * 128).data_ptr(), resp.data_ptr(), ist.data_ptr(), S.cuda_stream)
                tok = torch.cat([resp.view(m, 160)[:, :64], pre.view(m, 64)[:, 32:], pre.view(m, 64)[:, :32], cs], 1).contiguous()
                ch = torch.zeros(m, 32, dtype=torch.uint8, device=dev); ch[:, 0] = 7
                pf = torch.empty(m * PB, dtype=torch.uint8, device=dev); pr = torch.empty(m * 96, dtype=torch.uint8, device=dev)
                ps = torch.empty(m, dtype=torch.uint8, device=dev)
                e0.batch_prove_spend_dev(m, tok.data_ptr(), ch.data_ptr(), None, bytes(range(32)), lo, pf.data_ptr(), pr.data_ptr(), ps.data_ptr(), S.cuda_stream)
                hp[lo * PB:(lo + m) * PB].copy_(pf, non_blocking=True)
                hr[lo * 128:(lo + m) * 128].copy_(rb(m * 128), non_blocking=True)
                S.synchronize()
                assert bool((ps == 0).all()) and bool((ist == 0).all())
    return params, key, hp, hr


def step_leg(n, n_seen, reps, dev):
    t0 = time.time()
    params, key, hp, hr = make_proofs(n, dev)
    emit(leg="fixtures", proofs=n, seconds=round(time.time() - t0, 1))
    lib = act.load_library()
    href = torch.empty(n * 128, dtype=torch.uint8, pin_memory=True); hnul = torch.empty(n * 32, dtype=torch.uint8, pin_memory=True)
    hst = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    seen = torch.empty(n_seen * 32, dtype=torch.uint8, pin_memory=True)
    gen = torch.Generator(device=dev); gen.manual_seed(5)
    S = torch.cuda.Stream(device=dev)
    G = torch.cuda.device_count()
    # the multi-device handle over every GPU of the box; on a one-GPU box, two replicas on GPU 0 (the same gather path, no speed-up)
    for devices in ([dev.index], list(range(G)) if G > 1 else [dev.index, dev.index]):
        with act.Engine(params, key, devices=devices) as eng:
            times = {"recorded_store_1e8": [], "screened_seen_none": [], "screened_seen_1e8": []}
            accepted = {}
            for r in range(reps + 1):
                # _recorded needs a store of n_seen members that has not seen this batch yet: a fresh one per repetition (the
                # first repetition's keys are also the `seen` set of _screened)
                with act.NullifierStore(device=devices[0], capacity=n_seen + n) as store:
                    with torch.cuda.stream(S):
                        fill(store, n_seen, gen, dev, S, keep_host=seen if r == 0 else None)
                    cases = (
                        ("recorded_store_1e8", lambda: lib.act_batch_verify_spend_and_refund_recorded(
                            eng._h, store._h, n, hp.data_ptr(), hr.data_ptr(), href.data_ptr(), hnul.data_ptr(), hst.data_ptr())),
                        ("screened_seen_none", lambda: lib.act_batch_verify_spend_and_refund_screened(
                            eng._h, n, hp.data_ptr(), hr.data_ptr(), 0, None, href.data_ptr(), hnul.data_ptr(), hst.data_ptr())),
                        ("screened_seen_1e8", lambda: lib.act_batch_verify_spend_and_refund_screened(
                            eng._h, n, hp.data_ptr(), hr.data_ptr(), n_seen, seen.data_ptr(), href.data_ptr(), hnul.data_ptr(), hst.data_ptr())),
                    )
                    for name, fn in (cases if r % 2 == 0 else cases[::-1]):      # alternate the order between repetitions
                        t = time.perf_counter()
                        rc = fn()
                        dt = time.perf_counter() - t
                        assert rc == 0, lib.act_last_error().decode()
                        accepted[name] = int((hst.numpy() == 0).sum())
                        if r:
                            times[name].append(dt)
                    assert store.size == n_seen + accepted["recorded_store_1e8"]
            emit(leg="step", devices=devices, proofs=n, store_or_seen=n_seen, accepted=accepted,
                 **{f"{k}_s": [round(x, 4) for x in v] for k, v in times.items()},
                 **{f"{k}_proofs_per_s_median": round(n / float(np.median(v))) for k, v in times.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--proofs", type=int, default=1 << 20)
    ap.add_argument("--levels", default="0,1e8,1e9")
    ap.add_argument("--seen", type=float, default=1e8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-step", action="store_true")
    ap.add_argument("--skip-store", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nullifier_store_bench: needs a CUDA device (there is no CPU path)")
    emit(leg="gpu", info=gpu_info(), count=torch.cuda.device_count())
    dev = torch.device("cuda", 0)
    if not a.skip_store:
        store_leg([float(x) for x in a.levels.split(",")], a.reps, dev)
    if not a.skip_step:
        step_leg(a.proofs, int(a.seen), a.reps, dev)


if __name__ == "__main__":
    main()
