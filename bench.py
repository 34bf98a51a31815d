#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 batch engine (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--n-spend N] [--n-issue N] [--dump-outputs DIR]

One "step" = one pass of `batch_verify_spend_and_refund` over one batch of synthetic SpendProofs
(default 1,048,576 per GPU = BASELINE.json configs[2]; weak scaling, so N=8 is the 8M-proof batch of
configs[3]).  The inputs are generated from fixed seeds, so the same arguments give the same inputs in every run.
--dump-outputs DIR writes what the last timed step returned (see dump_outputs) so that two builds can be compared
output for output.  Prints ONE JSON line (rank 0):

  value      : spend verify+refund per second, whole job, inputs resident in HBM, device-timed
  e2e        : same metric through the C ABI with pinned HOST buffers (H2D + kernels + D2H in the timed region)
  issue      : batch_issue throughput (configs[1]) measured the same two ways
  roofline   : dominant kernel (spend_range_kernel) vs the measured integer-multiply roofline
  cpu_baseline: the oracle (port of the reference's algorithm) timed on this box's host cores

--impl reference times the reference's own CPU algorithm (the C oracle port: the crate itself cannot be built
in this image -- no Rust toolchain) with all host threads on a bounded sample.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True       # the tree may be read-only: the benchmark writes nothing there, bytecode caches included
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "spend_verify_refund_per_sec"
UNIT = "proofs/s"
# Algorithmic work per unit in 32x32+64->64 limb multiply-accumulates (field multiply M = 72, square S = 44), counted for
# the algorithm this engine implements (DESIGN.md section 4 has the breakdown; SURVEY.md 8d estimated 4.8e7 / 7.0e5 for
# a wNAF formulation -- the implemented shared-chain / wide-window / batched-encode algorithm needs less):
#   range kernel per com_j (bucket form, the default since round 2): 1266 S + 2525 M = 2.375e5 -> x128 = 3.04e7 per proof
#       (round 1's window form: 1506 S + 2583 M = 2.522e5 -> 3.23e7; the constant follows the algorithm that runs)
#       = the EXECUTED IMAD.WIDE lane count ncu reports for the kernel (3.0396e7 per proof, profiles/r02e_spend_range.txt)
#   the other stages: the executed IMAD.WIDE(.X) lane counts of one ncu capture each at the product launch shape
#   (profiles/r02f_*.txt): encode 5.40e5 (profiles/r02k_spend_encode_kernel.txt; 6.81e5 before r02j's 64-point batches), head 7.43e5, sign 3.40e5 per proof, issue 5.37e5 per request.  (Round 1's hand counts --
#   7.1e5 / 8.2e5 / 3.9e5 / 6.0e5 -- were 4-13 % too high; the constants below are what the kernels execute.)
LIMB_MACS_PER_SPEND_RANGE = 128 * (1266 * 44 + 2525 * 72)      # 3.040e7
LIMB_MACS_PER_SPEND_HEAD = 7.29e5       # 7.43e5 executed (r02f) - 3 x 63 T products (72 each) no longer computed: two vb_mul_pub, the A1 window loop (r02z)
LIMB_MACS_PER_SPEND_SIGN = 3.40e5
LIMB_MACS_PER_SPEND_ENCODE = 5.40e5     # executed at 64 points per inversion (profiles/r02k_spend_encode_kernel.txt); 6.81e5 at 16 per inversion (r02f)
LIMB_MACS_PER_SPEND = LIMB_MACS_PER_SPEND_RANGE + LIMB_MACS_PER_SPEND_ENCODE + LIMB_MACS_PER_SPEND_HEAD + LIMB_MACS_PER_SPEND_SIGN
LIMB_MACS_PER_ISSUE = 5.32e5            # 5.37e5 executed (r02f) - 63 T products of the public K*gamma (r02y)
MIXED_N_1GPU = 1 << 22               # BASELINE configs[4]: 4M requests on one GPU
STRONG_TOTAL = 1 << 23               # BASELINE configs[3]: the SAME 8M-proof batch split over 2/4/8 GPUs
# IMAD.WIDE.U32 issues at 32 lanes per clock per SM on sm_100 (ncu: 2 fma-heavy pipe cycles per warp instruction at
# 0.5 instructions/clock/SMSP; profiles/r01d_*.txt) -> integer-multiply roofline = SMs x 32 x SM clock
IMAD_WIDE_LANES_PER_CLK_PER_SM = 32
PROOF_BYTES = 16832
UNIQUE_PROOFS = 2048                 # valid proofs from the ORACLE prover: CPU baseline sample + cross-check of the engine
UNIQUE_REQUESTS = 16384
DUMP_ROWS = 65536                    # --dump-outputs: proofs sampled from the timed batch; 65536 x 161 float32 values = 42 MB


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)), "reasons": sorted(reasons), "samples": len(sm)}


def synth(ctx, n_unique_proofs, n_unique_req, threads):
    import corpus
    t0 = time.time()
    base = corpus.gen_valid(ctx, n_unique_proofs, seed=b"bench-spend", credits=(20, 1000), threads=threads)
    reqs = corpus.gen_valid(ctx, n_unique_req, seed=b"bench-issue", credits=(10, 1000), threads=threads, want_proofs=False)
    log(f"[bench] synthesised {n_unique_proofs} proofs + {n_unique_req} requests on {threads} host threads in {time.time() - t0:.1f}s")
    return base, reqs


def cpu_baseline(ctx, base, reqs, threads, budget_s=8.0):
    """Oracle (restated reference algorithm) on the host cores: typed refund()/issue() closures as in benches/benchmark.rs."""
    import corpus
    import oracle_lib
    if oracle_lib.use_native_build():      # time the -march=native build of the port; a new context binds to it
        ctx = corpus.make_ctx(corpus.BENCH_PARAMS)
    n1 = 24
    t1, ok = ctx.time_refund_typed(base["proofs"][:n1 * PROOF_BYTES], base["rnd"][:n1 * 128], threads=1, reps=1)
    assert ok == n1
    per = t1 / n1
    nall = min(len(base["proofs"]) // PROOF_BYTES, max(threads * 4, int(budget_s / per) * threads // 1))
    nall = max(threads, (nall // threads) * threads)
    tall, ok = ctx.time_refund_typed(base["proofs"][:nall * PROOF_BYTES], base["rnd"][:nall * 128], threads=threads, reps=1)
    assert ok == nall
    ni = 2048
    ti1, ok = ctx.time_issue_typed(reqs["req"][:ni * 128], reqs["cs"][:ni * 32], reqs["rnd"][:ni * 128], threads=1, reps=1)
    nia = min(len(reqs["req"]) // 128, 2048 * threads)
    tia, ok = ctx.time_issue_typed(reqs["req"][:nia * 128], reqs["cs"][:nia * 32], reqs["rnd"][:nia * 128], threads=threads, reps=4)
    out = {
        "value": nall / tall, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": f"{nall} typed refund() calls on {threads} threads ({tall:.2f}s); 1 thread: {n1} calls",
        "value_1thread": n1 / t1,
        "issue": {"value": nia * 4 / tia, "unit": "issues/s", "value_1thread": ni / ti1},
        "fidelity": "C port of the reference's algorithm (5x51-bit limbs, scalar code, no vector back end); the real crate would pick "
                    "curve25519-dalek's AVX2/IFMA back ends on hosts that have them, so ratios against this number overstate the margin "
                    "against the crate by whatever those back ends gain (typically 1.5-2x)",
    }
    out["libsodium_bound"] = libsodium_bound(out["value_1thread"])
    return out


def libsodium_bound(port_1thread):
    """Sanity bound of the port (BASELINE.md section 3): libsodium's ristretto255 per-op timings x the operation counts of one
    reference refund() (SURVEY 8a row a2: 395 constant-time variable-base multiplications, 265 fixed-base ones; libsodium's
    calls include a decode and an encode each, which stands in for the reference's 400 compressions)."""
    try:
        import refstack as R
        if not R.available():
            return {"unavailable": "libsodium with ristretto255 not found"}
        import ctypes as C
        sod = R._sodium
        p = R.mul_base(12345)
        sc = (0x1234567890abcdef1234567890abcdef1234567890abcdef1234567890abcde % R.ELL).to_bytes(32, "little")
        out = C.create_string_buffer(32)
        reps = 400
        t0 = time.perf_counter()
        for _ in range(reps):
            sod.crypto_scalarmult_ristretto255(out, sc, p)
        t_vb = (time.perf_counter() - t0) / reps
        t0 = time.perf_counter()
        for _ in range(reps):
            sod.crypto_scalarmult_ristretto255_base(out, sc)
        t_fb = (time.perf_counter() - t0) / reps
        est = 1.0 / (395 * t_vb + 265 * t_fb)
        return {"vb_mult_us": 1e6 * t_vb, "fb_mult_us": 1e6 * t_fb, "estimated_refunds_per_s_1thread": est,
                "port_over_estimate": port_1thread / est,
                "how": "1 / (395 x crypto_scalarmult_ristretto255 + 265 x crypto_scalarmult_ristretto255_base), timed here on one thread"}
    except Exception as ex:   # a sanity figure must never take the bench down
        return {"unavailable": repr(ex)}


def dump_outputs(out_dir, n, ref, nul, st):
    """What one call of batch_verify_spend_and_refund over the timed batch returns to its caller -- refund records (n x 128 B),
    nullifiers (n x 32 B) and statuses (n) -- for a fixed, seeded sample of DUMP_ROWS proofs (all of them when the batch is no
    larger), as DIR/{refund,nullifier,status}.npy with one byte per float32 value (exact) and the sampled proof indices as
    DIR/index.npy (float64)."""
    import torch
    m = min(n, DUMP_ROWS)
    idx = np.sort(np.random.RandomState(20261020).choice(n, size=m, replace=False)) if m < n else np.arange(n)
    sel = torch.as_tensor(idx, device=ref.device)
    arrays = {"index": idx.astype(np.float64),
              "refund": ref.view(n, 128)[sel].cpu().numpy().astype(np.float32),
              "nullifier": nul.view(n, 32)[sel].cpu().numpy().astype(np.float32),
              "status": st[sel].cpu().numpy().astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[bench] outputs of the last timed step ({m} of {n} proofs, {sum(a.nbytes for a in arrays.values()) / 2**20:.1f} MiB) written to {out_dir}")


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port) on all host threads, bounded sample per step."""
    if rank != 0:
        return
    import corpus
    threads = os.cpu_count() or 1
    import oracle_lib
    native = oracle_lib.use_native_build()
    ctx = corpus.make_ctx(corpus.BENCH_PARAMS)
    n = max(threads * 64, 512)   # per step: enough calls per thread that thread start-up and imbalance do not show
    base = corpus.gen_valid(ctx, n, seed=b"bench-spend", credits=(20, 1000), threads=threads)
    times = []
    for s in range(args.warmup + args.steps):
        t, ok = ctx.time_refund_typed(base["proofs"], base["rnd"], threads=threads, reps=1)
        assert ok == n
        if s >= args.warmup:
            times.append(t)
    tot = sum(times)
    v = n * len(times) / tot
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (int)",
        "data": "synthetic", "config": {"workload": f"PrivateKey::refund on {n} valid SpendProofs per step (bounded sample of configs[2]), L=128, bench params",
                                       "note": "reference crate is Rust with un-vendored deps; no cargo/rustc in this image -> C port of its algorithm (oracle/act_oracle.c), "
                                               "constant-time radix-16 scalar mults and the 128-mult K' as in src/lib.rs:781-869"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": f"{n} typed refund() calls per step on {threads} threads"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-spend", type=int, default=1 << 20, help="SpendProofs per GPU per step")
    ap.add_argument("--n-issue", type=int, default=1 << 20, help="IssuanceRequests per GPU per step")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mixed-frac", type=float, default=0.1, help="tampered fraction of the mixed adversarial batch (0 = skip)")
    ap.add_argument("--mixed-n", type=int, default=None, help="size of the mixed adversarial batch (default: 4194304 on one GPU = configs[4], n-spend per GPU otherwise)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling form of configs[3] (8M proofs split over the GPUs)")
    ap.add_argument("--no-multi-abi", action="store_true", help="skip the single-process multi-device C-ABI leg (N > 1)")
    ap.add_argument("--oracle-sample", type=int, default=1024, help="proofs of the timed batch re-verified and re-signed by the CPU oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (refunds, nullifiers, statuses of a fixed, seeded sample of "
                         f"{DUMP_ROWS} proofs; rank 0's shard when N > 1) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 engine's timed step")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # Only the JSON line may reach stdout: libraries (NCCL prints its version banner to fd 1) write to stderr instead.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    import corpus
    act = importlib.import_module("anonymous-credit-tokens_b200")
    act.load_library()                      # fails loudly if the CUDA extension is missing
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        cpu_group = dist.new_group(backend="gloo")     # host-side barrier for the leg in which rank 0 drives every GPU itself
    W, K = args.warmup, args.steps
    n, ni = args.n_spend, args.n_issue
    threads = max(1, (os.cpu_count() or 1) // world)

    # ---- synthetic inputs (oracle fixture generators), identical on every rank; each rank rotates its tiling ----
    ctx = corpus.make_ctx(corpus.BENCH_PARAMS)
    base, reqs = synth(ctx, UNIQUE_PROOFS, UNIQUE_REQUESTS, threads)
    params = act.Params.new(*corpus.BENCH_PARAMS, device=local)
    assert params.h == ctx.h, "Params::new differs from the oracle"
    key = act.PrivateKey(ctx.x, ctx.w)
    eng = act.Engine(params, key, device=local)
    sm_count = torch.cuda.get_device_properties(local).multi_processor_count

    # a real (non-default) stream: torch ops, the engine's launches and the timing events all go to it
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    # ---- device-side fixture generation (untimed): UNIQUE tokens are requested, issued and spent on this GPU by the engine's
    # client-side generators (act_batch_request -> act_batch_issue -> act_batch_prove_spend; bit-exact with the oracle prover,
    # tests/test_gpu_parity.py), so no proof in a batch repeats.  Seeds are fixed per rank.
    gen = torch.Generator(device=dev); gen.manual_seed(20261017 + rank)

    def rbytes(k):
        return torch.randint(0, 256, (k,), dtype=torch.uint8, device=dev, generator=gen)

    def le32(v, count):
        sh = 8 * torch.arange(2, device=dev)
        return torch.cat([((v.view(count, 1) >> sh) & 0xff).to(torch.uint8), torch.zeros(count, 30, dtype=torch.uint8, device=dev)], 1).reshape(-1)

    def make_requests(count):
        pre = rbytes(count * 64); pv = pre.view(count, 64); pv[:, 31] &= 0x0f; pv[:, 63] &= 0x0f   # PreIssuance r, k (< 2^252)
        req = torch.empty(count * 128, dtype=torch.uint8, device=dev)
        eng.batch_request_dev(count, pre.data_ptr(), rbytes(count * 128).data_ptr(), req.data_ptr(), stream)
        credits = torch.randint(20, 1000, (count,), device=dev, generator=gen)                     # benches/benchmark.rs:60,178
        torch.cuda.synchronize()
        return pre, req, credits

    def make_tokens(count, issuer):
        """count tokens issued by `issuer` (an Engine on this device): (tokens count x 160 [A|e|k|r|c], credits)."""
        pre, req, credits = make_requests(count)
        cs = le32(credits, count)
        resp = torch.empty(count * 160, dtype=torch.uint8, device=dev); ist = torch.empty(count, dtype=torch.uint8, device=dev)
        issuer.batch_issue_dev(count, req.data_ptr(), cs.data_ptr(), rbytes(count * 128).data_ptr(), resp.data_ptr(), ist.data_ptr(), stream)
        torch.cuda.synchronize()
        assert bool((ist == 0).all()), "fixture issuance rejected a request"
        tokens = torch.cat([resp.view(count, 160)[:, :64], pre.view(count, 64)[:, 32:], pre.view(count, 64)[:, :32], cs.view(count, 32)], 1).contiguous()
        return tokens, credits

    prove_calls = [0]

    def prove(tokens, charges_le, count, out=None):
        """count proofs from tokens (count x 160) and charges (count*32 LE) with a fresh derived RNG stream per call."""
        pf = out if out is not None else torch.empty(count * PROOF_BYTES, dtype=torch.uint8, device=dev)
        pr = torch.empty(count * 96, dtype=torch.uint8, device=dev); ps = torch.empty(count, dtype=torch.uint8, device=dev)
        prove_calls[0] += 1
        seed = bytes([(7 * i + rank + 31 * prove_calls[0]) & 0xff for i in range(32)])
        eng.batch_prove_spend_dev(count, tokens.data_ptr(), charges_le.data_ptr(), None, seed, (rank * 64 + prove_calls[0]) << 32, pf.data_ptr(), pr.data_ptr(), ps.data_ptr(), stream)
        torch.cuda.synchronize()
        assert bool((ps == 0).all())
        return pf

    def make_spend_batch(count):
        """count unique valid proofs with charges uniform in [1, c-1] (benchmark.rs:194-201): (proofs, tokens, rnd)."""
        tokens, credits = make_tokens(count, eng)
        spend = (torch.rand(count, device=dev, generator=gen) * (credits - 1)).long() + 1
        proofs = prove(tokens, le32(spend, count), count)
        return proofs, tokens, rbytes(count * 128)

    t_gen = time.time()
    d_proofs, d_tokens, d_rnd = make_spend_batch(n)
    log(f"[bench] rank {rank}: {n} unique tokens issued and spent on the device in {time.time() - t_gen:.1f}s")
    d_ref = torch.zeros(n * 128, dtype=torch.uint8, device=dev)
    d_nul = torch.zeros(n * 32, dtype=torch.uint8, device=dev)
    d_st = torch.zeros(n, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, warm, steps):
        for _ in range(warm):
            step_fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step_fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def spend_stepper(count, proofs, rnd, ref, nul, st):
        """One step = verify + refund of this rank's shard, then the one collective on the path (N > 1): the gather of accept
        bits and nullifiers, 33 B per proof."""
        if world > 1:
            g_st = torch.empty(world * count, dtype=torch.uint8, device=dev)
            g_nul = torch.empty(world * count * 32, dtype=torch.uint8, device=dev)

        def step():
            eng.batch_verify_spend_and_refund_dev(count, proofs.data_ptr(), rnd.data_ptr(), ref.data_ptr(), nul.data_ptr(), st.data_ptr(), stream)
            if world > 1:
                dist.all_gather_into_tensor(g_st, st)
                dist.all_gather_into_tensor(g_nul, nul)
        return step

    spend_step = spend_stepper(n, d_proofs, d_rnd, d_ref, d_nul, d_st)

    # ---- value: device-resident, device-timed ----
    for _ in range(W):
        spend_step()
    barrier()
    launches0 = eng.launch_count
    with ClockSampler(local) as clk:
        ms = timed(spend_step, 0, K)
    launches = eng.launch_count - launches0
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, n, d_ref, d_nul, d_st)
    value = world * n * K / (ms * 1e-3)
    sm_hz = 1e6 * (clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0)
    peak_model = sm_count * IMAD_WIDE_LANES_PER_CLK_PER_SM * sm_hz
    # the integer-multiply peak this box delivers, measured now (GPU warm, same clocks): pure IMAD.WIDE.U32 chains
    peak_measured = max(act.measure_int_mul_peak(local) for _ in range(3))
    peak = peak_measured
    # ---- roofline pass: the same work in slices of one pipeline chunk (the product's launch shape) on ONE stream (no
    # inter-chunk overlap), every launch bracketed by CUDA events on that stream, so that per-kernel durations are clean ----
    SL = 65536
    eng.set_timing(True)
    eng.get_timing()
    for off in range(0, n, SL):
        m = min(SL, n - off)
        eng.batch_verify_spend_and_refund_dev(m, d_proofs.data_ptr() + off * PROOF_BYTES, d_rnd.data_ptr() + off * 128, d_ref.data_ptr() + off * 128,
                                              d_nul.data_ptr() + off * 32, d_st.data_ptr() + off, stream)
    torch.cuda.synchronize()
    ktimes = eng.get_timing()
    eng.set_timing(False)
    # ---- parity guard inside the bench: every proof of the valid batch accepted; the CPU oracle verifies and re-signs a random
    # sample of the device-generated proofs with the same randomness: identical status, refund and nullifier bytes ----
    st_host = d_st.cpu().numpy()
    assert (st_host == 0).all(), f"bench batch not fully accepted: {np.unique(st_host, return_counts=True)}"
    chk = max(4, min(args.oracle_sample, n))
    rs = np.random.RandomState(1234 + rank)
    sidx = torch.as_tensor(np.sort(rs.choice(n, size=chk, replace=False)), device=dev)
    o_ref, o_nul, o_st, _ = ctx.batch_refund(d_proofs.view(n, PROOF_BYTES)[sidx].reshape(-1).cpu().numpy(), d_rnd.view(n, 128)[sidx].reshape(-1).cpu().numpy(), threads=threads)
    assert (o_st == 0).all(), "oracle rejects a device-generated proof"
    assert (d_ref.view(n, 128)[sidx].reshape(-1).cpu().numpy() == o_ref).all() and (d_nul.view(n, 32)[sidx].reshape(-1).cpu().numpy() == o_nul).all(), "bench output differs from oracle"
    # ... and the engine verifies a sample of the ORACLE prover's proofs (CPU fixtures) to the oracle's bytes
    c2 = min(256, UNIQUE_PROOFS)
    o2_ref, o2_nul, o2_st, _ = ctx.batch_refund(base["proofs"][:c2 * PROOF_BYTES], base["rnd"][:c2 * 128], threads=threads)
    g2 = eng.batch_verify_spend_and_refund(base["proofs"][:c2 * PROOF_BYTES], base["rnd"][:c2 * 128])
    assert (g2[2] == o2_st).all() and (g2[0] == o2_ref).all() and (g2[1] == o2_nul).all()
    oracle_checks = {"device_generated_proofs_rechecked_by_oracle": int(chk), "oracle_generated_proofs_checked_on_gpu": int(c2), "all_equal": True}
    rng_ms, rng_cnt = ktimes["spend_range"]
    per_launch_proofs = n / max(rng_cnt, 1)
    achieved = LIMB_MACS_PER_SPEND_RANGE * per_launch_proofs / (rng_ms / max(rng_cnt, 1) * 1e-3) if rng_ms else None
    total_kernel_ms = sum(v[0] for v in ktimes.values())
    hbm_bytes = n * K * (PROOF_BYTES + 128 + 161)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    # DRAM traffic of the dominant kernel per launch, from the committed `ncu --set full` capture (bytes per proof x proofs per launch)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = {"bytes_per_launch": tj["spend_range_dram_bytes_per_proof"] * per_launch_proofs, "bytes_per_proof": tj["spend_range_dram_bytes_per_proof"],
                   "algorithmic_bytes_per_proof": PROOF_BYTES + 128 * 96 + 256 * 128 + 128 * 32, "source": tj.get("source"), "note": tj.get("note")}
    except Exception:
        pass

    def kfrac(kind, work):
        t, c = ktimes[kind]
        return (work * n / (t * 1e-3) / peak) if t else None

    roofline = {
        "bound": "int_mul", "kernel": "spend_range_kernel", "achieved": achieved / 1e12 if achieved else None, "peak": peak / 1e12,
        "unit": "Tlimb-MAC/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
        "peak_source": "MEASURED on this GPU in this run by act_measure_int_mul_peak (16 independent IMAD.WIDE.U32 chains per thread, 64 warps per SM; "
                       "tests/test_abi.py checks that its SASS loop is 16 wide multiplies and nothing else on the multiply pipe); "
                       "there is no integer entry in MEASURED_PEAKS.json.  `frac` uses this number.",
        "peak_model": peak_model / 1e12,
        "peak_model_source": f"{sm_count} SMs x {IMAD_WIDE_LANES_PER_CLK_PER_SM} IMAD.WIDE lanes/clk x {sm_hz / 1e6:.0f} MHz (SM clock sampled under load); "
                             "pipe rate from ncu (sm__pipe_fmaheavy_cycles_active: 2 cycles per IMAD.WIDE warp instruction)",
        "frac_of_model": (achieved / peak_model) if achieved else None,
        "measured_over_model": peak_measured / peak_model,
        "work_per_unit": f"{LIMB_MACS_PER_SPEND_RANGE:.4g} limb-MACs per proof in this kernel = 128 x (1266 S x 44 + 2525 M x 72), the implemented (bucket) algorithm (DESIGN.md 4)",
        "timing": f"separate pass, one stream, slices of {SL} proofs (the product's chunk), CUDA events around every launch",
        "second_bound": "instruction issue: the IADD3 + IMAD.WIDE mix of a field multiplication tops out at 0.52-0.54 warp instructions per clock "
                        "per SM sub-partition on B200 (tools/issue_bench.cu, profiles/r01j_micro_issue_rate.txt)",
        "kernel_share_of_step": rng_ms / total_kernel_ms if total_kernel_ms else None,
        "kernel_ms": {k: round(v[0], 3) for k, v in ktimes.items() if v[1]},
        "other_kernels_frac": {"spend_head": kfrac("spend_head", LIMB_MACS_PER_SPEND_HEAD), "refund_sign": kfrac("refund_sign", LIMB_MACS_PER_SPEND_SIGN),
                               "spend_encode": kfrac("spend_encode", LIMB_MACS_PER_SPEND_ENCODE)},
        "step_over_range_kernel": (ms / K) / rng_ms if rng_ms else None,
        "whole_step": {"achieved": LIMB_MACS_PER_SPEND * n * K / (ms * 1e-3) / 1e12, "frac": LIMB_MACS_PER_SPEND * n * K / (ms * 1e-3) / peak,
                       "frac_of_model": LIMB_MACS_PER_SPEND * n * K / (ms * 1e-3) / peak_model},
        "hbm": {"achieved_gbs": hbm_bytes / (ms * 1e-3) / 1e9, "peak_gbs": hbm_peak, "frac": hbm_bytes / (ms * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650 GB/s"},
    }

    # ---- issue (configs[1]) device-resident ----
    _pre, d_req, icred = make_requests(ni)
    d_cs = le32(icred, ni)
    d_irnd = rbytes(ni * 128)
    del _pre
    d_resp = torch.zeros(ni * 160, dtype=torch.uint8, device=dev); d_ist = torch.zeros(ni, dtype=torch.uint8, device=dev)

    def issue_step():
        eng.batch_issue_dev(ni, d_req.data_ptr(), d_cs.data_ptr(), d_irnd.data_ptr(), d_resp.data_ptr(), d_ist.data_ptr(), stream)

    ims = timed(issue_step, W, K)
    eng.set_timing(True); eng.get_timing()
    issue_step(); torch.cuda.synchronize()
    issue_kernel_ms = eng.get_timing()["issue"][0]
    eng.set_timing(False)
    assert (d_ist.cpu().numpy() == 0).all()
    ichk = min(1024, ni)
    o_resp, o_ist, _ = ctx.batch_issue(d_req[:ichk * 128].cpu().numpy(), d_cs[:ichk * 32].cpu().numpy(), d_irnd[:ichk * 128].cpu().numpy(), threads=threads)
    assert (o_ist == 0).all() and (d_resp[:ichk * 160].cpu().numpy() == o_resp).all(), "issue output differs from oracle"
    oracle_checks["issue_responses_rechecked_by_oracle"] = int(ichk)
    issue_value = world * ni * K / (ims * 1e-3)

    # ---- client-side checks (SURVEY 8a rows a3, a4: the verification halves of the two to_credit_token), device-resident:
    # every response / refund just produced must verify ----
    d_K = d_req.view(ni, 128)[:, :32].contiguous().view(-1)
    d_cst = torch.full((ni,), 255, dtype=torch.uint8, device=dev)
    icms = timed(lambda: eng.batch_issuance_check_dev(ni, d_K.data_ptr(), d_resp.data_ptr(), d_cst.data_ptr(), stream), 1, K)
    assert (d_cst == 0).all(), "issuance_check rejected a response of batch_issue"
    nrc = min(n, 131072)
    d_com = d_proofs.view(n, PROOF_BYTES)[:nrc, 128:128 + 4096].contiguous().view(-1)
    d_rst = torch.full((nrc,), 255, dtype=torch.uint8, device=dev)
    rcms = timed(lambda: eng.batch_refund_check_dev(nrc, d_com.data_ptr(), d_ref.data_ptr(), d_rst.data_ptr(), stream), 1, K)
    assert (d_rst == 0).all(), "refund_check rejected a refund of batch_verify_spend_and_refund"
    client_checks = {"issuance_check": {"value": world * ni * K / (icms * 1e-3), "unit": "checks/s", "n": ni},
                     "refund_check": {"value": world * nrc * K / (rcms * 1e-3), "unit": "checks/s", "n": nrc}}
    del d_K, d_cst, d_com, d_rst

    # ---- e2e: pinned host buffers through the public C ABI (H2D + kernels + D2H inside the timed region) ----
    Ke = args.e2e_steps or K
    host_mem = "pinned"
    try:
        h_proofs = torch.empty(n * PROOF_BYTES, dtype=torch.uint8, pin_memory=True)
    except RuntimeError as ex:   # a box that cannot page-lock world x 17.6 GB: the same bytes from pageable memory (slower copies)
        log(f"[bench] rank {rank}: pinned allocation failed ({ex}); using pageable host memory for the e2e leg")
        h_proofs = torch.empty(n * PROOF_BYTES, dtype=torch.uint8)
        host_mem = "pageable (pinned allocation failed)"
    h_proofs.copy_(d_proofs)
    hq = torch.empty(ni * 128, dtype=torch.uint8, pin_memory=True); hq.copy_(d_req)
    h_rnd = d_rnd.cpu().pin_memory()
    h_ref = torch.empty(n * 128, dtype=torch.uint8, pin_memory=True); h_nul = torch.empty(n * 32, dtype=torch.uint8, pin_memory=True)
    h_st = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    ref_dev = d_ref.cpu().numpy().copy()      # the device-resident leg's refunds: the e2e leg must reproduce them byte for byte

    def e2e_step():
        eng.batch_verify_spend_and_refund_ptr(n, h_proofs.data_ptr(), h_rnd.data_ptr(), h_ref.data_ptr(), h_nul.data_ptr(), h_st.data_ptr())

    e2e_step()  # warm-up (allocates the staging buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_s = float(t.item())
    assert (h_st.numpy() == 0).all() and (h_ref.numpy() == ref_dev).all(), "e2e leg differs from the device-resident leg"
    e2e_value = world * n * Ke / e2e_s
    del ref_dev

    hc = d_cs.cpu().pin_memory(); hr = d_irnd.cpu().pin_memory()
    hresp = torch.empty(ni * 160, dtype=torch.uint8, pin_memory=True); hst = torch.empty(ni, dtype=torch.uint8, pin_memory=True)

    def e2e_issue():
        eng.batch_issue_ptr(ni, hq.data_ptr(), hc.data_ptr(), hr.data_ptr(), hresp.data_ptr(), hst.data_ptr())

    e2e_issue(); barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        e2e_issue()
    barrier()
    e2e_issue_s = time.perf_counter() - t0

    nm = max(1, min(262144, n // world))     # per-GPU shard of the multi-device leg: disjoint windows of rank 0's unique proofs
    m_keep = None
    if world > 1 and not args.no_multi_abi and rank == 0:
        mk_p = torch.empty(world * nm * PROOF_BYTES, dtype=torch.uint8, pin_memory=True); mk_p.copy_(h_proofs[:world * nm * PROOF_BYTES])
        mk_r = torch.empty(world * nm * 128, dtype=torch.uint8, pin_memory=True); mk_r.copy_(h_rnd[:world * nm * 128])
        m_keep = (mk_p, mk_r, h_ref[:nm * 128].clone())
    del h_proofs
    torch.cuda.empty_cache()

    # ---- mixed adversarial batch (BASELINE configs[4]: 4M requests on one GPU, 10 % tampered, malformed points, replayed
    # nullifiers).  Every tamper class of the reference's tests (SURVEY section 4) is planted on the device; expected statuses are
    # known by construction AND a sample of every class (>= 256 where the class has that many) is re-verified and re-signed by the
    # CPU oracle: status, refund and nullifier bytes must be equal.  Then the engine's replay screen over the batch. ----
    mixed = None
    if args.mixed_frac > 0:
        nmix = args.mixed_n or (MIXED_N_1GPU if world == 1 else n)
        if nmix == n:
            pv_all, tok_all, rnd_all = d_proofs, d_tokens, d_rnd
            m_ref_, m_nul_, m_st_ = d_ref, d_nul, d_st
        else:
            del d_proofs
            torch.cuda.empty_cache()
            t_gen = time.time()
            pv_all, tok_all, rnd_all = make_spend_batch(nmix)
            log(f"[bench] rank {rank}: mixed batch: {nmix} unique tokens issued and spent on the device in {time.time() - t_gen:.1f}s")
            m_ref_ = torch.zeros(nmix * 128, dtype=torch.uint8, device=dev); m_nul_ = torch.zeros(nmix * 32, dtype=torch.uint8, device=dev)
            m_st_ = torch.zeros(nmix, dtype=torch.uint8, device=dev)
        pv = pv_all.view(nmix, PROOF_BYTES)
        NCLS = 12
        sel = torch.rand(nmix, device=dev, generator=gen) < args.mixed_frac
        sel[0] = False
        tidx = torch.nonzero(sel).view(-1)
        cls = torch.randint(0, NCLS, (tidx.numel(),), device=dev, generator=gen)
        expect = torch.zeros(nmix, dtype=torch.uint8, device=dev)
        names = ["s changed", "A' = identity", "malformed com point (s = p)", "gamma bit flip", "exact replay of the neighbour",
                 "same token spent again with a different proof", "non-canonical scalar encodings (must accept)", "overspend (s > c)",
                 "token of another issuer key", "token with a, e replaced", "malformed A' (odd s)", "malformed B-bar (non-square)"]
        I = [tidx[cls == c] for c in range(NCLS)]
        pv[I[0], 32] ^= 1; expect[I[0]] = 7                                            # src/tests.rs:631-638 -> InvalidClientSpendProof
        pv[I[1], 64:96] = 0; expect[I[1]] = 6                                          # :868-872 -> IdentityPointError
        badp = torch.tensor(list(((1 << 255) - 19).to_bytes(32, "little")), dtype=torch.uint8, device=dev)
        pv[I[2], 128 + 32 * 77:128 + 32 * 78] = badp; expect[I[2]] = 0x81              # non-canonical field element -> decode error
        pv[I[3], 32 * 132 + 3] ^= 0x40; expect[I[3]] = 7                               # :1701-1708
        one_le = lambda m: le32(torch.ones(m, dtype=torch.int64, device=dev), m)

        def reprove(idx, tokens, charges_le):
            m = int(idx.numel())
            if m:
                pv[idx] = prove(tokens, charges_le, m).view(m, PROOF_BYTES)
            return m
        # same token spent twice with DIFFERENT proofs (same k, other charge and randomness): refund() says Ok, the screen must flag it
        m5 = reprove(I[5], tok_all[I[5] - 1].contiguous(), one_le(int(I[5].numel())))
        # non-canonical scalar encodings (k + l, r_bar + l, gamma0[5] + l): accepted after reduction, nullifier = the reduced k (src/cbor.rs:80-91)
        ell = torch.tensor(list(corpus.ELL.to_bytes(32, "little")), dtype=torch.int64, device=dev)
        k6 = pv[I[6], :32].clone()
        for item in (0, 137, 145):
            v = pv[I[6], 32 * item:32 * item + 32].to(torch.int64) + ell
            for b in range(31):
                v[:, b + 1] += v[:, b] >> 8
                v[:, b] &= 0xff
            assert bool((v[:, 31] < 256).all())
            pv[I[6], 32 * item:32 * item + 32] = v.to(torch.uint8)
        # overspend: the prover runs with s = c + 1 .. c + 100 (src/tests.rs:366-374, 1540-1547) -> InvalidClientSpendProof
        m7 = int(I[7].numel())
        if m7:
            c7 = tok_all[I[7]][:, 128:130].to(torch.int64); c7 = c7[:, 0] + 256 * c7[:, 1]
            reprove(I[7], tok_all[I[7]].contiguous(), le32(c7 + 1 + torch.randint(0, 100, (m7,), device=dev, generator=gen), m7)); expect[I[7]] = 7
        # a token issued under ANOTHER issuer key (src/tests.rs:1997-2033)
        m8 = int(I[8].numel())
        if m8:
            import oracle_lib as O_
            x2, w2 = O_.keygen(corpus.xof(b"bench-other-issuer", 64))
            with act.Engine(params, act.PrivateKey(x2, w2), device=local) as eng2:
                tok8, _ = make_tokens(m8, eng2)
            reprove(I[8], tok8, one_le(m8)); expect[I[8]] = 7
            del tok8
        # token tampering (src/tests.rs:1898-1927): a := another token's A (a valid point), e := random scalar bytes
        m9 = int(I[9].numel())
        if m9:
            tok9 = tok_all[I[9]].clone(); tok9[:, 0:32] = tok_all[I[9] - 1][:, 0:32]; tok9[:, 32:64] = rbytes(m9 * 32).view(m9, 32); tok9[:, 63] &= 0x0f
            reprove(I[9], tok9.contiguous(), one_le(m9)); expect[I[9]] = 7
            del tok9
        pv[I[10], 64] |= 1; expect[I[10]] = 0x81                                       # A': odd ("negative") s -> decode error
        nonsq = torch.tensor(list(bytes.fromhex("26948d35ca62e643e26a83177332e6b6afeb9d08e4268b650f1f5bbd8d81d371")), dtype=torch.uint8, device=dev)
        pv[I[11], 96:128] = nonsq; expect[I[11]] = 0x81                                # B-bar: RFC 9496 A.3 non-square
        # exact replay of the neighbour LAST, so that it copies whatever the neighbour has become (still Ok for refund() if that was)
        src4 = pv[I[4] - 1].clone(); exp4 = expect[I[4] - 1].clone()
        pv[I[4]] = src4; expect[I[4]] = exp4
        del src4
        mixed_step = spend_stepper(nmix, pv_all, rnd_all, m_ref_, m_nul_, m_st_)
        Km = min(K, 3)
        mms = timed(mixed_step, 1, Km)
        st_m = m_st_.clone()
        ok_status = bool((st_m == expect).all())
        ok_nul6 = bool((m_nul_.view(nmix, 32)[I[6]] == k6).all())
        ok_nul5 = bool((m_nul_.view(nmix, 32)[I[5]] == tok_all[I[5] - 1][:, 64:96]).all())
        d_flag = torch.empty_like(m_st_)
        eng.flag_replays_dev(nmix, m_st_.data_ptr(), m_nul_.data_ptr(), 0, None, d_flag.data_ptr(), stream)
        torch.cuda.synchronize()
        import replay_reference                                # tests/: sort-based torch formulation, the semantic reference of the screen
        flag_ref = replay_reference.flag_replays(m_st_, m_nul_)
        ok_flags = bool((d_flag == flag_ref).all())
        replays = int((d_flag == 3).sum().item())
        # oracle re-check: up to 256 of every class + 256 untouched proofs
        per_class = {}
        samp = [torch.nonzero(~sel).view(-1)[:256]]
        for c in range(NCLS):
            samp.append(I[c][:256]); per_class[names[c]] = {"planted": int(I[c].numel()), "oracle_checked": int(min(256, I[c].numel()))}
        samp = torch.cat(samp)
        sp_ = pv[samp].reshape(-1).cpu().numpy(); sr_ = rnd_all.view(nmix, 128)[samp].reshape(-1).cpu().numpy()
        o_refm, o_nulm, o_stm, _ = ctx.batch_refund(sp_, sr_, threads=threads)
        ok_oracle = bool((o_stm == st_m[samp].cpu().numpy()).all() and (o_refm.reshape(-1, 128) == m_ref_.view(nmix, 128)[samp].cpu().numpy()).all()
                         and (o_nulm.reshape(-1, 32) == m_nul_.view(nmix, 32)[samp].cpu().numpy()).all())
        mixed = {"value": world * nmix * Km / (mms * 1e-3), "unit": UNIT, "n_per_gpu": nmix, "steps": Km,
                 "workload": (f"BASELINE configs[4]: {nmix} SpendProofs on one GPU" if world == 1 else f"{nmix} SpendProofs per GPU") + f", {args.mixed_frac:.0%} tampered over {NCLS} classes",
                 "tampered_fraction": float(sel.float().mean().item()), "classes": per_class,
                 "status_matches_expectation": ok_status, "nullifiers_of_accepting_classes_match": ok_nul5 and ok_nul6,
                 "oracle_sample": int(samp.numel()), "oracle_sample_equal_status_refund_nullifier": ok_oracle,
                 "accepted": int((st_m == 0).sum().item()),
                 "rejected_by_status": {str(k): int((st_m == k).sum().item()) for k in (6, 7, 0x81)},
                 "replays_flagged_by_screen": replays, "replay_flags_equal_sort_based_reference": ok_flags,
                 "second_spends_planted": m5, "exact_replays_planted": int(I[4].numel())}
        assert ok_status, "mixed batch: a status differs from the class's expected status"
        assert ok_nul5 and ok_nul6, "mixed batch: nullifier of an accepted tampered class differs"
        assert ok_oracle, "mixed batch: the oracle disagrees with the engine on a sampled proof"
        assert ok_flags, "mixed batch: replay screen differs from the sort-based formulation"
        oracle_checks["mixed_batch_proofs_rechecked_by_oracle"] = int(samp.numel())
        del st_m, d_flag, expect, flag_ref, k6, pv, pv_all, tok_all, rnd_all, m_ref_, m_nul_, m_st_
        torch.cuda.synchronize()
    d_proofs = None
    torch.cuda.empty_cache()

    # ---- strong form of configs[3] (N = 2, 4): the SAME 8M-proof batch split over the GPUs, 8M / N unique proofs per GPU
    # (N = 8 is the weak run itself: 1M per GPU) ----
    strong = None
    per = STRONG_TOTAL // world if world > 1 else 0
    if world > 1 and not args.no_strong and per != n and per * PROOF_BYTES < 100e9:
        t_gen = time.time()
        s_proofs, s_tok, s_rnd = make_spend_batch(per)
        del s_tok
        log(f"[bench] rank {rank}: strong-scaling batch: {per} unique proofs in {time.time() - t_gen:.1f}s")
        s_ref = torch.zeros(per * 128, dtype=torch.uint8, device=dev); s_nul = torch.zeros(per * 32, dtype=torch.uint8, device=dev)
        s_st = torch.zeros(per, dtype=torch.uint8, device=dev)
        Ks = min(K, 2)
        sms_ = timed(spend_stepper(per, s_proofs, s_rnd, s_ref, s_nul, s_st), 1, Ks)
        assert bool((s_st == 0).all())
        strong = {"value": STRONG_TOTAL * Ks / (sms_ * 1e-3), "unit": UNIT, "total_proofs": STRONG_TOTAL, "per_gpu": per, "steps": Ks, "scaling": "strong",
                  "ms_per_step": sms_ / Ks, "workload": f"BASELINE configs[3]: one batch of {STRONG_TOTAL} unique SpendProofs split contiguously over {world} GPUs"}
        del s_proofs, s_rnd, s_ref, s_nul, s_st
        torch.cuda.empty_cache()
    elif world > 1 and per == n:
        strong = {"note": f"at N = {world} the weak run IS the {STRONG_TOTAL}-proof batch of configs[3] ({n} per GPU)"}

    # ---- single-process multi-device leg (N > 1), LAST: rank 0 alone drives every GPU of the box through ONE C-ABI handle
    # (act_engine_create_multi + act_batch_verify_spend_and_refund_screened: shards over per-device replicas, NVLink gather of
    # status + nullifiers to replica 0, replay screen).  The other ranks have nothing left to do and EXIT (code 0) first: an idle
    # process that still holds a CUDA context on a GPU makes the driver time-slice it against rank 0's replica there (measured at
    # N = 4: steps between 1.29 s and 2.08 s with the idle ranks alive, 1.286 s steady from a lone process,
    # profiles/r02m_multi_abi.txt) ----
    multi_abi = None
    if world > 1 and not args.no_multi_abi:
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)
        dist.destroy_process_group()          # every rank: no communicator is left that could notice a peer leaving
        if rank != 0:
            sys.stderr.flush()
            os._exit(0)
        eng.close()
        del d_ref, d_nul, d_st, d_rnd, d_tokens
        torch.cuda.empty_cache()
        time.sleep(8.0)                       # the exited ranks' contexts are torn down by the driver
        box = {}

        def multi_leg():
            try:
                mp_, mr_, ref0 = m_keep
                tot = world * nm
                m_ref = torch.empty(tot * 128, dtype=torch.uint8, pin_memory=True); m_nul = torch.empty(tot * 32, dtype=torch.uint8, pin_memory=True)
                m_st = torch.empty(tot, dtype=torch.uint8, pin_memory=True)
                with act.Engine(params, key, devices=list(range(world))) as meng:
                    def mstep():
                        meng.batch_verify_spend_and_refund_screened_ptr(tot, mp_.data_ptr(), mr_.data_ptr(), 0, None, m_ref.data_ptr(), m_nul.data_ptr(), m_st.data_ptr())
                    mstep(); mstep()
                    msteps = 5
                    step_s = []
                    for _ in range(msteps):
                        t0 = time.perf_counter()
                        mstep()
                        step_s.append(time.perf_counter() - t0)
                    m_s = sum(step_s)
                    med = sorted(step_s)[len(step_s) // 2]
                    stv = m_st.numpy()
                    box["r"] = {"value": tot / med, "unit": UNIT, "n": tot, "steps": msteps, "n_gpus": world, "step_s": [round(t, 4) for t in step_s],
                                 "value_is": "proofs per MEDIAN step (a step now and then is slowed by the tear-down of the exited ranks' contexts)",
                                 "mean_value": tot * msteps / m_s,
                                 "api": "act_engine_create_multi + act_batch_verify_spend_and_refund_screened: one process, one handle, pinned host buffers, "
                                        "shards over per-device replicas, cudaMemcpyPeerAsync gather of status + nullifiers to replica 0, replay screen",
                                 "accepted": int((stv == 0).sum()), "flagged_replays": int((stv == 3).sum()),
                                 "first_shard_equals_rank0_refunds": bool((m_ref[:nm * 128].numpy() == ref0.numpy()).all()),
                                 "note": "run last, after the other ranks have exited; tools/multi_abi_bench.py measures the same call from a "
                                         "lone process (profiles/r02m_multi_abi.txt)"}
                    assert box["r"]["first_shard_equals_rank0_refunds"], "multi-device leg differs from the per-rank leg"
                    assert int((stv == 0).sum()) == tot, "multi-device leg: a valid unique proof was rejected or flagged"
                del mp_, mr_, m_ref, m_nul, m_st

            except Exception as ex:
                box["r"] = {"unavailable": repr(ex)}

        # under a watchdog: whatever happens in this leg, rank 0 still prints its JSON line
        th = threading.Thread(target=multi_leg, daemon=True)
        th.start()
        th.join(timeout=240.0)
        multi_abi = box.get("r") or {"unavailable": "the multi-device leg did not finish within 240 s"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(ctx, base, reqs, os.cpu_count() or 1)

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (256-bit modular integer)",
            "data": "synthetic",
            "config": {"workload": f"batch_verify_spend_and_refund of {n} SpendProofs per GPU (BASELINE configs[2]; x{world} GPUs = configs[3] shape), L=128, bench params",
                       "fixtures": f"{n} unique tokens per GPU requested, issued and spent on the device by the engine's generators (bit-exact with the oracle prover); charges uniform in [1, c-1], c in [20, 1000)",
                       "l2": "inputs (17.6 GB per step) far larger than L2; no flush needed",
                       "collective": "all_gather of status+nullifiers (33 B/proof) inside the step" if world > 1 else "none (single GPU)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": world * n * (PROOF_BYTES + 128), "d2h_bytes_per_step": world * n * 161, "steps": Ke,
                    "api": f"act_batch_verify_spend_and_refund (C ABI, {host_mem} host buffers); refunds byte-identical to the device-resident leg"},
            "issue": {"metric": "issues_per_sec", "value": issue_value, "unit": "issues/s", "ms_per_step": ims / K, "n": ni,
                      "workload": f"batch_issue of {ni} IssuanceRequests per GPU (BASELINE configs[1])",
                      "e2e": {"value": world * ni * Ke / e2e_issue_s, "h2d_bytes_per_step": world * ni * 288, "d2h_bytes_per_step": world * ni * 161},
                      "kernel_ms": issue_kernel_ms,
                      "roofline_frac": LIMB_MACS_PER_ISSUE * ni / (issue_kernel_ms * 1e-3) / peak if issue_kernel_ms else None,
                      "roofline_frac_of_model": LIMB_MACS_PER_ISSUE * ni / (issue_kernel_ms * 1e-3) / peak_model if issue_kernel_ms else None,
                      "work_per_unit": f"{LIMB_MACS_PER_ISSUE:.3g} limb-MACs per request = the executed IMAD.WIDE(.X) lane count of issue_kernel (ncu, profiles/r02f_issue_kernel.txt)"},
            "mixed_adversarial": mixed,
            "strong_scaling": strong,
            "multi_abi": multi_abi,
            "client_checks": client_checks,
            "oracle_checks": oracle_checks,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        real_stdout.write(json.dumps(out) + "\n")
        real_stdout.flush()
    if world > 1 and not args.no_multi_abi:
        sys.stderr.flush()
        os._exit(0)                           # process group already destroyed, engine closed
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
