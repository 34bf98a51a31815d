"""Request-level sharding across the GPUs of one box (one process per GPU, torch.distributed).

The hot path has no cross-request arithmetic (the reference's issue/refund take &self and are pure,
/root/reference src/lib.rs:621,781), so a batch shards by contiguous index range with NO data-path
collective.  The only exchange is the gather of per-request status bytes and 32-byte nullifiers
(33 B / proof) so that every rank -- or the caller's nullifier database (src/lib.rs:741-745) -- sees the
whole batch's accept bits.  Works with NCCL on GPU tensors and with gloo on CPU tensors (tests).
"""
import torch
import torch.distributed as dist

_SIDE = {}   # device -> side stream used when torch's current stream is the legacy default stream


def shard_bounds(n, rank, world):
    """Contiguous range [lo, hi) of request indices owned by `rank`; sizes differ by at most one."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_gather_results(status, nullifiers, n_total, group=None):
    """All-gather the per-shard status (uint8[m]) and nullifiers (uint8[m*32]) into whole-batch tensors
    ordered by request index.  Shards may be ragged (shard_bounds)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return status, nullifiers
    sizes = [shard_bounds(n_total, r, world) for r in range(world)]
    mmax = max(hi - lo for lo, hi in sizes)
    pad_s = torch.zeros(mmax, dtype=torch.uint8, device=status.device); pad_s[:status.numel()] = status
    pad_n = torch.zeros(mmax * 32, dtype=torch.uint8, device=status.device); pad_n[:nullifiers.numel()] = nullifiers
    out_s = torch.empty(world * mmax, dtype=torch.uint8, device=status.device)
    out_n = torch.empty(world * mmax * 32, dtype=torch.uint8, device=status.device)
    dist.all_gather_into_tensor(out_s, pad_s, group=group)
    dist.all_gather_into_tensor(out_n, pad_n, group=group)
    if all(hi - lo == mmax for lo, hi in sizes):
        return out_s, out_n
    s = torch.cat([out_s[r * mmax:r * mmax + (hi - lo)] for r, (lo, hi) in enumerate(sizes)])
    nl = torch.cat([out_n[r * mmax * 32:(r * mmax + (hi - lo)) * 32] for r, (lo, hi) in enumerate(sizes)])
    return s, nl


def flag_replays(status, nullifiers, seen=None, engine=None):
    """Caller-side double-spend screen over a gathered batch (the reference leaves this to the caller:
    src/lib.rs:741-745, examples/act.rs:65-69, src/tests.rs:28-50).  Among ACCEPTED proofs (status 0) the first
    occurrence of a nullifier in slice order keeps status 0; later ones -- and any nullifier present in `seen`
    (uint8[k*32] of previously spent nullifiers) -- are flagged 3 (DoubleSpendError).  Refund outputs are not
    touched.  Returns a new status tensor.  Runs the engine's CUDA kernels (act_flag_replays_dev) on CUDA tensors; there is
    no other path in the product (the sort-based torch formulation the tests compare against lives in tests/replay_reference.py)."""
    n = status.numel()
    if n == 0:
        return status.clone()
    if engine is None or not status.is_cuda:
        raise RuntimeError("flag_replays needs the CUDA engine and CUDA tensors (no CPU path)")
    # the CUDA replay screen of the engine (act_flag_replays_dev: hash table of lowest index per key)
    out = torch.empty_like(status)
    status, nullifiers = status.contiguous(), nullifiers.contiguous()
    k = 0 if seen is None else seen.numel() // 32
    seen = seen.contiguous() if k else None
    sp = seen.data_ptr() if k else None
    cur = torch.cuda.current_stream(status.device)
    if cur.cuda_stream != 0:
        engine.flag_replays_dev(n, status.data_ptr(), nullifiers.data_ptr(), k, sp, out.data_ptr(), cur.cuda_stream)
    else:
        # torch is on the legacy default stream, whose handle (0) means "the engine's own stream" in the C ABI: run
        # on a side stream ordered after the producers of the inputs and before the consumers of the result
        side = _SIDE.get(status.device)
        if side is None:
            side = _SIDE[status.device] = torch.cuda.Stream(device=status.device)
        side.wait_stream(cur)
        engine.flag_replays_dev(n, status.data_ptr(), nullifiers.data_ptr(), k, sp, out.data_ptr(), side.cuda_stream)
        for t in (status, nullifiers, out) + ((seen,) if k else ()):
            t.record_stream(side)
        cur.wait_stream(side)
    return out


def screen_with_store(status, nullifiers, store, record=True):
    """The screen of flag_replays against a device-resident NullifierStore in place of `seen`, on torch's current stream; with
    `record` the nullifiers that keep status 0 are inserted into the store.  status uint8[n] and nullifiers uint8[n*32] are CUDA
    tensors on the store's device.  Returns a new status tensor (act_nullifier_store_screen_dev; no CPU path)."""
    n = status.numel()
    if n == 0:
        return status.clone()
    if not status.is_cuda:
        raise RuntimeError("screen_with_store needs CUDA tensors (no CPU path)")
    out = torch.empty_like(status)
    status, nullifiers = status.contiguous(), nullifiers.contiguous()
    cur = torch.cuda.current_stream(status.device)
    if cur.cuda_stream != 0:
        store.screen_dev(n, status.data_ptr(), nullifiers.data_ptr(), out.data_ptr(), record, cur.cuda_stream)
    else:
        # legacy default stream (handle 0 = the store's own stream in the C ABI): side stream ordered both ways, as in flag_replays
        side = _SIDE.get(status.device)
        if side is None:
            side = _SIDE[status.device] = torch.cuda.Stream(device=status.device)
        side.wait_stream(cur)
        store.screen_dev(n, status.data_ptr(), nullifiers.data_ptr(), out.data_ptr(), record, side.cuda_stream)
        for t in (status, nullifiers, out):
            t.record_stream(side)
        cur.wait_stream(side)
    return out
