// act_aux.cuh -- the rows either side of the hot path (SURVEY.md 8f), as HBM-bound byte/index kernels:
//
//  * batch nullifier replay screen (f-2): the reference leaves the double-spend check to the caller
//    (/root/reference src/lib.rs:741-745, examples/act.rs:65-69, NullifierDb in src/tests.rs:28-50).
//    Semantics here = that NullifierDb applied in slice order: among ACCEPTED proofs (status 0) the first
//    occurrence of a nullifier keeps 0, every later one -- and every nullifier present in the caller's
//    `seen` set -- becomes 3 (Error::DoubleSpendError, src/lib.rs:105).  Refund outputs are not touched.
//    Implementation: open-addressing hash table of "lowest index holding this key" (atomicCAS / atomicMin),
//    keys compared in place, so the result is deterministic whatever the thread order.
//
//  * canonical-CBOR fast path (f-3): the encodings ciborium produces for SpendProof / Refund /
//    IssuanceResponse / IssuanceRequest (src/cbor.rs:96-103,153-161,216-268,413-420) are fixed skeletons with
//    32-byte payloads at fixed offsets.  Unpack = compare every skeleton byte, gather the payloads; anything that
//    is not byte-for-byte the canonical skeleton gets status 0xFF and goes to the host's lenient parser
//    (act_pack_*_cbor: indefinite lengths, unknown / duplicate / reordered keys).  Encode = scatter.
#pragma once
#include <stdint.h>

#include "fe25519.cuh"

#define ACT_AUX_NOT_CANONICAL 0xFFu
#define ACT_CBOR_PROOF_LEN 18036
#define ACT_REC_PROOF_LEN 16832

// ---- canonical skeleton of a record type: for every CBOR byte either the expected constant or the record byte it carries
// skel[i] >= 0 : CBOR byte i is payload, = record byte index;  skel[i] < 0 : constant byte (-(int)value - 1)
static inline void act_build_skeleton(int32_t* skel, int kind /* 0 request, 1 response, 2 proof, 3 refund */) {
    size_t pos = 0, rec = 0;
    auto konst = [&](uint8_t v) { skel[pos++] = -(int32_t)v - 1; };
    auto bstr32 = [&]() { konst(0x58); konst(0x20); for (int i = 0; i < 32; i++) skel[pos++] = (int32_t)(rec++); };
    if (kind == 2) {
        konst(0xb1);
        for (int key = 1; key <= 17; key++) {
            konst((uint8_t)key);
            if (key == 5 || key == 14) { konst(0x98); konst(0x80); for (int j = 0; j < 128; j++) bstr32(); }
            else if (key == 15) { konst(0x98); konst(0x80); for (int j = 0; j < 128; j++) { konst(0x82); bstr32(); bstr32(); } }
            else bstr32();
        }
    } else {
        int fields = (kind == 1) ? 5 : 4;
        konst((uint8_t)(0xa0 | fields));
        for (int key = 1; key <= fields; key++) { konst((uint8_t)key); bstr32(); }
    }
}
static inline size_t act_cbor_len(int kind) { return kind == 2 ? 18036 : (kind == 1 ? 176 : 141); }
static inline size_t act_rec_len(int kind) { return kind == 2 ? 16832 : (kind == 1 ? 160 : 128); }

#if defined(__CUDACC__)
// one block per item (grid-stride): every thread walks a strided subset of the CBOR bytes
__global__ void __launch_bounds__(256) cbor_unpack_kernel(size_t n, const int32_t* __restrict__ skel, u32 clen, u32 rlen,
                                                          const u8* __restrict__ cbor, u8* __restrict__ rec, u8* __restrict__ status) {
    __shared__ u32 bad;
    for (size_t it = blockIdx.x; it < n; it += gridDim.x) {
        if (threadIdx.x == 0) bad = 0;
        __syncthreads();
        const u8* src = cbor + it * clen;
        u8* dst = rec + it * rlen;
        u32 mybad = 0;
        for (u32 i = threadIdx.x; i < clen; i += blockDim.x) {
            int32_t s = skel[i];
            u8 b = src[i];
            if (s >= 0) dst[s] = b;
            else if (b != (u8)(-(s + 1))) mybad = 1;
        }
        if (mybad) atomicOr(&bad, 1u);
        __syncthreads();
        if (threadIdx.x == 0) status[it] = bad ? (u8)ACT_AUX_NOT_CANONICAL : (u8)0;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) cbor_encode_kernel(size_t n, const int32_t* __restrict__ skel, u32 clen, u32 rlen,
                                                          const u8* __restrict__ rec, u8* __restrict__ cbor) {
    size_t total = n * clen;
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
        size_t it = g / clen;
        u32 i = (u32)(g - it * clen);
        int32_t s = skel[i];
        cbor[g] = (s >= 0) ? rec[it * rlen + s] : (u8)(-(s + 1));
    }
}

// ---- replay screen ----
#define ACT_RP_EMPTY 0xffffffffu
// key j < n_seen lives in `seen`, key n_seen + i in `nul`
__device__ __forceinline__ const uint4* rp_key(u32 id, u32 n_seen, const uint4* seen, const uint4* nul) {
    return id < n_seen ? seen + 2 * (size_t)id : nul + 2 * (size_t)(id - n_seen);
}
__device__ __forceinline__ bool rp_equal(const uint4* a, const uint4* b) {
    uint4 a0 = a[0], a1 = a[1], b0 = b[0], b1 = b[1];
    return ((a0.x ^ b0.x) | (a0.y ^ b0.y) | (a0.z ^ b0.z) | (a0.w ^ b0.w) | (a1.x ^ b1.x) | (a1.y ^ b1.y) | (a1.z ^ b1.z) | (a1.w ^ b1.w)) == 0;
}
// Keyed PRF over all 32 bytes: SipHash-1-3 under a 128-bit key the engine draws from the OS CSPRNG at creation (tweaked per call).
// Nullifiers are chosen by clients, so an unkeyed or predictable mix would let them aim many accepted proofs at one probe run
// (quadratic probing work inside one launch); under a secret key the slots of distinct nullifiers are unpredictable, and equal
// nullifiers never lengthen a run (they meet their own slot).
struct rp_key128 { u64 k0, k1; };
#define RP_ROTL(x, b) (((x) << (b)) | ((x) >> (64 - (b))))
#define RP_SIPROUND                                                                             \
    do {                                                                                        \
        v0 += v1; v1 = RP_ROTL(v1, 13); v1 ^= v0; v0 = RP_ROTL(v0, 32);                         \
        v2 += v3; v3 = RP_ROTL(v3, 16); v3 ^= v2;                                               \
        v0 += v3; v3 = RP_ROTL(v3, 21); v3 ^= v0;                                               \
        v2 += v1; v1 = RP_ROTL(v1, 17); v1 ^= v2; v2 = RP_ROTL(v2, 32);                         \
    } while (0)
__host__ __device__ __forceinline__ u64 rp_siphash13(const u64 m[4], rp_key128 key) {
    u64 v0 = key.k0 ^ 0x736f6d6570736575ull, v1 = key.k1 ^ 0x646f72616e646f6dull;
    u64 v2 = key.k0 ^ 0x6c7967656e657261ull, v3 = key.k1 ^ 0x7465646279746573ull;
#pragma unroll
    for (int i = 0; i < 4; i++) { v3 ^= m[i]; RP_SIPROUND; v0 ^= m[i]; }
    const u64 last = (u64)32 << 56;   // length byte, no tail bytes
    v3 ^= last; RP_SIPROUND; v0 ^= last;
    v2 ^= 0xff;
    RP_SIPROUND; RP_SIPROUND; RP_SIPROUND;
    return v0 ^ v1 ^ v2 ^ v3;
}
__device__ __forceinline__ u32 rp_hash(const uint4* k, rp_key128 key) {
    uint4 a = k[0], b = k[1];
    u64 m[4] = {(u64)a.x | ((u64)a.y << 32), (u64)a.z | ((u64)a.w << 32), (u64)b.x | ((u64)b.y << 32), (u64)b.z | ((u64)b.w << 32)};
    u64 h = rp_siphash13(m, key);
    return (u32)h ^ (u32)(h >> 32);
}
// insert pass: table[slot] = lowest id whose key hashes there.  ids 0..n_seen-1 are the caller's seen set (always "first").
__global__ void __launch_bounds__(256) replay_insert_kernel(u32 n, u32 n_seen, const u8* __restrict__ status, const uint4* __restrict__ seen,
                                                            const uint4* __restrict__ nul, u32* table, u32 mask, rp_key128 seed) {
    u32 id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= n + n_seen) return;
    if (id >= n_seen && status[id - n_seen] != 0) return;   // only accepted proofs take part
    const uint4* key = rp_key(id, n_seen, seen, nul);
    u32 slot = rp_hash(key, seed) & mask;
    for (;;) {
        u32 cur = table[slot];
        if (cur == ACT_RP_EMPTY) {
            u32 prev = atomicCAS(&table[slot], ACT_RP_EMPTY, id);
            if (prev == ACT_RP_EMPTY) return;
            cur = prev;
        }
        if (rp_equal(rp_key(cur, n_seen, seen, nul), key)) { atomicMin(&table[slot], id); return; }
        slot = (slot + 1) & mask;
    }
}
__global__ void __launch_bounds__(256) replay_resolve_kernel(u32 n, u32 n_seen, const u8* __restrict__ status, const uint4* __restrict__ seen,
                                                             const uint4* __restrict__ nul, const u32* __restrict__ table, u32 mask, rp_key128 seed,
                                                             u8* __restrict__ out) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u8 st = status[i];
    if (st == 0) {
        const uint4* key = nul + 2 * (size_t)i;
        u32 slot = rp_hash(key, seed) & mask;
        for (;;) {
            u32 cur = table[slot];   // never empty before the key is met: it was inserted by the first pass
            if (cur == ACT_RP_EMPTY) break;
            if (rp_equal(rp_key(cur, n_seen, seen, nul), key)) { if (cur != n_seen + i) st = 3; break; }
            slot = (slot + 1) & mask;
        }
    }
    out[i] = st;
}

// ---- per-store screen of a keyed batch: key id -> store index through a map of ACT_KEY_SLOTS bytes (0xFF = no store) ----
#ifndef ACT_KEY_SLOTS
#define ACT_KEY_SLOTS 16
#endif
struct act_store_map { u8 of_slot[ACT_KEY_SLOTS]; };
__device__ __forceinline__ u32 store_of(const act_store_map& m, u8 key_id) { return key_id < ACT_KEY_SLOTS ? m.of_slot[key_id] : 0xFFu; }
// the statuses store j screens: the proofs of other stores (and of no store) get a nonzero status, so they take no part
__global__ void __launch_bounds__(256) store_mask_kernel(size_t n, const u8* __restrict__ status, const u8* __restrict__ key_ids, act_store_map m, u32 j,
                                                         u8* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = store_of(m, key_ids[i]) == j ? status[i] : (u8)0xFF;
}
// store j's outcomes back into the batch's statuses
__global__ void __launch_bounds__(256) store_merge_kernel(size_t n, const u8* __restrict__ screened, const u8* __restrict__ key_ids, act_store_map m, u32 j,
                                                          u8* __restrict__ status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && store_of(m, key_ids[i]) == j) status[i] = screened[i];
}
#endif
