// act_store.cuh -- the device-resident nullifier store (act_nullifier_store_*): the set of nullifiers already spent, kept in
// HBM between calls so that the issuer's replay screen costs in proportion to the batch, not to the history.
//
// Layout: open addressing over a power-of-two array of 32-byte slots (two uint4), linear probing, load factor <= 1/2.  A slot
// holds the nullifier itself; the empty marker is all 0xFF.  Every key the store accepts is reduced mod l (the engine's
// nullifiers always are; the screen refuses others), so byte 31 <= 0x10 and the last 8-byte word of a key is never all-ones:
// that word alone tells an occupied slot from an empty one, and it is the word an insert claims with atomicCAS.  (The first
// word can be all-ones in a valid key, e.g. the key 2^64 - 1.)  The all-zero nullifier is an ordinary key.
//
// Slot index = SipHash-1-3 (rp_siphash13) of the 32 bytes under the store's secret 128-bit key, masked to the table: 64-bit, so
// the table is bounded by device memory, not by 2^32 slots.  Nullifiers are chosen by clients; under a secret key they cannot
// aim keys at one probe run.
//
// Inserts never compare keys: a recording call inserts only the survivors of its screen, which are distinct and absent from the
// store, and no lookup runs concurrently (stream order).  A thread claims the first empty slot of its probe sequence with
// atomicCAS on the last word and then writes the other 24 bytes; a loser moves on to the next slot.  Nothing waits on another
// thread's write.
#pragma once
#include <stdint.h>

#include "act_aux.cuh"

#define ACT_ST_EMPTY 0xffffffffffffffffull

#if defined(__CUDACC__)
__device__ __forceinline__ void st_words(const uint4* k, u64 m[4]) {
    uint4 a = k[0], b = k[1];
    m[0] = (u64)a.x | ((u64)a.y << 32); m[1] = (u64)a.z | ((u64)a.w << 32);
    m[2] = (u64)b.x | ((u64)b.y << 32); m[3] = (u64)b.z | ((u64)b.w << 32);
}
// key < l = 2^252 + 27742317777372353535851937790883648493 (little-endian 64-bit words, most significant first)
__device__ __forceinline__ bool st_reduced(const u64 m[4]) {
    const u64 l[4] = {0x5812631a5cf5d3edull, 0x14def9dea2f79cd6ull, 0ull, 0x1000000000000000ull};
#pragma unroll
    for (int w = 3; w >= 0; w--) {
        if (m[w] != l[w]) return m[w] < l[w];
    }
    return false;
}
// claim the first empty slot on the probe sequence of m (distinct, absent keys only: see the header comment)
__device__ __forceinline__ void st_claim(uint4* table, u64 mask, rp_key128 key, const u64 m[4]) {
    u64 slot = rp_siphash13(m, key) & mask;
    for (;;) {
        unsigned long long* w3 = reinterpret_cast<unsigned long long*>(table + 2 * slot) + 3;
        if (__ldcg(w3) == ACT_ST_EMPTY && atomicCAS(w3, ACT_ST_EMPTY, (unsigned long long)m[3]) == ACT_ST_EMPTY) {
            u64* s = reinterpret_cast<u64*>(table + 2 * slot);
            s[0] = m[0]; s[1] = m[1]; s[2] = m[2];
            return;
        }
        slot = (slot + 1) & mask;
    }
}

// step 1 of a screen: status-0 keys found in the store get 3, every other status is copied.  Also raises *bad when a status-0
// key is not reduced mod l (the call then fails as a whole before anything is written to the store).
__global__ void __launch_bounds__(256) store_lookup_kernel(u64 n, const u8* __restrict__ status, const uint4* __restrict__ nul,
                                                           const uint4* __restrict__ table, u64 mask, rp_key128 key, u8* __restrict__ out,
                                                           u32* __restrict__ bad) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u8 st = status[i];
    if (st == 0) {
        u64 m[4];
        st_words(nul + 2 * i, m);
        if (!st_reduced(m)) { atomicOr(bad, 1u); out[i] = st; return; }
        u64 slot = rp_siphash13(m, key) & mask;
        for (;;) {
            const uint4* s = table + 2 * slot;
            uint4 a = s[0], b = s[1];
            u64 s3 = (u64)b.z | ((u64)b.w << 32);
            if (s3 == ACT_ST_EMPTY) break;
            u64 s0 = (u64)a.x | ((u64)a.y << 32), s1 = (u64)a.z | ((u64)a.w << 32), s2 = (u64)b.x | ((u64)b.y << 32);
            if (((s0 ^ m[0]) | (s1 ^ m[1]) | (s2 ^ m[2]) | (s3 ^ m[3])) == 0) { st = 3; break; }
            slot = (slot + 1) & mask;
        }
    }
    out[i] = st;
}
// step 3 (recording calls): insert every key whose final status is 0; *count += the number inserted
__global__ void __launch_bounds__(256) store_insert_kernel(u64 n, const u8* __restrict__ status, const uint4* __restrict__ nul, uint4* table,
                                                           u64 mask, rp_key128 key, unsigned long long* count) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    bool mine = i < n && status[i] == 0;
    if (mine) {
        u64 m[4];
        st_words(nul + 2 * i, m);
        st_claim(table, mask, key, m);
    }
    unsigned b = __ballot_sync(0xffffffffu, mine);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(count, (unsigned long long)__popc(b));
}
// growth: every occupied slot of the old table into the new (larger) one, same lock-free insert
__global__ void __launch_bounds__(256) store_rehash_kernel(u64 old_slots, const uint4* __restrict__ old_table, uint4* table, u64 mask, rp_key128 key) {
    u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= old_slots) return;
    u64 m[4];
    st_words(old_table + 2 * j, m);
    if (m[3] != ACT_ST_EMPTY) st_claim(table, mask, key, m);
}
// export: the occupied slots of table[lo, lo + len) packed into out (order unspecified); *count += keys written
__global__ void __launch_bounds__(256) store_compact_kernel(u64 len, const uint4* __restrict__ table, uint4* __restrict__ out,
                                                            unsigned long long* count) {
    u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= len) return;
    uint4 a = table[2 * j], b = table[2 * j + 1];
    if (((u64)b.z | ((u64)b.w << 32)) == ACT_ST_EMPTY) return;
    unsigned long long k = atomicAdd(count, 1ull);
    out[2 * k] = a; out[2 * k + 1] = b;
}
#endif
