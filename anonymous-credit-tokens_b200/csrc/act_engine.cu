// act_engine.cu -- CUDA kernels (sm_100a) and the C-ABI engine of include/act_engine.h.
//
// One engine = one Params on one GPU with up to ACT_KEY_SLOTS issuer keys (one of them selected): generator tables, the secret
// scalars, two CUDA streams and the scratch buffers of the spend pipeline.  Batches are processed in chunks; the
// host-buffer entry points double-buffer H2D / compute / D2H across the two streams.
//
// There is no CPU path: every entry point needs a CUDA device and fails otherwise.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/random.h>

#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/act_engine.h"
#include "act_device.cuh"
#include "act_aux.cuh"
#include "act_prove.cuh"
#include "act_store.cuh"

// ---------------------------------------------------------------------------------------------------
// kernels: thin index wrappers around the per-thread bodies in act_device.cuh
// ---------------------------------------------------------------------------------------------------
// threads per block of the thread-per-request kernels; 512 threads (16 warps, 128 registers each) resident per SM
#ifndef ACT_ISSUE_BLOCK
#define ACT_ISSUE_BLOCK 128
#endif
#ifndef ACT_HEAD_BLOCK
#define ACT_HEAD_BLOCK 64
#endif
#ifndef ACT_SIGN_BLOCK
#define ACT_SIGN_BLOCK 64
#endif
#define ACT_HASH_BLOCK 128
#define ACT_ISSUE_BPS (512 / ACT_ISSUE_BLOCK)
#define ACT_HEAD_BPS (512 / ACT_HEAD_BLOCK)
#define ACT_SIGN_BPS (512 / ACT_SIGN_BLOCK)

__global__ void __launch_bounds__(ACT_ISSUE_BLOCK, ACT_ISSUE_BPS) issue_kernel(const act_ctx* C, size_t n, const u32* req, const u32* cs, const u32* rnd, u32* resp, u8* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) issue_thread(C, i, req, cs, rnd, resp, status);
}
// the two halves of issue for the sequential-RNG contract (act_batch_issue_seq)
__global__ void __launch_bounds__(ACT_ISSUE_BLOCK, ACT_ISSUE_BPS) issue_mode_kernel(const act_ctx* C, size_t n, const u32* req, const u32* cs, const u32* rnd, u32* resp, u8* status,
                                                                       int mode, const u32* rnd_index) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) issue_thread(C, i, req, cs, rnd, resp, status, mode, rnd_index);
}
__global__ void __launch_bounds__(ACT_SIGN_BLOCK, ACT_SIGN_BPS) refund_sign_seq_kernel(const act_ctx* C, size_t n, const u32* proofs, const u32* rnd, const u32* kprime, const u8* status,
                                                                           u32* refunds, u32* nullifiers, const u32* rnd_index, const u32* kwords) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) refund_sign_thread(C, p, proofs, rnd, kprime, status, refunds, nullifiers, rnd_index, kwords);
}
__global__ void __launch_bounds__(ACT_ISSUE_BLOCK, ACT_ISSUE_BPS) issuance_check_kernel(const act_ctx* C, size_t n, const u32* K, const u32* resp, u8* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) issuance_check_thread(C, i, K, resp, status);
}
// The range kernel: a thread owns one com_j and the pair C'_j0, C'_j1; a warp owns 32 consecutive j of one proof.  The grid
// is persistent and sized to the machine (SMs x resident blocks), so the per-thread window tables live in a scratch buffer
// indexed by (block, thread) whose size does not depend on the batch.
#ifndef ACT_RANGE_BLOCKS_PER_SM
#define ACT_RANGE_BLOCKS_PER_SM 4   // 128 registers per thread; measured 153k vs 146k proofs/s at 3
#endif
// Work distribution: the unit of work is one warp's quarter of a proof (32 of its 128 com_j).  Every resident warp draws
// the next unit from a per-launch counter.  Measured on B200 (profiles/r01i_range_trace.txt): with a static grid-stride
// assignment of whole proofs to blocks, the warps of one SM finish the SAME amount of work between 60 ms and 96 ms after
// launch -- the warp scheduler is not fair between warps -- so on average only 79 % of the launched warps were resident;
// drawing units on demand keeps 98 % resident (a favoured warp simply draws up to 3x the units of a starved one) and
// evens out whatever else differs between warps.  ACT_RANGE_DYNAMIC=0 is the static form (block = 128 only).
#ifndef ACT_RANGE_DYNAMIC
#define ACT_RANGE_DYNAMIC 1
#endif
// threads per block of the range kernel (a multiple of 32; the unit of work is a warp, so any block size works in the
// dynamic form) and resident blocks per SM
#ifndef ACT_RANGE_BLOCK
#define ACT_RANGE_BLOCK 128
#endif
#if !ACT_RANGE_DYNAMIC && ACT_RANGE_BLOCK != ACT_L
#error "the static work distribution needs one block per proof"
#endif
#define ACT_RANGE_UNITS (ACT_L / 32)    // units per proof
#if ACT_RANGE_TRACE
__device__ unsigned long long act_trace_buf[4096 * 4];   // per warp: smid, first/last globaltimer, units
__device__ __forceinline__ unsigned long long act_gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#endif
#ifdef ACT_RANGE_MAXREG   // explicit register cap instead of a resident-block target (block sizes of 32/64 threads)
#define ACT_RANGE_BOUNDS __maxnreg__(ACT_RANGE_MAXREG)
#else
#define ACT_RANGE_BOUNDS __launch_bounds__(ACT_RANGE_BLOCK, ACT_RANGE_BLOCKS_PER_SM)
#endif
__global__ void ACT_RANGE_BOUNDS spend_range_kernel(const act_ctx* C, size_t m, const u32* proofs, u32* items, u32* com_niels, u32* flags, vb_table* tabs, u32* cpts, u32* counter) {
    vb_table* mine = tabs + ((size_t)blockIdx.x * ACT_RANGE_BLOCK + threadIdx.x) * ACT_RANGE_SPLIT;
#if ACT_RANGE_TRACE
    unsigned long long t0 = act_gtime(), units = 0;
#endif
#if ACT_RANGE_DYNAMIC
    const u32 lane = threadIdx.x & 31u, total = (u32)m * ACT_RANGE_UNITS;
    for (;;) {
        u32 unit = 0;
        if (lane == 0) unit = atomicAdd(counter, 1u);
        unit = __shfl_sync(0xffffffffu, unit, 0);
        if (unit >= total) break;
        spend_range_thread(C, unit / ACT_RANGE_UNITS, (int)((unit % ACT_RANGE_UNITS) * 32 + lane), proofs, items, com_niels, flags, mine, cpts);
#if ACT_RANGE_TRACE
        units++;
#endif
    }
#else
    (void)counter;
    for (size_t p = blockIdx.x; p < m; p += gridDim.x) {
        spend_range_thread(C, p, threadIdx.x, proofs, items, com_niels, flags, mine, cpts);
#if ACT_RANGE_TRACE
        units++;
#endif
    }
#endif
#if ACT_RANGE_TRACE
    if ((threadIdx.x & 31) == 0) {
        unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        unsigned w = blockIdx.x * (ACT_RANGE_BLOCK / 32) + threadIdx.x / 32;
        if (w < 4096) { act_trace_buf[4 * w] = smid; act_trace_buf[4 * w + 1] = t0; act_trace_buf[4 * w + 2] = act_gtime(); act_trace_buf[4 * w + 3] = units; }
    }
#endif
}
#if ACT_RANGE_TRACE
// dev tool (tools/trace_range.py): not part of the ABI, only present in builds with -DACT_RANGE_TRACE=1
extern "C" __attribute__((visibility("default"))) int act_debug_read_trace(unsigned long long* out, size_t n) {
    return (int)cudaMemcpyFromSymbol(out, act_trace_buf, n * sizeof(unsigned long long));
}
#endif
// encodes the 256 commitments of each proof: one thread per 16 points (batched inversion)
#define ACT_ENC_BLOCK 128
#define ACT_ENC_PARTS (2 * ACT_L / ACT_ENC_BATCH)
__global__ void __launch_bounds__(ACT_ENC_BLOCK, 4) spend_encode_kernel(const act_ctx* C, size_t m, const u32* cpts, u32* items, int pts, int item0) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int parts = pts / ACT_ENC_BATCH;
    if (t < m * parts) spend_encode_thread(C, t / parts, (int)(t % parts), cpts, items, pts, item0);
}
// ---- client-side generators (act_prove.cuh) ----
__global__ void __launch_bounds__(ACT_L, 4) prove_range_kernel(const act_ctx* C, prove_rng R, size_t m, const u32* tokens, const u32* charges, u32* cpts) {
    for (size_t p = blockIdx.x; p < m; p += gridDim.x) prove_range_thread(C, &R, p, p, threadIdx.x, tokens, charges, cpts);
}
__global__ void __launch_bounds__(ACT_HEAD_BLOCK, ACT_HEAD_BPS) prove_head_kernel(const act_ctx* C, prove_rng R, size_t m, const u32* tokens, u32* items, u32* aux, u8* status) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < m) prove_head_thread(C, &R, p, p, tokens, items, aux, status);
}
__global__ void __launch_bounds__(ACT_HASH_BLOCK) prove_challenge_kernel(size_t m, const u32* cvs, u32* gammas) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < m) prove_challenge_thread(p, cvs, gammas);
}
__global__ void __launch_bounds__(ACT_L, 4) prove_finish_kernel(const act_ctx* C, prove_rng R, size_t m, const u32* tokens, const u32* charges, const u32* items,
                                                               const u32* aux, const u32* gammas, const u8* status, u32* proofs, u32* prerefunds) {
    for (size_t p = blockIdx.x; p < m; p += gridDim.x) prove_finish_thread(C, &R, p, p, threadIdx.x, tokens, charges, items, aux, gammas, status, proofs, prerefunds);
}
__global__ void __launch_bounds__(ACT_ISSUE_BLOCK, ACT_ISSUE_BPS) request_kernel(const act_ctx* C, size_t n, const u32* pre, const u32* rnd, u32* req) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) request_thread(C, i, pre, rnd, req);
}
__global__ void __launch_bounds__(ACT_HEAD_BLOCK, ACT_HEAD_BPS) spend_head_kernel(const act_ctx* C, size_t n, const u32* proofs, u32* items, const u32* com_niels, u32* kprime, u32* flags, u32* cpts) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) spend_head_thread(C, p, proofs, items, com_niels, kprime, flags, cpts);
}
// the keyed form: proof p is verified under the key of slot key_ids[p] (slots: ACT_KEY_SLOTS contexts, null = empty)
__global__ void __launch_bounds__(ACT_HEAD_BLOCK, ACT_HEAD_BPS) spend_head_keyed_kernel(const act_ctx* C, size_t n, const u32* proofs, u32* items, const u32* com_niels, u32* kprime,
                                                                                     u32* flags, u32* cpts, const u8* key_ids, const act_ctx* const* slots) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) spend_head_thread<true>(C, p, proofs, items, com_niels, kprime, flags, cpts, key_ids, slots);
}
__global__ void __launch_bounds__(ACT_HASH_BLOCK) spend_chunk_kernel(const act_ctx* C, size_t n, const u32* items, u32* cvs) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n * ACT_SPEND_CHUNKS) spend_chunk_thread(C, t / ACT_SPEND_CHUNKS, (int)(t % ACT_SPEND_CHUNKS), items, cvs);
}
__global__ void __launch_bounds__(ACT_HASH_BLOCK) spend_finish_kernel(const act_ctx* C, size_t n, const u32* proofs, const u32* cvs, const u32* flags, u8* status) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) spend_finish_thread(C, p, proofs, cvs, flags, status);
}
__global__ void __launch_bounds__(ACT_SIGN_BLOCK, ACT_SIGN_BPS) refund_sign_kernel(const act_ctx* C, size_t n, const u32* proofs, const u32* rnd, const u32* kprime, const u8* status, u32* refunds, u32* nullifiers) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) refund_sign_thread(C, p, proofs, rnd, kprime, status, refunds, nullifiers);
}
__global__ void __launch_bounds__(ACT_HEAD_BLOCK, ACT_HEAD_BPS) refund_check_kernel(const act_ctx* C, size_t n, const u32* com, const u32* refund, u8* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) refund_check_thread(C, i, com, refund, status);
}

// nullifiers of a verification-only pass: item 0 of the transcript is the reduced k (src/lib.rs:720-722); zero for rejected proofs
__global__ void __launch_bounds__(256) nullifier_kernel(size_t n, const u32* items, const u8* status, u32* nullifiers) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * 8) return;
    size_t p = t >> 3;
    nullifiers[t] = status[p] == ACT_ST_OK ? items[(size_t)ACT_ITEM_WORDS * p + (t & 7)] : 0u;
}
// Overwrites the local memory (stack frames, register spills) the signing kernels left behind: local memory is carved per
// resident thread slot out of one per-context pool and is NOT cleared between kernels, so a later kernel of the same process
// could read spilled fragments of alpha or (e+x)^-1.  Every thread slot of the machine (SMs x 2048) writes zeros over a frame
// larger than any kernel's in this library (ptxas.log: 8.6 KB for issue_kernel).
#define ACT_SCRUB_WORDS 3072
__global__ void __launch_bounds__(1024, 2) scrub_local_kernel(u32* sink) {
    volatile u32 frame[ACT_SCRUB_WORDS];
#pragma unroll 1
    for (int i = 0; i < ACT_SCRUB_WORDS; i++) frame[i] = 0u;
    if (sink && frame[threadIdx.x % ACT_SCRUB_WORDS] != 0u) *sink = 1u;   // keeps the frame alive; never true
}

// ---- set-up kernels ----
__global__ void params_derive_kernel(const u8* dom, u32 dlen, u32* out) {
    if (blockIdx.x == 0 && threadIdx.x == 0) params_derive_thread(dom, dlen, out);
}
// decodes H1,H2,H3,W into bases[1..4] (and W); bases[0] = G.  ok[0] = all valid
__global__ void setup_decode_kernel(const u32* enc /* 4 x 8 words: H1,H2,H3,W */, ge* bases /* ACT_FB_BASES */, ge* W, u32* ok) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        u32 v = 1;
        bases[0] = ge_basepoint();
        for (int i = 0; i < 4; i++) v &= ristretto_decode_(&bases[1 + i], enc + 8 * i);
        *W = bases[ACT_BASE_W];
        *ok = v;
    }
}
// the wide-window tables of G, H1, H2, H3: one thread per (base, window, part)
struct fb_layout { u32 bits[ACT_FB_BASES]; u32 first_thread[ACT_FB_BASES + 1]; size_t offset[ACT_FB_BASES]; };
__global__ void build_fb_tables_kernel(const ge* bases, ge_niels* tabs, fb_layout L) {
    u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= L.first_thread[ACT_FB_BASES]) return;
    int base = 0;
    while (t >= L.first_thread[base + 1]) base++;
    u32 r = t - L.first_thread[base], parts = fb_parts_of(L.bits[base]);
    build_fb_table_thread(&bases[base], L.bits[base], (int)(r / parts), (int)(r % parts), tabs + L.offset[base]);
}
static fb_layout make_fb_layout(size_t* total_entries) {
    fb_layout L;
    const u32 bits[ACT_FB_BASES] = {ACT_FB_BITS, ACT_FB_BITS_HOT, ACT_FB_BITS, ACT_FB_BITS_HOT, ACT_FB_BITS};   // G, H1, H2, H3, W
    size_t off = 0; u32 th = 0;
    for (int b = 0; b < ACT_FB_BASES; b++) {
        L.bits[b] = bits[b]; L.offset[b] = off; L.first_thread[b] = th;
        off += fb_size_of(bits[b]); th += fb_win_of(bits[b]) * fb_parts_of(bits[b]);
    }
    L.first_thread[ACT_FB_BASES] = th;
    *total_entries = off;
    return L;
}
__global__ void build_ct_table_kernel(const ge* bases, ge_niels* tab) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ACT_CT_WIN) build_table_thread<4, ACT_CT_ENT>(&bases[0], t, tab);
}
// reduce the stored secret mod l once and precompute W/2
// ... and check that the public key given is the public key of the secret: ok = (encode(G*x) == encode(W))
__global__ void finalize_ctx_kernel(act_ctx* C, const u32* w_enc, u32* ok) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        ctx_finalize_thread(C);
        ge W = fb_accumulate_ct(ge_identity(), C->ct_g, C->x);
        u32 enc[8], same = 1;
        ristretto_encode_(enc, &W);
        for (int i = 0; i < 8; i++) same &= (enc[i] == w_enc[i]);
        *ok = same;
    }
}
__global__ void public_key_kernel(const ge_niels* ct_g, const u32* x, u32* out) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        sc s = sc_from_words(x);
        ge W = fb_accumulate_ct(ge_identity(), ct_g, s);
        ristretto_encode_(out, &W);
    }
}

// ---- device self-test: PTX field arithmetic against the portable formulation, plus known answers ----
__device__ void selftest_mul_portable(u32* r, const fe& a, const fe& b) {
    for (int i = 0; i < 16; i++) r[i] = 0;
    for (int i = 0; i < 8; i++) {
        u64 c = 0;
        for (int j = 0; j < 8; j++) { c += (u64)a.v[j] * b.v[i] + r[i + j]; r[i + j] = (u32)c; c >>= 32; }
        r[i + 8] = (u32)c;
    }
}
__device__ u32 selftest_rng(u32& s) { s ^= s << 13; s ^= s >> 17; s ^= s << 5; return s; }
__global__ void selftest_kernel(u32* fail) {
    u32 seed = 0x9e3779b9u * (blockIdx.x * blockDim.x + threadIdx.x + 1);
    u32 bad = 0;
    for (int it = 0; it < 64; it++) {
        fe a, b;
        for (int i = 0; i < 8; i++) { a.v[i] = selftest_rng(seed); b.v[i] = selftest_rng(seed); }
        if (it % 8 == 1) for (int i = 0; i < 8; i++) a.v[i] = 0xffffffffu;
        if (it % 8 == 2) for (int i = 0; i < 8; i++) b.v[i] = 0xffffffffu;
        if (it % 8 == 3) for (int i = 1; i < 8; i++) a.v[i] = 0;
        // mul: compare canonical(PTX product) with canonical(portable product reduced by the generic path)
        u32 r[16], t[9];
        selftest_mul_portable(r, a, b);
        u64 c = 0;
        for (int i = 0; i < 8; i++) { c += (u64)r[i] + (u64)r[8 + i] * 38u; t[i] = (u32)c; c >>= 32; }
        u64 c2 = c * 38u;
        fe ref;
        for (int i = 0; i < 8; i++) { c2 += t[i]; ref.v[i] = (u32)c2; c2 >>= 32; }
        ref.v[0] += (u32)c2 * 38u;  // cannot carry: value wrapped
        fe got = fe_mul(a, b);
        if (!fe_eq(got, ref)) bad |= 1;
        // add / sub consistency with big-int emulation through canon: (a+b)-b == a, (a-b)+b == a
        if (!fe_eq(fe_sub(fe_add(a, b), b), a)) bad |= 2;
        if (!fe_eq(fe_add(fe_sub(a, b), b), a)) bad |= 4;
        // a * a^-1 == 1 (skip zero)
        if (!fe_is_zero(a)) { if (!fe_eq(fe_mul(a, fe_invert(a)), fe_one())) bad |= 8; }
        if (!fe_eq(fe_sq(a), fe_mul(a, a))) bad |= 16;
        // products are tight, and the one-pass sum / double of two products agree with the general add
        fe sq = fe_sq(a);
        if (!fe_is_tight_(got) || !fe_is_tight_(sq)) bad |= 256;
        if (!fe_eq(fe_add_tt(got, sq), fe_add(got, sq)) || !fe_eq(fe_dbl_tt(got), fe_add(got, got))) bad |= 512;
        // the wrap-around branch of the tight operations: operands at the top of the tight range
        fe hi1 = fe_zero(), hi2 = fe_zero();
        hi1.v[7] = 0x80000000u; hi1.v[0] = 2047u - (u32)(it & 31);            // 2^255 + (2047 - k)
        hi2.v[7] = 0x7fffffffu; for (int i = 0; i < 7; i++) hi2.v[i] = 0xffffffffu - (u32)(it * i);   // just below 2^255
        if (!fe_eq(fe_add_tt(hi1, hi2), fe_add(hi1, hi2)) || !fe_eq(fe_add_tt(hi1, hi1), fe_add(hi1, hi1))) bad |= 1024;
        if (!fe_eq(fe_dbl_tt(hi1), fe_add(hi1, hi1)) || !fe_eq(fe_dbl_tt(hi2), fe_add(hi2, hi2))) bad |= 2048;
        // the variable-time add / sub forms (public data) equal the two-pass forms word for word: on random operands and on
        // operands that take the out-of-line branch (single ripple, and the ripple that wraps a second time)
        {
            fe x[6], y[6];
            x[0] = a; y[0] = b;
            for (int i = 0; i < 8; i++) { x[1].v[i] = 0xffffffffu; y[1].v[i] = b.v[i]; }
            y[1].v[0] = 0xfffffff0u - (u32)(it & 7);                                      // sum wraps, low word lands within 38 of 2^32
            x[2] = x[1]; for (int i = 0; i < 8; i++) y[2].v[i] = 0xffffffffu; y[2].v[0] = 0xfffffff0u + (u32)(it & 7);   // ... and ripples to the top
            x[3] = fe_zero(); x[3].v[0] = 5u + (u32)(it & 7); for (int i = 0; i < 8; i++) y[3].v[i] = 0xffffffffu;      // difference borrows twice
            x[4] = a; x[4].v[0] = (u32)(it & 31); x[4].v[7] &= 0x7fffffffu; y[4] = fe_zero(); y[4].v[7] = 0x80000000u | b.v[7];   // one borrow, low word below 38
            x[5] = fe_zero(); y[5] = fe_zero(); y[5].v[0] = 1u + (u32)(it & 1);           // 0 - 1, 0 - 2
            for (int k = 0; k < 6; k++) {
                fe s1 = fe_add_v(x[k], y[k]), s2 = fe_add(x[k], y[k]), d1 = fe_sub_v(x[k], y[k]), d2 = fe_sub(x[k], y[k]);
                fe e1 = fe_sub_v(y[k], x[k]), e2 = fe_sub(y[k], x[k]);
                for (int i = 0; i < 8; i++) if (s1.v[i] != s2.v[i] || d1.v[i] != d2.v[i] || e1.v[i] != e2.v[i]) bad |= 4096;
            }
            // the point operations instantiated for public data equal the branch-free instances on the same (arbitrary) coordinates,
            // with operands that make their first sums / differences take the rare paths in either order
            for (int k = 0; k < 12; k++) {
                ge P; P.X = (k & 1) ? y[k >> 1] : x[k >> 1]; P.Y = (k & 1) ? x[k >> 1] : y[k >> 1]; P.Z = a; P.T = b;
                ge_cached Q; Q.YpX = b; Q.YmX = a; Q.Z = x[0]; Q.T2d = y[4];
                ge_niels N; N.ypx = a; N.ymx = y[4]; N.xy2d = b;
                ge r1 = ge_dbl_u<true>(P, true), r2 = ge_dbl_u<false>(P, true);
                ge r3 = ge_add_cached_u<true>(P, Q, (u32)(k & 1), true), r4 = ge_add_cached_u<false>(P, Q, (u32)(k & 1), true);
                ge r5 = ge_add_niels_n<true>(P, N, (u32)(k & 1)), r6 = ge_add_niels_n<false>(P, N, (u32)(k & 1));
                if (!(fe_eq(r1.X, r2.X) & fe_eq(r1.Y, r2.Y) & fe_eq(r1.Z, r2.Z) & fe_eq(r1.T, r2.T))) bad |= 8192;
                if (!(fe_eq(r3.X, r4.X) & fe_eq(r3.Y, r4.Y) & fe_eq(r3.Z, r4.Z) & fe_eq(r3.T, r4.T))) bad |= 8192;
                if (!(fe_eq(r5.X, r6.X) & fe_eq(r5.Y, r6.Y) & fe_eq(r5.Z, r6.Z) & fe_eq(r5.T, r6.T))) bad |= 8192;
            }
        }
    }
    // basepoint encodes to the RFC 9496 generator
    {
        const u32 gen[8] = {0x0aaef2e2u, 0x714ebc6au, 0x61a984a8u, 0x5f5100c5u, 0x6a0be358u, 0x8ddd82a5u, 0x4559a6b6u, 0x762d8de0u};
        ge B = ge_basepoint();
        u32 w[8];
        ristretto_encode_(w, &B);
        for (int i = 0; i < 8; i++) if (w[i] != gen[i]) bad |= 32;
        ge D;
        if (!ristretto_decode_(&D, gen)) bad |= 64;
        ristretto_encode_(w, &D);
        for (int i = 0; i < 8; i++) if (w[i] != gen[i]) bad |= 128;
    }
    if (bad) atomicOr(fail, bad);
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(const char* what, cudaError_t e) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return -2;
}
static int fail_msg(const char* what) { g_err = what; return -1; }
#define CK(call)                                       \
    do {                                               \
        cudaError_t e_ = (call);                       \
        if (e_ != cudaSuccess) return fail(#call, e_); \
    } while (0)
// returns the nonzero result of a call that reports its own error
#define TRY(call)              \
    do {                       \
        int rc_ = (call);      \
        if (rc_) return rc_;   \
    } while (0)

// One device allocation and its size in bytes.  The destructor frees it; it can be moved but not copied.  Create and destroy it
// with its device current.  It converts to T*, so it passes to kernels and copies as the pointer itself.
template <typename T>
struct dev_buf {
    T* p = nullptr;
    size_t bytes = 0;
    dev_buf() = default;
    dev_buf(const dev_buf&) = delete;
    dev_buf(dev_buf&& o) noexcept { *this = std::move(o); }
    dev_buf& operator=(dev_buf&& o) noexcept { std::swap(p, o.p); std::swap(bytes, o.bytes); return *this; }   // o frees what was here
    ~dev_buf() { if (p) cudaFree(p); }
    operator T*() const { return p; }
};
// Gives `b` at least `bytes` bytes; the contents are not kept.  `drain` (if not null) is synchronised before the old buffer is
// freed, for work queued there that may still read it.  A failed allocation leaves `b` empty and clears the runtime's last error,
// which the next launch check on this thread would otherwise report.
template <typename T>
static int ensure(dev_buf<T>& b, size_t bytes, cudaStream_t drain = nullptr) {
    if (b.bytes >= bytes) return 0;
    if (drain) CK(cudaStreamSynchronize(drain));
    b = dev_buf<T>();
    cudaError_t e = cudaMalloc((void**)&b.p, bytes);
    if (e != cudaSuccess) {
        b.p = nullptr;
        cudaGetLastError();
        return fail(("cudaMalloc(" + std::to_string(bytes) + " bytes)").c_str(), e);
    }
    b.bytes = bytes;
    return 0;
}
// Zero-fills a device buffer that held secret material, on `st`, and waits for it: on every way out of the scope that declares
// it.  A path that has already queued the wipe in its own stream order sets p to null.
struct wipe_dev_on_exit {
    void* p; size_t n; cudaStream_t st;
    ~wipe_dev_on_exit() { if (p) { cudaMemsetAsync(p, 0, n, st); cudaStreamSynchronize(st); } }
};

// Proofs per pipeline chunk (default; act_engine_set_spend_chunk or the environment variable ACT_SPEND_CHUNK change it per
// engine).  The thread-per-proof stages (head, sign) need about 2 368 warps to fill the machine (148 SMs x 16 warps at 128
// registers): 65 536 proofs per chunk give 2 048.  Round 1 used 16 384 (3.5 warps per SM in those stages:
// profiles/r01g_other_kernels.txt); measured on 262 144 proofs (profiles/r02a_chunk_size.txt): 200.6k proofs/s at 16 384,
// 204.1k at 32 768, 204.8k at 65 536, 205.2k at 131 072.
#ifndef ACT_SPEND_CHUNK
#define ACT_SPEND_CHUNK 65536
#endif
#define ACT_SMALL_CHUNK 262144  // requests per chunk for the light-weight paths

struct spend_scratch {
    dev_buf<u32> items, com_niels, kprime, flags, cvs;
    dev_buf<u32> cpts;          // half-commitments C'/2 in extended coordinates: m x 256 x 128 B
    dev_buf<vb_table> tabs;     // window tables of the range kernel: grid x 128 threads x ACT_RANGE_SPLIT
    dev_buf<u32> counter;       // work counter of the range kernel (units drawn so far in the current launch)
    unsigned range_grid = 0;
    // recorded after every pipeline that used this scratch set; the next user (possibly on another stream) waits on it
    cudaEvent_t done = nullptr; bool used = false;
};
struct io_slot {  // device staging for the host-buffer entry points, indexed like host_io (st: status)
    dev_buf<u8> in[3], out[2], st;
};

// One issuer key: its device context -- the shared tables of the engine, its own x, W, W/2 and W table -- and that W table.
// The creation key's W table lies in the engine's d_tables; a key installed later has one of its own (2^13 wide, 7.9 MB).
struct key_slot {
    dev_buf<act_ctx> ctx;
    dev_buf<ge_niels> w_table;
};

#define ACT_IO_SLOTS 3
struct act_engine {
    int device = 0;
    cudaStream_t stream[2] = {nullptr, nullptr};
    cudaEvent_t fork = nullptr, join[2] = {nullptr, nullptr};
    key_slot key[ACT_KEY_SLOTS];      // slot 0 holds the creation key
    int selected = 0;                 // the slot every single-key entry point uses
    dev_buf<const act_ctx*> d_slots;  // ctx of every slot, null when empty: what the keyed head reads
    act_ctx pub;                      // host template of a slot's context: table pointers, H encodings, prefixes; no key
    dev_buf<ge_niels> d_tables;
    dev_buf<ge> d_bases;
    spend_scratch scratch[2];
    // host-buffer entry points: ACT_IO_SLOTS staging sets filled on a copy stream of their own, so that the H2D of chunk
    // i+1 is already under way while chunk i computes and chunk i-1 drains (the two compute streams alternate as before)
    io_slot io[ACT_IO_SLOTS];
    cudaStream_t copy = nullptr;
    cudaEvent_t io_ready[ACT_IO_SLOTS] = {}, io_done[ACT_IO_SLOTS] = {};
    uint64_t launches = 0;
    size_t spend_chunk = ACT_SPEND_CHUNK;
    // multi-device engine (act_engine_create_multi): one single-device engine per GPU; host-buffer calls shard over them
    std::vector<act_engine*> replicas;
    // device copy of a call's status + nullifiers (33 B per proof), kept when a screened multi-device call asks for it:
    // what the NVLink gather to replica 0 reads (act_batch_verify_spend_and_refund_screened)
    dev_buf<u8> g_st, g_nul; bool g_keep = false;
    dev_buf<int32_t> d_skel[4];                        // canonical CBOR skeletons (request, response, proof, refund)
    dev_buf<u32> d_rp_table;                           // replay-screen hash table
    rp_key128 rp_key = {0, 0}; uint64_t rp_calls = 0;  // its PRF key (OS CSPRNG, drawn at creation) and a per-call tweak
    // prover scratch (one chunk): transcript items, half-points, chunk CVs, challenges, r3
    dev_buf<u32> pv_items, pv_cpts, pv_cvs, pv_gammas, pv_aux;
    // optional per-kernel device timing (CUDA events on the launching stream)
    bool timing = false;
    struct timed { int kind; cudaEvent_t a, b; };
    std::vector<timed> events;
};
static inline bool is_multi(const act_engine* e) { return !e->replicas.empty(); }
static inline act_ctx* sel_ctx(const act_engine* e) { return e->key[e->selected].ctx; }
#define NOT_MULTI(e, what) do { if (is_multi(e)) return fail_msg(what ": device-buffer calls need a single-device engine (act_engine_replica)"); } while (0)
// call(replica, first index of its shard, shard length) on every replica, each from its own host thread: contiguous shards
// (bounds of sharding.shard_bounds), no cross-GPU arithmetic (SURVEY 8e)
// first index of shard g of G: sizes differ by at most one, the first n % G shards take the extra request (sharding.shard_bounds)
static inline size_t shard_lo(size_t n, size_t g, size_t G) { size_t base = n / G, rem = n % G; return g * base + (g < rem ? g : rem); }
template <typename F>
static int shard_over(const std::vector<act_engine*>& reps, size_t n, F call) {
    size_t G = reps.size();
    std::vector<int> rcs(G, 0);
    std::vector<std::string> errs(G);
    std::vector<std::thread> th;
    for (size_t g = 0; g < G; g++) {
        size_t lo = shard_lo(n, g, G), hi = shard_lo(n, g + 1, G);
        th.emplace_back([&, g, lo, hi] {
            rcs[g] = hi > lo ? call(reps[g], lo, hi - lo) : 0;
            if (rcs[g]) errs[g] = g_err;
        });
    }
    for (auto& t : th) t.join();
    for (size_t g = 0; g < G; g++) if (rcs[g]) { g_err = "replica " + std::to_string(g) + " (device " + std::to_string(reps[g]->device) + "): " + errs[g]; return rcs[g]; }
    return 0;
}
template <typename F>
static int shard_over_replicas(act_engine* e, size_t n, F call) { return shard_over(e->replicas, n, call); }

enum { K_RANGE = 0, K_HEAD, K_CHUNK, K_FINISH, K_SIGN, K_ISSUE, K_ISSUANCE_CHECK, K_REFUND_CHECK, K_ENCODE, K_KINDS };

// LAUNCH(e, kind, stream, kernel<<<...>>>(...)) : counts the launch and, when timing is on, brackets it with events
#define LAUNCH(e, kind, st, ...)                                                              \
    do {                                                                                      \
        act_engine::timed t_{kind, nullptr, nullptr};                                         \
        if ((e)->timing) { cudaEventCreate(&t_.a); cudaEventCreate(&t_.b); cudaEventRecord(t_.a, st); } \
        __VA_ARGS__;                                                                          \
        if ((e)->timing) { cudaEventRecord(t_.b, st); (e)->events.push_back(t_); }            \
        (e)->launches += 1;                                                                   \
    } while (0)

// one scratch set for chunks of up to n proofs
static int ensure_scratch(spend_scratch* s, size_t n) {
    if (!s->range_grid) {
        int dev = 0, sms = 0, per_sm = 0;
        CK(cudaGetDevice(&dev));
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, spend_range_kernel, ACT_RANGE_BLOCK, 0));
        if (per_sm < 1) per_sm = 1;
        s->range_grid = (unsigned)(sms * per_sm);
    }
    TRY(ensure(s->tabs, (size_t)s->range_grid * ACT_RANGE_BLOCK * ACT_RANGE_SPLIT * sizeof(vb_table)));
    TRY(ensure(s->counter, 4));
    if (!s->done) CK(cudaEventCreateWithFlags(&s->done, cudaEventDisableTiming));
    TRY(ensure(s->cpts, n * 2 * ACT_L * 128));
    TRY(ensure(s->items, n * ACT_ITEM_WORDS * 4));
    TRY(ensure(s->com_niels, n * ACT_L * 96));
    TRY(ensure(s->kprime, n * 128));
    TRY(ensure(s->flags, n * 4));
    TRY(ensure(s->cvs, n * ACT_SPEND_CHUNKS * 32));
    return 0;
}
// the scratch sets a spend batch of n proofs uses, at the size of its largest chunk: set 1 only if the batch spans chunks
static int ensure_spend_scratch(act_engine* e, size_t n) {
    size_t cap = n < e->spend_chunk ? n : e->spend_chunk;
    TRY(ensure_scratch(&e->scratch[0], cap));
    if (n > e->spend_chunk) TRY(ensure_scratch(&e->scratch[1], cap));
    return 0;
}
// n bytes from the OS CSPRNG; false if it fails
static bool os_random(void* out, size_t n) {
    size_t got = 0;
    while (got < n) {
        ssize_t r = getrandom(static_cast<char*>(out) + got, n - got, 0);
        if (r <= 0) return false;
        got += (size_t)r;
    }
    return true;
}

extern "C" const char* act_last_error(void) { return g_err.c_str(); }
extern "C" int act_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}
extern "C" void* act_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
extern "C" void act_host_free(void* p) { if (p) cudaFreeHost(p); }

extern "C" int act_params_derive(int device, const char* org, const char* svc, const char* dep, const char* ver, uint8_t h[96]) {
    if (!org || !svc || !dep || !ver || !h) return fail_msg("act_params_derive: null argument");
    std::string dom = std::string("ACT-v1:") + org + ":" + svc + ":" + dep + ":" + ver;  // src/lib.rs:293-296
    if (dom.size() > 900) return fail_msg("act_params_derive: domain separator longer than 900 bytes");
    CK(cudaSetDevice(device));
    dev_buf<u8> d_dom; dev_buf<u32> d_out;
    TRY(ensure(d_dom, dom.size() + 1));
    TRY(ensure(d_out, 96));
    CK(cudaMemcpy(d_dom, dom.data(), dom.size(), cudaMemcpyHostToDevice));
    params_derive_kernel<<<1, 1>>>(d_dom, (u32)dom.size(), d_out);
    CK(cudaGetLastError());
    CK(cudaMemcpy(h, d_out, 96, cudaMemcpyDeviceToHost));
    return 0;
}

static void build_prefix(act_ctx* c, int which, const char* label, const uint8_t h[96]) {
    // src/transcript.rs:54-74: u64be(43) | version | 3 x (u64be(32) | enc(H_i)) | u64be(len(label)) | label
    static const char ver[] = "curve25519-ristretto anonymous-credits v1.0";
    uint8_t buf[192];
    memset(buf, 0, sizeof buf);
    size_t n = 0;
    buf[7] = 43; n = 8;
    memcpy(buf + n, ver, 43); n += 43;
    for (int i = 0; i < 3; i++) { buf[n + 7] = 32; n += 8; memcpy(buf + n, h + 32 * i, 32); n += 32; }
    size_t ll = strlen(label);
    buf[n + 7] = (uint8_t)ll; n += 8;
    memcpy(buf + n, label, ll); n += ll;
    memcpy(c->prefix[which], buf, 192);
    c->prefix_len[which] = (u32)n;
}

extern "C" void act_engine_destroy(act_engine* e) {
    if (!e) return;
    if (!e->replicas.empty()) {
        for (act_engine* r : e->replicas) act_engine_destroy(r);
        delete e;
        return;
    }
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    if (e->stream[0]) {   // every staging copy of signer randomness, and the local memory of the signing kernels
        for (int which = 0; which < 3; which++) {
            for (io_slot& io : e->io) {
                dev_buf<u8>& b = io.in[which];
                if (b.p) cudaMemsetAsync(b, 0, b.bytes, e->stream[0]);
            }
        }
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device) == cudaSuccess && sms > 0)
            scrub_local_kernel<<<sms * 2, 1024, 0, e->stream[0]>>>(nullptr);
        cudaStreamSynchronize(e->stream[0]);
    }
    for (key_slot& k : e->key) if (k.ctx.p) cudaMemset(k.ctx, 0, sizeof(act_ctx));  // zeroise every x on the device
    if (e->fork) cudaEventDestroy(e->fork);
    for (int s = 0; s < 2; s++) if (e->join[s]) cudaEventDestroy(e->join[s]);
    for (int s = 0; s < 2; s++) {
        if (e->scratch[s].done) cudaEventDestroy(e->scratch[s].done);
        if (e->stream[s]) cudaStreamDestroy(e->stream[s]);
    }
    for (int k = 0; k < ACT_IO_SLOTS; k++) {
        if (e->io_ready[k]) cudaEventDestroy(e->io_ready[k]);
        if (e->io_done[k]) cudaEventDestroy(e->io_done[k]);
    }
    if (e->copy) cudaStreamDestroy(e->copy);
    delete e;   // frees every device buffer
}

// the slot table the keyed head reads; the device has no work in flight that reads it (callers synchronise first)
static int upload_slots(act_engine* e) {
    const act_ctx* h[ACT_KEY_SLOTS];
    for (int k = 0; k < ACT_KEY_SLOTS; k++) h[k] = e->key[k].ctx;
    CK(cudaMemcpy(e->d_slots, h, sizeof h, cudaMemcpyHostToDevice));
    return 0;
}
// streams, events, tables and the device context of a new engine; the caller destroys e if this fails
static int engine_init(act_engine* e, const uint8_t h[96], const uint8_t sk_x[32], const uint8_t pk_w[32]) {
    CK(cudaStreamCreateWithFlags(&e->stream[0], cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&e->stream[1], cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&e->copy, cudaStreamNonBlocking));
    for (int k = 0; k < ACT_IO_SLOTS; k++) {
        if (cudaEventCreateWithFlags(&e->io_ready[k], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&e->io_done[k], cudaEventDisableTiming) != cudaSuccess) return fail_msg("cudaEventCreate (io slots)");
    }
    CK(cudaEventCreateWithFlags(&e->fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->join[0], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->join[1], cudaEventDisableTiming));
    TRY(ensure(e->key[0].ctx, sizeof(act_ctx)));
    // replay-screen PRF key
    if (!os_random(&e->rp_key, sizeof e->rp_key)) return fail_msg("act_engine_create: the OS random source (getrandom) failed");
    size_t fb_entries = 0;
    fb_layout L = make_fb_layout(&fb_entries);
    TRY(ensure(e->d_tables, sizeof(ge_niels) * (fb_entries + ACT_CT_SIZE)));
    TRY(ensure(e->d_bases, sizeof(ge) * ACT_FB_BASES));
    dev_buf<u32> d_enc, d_ok;
    dev_buf<ge> d_W;
    TRY(ensure(d_enc, 128));
    TRY(ensure(d_ok, 4));
    TRY(ensure(d_W, sizeof(ge)));
    CK(cudaMemcpy(d_enc, h, 96, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_enc.p + 24, pk_w, 32, cudaMemcpyHostToDevice));
    setup_decode_kernel<<<1, 1>>>(d_enc, e->d_bases, d_W, d_ok);
    build_fb_tables_kernel<<<(L.first_thread[ACT_FB_BASES] + 31) / 32, 32>>>(e->d_bases, e->d_tables, L);
    build_ct_table_kernel<<<1, ACT_CT_WIN>>>(e->d_bases, e->d_tables.p + fb_entries);
    CK(cudaGetLastError());
    u32 ok = 0;
    CK(cudaMemcpy(&ok, d_ok, 4, cudaMemcpyDeviceToHost));
    if (!ok) return fail_msg("act_engine_create: H1/H2/H3/W is not a valid ristretto255 encoding");
    // context
    act_ctx hc;
    struct wipe_on_exit { void* p; size_t n; ~wipe_on_exit() { explicit_bzero(p, n); } } hc_guard{&hc, sizeof hc};   // every way out of this function
    memset(&hc, 0, sizeof hc);
    for (int b = 0; b < ACT_FB_BASES; b++) { hc.fb[b].p = e->d_tables.p + L.offset[b]; hc.fb[b].bits = L.bits[b]; hc.fb[b].win = fb_win_of(L.bits[b]); hc.fb[b].ent = fb_ent_of(L.bits[b]); }
    hc.ct_g = e->d_tables.p + fb_entries;
    memcpy(hc.h_enc, h, 96);
    build_prefix(&hc, ACT_TR_REQUEST, "request", h);
    build_prefix(&hc, ACT_TR_RESPOND, "respond", h);
    build_prefix(&hc, ACT_TR_REFUND, "refund", h);
    build_prefix(&hc, ACT_TR_SPEND, "spend", h);
    e->pub = hc;   // before any key material enters hc
    e->pub.fb[ACT_BASE_W] = fb_tab{};
    CK(cudaMemcpy(&hc.W, d_W, sizeof(ge), cudaMemcpyDeviceToHost));
    // raw key words; finalize_ctx_kernel reduces them mod l on the device
    memcpy(hc.x.v, sk_x, 32);
    CK(cudaMemcpy(e->key[0].ctx, &hc, sizeof hc, cudaMemcpyHostToDevice));
    explicit_bzero(&hc, sizeof hc);
    finalize_ctx_kernel<<<1, 1>>>(e->key[0].ctx, d_enc.p + 24, d_ok);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(&ok, d_ok, 4, cudaMemcpyDeviceToHost));
    if (!ok) return fail_msg("act_engine_create: pk_w is not the public key of sk_x (W != G*x)");
    TRY(ensure(e->d_slots, sizeof(const act_ctx*) * ACT_KEY_SLOTS));
    return upload_slots(e);
}
extern "C" int act_engine_create(act_engine** out, int device, const uint8_t h[96], const uint8_t sk_x[32], const uint8_t pk_w[32]) {
    if (!out || !h || !sk_x || !pk_w) return fail_msg("act_engine_create: null argument");
    *out = nullptr;
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) return fail_msg("act_engine_create: no CUDA device (this engine has no CPU path)");
    if (device < 0 || device >= ndev) return fail_msg("act_engine_create: bad device index");
    CK(cudaSetDevice(device));
    act_engine* e = new act_engine();
    e->device = device;
    if (int rc = engine_init(e, h, sk_x, pk_w)) { act_engine_destroy(e); return rc; }
    e->launches += 3;
    if (const char* env = getenv("ACT_SPEND_CHUNK")) {
        long v = atol(env);
        if (v >= 1 && v <= (1l << 22)) e->spend_chunk = (size_t)v;
    }
    *out = e;
    return 0;
}
extern "C" int act_engine_device(const act_engine* e) { return e ? e->device : -1; }
extern "C" int act_engine_set_spend_chunk(act_engine* e, size_t proofs) {
    if (!e) return fail_msg("null engine");
    if (proofs < 1 || proofs > ((size_t)1 << 22)) return fail_msg("act_engine_set_spend_chunk: 1 .. 4194304 proofs per chunk");
    for (act_engine* r : e->replicas) r->spend_chunk = proofs;
    e->spend_chunk = proofs;
    return 0;
}
extern "C" uint64_t act_engine_launch_count(const act_engine* e) {
    if (!e) return 0;
    uint64_t t = e->launches;
    for (const act_engine* r : e->replicas) t += r->launches;
    return t;
}

extern "C" int act_public_key(int device, const uint8_t sk_x[32], uint8_t pk_w[32]) {
    if (!sk_x || !pk_w) return fail_msg("act_public_key: null argument");
    CK(cudaSetDevice(device));
    dev_buf<ge> d_b, d_W; dev_buf<ge_niels> d_t; dev_buf<u32> d_x, d_o, d_enc, d_ok;
    // the device copy of the secret is overwritten before it is freed, whatever fails below (everything runs on the NULL stream)
    wipe_dev_on_exit x_wipe{nullptr, 32, nullptr};
    TRY(ensure(d_b, sizeof(ge) * ACT_FB_BASES));
    TRY(ensure(d_t, sizeof(ge_niels) * ACT_CT_SIZE));
    TRY(ensure(d_x, 32)); x_wipe.p = d_x;
    TRY(ensure(d_o, 32));
    // bases[0] = G via the set-up kernel with dummy (identity) encodings
    TRY(ensure(d_enc, 128)); CK(cudaMemset(d_enc, 0, 128));
    TRY(ensure(d_ok, 4)); TRY(ensure(d_W, sizeof(ge)));
    CK(cudaMemcpy(d_x, sk_x, 32, cudaMemcpyHostToDevice));
    setup_decode_kernel<<<1, 1>>>(d_enc, d_b, d_W, d_ok);
    build_ct_table_kernel<<<1, ACT_CT_WIN>>>(d_b, d_t);
    public_key_kernel<<<1, 1>>>(d_t, d_x, d_o);
    CK(cudaGetLastError());
    CK(cudaMemcpy(pk_w, d_o, 32, cudaMemcpyDeviceToHost));
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// issuer key slots: every slot shares the engine's Params, tables and scratch and holds its own x, W and W table
// ---------------------------------------------------------------------------------------------------
// a one-base layout of build_fb_tables_kernel: the W table alone, 2^ACT_FB_BITS wide
static fb_layout w_layout() {
    fb_layout L;
    memset(&L, 0, sizeof L);
    L.bits[0] = ACT_FB_BITS;
    u32 threads = fb_win_of(ACT_FB_BITS) * fb_parts_of(ACT_FB_BITS);
    for (int b = 1; b <= ACT_FB_BASES; b++) L.first_thread[b] = threads;
    return L;
}
static int slot_install(act_engine* e, int slot, const uint8_t sk_x[32], const uint8_t pk_w[32]) {
    CK(cudaSetDevice(e->device));
    key_slot k;
    TRY(ensure(k.ctx, sizeof(act_ctx)));
    TRY(ensure(k.w_table, sizeof(ge_niels) * fb_size_of(ACT_FB_BITS)));
    dev_buf<u32> d_enc, d_ok;
    dev_buf<ge> d_bases, d_W;
    TRY(ensure(d_enc, 128)); TRY(ensure(d_ok, 4));
    TRY(ensure(d_bases, sizeof(ge) * ACT_FB_BASES)); TRY(ensure(d_W, sizeof(ge)));
    CK(cudaMemcpy(d_enc, e->pub.h_enc, 96, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_enc.p + 24, pk_w, 32, cudaMemcpyHostToDevice));
    fb_layout L = w_layout();
    setup_decode_kernel<<<1, 1>>>(d_enc, d_bases, d_W, d_ok);
    build_fb_tables_kernel<<<(L.first_thread[ACT_FB_BASES] + 31) / 32, 32>>>(d_bases.p + ACT_BASE_W, k.w_table, L);
    CK(cudaGetLastError());
    u32 ok = 0;
    CK(cudaMemcpy(&ok, d_ok, 4, cudaMemcpyDeviceToHost));
    if (!ok) return fail_msg("act_engine_set_key: pk_w is not a valid ristretto255 encoding");
    act_ctx hc = e->pub;
    struct wipe_on_exit { void* p; size_t n; ~wipe_on_exit() { explicit_bzero(p, n); } } hc_guard{&hc, sizeof hc};
    hc.fb[ACT_BASE_W] = fb_tab{k.w_table.p, ACT_FB_BITS, fb_win_of(ACT_FB_BITS), fb_ent_of(ACT_FB_BITS)};
    CK(cudaMemcpy(&hc.W, d_W, sizeof(ge), cudaMemcpyDeviceToHost));
    memcpy(hc.x.v, sk_x, 32);
    wipe_dev_on_exit ctx_wipe{k.ctx.p, sizeof(act_ctx), nullptr};   // the new context holds x from here on; wiped unless installed
    CK(cudaMemcpy(k.ctx, &hc, sizeof hc, cudaMemcpyHostToDevice));
    explicit_bzero(&hc, sizeof hc);
    finalize_ctx_kernel<<<1, 1>>>(k.ctx, d_enc.p + 24, d_ok);
    CK(cudaGetLastError());
    CK(cudaMemcpy(&ok, d_ok, 4, cudaMemcpyDeviceToHost));
    if (!ok) return fail_msg("act_engine_set_key: pk_w is not the public key of sk_x (W != G*x)");
    // in-flight work (also _dev calls on callers' streams) may still read the slot's old key and table
    CK(cudaDeviceSynchronize());
    key_slot& old = e->key[slot];
    if (old.ctx.p) CK(cudaMemset(old.ctx, 0, sizeof(act_ctx)));
    ctx_wipe.p = nullptr;
    std::swap(old, k);   // k takes the old key and frees it
    return upload_slots(e);
}
static int slot_clear(act_engine* e, int slot) {
    CK(cudaSetDevice(e->device));
    CK(cudaDeviceSynchronize());
    key_slot& k = e->key[slot];
    CK(cudaMemset(k.ctx, 0, sizeof(act_ctx)));
    k = key_slot();   // frees the context and the W table
    return upload_slots(e);
}
static uint32_t slots_held(const act_engine* e) {
    uint32_t m = 0;
    for (int k = 0; k < ACT_KEY_SLOTS; k++) if (e->key[k].ctx.p) m |= 1u << k;
    return m;
}
static inline const act_engine* replica0(const act_engine* e) { return is_multi(e) ? e->replicas[0] : e; }
extern "C" int act_engine_set_key(act_engine* e, int slot, const uint8_t sk_x[32], const uint8_t pk_w[32]) {
    if (!e) return fail_msg("null engine");
    if (!sk_x || !pk_w) return fail_msg("act_engine_set_key: null argument");
    if (slot < 0 || slot >= ACT_KEY_SLOTS) return fail_msg("act_engine_set_key: slot out of range (0 .. ACT_KEY_SLOTS - 1)");
    if (!is_multi(e)) return slot_install(e, slot, sk_x, pk_w);
    for (act_engine* r : e->replicas) TRY(slot_install(r, slot, sk_x, pk_w));   // replica 0 checks the key before any other changes
    return 0;
}
extern "C" int act_engine_clear_key(act_engine* e, int slot) {
    if (!e) return fail_msg("null engine");
    if (slot < 0 || slot >= ACT_KEY_SLOTS) return fail_msg("act_engine_clear_key: slot out of range (0 .. ACT_KEY_SLOTS - 1)");
    const act_engine* r0 = replica0(e);
    if (slot == r0->selected) return fail_msg("act_engine_clear_key: the selected slot cannot be cleared (select another first)");
    if (!(slots_held(r0) >> slot & 1u)) return fail_msg("act_engine_clear_key: the slot holds no key");
    if (!is_multi(e)) return slot_clear(e, slot);
    for (act_engine* r : e->replicas) TRY(slot_clear(r, slot));
    return 0;
}
extern "C" int act_engine_select_key(act_engine* e, int slot) {
    if (!e) return fail_msg("null engine");
    if (slot < 0 || slot >= ACT_KEY_SLOTS) return fail_msg("act_engine_select_key: slot out of range (0 .. ACT_KEY_SLOTS - 1)");
    if (!(slots_held(replica0(e)) >> slot & 1u)) return fail_msg("act_engine_select_key: the slot holds no key");
    for (act_engine* r : e->replicas) r->selected = slot;
    e->selected = slot;
    return 0;
}
extern "C" int act_engine_selected_key(const act_engine* e) { return e ? replica0(e)->selected : -1; }
extern "C" uint32_t act_engine_key_slots(const act_engine* e) { return e ? slots_held(replica0(e)) : 0u; }

extern "C" int act_engine_set_timing(act_engine* e, int enable) {
    if (!e) return fail_msg("null engine");
    for (act_engine* r : e->replicas) r->timing = enable != 0;
    e->timing = enable != 0;
    return 0;
}
// Sums (and clears) the device time of every launch recorded since the last call, per kernel kind:
// 0 spend_range, 1 spend_head, 2 spend_chunk(hash), 3 spend_finish, 4 refund_sign, 5 issue, 6 issuance_check, 7 refund_check,
// 8 spend_encode.
extern "C" int act_engine_get_timing(act_engine* e, double ms[9], uint64_t count[9]) {
    if (!e || !ms || !count) return fail_msg("act_engine_get_timing: null argument");
    if (is_multi(e)) {   // sums over the replicas
        for (int k = 0; k < K_KINDS; k++) { ms[k] = 0; count[k] = 0; }
        for (act_engine* r : e->replicas) {
            double m1[K_KINDS]; uint64_t c1[K_KINDS];
            int rc = act_engine_get_timing(r, m1, c1);
            if (rc) return rc;
            for (int k = 0; k < K_KINDS; k++) { ms[k] += m1[k]; count[k] += c1[k]; }
        }
        return 0;
    }
    CK(cudaSetDevice(e->device));
    for (int k = 0; k < K_KINDS; k++) { ms[k] = 0; count[k] = 0; }
    for (auto& t : e->events) {
        CK(cudaEventSynchronize(t.b));
        float f = 0;
        CK(cudaEventElapsedTime(&f, t.a, t.b));
        ms[t.kind] += f; count[t.kind] += 1;
        cudaEventDestroy(t.a); cudaEventDestroy(t.b);
    }
    e->events.clear();
    return 0;
}

// Integer-multiply roofline of this GPU, MEASURED: sustained rate of 32x32+64->64 multiply-adds (IMAD.WIDE.U32 with a
// 64-bit addend, the instruction the field arithmetic is made of), in limb-MACs per second.
// Sixteen chains per thread, (hi:lo)_i <- hi_{i+1} * b + (hi:lo)_i: the multiplicand of every step is the high word a
// neighbouring chain produced one step earlier, so no product is loop-invariant (a hoisted product would time 64-bit
// additions) and no other instruction is needed to keep it so (round 1 xor-ed the accumulators into the operands: one ALU
// instruction per multiply, and it read 5.0 T, below what the range kernel sustains).  The loop body is 16 IMAD.WIDE.U32,
// two register moves on the ALU pipe and uniform-datapath loop control (tests/test_abi.py checks the SASS); 16 warps per SM
// sub-partition hide the 4-cycle issue interval many times over.
#define PEAK_ITER 2048
#define PEAK_CHAINS 16
__global__ void __launch_bounds__(256) int_mul_peak_kernel(u32* out, u32 b0) {
    u32 lo[PEAK_CHAINS], hi[PEAK_CHAINS];
    const u32 b = (b0 + 2u * blockIdx.x) | 1u;
#pragma unroll
    for (int i = 0; i < PEAK_CHAINS; i++) { lo[i] = 0x9e3779b9u * (threadIdx.x + 1u) + (u32)i; hi[i] = (u32)i; }
#pragma unroll 1
    for (int it = 0; it < PEAK_ITER; it++) {
#pragma unroll
        for (int i = 0; i < PEAK_CHAINS; i++) {
            // the mad.lo.cc / madc.hi pair is what fe_mul uses; ptxas fuses it into one IMAD.WIDE.U32 with a 64-bit addend
            asm volatile("mad.lo.cc.u32 %0, %2, %3, %0;\n\tmadc.hi.u32 %1, %2, %3, %1;" : "+r"(lo[i]), "+r"(hi[i]) : "r"(hi[(i + 1) % PEAK_CHAINS]), "r"(b));
        }
    }
    u32 s = 0;
#pragma unroll
    for (int i = 0; i < PEAK_CHAINS; i++) s ^= lo[i] ^ hi[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
extern "C" int act_measure_int_mul_peak(int device, double* limb_macs_per_s) {
    if (!limb_macs_per_s) return fail_msg("null argument");
    CK(cudaSetDevice(device));
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device));
    int blocks = p.multiProcessorCount * 8;     // 8 x 256 threads = 64 warps per SM, one wave
    dev_buf<u32> out;
    TRY(ensure(out, (size_t)blocks * 256 * 4));
    cudaEvent_t a = nullptr, b = nullptr;
    double best = 1e30;
    auto timed = [&]() -> int {
        CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
        for (int r = 0; r < 8; r++) {   // the first launches also bring the clocks up
            CK(cudaEventRecord(a));
            int_mul_peak_kernel<<<blocks, 256>>>(out, 3);
            CK(cudaEventRecord(b));
            CK(cudaEventSynchronize(b));
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, a, b));
            if (r > 1 && ms < best) best = ms;
        }
        return 0;
    };
    int rc = timed();
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
    if (rc) return rc;
    *limb_macs_per_s = (double)blocks * 256 * PEAK_ITER * PEAK_CHAINS / (best * 1e-3);
    return 0;
}

extern "C" int act_selftest(int device) {
    CK(cudaSetDevice(device));
    dev_buf<u32> d_fail;
    TRY(ensure(d_fail, 4));
    CK(cudaMemset(d_fail, 0, 4));
    selftest_kernel<<<8, 64>>>(d_fail);
    CK(cudaGetLastError());
    u32 f = 0;
    CK(cudaMemcpy(&f, d_fail, 4, cudaMemcpyDeviceToHost));
    if (f) { char b[64]; snprintf(b, sizeof b, "act_selftest: failure mask 0x%x", f); g_err = b; return (int)f; }
    return 0;
}

static inline unsigned nblocks(size_t n, unsigned bs) { return (unsigned)((n + bs - 1) / bs); }
// device-buffer entry points move records with 16-byte vector accesses: a misaligned pointer would fault inside a kernel
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
#define NEED_ALIGNED(what, ...)                                                                                     \
    do {                                                                                                            \
        const void* ps_[] = {__VA_ARGS__};                                                                          \
        for (const void* p_ : ps_) if (p_ && !aligned16(p_)) return fail_msg(what ": device buffers must be 16-byte aligned"); \
    } while (0)

// ---- device-buffer entry points ----
extern "C" int act_batch_issue_dev(act_engine* e, size_t n, const void* req, const void* c, const void* rnd, void* resp, void* status, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_batch_issue_dev");
    if (n == 0) return 0;
    if (!req || !c || !rnd || !resp || !status) return fail_msg("act_batch_issue_dev: null buffer");
    NEED_ALIGNED("act_batch_issue_dev", req, c, rnd, resp);
    CK(cudaSetDevice(e->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream[0];
    LAUNCH(e, K_ISSUE, st, (issue_kernel<<<nblocks(n, ACT_ISSUE_BLOCK), ACT_ISSUE_BLOCK, 0, st>>>(sel_ctx(e), n, (const u32*)req, (const u32*)c, (const u32*)rnd, (u32*)resp, (u8*)status)));
    CK(cudaGetLastError());
    return 0;
}
extern "C" int act_batch_issuance_check_dev(act_engine* e, size_t n, const void* K, const void* resp, void* status, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_batch_issuance_check_dev");
    if (n == 0) return 0;
    if (!K || !resp || !status) return fail_msg("act_batch_issuance_check_dev: null buffer");
    NEED_ALIGNED("act_batch_issuance_check_dev", K, resp);
    CK(cudaSetDevice(e->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream[0];
    LAUNCH(e, K_ISSUANCE_CHECK, st, (issuance_check_kernel<<<nblocks(n, ACT_ISSUE_BLOCK), ACT_ISSUE_BLOCK, 0, st>>>(sel_ctx(e), n, (const u32*)K, (const u32*)resp, (u8*)status)));
    CK(cudaGetLastError());
    return 0;
}
extern "C" int act_batch_refund_check_dev(act_engine* e, size_t n, const void* com, const void* refund, void* status, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_batch_refund_check_dev");
    if (n == 0) return 0;
    if (!com || !refund || !status) return fail_msg("act_batch_refund_check_dev: null buffer");
    NEED_ALIGNED("act_batch_refund_check_dev", com, refund);
    CK(cudaSetDevice(e->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream[0];
    LAUNCH(e, K_REFUND_CHECK, st, (refund_check_kernel<<<nblocks(n, ACT_HEAD_BLOCK), ACT_HEAD_BLOCK, 0, st>>>(sel_ctx(e), n, (const u32*)com, (const u32*)refund, (u8*)status)));
    CK(cudaGetLastError());
    return 0;
}
// one chunk of the spend pipeline on one stream with one scratch set
// kprime_out != nullptr: verification only -- K' of every proof goes to kprime_out (m x 128 B) and the signing stage is left
// to the caller (sequential-RNG contract)
// key_ids != nullptr: keyed verification (one key id per proof; the refund is signed under the selected key)
static int spend_chunk_launch(act_engine* e, spend_scratch* s, cudaStream_t st, size_t m, const u32* proofs, const u32* rnd,
                              u32* refunds, u32* nullifiers, u8* status, u32* kprime_out = nullptr, const u8* key_ids = nullptr) {
    if (s->used) CK(cudaStreamWaitEvent(st, s->done, 0));   // the previous pipeline on this scratch set (any stream) has drained
    CK(cudaMemsetAsync(s->flags, 0, m * 4, st));
    CK(cudaMemsetAsync(s->counter, 0, 4, st));
    size_t rblocks = (m * ACT_L + ACT_RANGE_BLOCK - 1) / ACT_RANGE_BLOCK;   // blocks that would hold one thread per com_j
    unsigned rgrid = rblocks < s->range_grid ? (unsigned)rblocks : s->range_grid;
    LAUNCH(e, K_RANGE, st, (spend_range_kernel<<<rgrid, ACT_RANGE_BLOCK, 0, st>>>(sel_ctx(e), m, proofs, s->items, s->com_niels, s->flags, s->tabs, s->cpts, s->counter)));
    // head before encode: it completes the two half-commitments of j = 0 (their h2 terms) that the encode stage then reads
    u32* kp = kprime_out ? kprime_out : s->kprime;
    if (key_ids)
        LAUNCH(e, K_HEAD, st, (spend_head_keyed_kernel<<<nblocks(m, ACT_HEAD_BLOCK), ACT_HEAD_BLOCK, 0, st>>>(sel_ctx(e), m, proofs, s->items, s->com_niels, kp, s->flags, s->cpts,
                                                                                                           key_ids, e->d_slots)));
    else
        LAUNCH(e, K_HEAD, st, (spend_head_kernel<<<nblocks(m, ACT_HEAD_BLOCK), ACT_HEAD_BLOCK, 0, st>>>(sel_ctx(e), m, proofs, s->items, s->com_niels, kp, s->flags, s->cpts)));
    LAUNCH(e, K_ENCODE, st, (spend_encode_kernel<<<nblocks(m * ACT_ENC_PARTS, ACT_ENC_BLOCK), ACT_ENC_BLOCK, 0, st>>>(sel_ctx(e), m, s->cpts, s->items, 2 * ACT_L, 133)));
    LAUNCH(e, K_CHUNK, st, (spend_chunk_kernel<<<nblocks(m * ACT_SPEND_CHUNKS, ACT_HASH_BLOCK), ACT_HASH_BLOCK, 0, st>>>(sel_ctx(e), m, s->items, s->cvs)));
    LAUNCH(e, K_FINISH, st, (spend_finish_kernel<<<nblocks(m, ACT_HASH_BLOCK), ACT_HASH_BLOCK, 0, st>>>(sel_ctx(e), m, proofs, s->cvs, s->flags, status)));
    if (!kprime_out)
        LAUNCH(e, K_SIGN, st, (refund_sign_kernel<<<nblocks(m, ACT_SIGN_BLOCK), ACT_SIGN_BLOCK, 0, st>>>(sel_ctx(e), m, proofs, rnd, s->kprime, status, refunds, nullifiers)));
    else if (nullifiers) {   // verification-only pass that also delivers nullifier() of every accepted proof
        nullifier_kernel<<<nblocks(m * 8, 256), 256, 0, st>>>(m, s->items, status, nullifiers);
        e->launches += 1;
    }
    CK(cudaGetLastError());
    CK(cudaEventRecord(s->done, st));
    s->used = true;
    return 0;
}
// the body of act_batch_verify_spend_and_refund_dev and of its keyed form (key_ids != nullptr)
static int verify_spend_dev(act_engine* e, size_t n, const void* proofs, const u8* key_ids, const void* rnd, void* refunds, void* nullifiers,
                            void* status, void* stream) {
    CK(cudaSetDevice(e->device));
    cudaStream_t user = stream ? (cudaStream_t)stream : e->stream[0];
    const size_t ACT_SPEND_CHUNK_RT = e->spend_chunk;
    // chunks alternate over the engine's two streams (each with its own scratch) so that the thread-per-proof
    // kernels of one chunk overlap the range kernel of the next; fork from / join into the caller's stream.
    bool two = n > ACT_SPEND_CHUNK_RT;
    TRY(ensure_spend_scratch(e, n));
    if (two) {
        CK(cudaEventRecord(e->fork, user));
        CK(cudaStreamWaitEvent(e->stream[0], e->fork, 0));
        CK(cudaStreamWaitEvent(e->stream[1], e->fork, 0));
    }
    size_t ci = 0;
    for (size_t off = 0; off < n; off += ACT_SPEND_CHUNK_RT, ci++) {
        size_t m = n - off < ACT_SPEND_CHUNK_RT ? n - off : ACT_SPEND_CHUNK_RT;
        int slot = two ? (int)(ci & 1) : 0;
        cudaStream_t st = two ? e->stream[slot] : user;
        TRY(spend_chunk_launch(e, &e->scratch[slot], st, m, (const u32*)proofs + off * ACT_PROOF_WORDS, (const u32*)rnd + off * 32,
                               (u32*)refunds + off * 32, (u32*)nullifiers + off * 8, (u8*)status + off, nullptr, key_ids ? key_ids + off : nullptr));
    }
    if (two) {
        CK(cudaEventRecord(e->join[0], e->stream[0]));
        CK(cudaEventRecord(e->join[1], e->stream[1]));
        CK(cudaStreamWaitEvent(user, e->join[0], 0));
        CK(cudaStreamWaitEvent(user, e->join[1], 0));
    }
    return 0;
}
extern "C" int act_batch_verify_spend_and_refund_dev(act_engine* e, size_t n, const void* proofs, const void* rnd, void* refunds,
                                                      void* nullifiers, void* status, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_batch_verify_spend_and_refund_dev");
    if (n == 0) return 0;
    if (!proofs || !rnd || !refunds || !nullifiers || !status) return fail_msg("act_batch_verify_spend_and_refund_dev: null buffer");
    NEED_ALIGNED("act_batch_verify_spend_and_refund_dev", proofs, rnd, refunds, nullifiers);
    return verify_spend_dev(e, n, proofs, nullptr, rnd, refunds, nullifiers, status, stream);
}
extern "C" int act_batch_verify_spend_and_refund_keyed_dev(act_engine* e, size_t n, const void* proofs, const void* key_ids, const void* rnd, void* refunds,
                                                            void* nullifiers, void* status, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_batch_verify_spend_and_refund_keyed_dev");
    if (n == 0) return 0;
    if (!proofs || !key_ids || !rnd || !refunds || !nullifiers || !status) return fail_msg("act_batch_verify_spend_and_refund_keyed_dev: null buffer");
    NEED_ALIGNED("act_batch_verify_spend_and_refund_keyed_dev", proofs, rnd, refunds, nullifiers);   // key ids are read byte by byte
    return verify_spend_dev(e, n, proofs, (const u8*)key_ids, rnd, refunds, nullifiers, status, stream);
}

// ---- host-buffer entry points: chunked, double-buffered over the engine's two streams ----
struct host_io {
    const uint8_t* in[3]; size_t in_stride[3];
    uint8_t* out[3]; size_t out_stride[3];  // out[2] = status (stride 1)
    int secret_in = -1;                     // index of the input that carries signer randomness (e_wide | alpha_wide), or -1
};
// Leaves no signer randomness behind on the device: zero-fills the staging copies of `rnd` (alpha together with the public
// (z, gamma, e) yields x) and overwrites the local memory the signing kernels used.  Runs on `st`, asynchronously.
static int scrub_after_signing(act_engine* e, cudaStream_t st, int secret_in) {
    for (int k = 0; k < ACT_IO_SLOTS && secret_in >= 0; k++) {
        dev_buf<u8>& b = e->io[k].in[secret_in];
        if (b.p) CK(cudaMemsetAsync(b, 0, b.bytes, st));
    }
    int sms = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device));
    scrub_local_kernel<<<sms * 2, 1024, 0, st>>>(nullptr);
    e->launches += 1;
    CK(cudaGetLastError());
    return 0;
}
// Chunk boundaries of a host-buffer call: full chunks, except that a batch of more than one chunk starts with a short ramp
// (chunk/8, chunk/2) so that the first kernels start after a small H2D copy instead of after a whole chunk's (1.1 GB for
// 65 536 proofs); the copy stream runs ahead of the compute streams from then on.
static void chunk_plan(size_t n, size_t chunk, bool ramp, std::vector<size_t>& sizes) {
    sizes.clear();
    size_t off = 0;
    if (ramp && n > chunk && chunk >= 4096) {
        for (size_t m : {chunk / 8, chunk / 2}) { sizes.push_back(m); off += m; }
    }
    while (off < n) { size_t m = n - off < chunk ? n - off : chunk; sizes.push_back(m); off += m; }
}
template <typename F>
static int run_chunked(act_engine* e, size_t n, size_t chunk, const host_io& h, F launch, bool ramp = false) {
    CK(cudaSetDevice(e->device));
    std::vector<size_t> sizes;
    chunk_plan(n, chunk, ramp, sizes);
    size_t nchunks = sizes.size(), maxm = 0;
    for (size_t m : sizes) maxm = m > maxm ? m : maxm;
    // staging of every slot this call will use, sized for its largest chunk BEFORE anything is in flight (growing a slot later
    // would free memory a running kernel still reads)
    for (size_t k = 0; k < (nchunks < ACT_IO_SLOTS ? nchunks : (size_t)ACT_IO_SLOTS); k++) {
        io_slot& io = e->io[k];
        for (int i = 0; i < 3; i++) if (h.in[i]) TRY(ensure(io.in[i], maxm * h.in_stride[i] + 16));
        for (int i = 0; i < 2; i++) if (h.out[i]) TRY(ensure(io.out[i], maxm * h.out_stride[i] + 16));
        TRY(ensure(io.st, maxm + 16));
    }
    size_t off = 0;
    for (size_t ci = 0; ci < nchunks; ci++) {
        int s = (int)(ci & 1), k = (int)(ci % ACT_IO_SLOTS);
        io_slot& io = e->io[k];
        cudaStream_t st = e->stream[s];
        size_t m = sizes[ci];
        if (ci >= ACT_IO_SLOTS) CK(cudaEventSynchronize(e->io_done[k]));  // slot reuse: chunk ci-3 fully drained (incl. D2H)
        for (int i = 0; i < 3; i++)
            if (h.in[i]) CK(cudaMemcpyAsync(io.in[i], h.in[i] + off * h.in_stride[i], m * h.in_stride[i], cudaMemcpyHostToDevice, e->copy));
        CK(cudaEventRecord(e->io_ready[k], e->copy));
        CK(cudaStreamWaitEvent(st, e->io_ready[k], 0));
        TRY(launch(s, st, m, io));
        if (e->g_keep) {   // screened call: status + nullifiers of the whole shard stay on the device for the gather
            CK(cudaMemcpyAsync(e->g_st.p + off, io.st, m, cudaMemcpyDeviceToDevice, st));
            CK(cudaMemcpyAsync(e->g_nul.p + off * 32, io.out[1], m * 32, cudaMemcpyDeviceToDevice, st));
        }
        for (int i = 0; i < 2; i++)
            if (h.out[i]) CK(cudaMemcpyAsync(h.out[i] + off * h.out_stride[i], io.out[i], m * h.out_stride[i], cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(h.out[2] + off, io.st, m, cudaMemcpyDeviceToHost, st));
        CK(cudaEventRecord(e->io_done[k], st));
        off += m;
    }
    CK(cudaStreamSynchronize(e->stream[0]));
    CK(cudaStreamSynchronize(e->stream[1]));
    if (h.secret_in >= 0) {
        TRY(scrub_after_signing(e, e->stream[0], h.secret_in));
        CK(cudaStreamSynchronize(e->stream[0]));
    }
    return 0;
}

extern "C" int act_batch_issue(act_engine* e, size_t n, const uint8_t* req, const uint8_t* c, const uint8_t* rnd, uint8_t* resp, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!req || !c || !rnd || !resp || !status) return fail_msg("act_batch_issue: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_issue(r, m, req + lo * 128, c + lo * 32, rnd + lo * 128, resp + lo * 160, status + lo); });
    host_io h = {{req, c, rnd}, {128, 32, 128}, {resp, nullptr, status}, {160, 0, 1}, 2};
    return run_chunked(e, n, ACT_SMALL_CHUNK, h, [&](int, cudaStream_t st, size_t m, io_slot& io) {
        return act_batch_issue_dev(e, m, io.in[0], io.in[1], io.in[2], io.out[0], io.st, st);
    }, true);
}
extern "C" int act_batch_issuance_check(act_engine* e, size_t n, const uint8_t* K, const uint8_t* resp, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!K || !resp || !status) return fail_msg("act_batch_issuance_check: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_issuance_check(r, m, K + lo * 32, resp + lo * 160, status + lo); });
    host_io h = {{K, resp, nullptr}, {32, 160, 0}, {nullptr, nullptr, status}, {0, 0, 1}};
    return run_chunked(e, n, ACT_SMALL_CHUNK, h, [&](int, cudaStream_t st, size_t m, io_slot& io) {
        return act_batch_issuance_check_dev(e, m, io.in[0], io.in[1], io.st, st);
    });
}
extern "C" int act_batch_refund_check(act_engine* e, size_t n, const uint8_t* com, const uint8_t* refund, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!com || !refund || !status) return fail_msg("act_batch_refund_check: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_refund_check(r, m, com + lo * 4096, refund + lo * 128, status + lo); });
    host_io h = {{com, refund, nullptr}, {4096, 128, 0}, {nullptr, nullptr, status}, {0, 0, 1}};
    return run_chunked(e, n, e->spend_chunk, h, [&](int, cudaStream_t st, size_t m, io_slot& io) {
        return act_batch_refund_check_dev(e, m, io.in[0], io.in[1], io.st, st);
    });
}
// one replica's host-buffer verify + refund; key_ids (one byte per proof, optional) travel with the proofs
static int verify_spend_host(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* key_ids, const uint8_t* rnd, uint8_t* refunds,
                             uint8_t* nullifiers, uint8_t* status) {
    host_io h = {{proofs, rnd, key_ids}, {ACT_PROOF_BYTES, 128, 1}, {refunds, nullifiers, status}, {128, 32, 1}, 1};
    // the scratch sets before anything is in flight
    CK(cudaSetDevice(e->device));
    TRY(ensure_spend_scratch(e, n));
    return run_chunked(e, n, e->spend_chunk, h, [&](int s, cudaStream_t st, size_t m, io_slot& io) {
        return spend_chunk_launch(e, &e->scratch[s], st, m, (const u32*)io.in[0].p, (const u32*)io.in[1].p, (u32*)io.out[0].p, (u32*)io.out[1].p, io.st,
                                  nullptr, key_ids ? io.in[2].p : nullptr);
    }, true);
}
extern "C" int act_batch_verify_spend_and_refund(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* rnd, uint8_t* refunds,
                                                  uint8_t* nullifiers, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!proofs || !rnd || !refunds || !nullifiers || !status) return fail_msg("act_batch_verify_spend_and_refund: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_verify_spend_and_refund(r, m, proofs + lo * ACT_PROOF_BYTES, rnd + lo * 128, refunds + lo * 128, nullifiers + lo * 32, status + lo); });
    return verify_spend_host(e, n, proofs, nullptr, rnd, refunds, nullifiers, status);
}

// ---------------------------------------------------------------------------------------------------
// rows either side of the hot path (act_aux.cuh): replay screen and the canonical-CBOR fast path
// ---------------------------------------------------------------------------------------------------
extern "C" int act_flag_replays_dev(act_engine* e, size_t n, const void* status, const void* nullifiers, size_t n_seen, const void* seen,
                                    void* status_out, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_flag_replays_dev");
    if (n == 0) return 0;
    if (!status || !nullifiers || !status_out || (n_seen && !seen)) return fail_msg("act_flag_replays_dev: null buffer");
    if (n + n_seen >= 0x7fffffffu) return fail_msg("act_flag_replays_dev: batch too large");
    CK(cudaSetDevice(e->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream[0];
    size_t slots = 1024;
    while (slots < 2 * (n + n_seen)) slots <<= 1;
    TRY(ensure(e->d_rp_table, slots * 4, st));
    CK(cudaMemsetAsync(e->d_rp_table, 0xff, slots * 4, st));
    // secret per-engine key, tweaked per call: slots are unpredictable to whoever chose the nullifiers
    rp_key128 seed = {e->rp_key.k0 ^ (++e->rp_calls * 0x9e3779b97f4a7c15ull), e->rp_key.k1};
    u32 total = (u32)(n + n_seen);
    replay_insert_kernel<<<nblocks(total, 256), 256, 0, st>>>((u32)n, (u32)n_seen, (const u8*)status, (const uint4*)seen, (const uint4*)nullifiers,
                                                             e->d_rp_table, (u32)(slots - 1), seed);
    replay_resolve_kernel<<<nblocks(n, 256), 256, 0, st>>>((u32)n, (u32)n_seen, (const u8*)status, (const uint4*)seen, (const uint4*)nullifiers,
                                                           e->d_rp_table, (u32)(slots - 1), seed, (u8*)status_out);
    e->launches += 2;
    CK(cudaGetLastError());
    return 0;
}
extern "C" int act_flag_replays(act_engine* e, size_t n, const uint8_t* status, const uint8_t* nullifiers, size_t n_seen, const uint8_t* seen,
                                uint8_t* status_out) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!status || !nullifiers || !status_out || (n_seen && !seen)) return fail_msg("act_flag_replays: null buffer");
    if (is_multi(e)) return act_flag_replays(e->replicas[0], n, status, nullifiers, n_seen, seen, status_out);   // the screen is global: one device
    CK(cudaSetDevice(e->device));
    dev_buf<u8> d_st, d_nul, d_seen, d_out;
    TRY(ensure(d_st, n)); TRY(ensure(d_nul, n * 32)); TRY(ensure(d_out, n));
    if (n_seen) { TRY(ensure(d_seen, n_seen * 32)); CK(cudaMemcpyAsync(d_seen, seen, n_seen * 32, cudaMemcpyHostToDevice, e->stream[0])); }
    CK(cudaMemcpyAsync(d_st, status, n, cudaMemcpyHostToDevice, e->stream[0]));
    CK(cudaMemcpyAsync(d_nul, nullifiers, n * 32, cudaMemcpyHostToDevice, e->stream[0]));
    TRY(act_flag_replays_dev(e, n, d_st, d_nul, n_seen, d_seen, d_out, e->stream[0]));
    CK(cudaMemcpyAsync(status_out, d_out, n, cudaMemcpyDeviceToHost, e->stream[0]));
    CK(cudaStreamSynchronize(e->stream[0]));
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// device-resident nullifier store (act_store.cuh): the spent set, kept on one GPU between calls
// ---------------------------------------------------------------------------------------------------
struct act_nullifier_store {
    int device = 0;
    cudaStream_t stream = nullptr;        // the stream of calls that pass NULL
    cudaEvent_t done = nullptr;           // recorded after every call: the next one (any stream) waits on it
    dev_buf<uint4> table; size_t slots = 0;
    rp_key128 key = {0, 0}; uint64_t calls = 0;   // slot PRF key (OS CSPRNG, drawn at creation); per-call tweak of the dedupe table's
    // d_misc: [0] exact size, [1] bad-key flag, [2] export counter;  h_misc: pinned read-back of [0..1]
    dev_buf<unsigned long long> d_misc; unsigned long long* h_misc = nullptr;
    dev_buf<u32> dd_table;   // in-batch dedupe (replay_insert/resolve_kernel)
    dev_buf<u8> st_tmp;      // statuses after the store lookup
};
#define ACT_STORE_MIN_SLOTS 1024
// slots for `keys` members at load <= 1/2; 0 when that is not representable
static size_t store_slots_for(size_t keys) {
    size_t s = ACT_STORE_MIN_SLOTS;
    while (s / 2 < keys) { if (s > ((size_t)1 << 58)) return 0; s <<= 1; }
    return s;
}
extern "C" void act_nullifier_store_destroy(act_nullifier_store* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->done) cudaEventSynchronize(s->done);
    if (s->h_misc) cudaFreeHost(s->h_misc);
    if (s->done) cudaEventDestroy(s->done);
    if (s->stream) cudaStreamDestroy(s->stream);
    explicit_bzero(&s->key, sizeof s->key);
    delete s;   // frees every device buffer
}
// key, stream, event and an empty table of `slots` slots for a new store; the caller destroys s if this fails
static int store_init(act_nullifier_store* s, size_t slots) {
    if (!os_random(&s->key, sizeof s->key)) return fail_msg("act_nullifier_store_create: the OS random source (getrandom) failed");
    CK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&s->done, cudaEventDisableTiming));
    TRY(ensure(s->d_misc, 4 * sizeof(unsigned long long)));
    CK(cudaHostAlloc((void**)&s->h_misc, 4 * sizeof(unsigned long long), cudaHostAllocDefault));
    TRY(ensure(s->table, slots * 32));
    s->slots = slots;
    CK(cudaMemsetAsync(s->table, 0xff, slots * 32, s->stream));
    CK(cudaMemsetAsync(s->d_misc, 0, 4 * sizeof(unsigned long long), s->stream));
    CK(cudaEventRecord(s->done, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    return 0;
}
extern "C" int act_nullifier_store_create(act_nullifier_store** out, int device, size_t capacity) {
    if (!out) return fail_msg("act_nullifier_store_create: null argument");
    *out = nullptr;
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) return fail_msg("act_nullifier_store_create: no CUDA device (the store has no CPU path)");
    if (device < 0 || device >= ndev) return fail_msg("act_nullifier_store_create: bad device index");
    size_t slots = store_slots_for(capacity);
    if (!slots) return fail_msg("act_nullifier_store_create: capacity too large");
    CK(cudaSetDevice(device));
    act_nullifier_store* s = new act_nullifier_store();
    s->device = device;
    if (int rc = store_init(s, slots)) { act_nullifier_store_destroy(s); return rc; }
    *out = s;
    return 0;
}
extern "C" int act_nullifier_store_device(const act_nullifier_store* s) { return s ? s->device : -1; }
// exact member count; waits for the store's last call
static int store_count(act_nullifier_store* s, size_t* count) {
    CK(cudaSetDevice(s->device));
    CK(cudaStreamWaitEvent(s->stream, s->done, 0));
    CK(cudaMemcpyAsync(s->h_misc, s->d_misc, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    *count = (size_t)s->h_misc[0];
    return 0;
}
extern "C" size_t act_nullifier_store_size(const act_nullifier_store* s) {
    size_t c = 0;
    if (!s || store_count(const_cast<act_nullifier_store*>(s), &c)) return 0;
    return c;
}
// a table of at least `slots` slots holding every current member; the old one is freed only once the new one is complete, so a
// failed allocation leaves the store as it was.  `st` is idle when this runs (act_nullifier_store_screen_dev has synchronised it).
static int store_grow(act_nullifier_store* s, size_t slots, cudaStream_t st) {
    dev_buf<uint4> t;
    TRY(ensure(t, slots * 32));
    CK(cudaMemsetAsync(t, 0xff, slots * 32, st));
    store_rehash_kernel<<<nblocks(s->slots, 256), 256, 0, st>>>((u64)s->slots, s->table, t, (u64)(slots - 1), s->key);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    s->table = std::move(t);   // t takes the old table and frees it
    s->slots = slots;
    return 0;
}
// slots of the in-batch dedupe table for n keys
static size_t dedupe_slots(size_t n) {
    size_t dd = ACT_STORE_MIN_SLOTS;
    while (dd < 2 * n) dd <<= 1;
    return dd;
}
// A screen of n (status, nullifier) pairs against the store and the batch itself, then (record != 0) insertion of the survivors,
// in two halves.  The first does everything that can fail: scratch, the lookup (+ key check), one 16-byte read-back (bad-key flag
// and exact size), growth if `adds` more members could cross the load limit.  It leaves the membership as it was.  The second
// launches the in-batch dedupe and the insert and cannot fail but for a launch error.  A call over several stores prepares every
// store before it commits the first.
static int store_prepare(act_nullifier_store* s, size_t n, const void* status, const void* nullifiers, int record, size_t adds, cudaStream_t st) {
    CK(cudaStreamWaitEvent(st, s->done, 0));
    // growing drains st first: the store's previous call has then finished with its scratch
    TRY(ensure(s->st_tmp, n, st));
    TRY(ensure(s->dd_table, dedupe_slots(n) * 4, st));
    CK(cudaMemsetAsync(s->d_misc.p + 1, 0, sizeof(unsigned long long), st));
    store_lookup_kernel<<<nblocks(n, 256), 256, 0, st>>>((u64)n, (const u8*)status, (const uint4*)nullifiers, s->table, (u64)(s->slots - 1), s->key,
                                                        s->st_tmp, reinterpret_cast<u32*>(s->d_misc.p + 1));
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(s->h_misc, s->d_misc, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (s->h_misc[1]) {
        CK(cudaEventRecord(s->done, st));
        return fail_msg("act_nullifier_store_screen_dev: a nullifier with status 0 is not reduced mod l");
    }
    size_t size = (size_t)s->h_misc[0];
    if (record && size + adds > s->slots / 2) {
        size_t want = store_slots_for(size + adds);
        if (!want) return fail_msg("act_nullifier_store_screen_dev: store too large");
        int rc = store_grow(s, want, st);
        if (rc) { cudaEventRecord(s->done, st); return rc; }
    }
    return 0;
}
static int store_commit(act_nullifier_store* s, size_t n, const void* nullifiers, void* status_out, int record, cudaStream_t st) {
    size_t dd = dedupe_slots(n);
    CK(cudaMemsetAsync(s->dd_table, 0xff, dd * 4, st));
    rp_key128 seed = {s->key.k0 ^ (++s->calls * 0x9e3779b97f4a7c15ull), s->key.k1};
    replay_insert_kernel<<<nblocks(n, 256), 256, 0, st>>>((u32)n, 0, s->st_tmp, nullptr, (const uint4*)nullifiers, s->dd_table, (u32)(dd - 1), seed);
    replay_resolve_kernel<<<nblocks(n, 256), 256, 0, st>>>((u32)n, 0, s->st_tmp, nullptr, (const uint4*)nullifiers, s->dd_table, (u32)(dd - 1), seed,
                                                           (u8*)status_out);
    if (record)
        store_insert_kernel<<<nblocks(n, 256), 256, 0, st>>>((u64)n, (const u8*)status_out, (const uint4*)nullifiers, s->table, (u64)(s->slots - 1),
                                                            s->key, s->d_misc);
    CK(cudaGetLastError());
    CK(cudaEventRecord(s->done, st));
    return 0;
}
// Screen of n (status, nullifier) pairs against the store and the batch itself, then (record != 0) insertion of the survivors.
// In stream order: lookup (+ key check) -> one 16-byte read-back (bad-key flag and exact size) -> growth if the survivors could
// cross the load limit -> in-batch dedupe -> insert.  Everything that can fail is decided before the insert is launched.
extern "C" int act_nullifier_store_screen_dev(act_nullifier_store* s, size_t n, const void* status, const void* nullifiers, void* status_out,
                                              int record, void* stream) {
    if (!s) return fail_msg("null store");
    if (n == 0) return 0;
    if (!status || !nullifiers || !status_out) return fail_msg("act_nullifier_store_screen_dev: null buffer");
    NEED_ALIGNED("act_nullifier_store_screen_dev", nullifiers);   // status bytes are read one by one
    if (n >= 0x7fffffffu) return fail_msg("act_nullifier_store_screen_dev: batch too large (at most 2^31 - 2 keys per call)");
    CK(cudaSetDevice(s->device));
    for (const void* p : {status, nullifiers, (const void*)status_out}) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return fail_msg("act_nullifier_store_screen_dev: not a device pointer"); }
        if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != s->device)
            return fail_msg("act_nullifier_store_screen_dev: buffers must be device memory on the store's device");
    }
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    TRY(store_prepare(s, n, status, nullifiers, record, n, st));
    return store_commit(s, n, nullifiers, status_out, record, st);
}
extern "C" int act_nullifier_store_screen(act_nullifier_store* s, size_t n, const uint8_t* status, const uint8_t* nullifiers, uint8_t* status_out,
                                          int record) {
    if (!s) return fail_msg("null store");
    if (n == 0) return 0;
    if (!status || !nullifiers || !status_out) return fail_msg("act_nullifier_store_screen: null buffer");
    CK(cudaSetDevice(s->device));
    dev_buf<u8> d_st, d_nul, d_out;
    TRY(ensure(d_st, n)); TRY(ensure(d_nul, n * 32)); TRY(ensure(d_out, n));
    CK(cudaMemcpyAsync(d_st, status, n, cudaMemcpyHostToDevice, s->stream));
    CK(cudaMemcpyAsync(d_nul, nullifiers, n * 32, cudaMemcpyHostToDevice, s->stream));
    TRY(act_nullifier_store_screen_dev(s, n, d_st, d_nul, d_out, record, s->stream));
    CK(cudaMemcpyAsync(status_out, d_out, n, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    return 0;
}
#define ACT_STORE_EXPORT_SLOTS ((size_t)1 << 24)   // table slots compacted per round trip (512 MB of table, at most as much of keys)
extern "C" int act_nullifier_store_export(act_nullifier_store* s, uint8_t* out, size_t cap, size_t* count) {
    if (!s) return fail_msg("null store");
    if (!count || (cap && !out)) return fail_msg("act_nullifier_store_export: null argument");
    size_t size = 0;
    int rc = store_count(s, &size);
    if (rc) return rc;
    *count = size;
    if (cap < size) return fail_msg("act_nullifier_store_export: the output holds fewer keys than the store");
    if (size == 0) return 0;
    cudaStream_t st = s->stream;
    size_t chunk = s->slots < ACT_STORE_EXPORT_SLOTS ? s->slots : ACT_STORE_EXPORT_SLOTS;
    size_t written = 0;
    auto rounds = [&]() -> int {
        dev_buf<uint4> d_out;
        TRY(ensure(d_out, chunk * 32));
        for (size_t lo = 0; lo < s->slots; lo += chunk) {
            CK(cudaMemsetAsync(s->d_misc.p + 2, 0, sizeof(unsigned long long), st));
            store_compact_kernel<<<nblocks(chunk, 256), 256, 0, st>>>((u64)chunk, s->table.p + 2 * lo, d_out, s->d_misc.p + 2);
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(s->h_misc + 2, s->d_misc.p + 2, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            size_t k = (size_t)s->h_misc[2];
            if (written + k > size) return fail_msg("act_nullifier_store_export: more occupied slots than members");
            CK(cudaMemcpyAsync(out + written * 32, d_out, k * 32, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            written += k;
        }
        return 0;
    };
    rc = rounds();
    cudaEventRecord(s->done, st);   // on every way out: the next call waits for whatever the rounds queued
    if (!rc && written != size) rc = fail_msg("act_nullifier_store_export: fewer occupied slots than members");
    return rc;
}

static int ensure_skeleton(act_engine* e, int kind) {
    if (kind < 0 || kind > 3) return fail_msg("bad record kind (0 request, 1 response, 2 proof, 3 refund)");
    if (e->d_skel[kind].p) return 0;
    size_t len = act_cbor_len(kind);
    std::vector<int32_t> h(len);
    act_build_skeleton(h.data(), kind);
    dev_buf<int32_t> d;
    TRY(ensure(d, len * 4));
    CK(cudaMemcpy(d, h.data(), len * 4, cudaMemcpyHostToDevice));
    e->d_skel[kind] = std::move(d);   // only once it holds the skeleton
    return 0;
}
extern "C" int act_unpack_cbor_dev(act_engine* e, int kind, size_t n, const void* cbor, void* records, void* status, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_unpack_cbor_dev");
    if (n == 0) return 0;
    if (!cbor || !records || !status) return fail_msg("act_unpack_cbor_dev: null buffer");
    CK(cudaSetDevice(e->device));
    TRY(ensure_skeleton(e, kind));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream[0];
    unsigned grid = (unsigned)(n < 148 * 8 ? n : 148 * 8);
    cbor_unpack_kernel<<<grid, 256, 0, st>>>(n, e->d_skel[kind], (u32)act_cbor_len(kind), (u32)act_rec_len(kind), (const u8*)cbor, (u8*)records, (u8*)status);
    e->launches += 1;
    CK(cudaGetLastError());
    return 0;
}
extern "C" int act_encode_cbor_dev(act_engine* e, int kind, size_t n, const void* records, void* cbor, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_encode_cbor_dev");
    if (n == 0) return 0;
    if (!cbor || !records) return fail_msg("act_encode_cbor_dev: null buffer");
    CK(cudaSetDevice(e->device));
    TRY(ensure_skeleton(e, kind));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream[0];
    size_t total = n * act_cbor_len(kind);
    unsigned grid = (unsigned)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    cbor_encode_kernel<<<grid, 256, 0, st>>>(n, e->d_skel[kind], (u32)act_cbor_len(kind), (u32)act_rec_len(kind), (const u8*)records, (u8*)cbor);
    e->launches += 1;
    CK(cudaGetLastError());
    return 0;
}
// host-buffer forms (one staging round trip; meant for ingest/egress next to the batch calls)
static int cbor_host_roundtrip(act_engine* e, int kind, size_t n, const uint8_t* in, size_t in_rec, uint8_t* out, size_t out_rec, uint8_t* status, bool unpack) {
    CK(cudaSetDevice(e->device));
    dev_buf<u8> d_in, d_out, d_st;
    TRY(ensure(d_in, n * in_rec)); TRY(ensure(d_out, n * out_rec));
    if (unpack) TRY(ensure(d_st, n));
    CK(cudaMemcpyAsync(d_in, in, n * in_rec, cudaMemcpyHostToDevice, e->stream[0]));
    TRY(unpack ? act_unpack_cbor_dev(e, kind, n, d_in, d_out, d_st, e->stream[0]) : act_encode_cbor_dev(e, kind, n, d_in, d_out, e->stream[0]));
    CK(cudaMemcpyAsync(out, d_out, n * out_rec, cudaMemcpyDeviceToHost, e->stream[0]));
    if (unpack) CK(cudaMemcpyAsync(status, d_st, n, cudaMemcpyDeviceToHost, e->stream[0]));
    CK(cudaStreamSynchronize(e->stream[0]));
    return 0;
}
extern "C" int act_unpack_cbor(act_engine* e, int kind, size_t n, const uint8_t* cbor, uint8_t* records, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (kind < 0 || kind > 3) return fail_msg("bad record kind");
    if (!cbor || !records || !status) return fail_msg("act_unpack_cbor: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_unpack_cbor(r, kind, m, cbor + lo * act_cbor_len(kind), records + lo * act_rec_len(kind), status + lo); });
    return cbor_host_roundtrip(e, kind, n, cbor, act_cbor_len(kind), records, act_rec_len(kind), status, true);
}
extern "C" int act_encode_cbor(act_engine* e, int kind, size_t n, const uint8_t* records, uint8_t* cbor) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (kind < 0 || kind > 3) return fail_msg("bad record kind");
    if (!cbor || !records) return fail_msg("act_encode_cbor: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_encode_cbor(r, kind, m, records + lo * act_rec_len(kind), cbor + lo * act_cbor_len(kind)); });
    return cbor_host_roundtrip(e, kind, n, records, act_rec_len(kind), cbor, act_cbor_len(kind), nullptr, false);
}

// ---------------------------------------------------------------------------------------------------
// client-side batch generators (act_prove.cuh): PreIssuance::request and CreditToken::prove_spend
// ---------------------------------------------------------------------------------------------------
#define ACT_PROVE_CHUNK 8192
extern "C" int act_batch_request_dev(act_engine* e, size_t n, const void* pre, const void* rnd, void* req, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_batch_request_dev");
    if (n == 0) return 0;
    if (!pre || !rnd || !req) return fail_msg("act_batch_request_dev: null buffer");
    CK(cudaSetDevice(e->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream[0];
    request_kernel<<<nblocks(n, ACT_ISSUE_BLOCK), ACT_ISSUE_BLOCK, 0, st>>>(sel_ctx(e), n, (const u32*)pre, (const u32*)rnd, (u32*)req);
    e->launches += 1;
    CK(cudaGetLastError());
    return 0;
}
extern "C" int act_batch_prove_spend_dev(act_engine* e, size_t n, const void* tokens, const void* charges, const void* rnd, const uint8_t seed[32],
                                         uint64_t first_index, void* proofs, void* prerefunds, void* status, void* stream) {
    if (!e) return fail_msg("null engine");
    NOT_MULTI(e, "act_batch_prove_spend_dev");
    if (n == 0) return 0;
    if (!tokens || !charges || !proofs || !prerefunds || !status || (!rnd && !seed)) return fail_msg("act_batch_prove_spend_dev: null buffer");
    CK(cudaSetDevice(e->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream[0];
    size_t cap = n < ACT_PROVE_CHUNK ? n : ACT_PROVE_CHUNK;
    TRY(ensure(e->pv_items, cap * ACT_ITEM_WORDS * 4, st));
    TRY(ensure(e->pv_cpts, cap * ACT_PROVE_PTS * 128, st));
    TRY(ensure(e->pv_cvs, cap * ACT_SPEND_CHUNKS * 32, st));
    TRY(ensure(e->pv_gammas, cap * 32, st));
    TRY(ensure(e->pv_aux, cap * 32, st));
    int sms = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device));
    for (size_t off = 0; off < n; off += ACT_PROVE_CHUNK) {
        size_t m = n - off < ACT_PROVE_CHUNK ? n - off : ACT_PROVE_CHUNK;
        prove_rng R;
        memset(&R, 0, sizeof R);
        R.rnd = rnd ? (const u32*)rnd + off * ACT_PROVE_SCALARS * 16 : nullptr;
        if (seed) memcpy(R.seed, seed, 32);
        R.first_index = first_index + off;
        const u32* tk = (const u32*)tokens + off * 40;
        const u32* ch = (const u32*)charges + off * 8;
        u8* stt = (u8*)status + off;
        unsigned grid = (unsigned)(m < (size_t)sms * 4 ? m : (size_t)sms * 4);
        prove_range_kernel<<<grid, ACT_L, 0, st>>>(sel_ctx(e), R, m, tk, ch, e->pv_cpts);
        spend_encode_kernel<<<nblocks(m * ACT_PROVE_PARTS, ACT_ENC_BLOCK), ACT_ENC_BLOCK, 0, st>>>(sel_ctx(e), m, e->pv_cpts, e->pv_items, ACT_PROVE_PTS, 5);
        prove_head_kernel<<<nblocks(m, ACT_HEAD_BLOCK), ACT_HEAD_BLOCK, 0, st>>>(sel_ctx(e), R, m, tk, e->pv_items, e->pv_aux, stt);
        spend_chunk_kernel<<<nblocks(m * ACT_SPEND_CHUNKS, ACT_HASH_BLOCK), ACT_HASH_BLOCK, 0, st>>>(sel_ctx(e), m, e->pv_items, e->pv_cvs);
        prove_challenge_kernel<<<nblocks(m, ACT_HASH_BLOCK), ACT_HASH_BLOCK, 0, st>>>(m, e->pv_cvs, e->pv_gammas);
        prove_finish_kernel<<<grid, ACT_L, 0, st>>>(sel_ctx(e), R, m, tk, ch, e->pv_items, e->pv_aux, e->pv_gammas, stt,
                                                   (u32*)proofs + off * ACT_PROOF_WORDS, (u32*)prerefunds + off * 24);
        e->launches += 6;
        CK(cudaGetLastError());
    }
    return 0;
}
// host-buffer forms
extern "C" int act_batch_request(act_engine* e, size_t n, const uint8_t* pre, const uint8_t* rnd, uint8_t* req) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!pre || !rnd || !req) return fail_msg("act_batch_request: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_request(r, m, pre + lo * 64, rnd + lo * 128, req + lo * 128); });
    CK(cudaSetDevice(e->device));
    dev_buf<u8> d_pre, d_rnd, d_req;
    TRY(ensure(d_pre, n * 64)); TRY(ensure(d_rnd, n * 128)); TRY(ensure(d_req, n * 128));
    CK(cudaMemcpyAsync(d_pre, pre, n * 64, cudaMemcpyHostToDevice, e->stream[0]));
    CK(cudaMemcpyAsync(d_rnd, rnd, n * 128, cudaMemcpyHostToDevice, e->stream[0]));
    TRY(act_batch_request_dev(e, n, d_pre, d_rnd, d_req, e->stream[0]));
    CK(cudaMemcpyAsync(req, d_req, n * 128, cudaMemcpyDeviceToHost, e->stream[0]));
    CK(cudaStreamSynchronize(e->stream[0]));
    return 0;
}
extern "C" int act_batch_prove_spend(act_engine* e, size_t n, const uint8_t* tokens, const uint8_t* charges, const uint8_t* rnd, const uint8_t seed[32],
                                     uint64_t first_index, uint8_t* proofs, uint8_t* prerefunds, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!tokens || !charges || !proofs || !prerefunds || !status || (!rnd && !seed)) return fail_msg("act_batch_prove_spend: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_prove_spend(r, m, tokens + lo * 160, charges + lo * 32, rnd ? rnd + lo * (size_t)ACT_PROVE_SCALARS * 64 : nullptr, seed, first_index + lo,
                                     proofs + lo * ACT_PROOF_BYTES, prerefunds + lo * 96, status + lo); });
    CK(cudaSetDevice(e->device));
    dev_buf<u8> d_tk, d_ch, d_rnd, d_pf, d_pr, d_st;
    TRY(ensure(d_tk, n * 160)); TRY(ensure(d_ch, n * 32)); TRY(ensure(d_pf, n * ACT_PROOF_BYTES));
    TRY(ensure(d_pr, n * 96)); TRY(ensure(d_st, n));
    if (rnd) { TRY(ensure(d_rnd, n * ACT_PROVE_SCALARS * 64)); CK(cudaMemcpyAsync(d_rnd, rnd, n * ACT_PROVE_SCALARS * 64, cudaMemcpyHostToDevice, e->stream[0])); }
    CK(cudaMemcpyAsync(d_tk, tokens, n * 160, cudaMemcpyHostToDevice, e->stream[0]));
    CK(cudaMemcpyAsync(d_ch, charges, n * 32, cudaMemcpyHostToDevice, e->stream[0]));
    TRY(act_batch_prove_spend_dev(e, n, d_tk, d_ch, d_rnd, seed, first_index, d_pf, d_pr, d_st, e->stream[0]));
    CK(cudaMemcpyAsync(proofs, d_pf, n * ACT_PROOF_BYTES, cudaMemcpyDeviceToHost, e->stream[0]));
    CK(cudaMemcpyAsync(prerefunds, d_pr, n * 96, cudaMemcpyDeviceToHost, e->stream[0]));
    CK(cudaMemcpyAsync(status, d_st, n, cudaMemcpyDeviceToHost, e->stream[0]));
    CK(cudaStreamSynchronize(e->stream[0]));
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// multi-device engine: one replica per GPU, contiguous shards, no cross-GPU arithmetic (SURVEY 8e)
// ---------------------------------------------------------------------------------------------------
extern "C" int act_engine_create_multi(act_engine** out, const int* devices, int n_devices, const uint8_t h[96], const uint8_t sk_x[32], const uint8_t pk_w[32]) {
    if (!out || !devices || n_devices < 1 || !h || !sk_x || !pk_w) return fail_msg("act_engine_create_multi: bad argument");
    *out = nullptr;
    // (a device listed twice gets two replicas: wasteful, but it lets a one-GPU box exercise the sharded path)
    act_engine* m = new act_engine();
    m->device = devices[0];
    for (int i = 0; i < n_devices; i++) {
        act_engine* r = nullptr;
        int rc = act_engine_create(&r, devices[i], h, sk_x, pk_w);
        if (rc) { act_engine_destroy(m); return rc; }
        m->replicas.push_back(r);
        m->spend_chunk = r->spend_chunk;
    }
    // direct NVLink copies into replica 0 for the gather of status + nullifiers (33 B per proof)
    cudaSetDevice(devices[0]);
    for (int i = 1; i < n_devices; i++) {
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, devices[0], devices[i]) == cudaSuccess && can) {
            cudaError_t pe = cudaDeviceEnablePeerAccess(devices[i], 0);
            if (pe != cudaSuccess) cudaGetLastError();   // already enabled, or unsupported: cudaMemcpyPeerAsync stages instead
        }
    }
    *out = m;
    return 0;
}
extern "C" int act_engine_replica_count(const act_engine* e) { return e ? (e->replicas.empty() ? 1 : (int)e->replicas.size()) : 0; }
extern "C" act_engine* act_engine_replica(act_engine* e, int i) {
    if (!e) return nullptr;
    if (e->replicas.empty()) return i == 0 ? e : nullptr;
    return (i >= 0 && (size_t)i < e->replicas.size()) ? e->replicas[(size_t)i] : nullptr;
}

// ---------------------------------------------------------------------------------------------------
// two-pass forms: verification and signing as separate calls.  A host that owns ONE RNG (the reference's
// `impl CryptoRngCore`, src/lib.rs:626,785) verifies, counts the accepted requests, draws exactly 128 bytes for each of
// them in slice order -- what a loop of issue() / refund() calls would have drawn (:638-643, 842-846) -- and signs.
// ---------------------------------------------------------------------------------------------------
// accepted-before-i positions in the compact randomness; fails if it is shorter than 128 bytes per accepted request
static int seq_positions(const uint8_t* st, size_t n, std::vector<u32>& idx, size_t stream_len, size_t* consumed) {
    size_t acc = 0;
    idx.resize(n);
    for (size_t i = 0; i < n; i++) { idx[i] = (u32)acc; if (st[i] == 0) acc++; }
    if (consumed) *consumed = acc * 128;
    if (acc * 128 > stream_len) return fail_msg("signing pass: the randomness is shorter than 128 bytes per accepted request");
    return 0;
}
static size_t count_accepted(const uint8_t* st, size_t n) { size_t a = 0; for (size_t i = 0; i < n; i++) a += st[i] == 0; return a; }

extern "C" int act_batch_issue_verify(act_engine* e, size_t n, const uint8_t* req, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!req || !status) return fail_msg("act_batch_issue_verify: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) { return act_batch_issue_verify(r, m, req + lo * 128, status + lo); });
    host_io h = {{req, nullptr, nullptr}, {128, 0, 0}, {nullptr, nullptr, status}, {0, 0, 1}};
    return run_chunked(e, n, ACT_SMALL_CHUNK, h, [&](int, cudaStream_t st, size_t m, io_slot& io) {
        issue_mode_kernel<<<nblocks(m, ACT_ISSUE_BLOCK), ACT_ISSUE_BLOCK, 0, st>>>(sel_ctx(e), m, (const u32*)io.in[0].p, nullptr, nullptr, nullptr, io.st, ACT_MODE_VERIFY, nullptr);
        e->launches += 1;
        CK(cudaGetLastError());
        return 0;
    });
}
extern "C" int act_batch_issue_sign(act_engine* e, size_t n, const uint8_t* req, const uint8_t* c, const uint8_t* status, const uint8_t* rnd, size_t rnd_len,
                                    uint8_t* resp) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!req || !c || !status || !resp || (!rnd && rnd_len)) return fail_msg("act_batch_issue_sign: null buffer");
    if (n >= 0xffffffffu) return fail_msg("act_batch_issue_sign: batch too large");
    if (is_multi(e)) {
        if (count_accepted(status, n) * 128 > rnd_len) return fail_msg("signing pass: the randomness is shorter than 128 bytes per accepted request");
        return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
            size_t before = count_accepted(status, lo), mine = count_accepted(status + lo, m);
            return act_batch_issue_sign(r, m, req + lo * 128, c + lo * 32, status + lo, rnd + before * 128, mine * 128, resp + lo * 160);
        });
    }
    CK(cudaSetDevice(e->device));
    std::vector<u32> idx;
    size_t used = 0;
    TRY(seq_positions(status, n, idx, rnd_len, &used));
    cudaStream_t st = e->stream[0];
    size_t rnd_bytes = used ? used : 128;
    dev_buf<u8> d_req, d_c, d_rnd, d_resp, d_st; dev_buf<u32> d_idx;
    wipe_dev_on_exit rnd_wipe{nullptr, rnd_bytes, st};   // the device copy of the signer randomness, if a step below fails
    TRY(ensure(d_req, n * 128)); TRY(ensure(d_c, n * 32)); TRY(ensure(d_resp, n * 160));
    TRY(ensure(d_st, n)); TRY(ensure(d_idx, n * 4)); TRY(ensure(d_rnd, rnd_bytes));
    rnd_wipe.p = d_rnd;
    CK(cudaMemcpyAsync(d_req, req, n * 128, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_c, c, n * 32, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_st, status, n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_idx, idx.data(), n * 4, cudaMemcpyHostToDevice, st));
    if (used) CK(cudaMemcpyAsync(d_rnd, rnd, used, cudaMemcpyHostToDevice, st));
    issue_mode_kernel<<<nblocks(n, ACT_ISSUE_BLOCK), ACT_ISSUE_BLOCK, 0, st>>>(sel_ctx(e), n, (const u32*)d_req.p, (const u32*)d_c.p, (const u32*)d_rnd.p, (u32*)d_resp.p, d_st, ACT_MODE_SIGN, d_idx);
    e->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(resp, d_resp, n * 160, cudaMemcpyDeviceToHost, st));
    CK(cudaMemsetAsync(d_rnd, 0, rnd_bytes, st));     // the device copy of the signer randomness
    rnd_wipe.p = nullptr;
    TRY(scrub_after_signing(e, st, -1));
    CK(cudaStreamSynchronize(st));
    return 0;
}
// one replica's verification pass (key_ids optional)
static int spend_verify_host(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* key_ids, uint8_t* nullifiers, uint8_t* status, uint8_t* kprime) {
    CK(cudaSetDevice(e->device));
    TRY(ensure_spend_scratch(e, n));
    host_io h = {{proofs, key_ids, nullptr}, {ACT_PROOF_BYTES, 1, 0}, {kprime, nullifiers, status}, {128, 32, 1}};
    return run_chunked(e, n, e->spend_chunk, h, [&](int s, cudaStream_t st, size_t m, io_slot& io) {
        return spend_chunk_launch(e, &e->scratch[s], st, m, (const u32*)io.in[0].p, nullptr, nullptr, (u32*)io.out[1].p, io.st, (u32*)io.out[0].p,
                                  key_ids ? io.in[1].p : nullptr);
    }, true);
}
extern "C" int act_batch_spend_verify(act_engine* e, size_t n, const uint8_t* proofs, uint8_t* nullifiers, uint8_t* status, uint8_t* kprime) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!proofs || !nullifiers || !status || !kprime) return fail_msg("act_batch_spend_verify: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_spend_verify(r, m, proofs + lo * ACT_PROOF_BYTES, nullifiers + lo * 32, status + lo, kprime + lo * 128); });
    return spend_verify_host(e, n, proofs, nullptr, nullifiers, status, kprime);
}
extern "C" int act_batch_spend_verify_keyed(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* key_ids, uint8_t* nullifiers, uint8_t* status,
                                            uint8_t* kprime) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!proofs || !key_ids || !nullifiers || !status || !kprime) return fail_msg("act_batch_spend_verify_keyed: null buffer");
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_spend_verify_keyed(r, m, proofs + lo * ACT_PROOF_BYTES, key_ids + lo, nullifiers + lo * 32, status + lo, kprime + lo * 128); });
    return spend_verify_host(e, n, proofs, key_ids, nullifiers, status, kprime);
}
extern "C" int act_batch_refund_sign(act_engine* e, size_t n, const uint8_t* kprime, const uint8_t* status, const uint8_t* rnd, size_t rnd_len, uint8_t* refunds) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!kprime || !status || !refunds || (!rnd && rnd_len)) return fail_msg("act_batch_refund_sign: null buffer");
    if (n >= 0xffffffffu) return fail_msg("act_batch_refund_sign: batch too large");
    if (is_multi(e)) {
        if (count_accepted(status, n) * 128 > rnd_len) return fail_msg("signing pass: the randomness is shorter than 128 bytes per accepted request");
        return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
            size_t before = count_accepted(status, lo), mine = count_accepted(status + lo, m);
            return act_batch_refund_sign(r, m, kprime + lo * 128, status + lo, rnd + before * 128, mine * 128, refunds + lo * 128);
        });
    }
    CK(cudaSetDevice(e->device));
    std::vector<u32> idx;
    size_t used = 0;
    TRY(seq_positions(status, n, idx, rnd_len, &used));
    cudaStream_t st = e->stream[0];
    size_t rnd_bytes = used ? used : 128;
    dev_buf<u8> d_kp, d_rnd, d_ref, d_st; dev_buf<u32> d_idx;
    wipe_dev_on_exit rnd_wipe{nullptr, rnd_bytes, st};   // the device copy of the signer randomness, if a step below fails
    TRY(ensure(d_kp, n * 128)); TRY(ensure(d_ref, n * 128)); TRY(ensure(d_st, n));
    TRY(ensure(d_idx, n * 4)); TRY(ensure(d_rnd, rnd_bytes));
    rnd_wipe.p = d_rnd;
    CK(cudaMemcpyAsync(d_kp, kprime, n * 128, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_st, status, n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_idx, idx.data(), n * 4, cudaMemcpyHostToDevice, st));
    if (used) CK(cudaMemcpyAsync(d_rnd, rnd, used, cudaMemcpyHostToDevice, st));
    refund_sign_seq_kernel<<<nblocks(n, ACT_SIGN_BLOCK), ACT_SIGN_BLOCK, 0, st>>>(sel_ctx(e), n, nullptr, (const u32*)d_rnd.p, (const u32*)d_kp.p, d_st, (u32*)d_ref.p, nullptr, d_idx, nullptr);
    e->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(refunds, d_ref, n * 128, cudaMemcpyDeviceToHost, st));
    CK(cudaMemsetAsync(d_rnd, 0, rnd_bytes, st));
    rnd_wipe.p = nullptr;
    TRY(scrub_after_signing(e, st, -1));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// sequential-RNG contract (SURVEY H5): outputs identical to a loop of issue() / refund() calls over ONE shared RNG whose
// bytes the caller has already laid out as a stream: request i uses the 128 bytes at offset 128 * (accepted requests before i).
// = verification pass, host scan of the accept bits, signing pass.
// ---------------------------------------------------------------------------------------------------
extern "C" int act_batch_issue_seq(act_engine* e, size_t n, const uint8_t* req, const uint8_t* c, const uint8_t* rnd_stream, size_t rnd_stream_len,
                                   uint8_t* resp, uint8_t* status, size_t* consumed) {
    if (!e) return fail_msg("null engine");
    if (consumed) *consumed = 0;
    if (n == 0) return 0;
    if (!req || !c || !resp || !status || (!rnd_stream && rnd_stream_len)) return fail_msg("act_batch_issue_seq: null buffer");
    int rc = act_batch_issue_verify(e, n, req, status);
    if (rc) return rc;
    size_t used = count_accepted(status, n) * 128;
    if (used > rnd_stream_len) return fail_msg("sequential-RNG call: the RNG stream is shorter than 128 bytes per accepted request");
    if ((rc = act_batch_issue_sign(e, n, req, c, status, rnd_stream, used, resp))) return rc;
    if (consumed) *consumed = used;
    return 0;
}
extern "C" int act_batch_verify_spend_and_refund_seq(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* rnd_stream, size_t rnd_stream_len,
                                                      uint8_t* refunds, uint8_t* nullifiers, uint8_t* status, size_t* consumed) {
    if (!e) return fail_msg("null engine");
    if (consumed) *consumed = 0;
    if (n == 0) return 0;
    if (!proofs || !refunds || !nullifiers || !status || (!rnd_stream && rnd_stream_len)) return fail_msg("act_batch_verify_spend_and_refund_seq: null buffer");
    std::vector<uint8_t> kprime(n * 128);
    int rc = act_batch_spend_verify(e, n, proofs, nullifiers, status, kprime.data());
    if (rc) return rc;
    size_t used = count_accepted(status, n) * 128;
    if (used > rnd_stream_len) return fail_msg("sequential-RNG call: the RNG stream is shorter than 128 bytes per accepted request");
    if ((rc = act_batch_refund_sign(e, n, kprime.data(), status, rnd_stream, used, refunds))) return rc;
    if (consumed) *consumed = used;
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// the issuer's whole batch step in one call: verify + refund on every replica, gather of status + nullifiers (33 B per
// proof) to replica 0 over NVLink (cudaMemcpyPeerAsync from each replica's device copy), replay screen there.
// What examples/act.rs:60-77 does per request -- nullifier check, then refund -- for a slice; a proof whose nullifier
// occurred earlier in the slice or in `seen` gets status 3 (DoubleSpendError) and NO refund (zero-filled, as the reference
// never calls refund() for it); its nullifier is kept so that the caller can tell which token was replayed.
// ---------------------------------------------------------------------------------------------------
// The screen of a keyed batch: proof i against the store of its key's slot (map), each store in slice order over its own proofs.
// Every store is prepared (lookup, key check, growth) before the first is committed, so a call that fails changes no store.
static int screen_stores_keyed(act_engine* r0, size_t n, const uint8_t* key_ids, const u8* g_st, const u8* g_nul,
                               const std::vector<act_nullifier_store*>& stores, const act_store_map& map, u8* d_out, cudaStream_t st) {
    size_t D = stores.size();
    std::vector<size_t> adds(D, 0);   // proofs per store: a bound on what it may record
    for (size_t i = 0; i < n; i++) {
        u8 j = key_ids[i] < ACT_KEY_SLOTS ? map.of_slot[key_ids[i]] : 0xFF;
        if (j != 0xFF) adds[j]++;
    }
    dev_buf<u8> d_kid;
    std::vector<dev_buf<u8>> masked(D);
    TRY(ensure(d_kid, n));
    for (size_t j = 0; j < D; j++) if (adds[j]) TRY(ensure(masked[j], n));
    CK(cudaMemcpyAsync(d_kid, key_ids, n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_out, g_st, n, cudaMemcpyDeviceToDevice, st));
    for (size_t j = 0; j < D; j++) {
        if (!adds[j]) continue;
        store_mask_kernel<<<nblocks(n, 256), 256, 0, st>>>(n, g_st, d_kid, map, (u32)j, masked[j]);
        r0->launches += 1;
        CK(cudaGetLastError());
        TRY(store_prepare(stores[j], n, masked[j], g_nul, 1, adds[j], st));
    }
    for (size_t j = 0; j < D; j++) {
        if (!adds[j]) continue;
        TRY(store_commit(stores[j], n, g_nul, masked[j], 1, st));
        store_merge_kernel<<<nblocks(n, 256), 256, 0, st>>>(n, masked[j], d_kid, map, (u32)j, d_out);
        r0->launches += 1;
        CK(cudaGetLastError());
    }
    return 0;
}
static int ensure_gather(act_engine* r, size_t m) {
    CK(cudaSetDevice(r->device));
    TRY(ensure(r->g_st, m + 16));
    TRY(ensure(r->g_nul, m * 32 + 16));
    return 0;
}
// The screen runs against `seen` (n_seen keys, host memory) when stores is null.  Otherwise it runs against stores[0] for every
// proof (key_ids null), or proof i against stores[key_ids[i]] (ACT_KEY_SLOTS entries: the keyed call), recording the survivors.
static int verify_refund_and_screen(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* key_ids, const uint8_t* rnd, size_t n_seen,
                                    const uint8_t* seen, act_nullifier_store* const* stores, uint8_t* refunds, uint8_t* nullifiers, uint8_t* status) {
    std::vector<act_engine*> reps = e->replicas.empty() ? std::vector<act_engine*>{e} : e->replicas;
    // the stores this call screens against, and (keyed) the index of each slot's store among them (0xFF: slot without a key)
    std::vector<act_nullifier_store*> distinct;
    act_store_map map;
    memset(map.of_slot, 0xff, sizeof map.of_slot);
    if (stores && !key_ids) distinct.push_back(stores[0]);
    if (stores && key_ids) {
        uint32_t held = slots_held(reps[0]);
        for (int k = 0; k < ACT_KEY_SLOTS; k++) {
            if (!(held >> k & 1u)) continue;
            if (!stores[k]) return fail_msg(("act_batch_verify_spend_and_refund_keyed: slot " + std::to_string(k) + " holds a key but has no store").c_str());
            size_t j = 0;
            while (j < distinct.size() && distinct[j] != stores[k]) j++;
            if (j == distinct.size()) distinct.push_back(stores[k]);
            map.of_slot[k] = (u8)j;
        }
    }
    for (act_nullifier_store* s : distinct)
        if (s->device != reps[0]->device)
            return fail_msg(key_ids ? "act_batch_verify_spend_and_refund_keyed: every store must be on the device of replica 0 (where the gather lands)"
                                    : "act_batch_verify_spend_and_refund_recorded: the store must be on the device of replica 0 (where the gather lands)");
    size_t G = reps.size();
    for (size_t g = 0; g < G; g++) TRY(ensure_gather(reps[g], shard_lo(n, g + 1, G) - shard_lo(n, g, G)));
    int rc;
    for (auto* r : reps) r->g_keep = true;
    if (G == 1) rc = verify_spend_host(reps[0], n, proofs, key_ids, rnd, refunds, nullifiers, status);
    else {
        rc = shard_over(reps, n, [&](act_engine* r, size_t lo, size_t m) {
            return verify_spend_host(r, m, proofs + lo * ACT_PROOF_BYTES, key_ids ? key_ids + lo : nullptr, rnd + lo * 128, refunds + lo * 128,
                                     nullifiers + lo * 32, status + lo); });
    }
    for (auto* r : reps) r->g_keep = false;
    if (rc) return rc;
    act_engine* r0 = reps[0];
    CK(cudaSetDevice(r0->device));
    cudaStream_t st = r0->stream[0];
    dev_buf<u8> d_st, d_nul, d_seen, d_out;
    if (G > 1) {
        TRY(ensure(d_st, n)); TRY(ensure(d_nul, n * 32));
        for (size_t g = 0; g < G; g++) {
            size_t lo = shard_lo(n, g, G), m = shard_lo(n, g + 1, G) - lo;
            if (!m) continue;
            CK(cudaMemcpyPeerAsync(d_st.p + lo, r0->device, reps[g]->g_st, reps[g]->device, m, st));
            CK(cudaMemcpyPeerAsync(d_nul.p + lo * 32, r0->device, reps[g]->g_nul, reps[g]->device, m * 32, st));
        }
    }
    TRY(ensure(d_out, n));
    if (n_seen) { TRY(ensure(d_seen, n_seen * 32)); CK(cudaMemcpyAsync(d_seen, seen, n_seen * 32, cudaMemcpyHostToDevice, st)); }
    const u8* g_st = G > 1 ? d_st.p : r0->g_st.p;
    const u8* g_nul = G > 1 ? d_nul.p : r0->g_nul.p;
    if (!stores) TRY(act_flag_replays_dev(r0, n, g_st, g_nul, n_seen, d_seen, d_out, st));
    else if (!key_ids) TRY(act_nullifier_store_screen_dev(distinct[0], n, g_st, g_nul, d_out, 1, st));
    else TRY(screen_stores_keyed(r0, n, key_ids, g_st, g_nul, distinct, map, d_out, st));
    CK(cudaMemcpyAsync(status, d_out, n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (size_t i = 0; i < n; i++) if (status[i] == 3) memset(refunds + i * 128, 0, 128);
    return 0;
}
extern "C" int act_batch_verify_spend_and_refund_screened(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* rnd, size_t n_seen, const uint8_t* seen,
                                                           uint8_t* refunds, uint8_t* nullifiers, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!proofs || !rnd || !refunds || !nullifiers || !status || (n_seen && !seen)) return fail_msg("act_batch_verify_spend_and_refund_screened: null buffer");
    return verify_refund_and_screen(e, n, proofs, nullptr, rnd, n_seen, seen, nullptr, refunds, nullifiers, status);
}
extern "C" int act_batch_verify_spend_and_refund_recorded(act_engine* e, act_nullifier_store* s, size_t n, const uint8_t* proofs, const uint8_t* rnd,
                                                           uint8_t* refunds, uint8_t* nullifiers, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (!s) return fail_msg("null store");
    if (n == 0) return 0;
    if (!proofs || !rnd || !refunds || !nullifiers || !status) return fail_msg("act_batch_verify_spend_and_refund_recorded: null buffer");
    return verify_refund_and_screen(e, n, proofs, nullptr, rnd, 0, nullptr, &s, refunds, nullifiers, status);
}
extern "C" int act_batch_verify_spend_and_refund_keyed(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* key_ids, const uint8_t* rnd,
                                                        act_nullifier_store* const* stores, uint8_t* refunds, uint8_t* nullifiers, uint8_t* status) {
    if (!e) return fail_msg("null engine");
    if (n == 0) return 0;
    if (!proofs || !key_ids || !rnd || !refunds || !nullifiers || !status) return fail_msg("act_batch_verify_spend_and_refund_keyed: null buffer");
    if (stores) return verify_refund_and_screen(e, n, proofs, key_ids, rnd, 0, nullptr, stores, refunds, nullifiers, status);
    if (is_multi(e)) return shard_over_replicas(e, n, [&](act_engine* r, size_t lo, size_t m) {
        return act_batch_verify_spend_and_refund_keyed(r, m, proofs + lo * ACT_PROOF_BYTES, key_ids + lo, rnd + lo * 128, nullptr, refunds + lo * 128,
                                                       nullifiers + lo * 32, status + lo); });
    return verify_spend_host(e, n, proofs, key_ids, rnd, refunds, nullifiers, status);
}
