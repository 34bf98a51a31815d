// act_device.cuh -- per-thread bodies of the batch kernels: scalar multiplication strategies,
// transcript assembly, and the issue / refund / to_credit_token equations.
//
// Every `*_thread` function is the whole body of one CUDA thread of the kernel of the same name in
// act_kernels.cu; they are plain functions of (context, index, buffers) so that tests/hostsim can
// run the identical logic on the CPU for small cases.  Reference equations: /root/reference
// src/lib.rs:621-663 (issue), :781-869 (refund), :528-562 and :1217-1253 (client checks),
// src/transcript.rs:54-155 (transcript layout).
//
// Secret-dependent work (x, alpha, (e+x)^-1) uses the *_ct routines: signed fixed windows, table
// selection by a full masked scan, no secret-dependent branch or address.  Public data (everything
// in a proof, gamma, e) uses direct table indexing.
#pragma once
#include "blake3.cuh"
#include "fe25519.cuh"
#include "ge25519.cuh"
#include "sc25519.cuh"

// ---- status codes (include/act_engine.h) ----------------------------------------------------------
#define ACT_ST_OK 0
#define ACT_ST_INVALID_ISSUANCE_REQUEST_PROOF 1
#define ACT_ST_INVALID_ISSUANCE_RESPONSE_PROOF 2
#define ACT_ST_INVALID_REFUND_PROOF 4
#define ACT_ST_IDENTITY_POINT 6
#define ACT_ST_INVALID_CLIENT_SPEND_PROOF 7
#define ACT_ST_DECODE_INVALID_POINT 0x81

#define ACT_FLAG_BAD_POINT 1u
#define ACT_FLAG_IDENTITY 2u
#define ACT_FLAG_BAD_PROOF 4u
#define ACT_FLAG_NO_KEY 8u          // keyed verification: the proof's key id names no key (finish: status 7)

// issuer key slots of an engine (include/act_engine.h); a keyed spend names one per proof
#ifndef ACT_KEY_SLOTS
#define ACT_KEY_SLOTS 16
#endif

// ---- layout constants -----------------------------------------------------------------------------
#define ACT_L 128
#define ACT_PROOF_WORDS (526 * 8)
#define ACT_ITEMS 390               // "spend" transcript items: k, A', B, A1, A2, com[128], C'[128][2], C
#define ACT_ITEM_WORDS (ACT_ITEMS * 8)
#define ACT_SPEND_BYTES 15784u      // 184 + 40*390
#define ACT_SPEND_CHUNKS 16

// fixed-base tables (public scalars): signed radix 2^bits, entry |d| in 0..2^(bits-1) (0 = identity), affine Niels,
// ceil(254/bits) windows -> that many mixed additions per scalar multiplication and no doublings.  The width is a
// property of each table (fb_tab): the two bases every range-proof commitment touches (H1, H3) get 2^16 windows
// (16 additions, 50 MB per base), G and H2 get 2^13 (20 additions, 7.9 MB per base); all L2/HBM resident.
#ifndef ACT_FB_BITS
#define ACT_FB_BITS 13          // G, H2
#endif
#ifndef ACT_FB_BITS_HOT
#define ACT_FB_BITS_HOT 16      // H1, H3
#endif
// table construction: one thread per (window, part of ACT_FB_PART entries), entries converted to affine with batched
// inversions of ACT_FB_BATCH points
#define ACT_FB_PART 512
#define ACT_FB_BATCH 16
#if defined(__CUDACC__)
#define ACT_HD __host__ __device__ __forceinline__
#else
#define ACT_HD static inline
#endif
struct fb_tab {
    const ge_niels* p;
    u32 bits, win, ent;     // window width, number of windows, entries per window (2^(bits-1) + 1)
};
ACT_HD u32 fb_win_of(u32 bits) { return (253u + bits) / bits; }
ACT_HD u32 fb_ent_of(u32 bits) { return (1u << (bits - 1)) + 1u; }
ACT_HD size_t fb_size_of(u32 bits) { return (size_t)fb_win_of(bits) * fb_ent_of(bits); }
ACT_HD u32 fb_parts_of(u32 bits) { u32 n = fb_ent_of(bits) - 1; return n >= ACT_FB_PART ? n / ACT_FB_PART : 1; }
// constant-time basepoint table: signed radix-16, 64 windows, |d| in 0..8
#define ACT_CT_WIN 64
#define ACT_CT_ENT 9
#define ACT_CT_SIZE (ACT_CT_WIN * ACT_CT_ENT)

// number of parts the range-proof scalars are split into (shared doubling chain), 1, 2 or 4
#ifndef ACT_RANGE_SPLIT
#define ACT_RANGE_SPLIT 4
#endif

#define ACT_BASE_G 0
#define ACT_BASE_H1 1
#define ACT_BASE_H2 2
#define ACT_BASE_H3 3
#define ACT_BASE_W 4     // the issuer's public key: fixed per engine, so the client-side checks use a table for it too
#define ACT_FB_BASES 5

struct act_ctx {
    fb_tab fb[ACT_FB_BASES]; // vartime fixed-base tables for G, H1, H2, H3, W (global memory, L2 resident)
    const ge_niels* ct_g;    // constant-time table for G
    sc x;                    // issuer secret
    ge W;                    // issuer public key
    ge W_half;               // (1/2 mod l) * W: lets X_G = G*e + W be produced as a half for the batched encode
    u32 h_enc[3][8];         // encodings of H1..H3
    u32 prefix[4][48];       // transcript prefixes "request","respond","refund","spend" as LE words, zero padded
    u32 prefix_len[4];       // 186, 186, 185, 184 bytes
};
#define ACT_TR_REQUEST 0
#define ACT_TR_RESPOND 1
#define ACT_TR_REFUND 2
#define ACT_TR_SPEND 3

#if ACT_PTX
#define ACT_ATOMIC_OR(p, v) atomicOr((p), (v))
#else
#define ACT_ATOMIC_OR(p, v) (*(p) |= (v))
#endif

// ---- 32-byte loads/stores ---------------------------------------------------------------------------
ACT_FN void load8(u32* w, const u32* p) {
#if ACT_PTX
    uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
    uint4 b = __ldg(reinterpret_cast<const uint4*>(p) + 1);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
#else
    for (int i = 0; i < 8; i++) w[i] = p[i];
#endif
}
ACT_FN void store8(u32* p, const u32* w) {
#if ACT_PTX
    reinterpret_cast<uint4*>(p)[0] = make_uint4(w[0], w[1], w[2], w[3]);
    reinterpret_cast<uint4*>(p)[1] = make_uint4(w[4], w[5], w[6], w[7]);
#else
    for (int i = 0; i < 8; i++) p[i] = w[i];
#endif
}
// plain (coherent) 32-byte load: for scratch written earlier by the same kernel (never __ldg there)
ACT_FN void load8_rw(u32* w, const u32* p) {
#if ACT_PTX
    uint4 a = reinterpret_cast<const uint4*>(p)[0];
    uint4 b = reinterpret_cast<const uint4*>(p)[1];
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
#else
    for (int i = 0; i < 8; i++) w[i] = p[i];
#endif
}
ACT_FN void store8_zero(u32* p) {
    u32 z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    store8(p, z);
}
ACT_FN sc load_scalar(const u32* p) { u32 w[8]; load8(w, p); return sc_from_words(w); }
ACT_FN void store_scalar(u32* p, const sc& s) { store8(p, s.v); }
ACT_FN u32 load_point(ge* out, const u32* p) { u32 w[8]; load8(w, p); return ristretto_decode_(out, w); }
ACT_FN void store_point(u32* p, const ge& q) { u32 w[8]; ristretto_encode_(w, &q); store8(p, w); }
ACT_FN void load_fe(fe* f, const u32* p) { load8(f->v, p); }
ACT_FN void store_fe(u32* p, const fe& f) { store8(p, f.v); }
ACT_FN ge_niels load_niels(const ge_niels* p) {
    ge_niels r;
    const u32* q = reinterpret_cast<const u32*>(p);
    load8(r.ypx.v, q); load8(r.ymx.v, q + 8); load8(r.xy2d.v, q + 16);
    return r;
}

// L1 prefetch of a table line that a later step of the same thread will read (no register is tied up while the
// line travels from L2 / HBM)
#ifndef ACT_PREFETCH
#define ACT_PREFETCH 1
#endif
ACT_FN void prefetch_line(const void* p) {
#if ACT_PTX && ACT_PREFETCH
    asm volatile("prefetch.L1 [%0];" ::"l"(p));
#else
    (void)p;
#endif
}

// ---- fixed-base accumulation (public scalars) ---------------------------------------------------------
// signed radix-2^W digit i of a scalar s < 2^253: raw window plus the carry of the window below, mapped to
// (-2^(W-1), 2^(W-1)].  Public scalars only (the carry is data dependent).
ACT_FN int fb_digit(const sc& s, u32 W, int i, u32* carry) {
    u32 bit = W * (u32)i, w = bit >> 5, sh = bit & 31u;
    u32 lo = s.v[w], hi = (w + 1 < 8) ? s.v[w + 1] : 0u;
    u32 raw = (sh ? ((lo >> sh) | (hi << (32u - sh))) : lo) & ((1u << W) - 1u);
    int d = (int)(raw + *carry);
    *carry = (d > (1 << (W - 1))) ? 1u : 0u;
    return d - (int)(*carry << W);
}
// acc += (negate ? -s : s) * B using the wide-window table of B: T.win mixed additions, no doublings.
ACT_FN ge fb_accumulate(ge acc, const fb_tab& T, const sc& s, bool negate) {
    u32 carry = 0;
    int d = fb_digit(s, T.bits, 0, &carry);
    ACT_NOUNROLL for (u32 i = 0; i < T.win; i++) {
        u32 neg = (d < 0) ? 1u : 0u;
        u32 idx = (u32)(d < 0 ? -d : d);
        if (negate) neg ^= 1u;
        const ge_niels* cur = T.p + (size_t)i * T.ent + idx;
        if (i + 1 < T.win) {   // next window's entry (96 B: may straddle two lines) travels while this addition runs
            d = fb_digit(s, T.bits, (int)i + 1, &carry);
            const ge_niels* nxt = T.p + (size_t)(i + 1) * T.ent + (u32)(d < 0 ? -d : d);
            prefetch_line(nxt); prefetch_line(reinterpret_cast<const u8*>(nxt) + 95);
        }
        acc = ge_add_niels_n<true>(acc, load_niels(cur), neg);    // public scalars: the variable-time add/sub forms
    }
    return acc;
}
// acc += alpha * G with a secret alpha: radix-16, all 9 entries of each window scanned
ACT_FN ge fb_accumulate_ct(ge acc, const ge_niels* tab, const sc& s) {
    sc b = sc_bias<4>(s);
    ACT_NOUNROLL for (int i = 0; i < ACT_CT_WIN; i++) {
        int d = sc_digit<4>(b, i);
        u32 neg = ((u32)d) >> 31;
        u32 idx = (u32)((d ^ (d >> 31)) - (d >> 31));
        ge_niels e = ge_niels_identity();
        ACT_NOUNROLL for (u32 k = 1; k < ACT_CT_ENT; k++) {
            ge_niels t = load_niels(tab + i * ACT_CT_ENT + k);
            u32 hit = (idx == k);
            e.ypx = fe_select(e.ypx, t.ypx, hit); e.ymx = fe_select(e.ymx, t.ymx, hit); e.xy2d = fe_select(e.xy2d, t.xy2d, hit);
        }
        acc = ge_add_niels(acc, ge_niels_cneg(e, neg));
    }
    return acc;
}

// ---- variable-base: signed radix-16 windows over a per-thread table of 0..8 multiples -------------------
// One entry = 128 contiguous bytes = one cache line, moved with 16-byte vector accesses.  (As a plain
// per-thread array in local memory the divergent lookups fetched a 32-byte sector for every 4 bytes
// used -- ncu: 1.6 B/sector, 8 MB of DRAM reads per proof -- so the range kernel keeps its tables in a
// global scratch buffer instead; the small kernels keep them on the stack through the same accessors.)
struct alignas(16) vb_table { ge_cached e[9]; };

ACT_FN void tab_store(vb_table* t, u32 idx, const ge_cached& c) {
    u32* q = reinterpret_cast<u32*>(&t->e[idx]);
    store8(q, c.YpX.v); store8(q + 8, c.YmX.v); store8(q + 16, c.Z.v); store8(q + 24, c.T2d.v);
}
ACT_FN ge_cached tab_load(const vb_table* t, u32 idx) {
    ge_cached c;
    const u32* q = reinterpret_cast<const u32*>(&t->e[idx]);
    load8_rw(c.YpX.v, q); load8_rw(c.YmX.v, q + 8); load8_rw(c.Z.v, q + 16); load8_rw(c.T2d.v, q + 24);
    return c;
}
ACT_FN void vb_table_build(vb_table* t, const ge& P) {
    ge_cached c1 = ge_to_cached(P);
    tab_store(t, 0, ge_cached_identity());
    tab_store(t, 1, c1);
    ge Q = P;
    ACT_NOUNROLL for (int k = 2; k <= 8; k++) {
        Q = ge_add_cached(Q, c1);
        tab_store(t, k, ge_to_cached(Q));
    }
}
ACT_FN ge_cached vb_lookup(const vb_table* t, int d, bool negate) {
    u32 neg = (d < 0) ? 1u : 0u;
    u32 idx = (u32)(d < 0 ? -d : d);
    if (negate) neg ^= 1u;
    return ge_cached_cneg(tab_load(t, idx), neg);
}
ACT_FN ge_cached vb_lookup_ct(const vb_table* t, int d) {
    u32 neg = ((u32)d) >> 31;
    u32 idx = (u32)((d ^ (d >> 31)) - (d >> 31));
    ge_cached e = ge_cached_identity();
    ACT_NOUNROLL for (u32 k = 1; k <= 8; k++) {
        u32 hit = (idx == k);
        ge_cached c = tab_load(t, k);
        e.YpX = fe_select(e.YpX, c.YpX, hit); e.YmX = fe_select(e.YmX, c.YmX, hit);
        e.Z = fe_select(e.Z, c.Z, hit); e.T2d = fe_select(e.T2d, c.T2d, hit);
    }
    return ge_cached_cneg(e, neg);
}
// sum_k (neg_k ? -s_k : s_k) * P_k for N public scalars sharing one doubling chain (Straus)
template <int N>
ACT_FN ge vb_mul_multi(const vb_table* t, const sc* s, const bool* negate) {
    sc b[N];
    ACT_UNROLL for (int k = 0; k < N; k++) b[k] = sc_bias<4>(s[k]);
    ge acc = ge_identity();
    ACT_NOUNROLL for (int i = 63; i >= 0; i--) {
        if (i != 63) {
            acc = ge_dbl(acc, false); acc = ge_dbl(acc, false); acc = ge_dbl(acc, false); acc = ge_dbl(acc, true);
        }
        ACT_UNROLL for (int k = 0; k < N; k++) acc = ge_add_cached(acc, vb_lookup(&t[k], sc_digit<4>(b[k], i), negate[k]));
    }
    return acc;
}
ACT_FN ge vb_mul(const vb_table* t, const sc& s, bool negate) { return vb_mul_multi<1>(t, &s, &negate); }
// (negate ? -s : s) * P for ONE public scalar: the entry of the coming addition is prefetched before the four doublings, the point
// operations are the public-data forms, and T is only produced by the last addition (a doubling does not read it).  Same group
// element as vb_mul.  (Measured for issue_kernel, profiles/r02y_variants_issue_pub.txt: +0.7 %; moving the table from the stack to a
// per-resident-thread global scratch needs a persistent grid, whose static grid-stride loop lost 6 % to uneven warp progress.)
ACT_FN ge vb_mul_pub(const vb_table* t, const sc& s, bool negate) {
    sc b = sc_bias<4>(s);
    ge a = ge_identity();
    ACT_NOUNROLL for (int i = 63; i >= 0; i--) {
        int d = sc_digit<4>(b, i);
        u32 ad = (u32)(d < 0 ? -d : d);
        prefetch_line(&t->e[ad]);
        if (i != 63) {
            ACT_NOUNROLL for (int k = 0; k < 4; k++) a = ge_dbl_u<true>(a, k == 3);
        }
        u32 neg = ((d < 0) ? 1u : 0u) ^ (negate ? 1u : 0u);
        a = ge_add_cached_u<true>(a, tab_load(t, ad), neg, i == 0);
    }
    return a;
}

// Two public scalars on ONE base with separate results (the range-proof pair com_j*gamma0_j, com_j*gamma01_j): the
// base's doubling chain is shared.  With P_k = 2^(256k/M) P precomputed once (256(M-1)/M doublings, M window tables),
// each scalar costs only 256/M doublings:  s*P = sum_k 2^(256k/M) * (sum_i 16^i d_{k*WIN+i}) P.
// M = 4: 192 + 2*64 doublings instead of 2*256.  The tables are built once, then each scalar is processed on its own
// (one accumulator live at a time: fewer registers, 4 resident blocks per SM).
template <int M, bool VT = false>
ACT_FN void vb_split_tables(const ge& P, vb_table* t) {
    const int WIN = 64 / M;
    ge Q = P;
    ACT_NOUNROLL for (int k = 0; k < M; k++) {
        vb_table_build(&t[k], Q);
        if (k < M - 1) {
            ACT_NOUNROLL for (int d = 0; d < 4 * WIN; d++) Q = ge_dbl_u<VT>(Q, d == 4 * WIN - 1);
        }
    }
}
// -s * P from the tables of vb_split_tables
template <int M>
ACT_FN ge vb_mul_split_neg(const vb_table* t, const sc& s) {
    const int WIN = 64 / M;
    sc b = sc_bias<4>(s);
    ge a = ge_identity();
    ACT_NOUNROLL for (int i = WIN - 1; i >= 0; i--) {
        if (i != WIN - 1) {
            ACT_NOUNROLL for (int d = 0; d < 4; d++) {
#if ACT_PREFETCH >= 2
                if (d == 3) {   // the first table's entry of this window travels during the last doubling
                    int d0 = sc_digit<4>(b, i);
                    prefetch_line(&t[0].e[d0 < 0 ? -d0 : d0]);
                }
#endif
                a = ge_dbl_u<true>(a, d == 3);
            }
        }
        ACT_NOUNROLL for (int k = 0; k < M; k++) {
            if (k + 1 < M) {   // the next table's entry travels to L1 while this addition runs
                int dn = sc_digit<4>(b, (k + 1) * WIN + i);
                prefetch_line(&t[k + 1].e[dn < 0 ? -dn : dn]);
            }
            // the doubling that follows the last addition of a window does not read T (the very last window's does: T goes on)
            int dk = sc_digit<4>(b, k * WIN + i);
            a = ge_add_cached_u<true>(a, tab_load(&t[k], (u32)(dk < 0 ? -dk : dk)), dk < 0 ? 0u : 1u, k + 1 < M || i == 0);   // -|d| * sign
        }
    }
    return a;
}
// ---- the form the range kernel uses (ACT_RANGE_BUCKETS=1, the default since round 2: 215.5k vs 207.3k proofs/s in the kernel on
// B200, profiles/r02a_variants_buckets.txt; ACT_RANGE_BUCKETS=0 keeps the window form above for A/B runs) ------------------
// Right-to-left evaluation of the range-proof pair: the two results -s0*P and -s1*P share ALL doublings.  Q_i = 16^i P is
// formed once (252 doublings instead of 192 + 2 x 60); each result collects -sign(d_i) Q_i into the bucket of |d_i| (9 buckets
// per result, bucket 0 absorbs the zero digits so that every lane adds at every step) and sum_d d * bucket_d closes it
// (running sums, 14 additions).  Buckets live in the thread's table scratch (18 of its 36 entries), extended coordinates.
// Same group elements as vb_mul_split_neg, so the encoded commitments are identical (tests/hostsim builds this form too).
#ifndef ACT_RANGE_BUCKETS
#define ACT_RANGE_BUCKETS 1
#endif
#if ACT_RANGE_BUCKETS
ACT_FN u32* bucket_ptr(vb_table* t, u32 idx) { return reinterpret_cast<u32*>(&t[idx / 9].e[idx % 9]); }
ACT_FN void bucket_store(vb_table* t, u32 idx, const ge& p) {
    u32* q = bucket_ptr(t, idx);
    store8(q, p.X.v); store8(q + 8, p.Y.v); store8(q + 16, p.Z.v); store8(q + 24, p.T.v);
}
ACT_FN ge bucket_load(vb_table* t, u32 idx) {
    ge p;
    const u32* q = bucket_ptr(t, idx);
    load8_rw(p.X.v, q); load8_rw(p.Y.v, q + 8); load8_rw(p.Z.v, q + 16); load8_rw(p.T.v, q + 24);
    return p;
}
#ifndef ACT_BUCKET_SKIP0
#define ACT_BUCKET_SKIP0 0
#endif
ACT_FN void vb_pair_buckets_fill(const ge& P, const sc& s0, const sc& s1, vb_table* t) {
    sc b0 = sc_bias<4>(s0), b1 = sc_bias<4>(s1);
    {
        ge id = ge_identity();
        ACT_NOUNROLL for (u32 k = 0; k < 18; k++) bucket_store(t, k, id);
    }
    ge Q = P;
    ACT_NOUNROLL for (int i = 0; i < 64; i++) {
        ge_cached Qc = ge_to_cached(Q);
        ACT_NOUNROLL for (int r = 0; r < 2; r++) {
            int d = sc_digit<4>(r ? b1 : b0, i);
#if ACT_BUCKET_SKIP0
            // a zero digit adds into a copy of bucket 1 that is never stored: every lane still adds at every step (lock-step), but
            // bucket 0 does not exist and one store in sixteen is predicated off
            u32 ad = (u32)(d < 0 ? -d : d);
            u32 idx = 9u * (u32)r + (ad ? ad : 1u);
            if (i + 1 < 64 || r == 0) {
                int dn = r ? sc_digit<4>(b0, i + 1) : sc_digit<4>(b1, i);
                u32 an = (u32)(dn < 0 ? -dn : dn);
                prefetch_line(bucket_ptr(t, 9u * (u32)(r ^ 1) + (an ? an : 1u)));
            }
            ge B = bucket_load(t, idx);
            B = ge_add_cached_u<true>(B, Qc, d < 0 ? 0u : 1u, true);
            if (ad) bucket_store(t, idx, B);
#else
            u32 idx = 9u * (u32)r + (u32)(d < 0 ? -d : d);
            if (i + 1 < 64 || r == 0) {   // the bucket of the next addition travels to L1 while this one runs
                int dn = r ? sc_digit<4>(b0, i + 1) : sc_digit<4>(b1, i);
                prefetch_line(bucket_ptr(t, 9u * (u32)(r ^ 1) + (u32)(dn < 0 ? -dn : dn)));
            }
            ge B = bucket_load(t, idx);
            B = ge_add_cached_u<true>(B, Qc, d < 0 ? 0u : 1u, true);      // bucket += -sign(d) Q_i
            bucket_store(t, idx, B);
#endif
        }
        if (i + 1 < 64) {
            ACT_NOUNROLL for (int k = 0; k < 4; k++) Q = ge_dbl_u<true>(Q, k == 3);
        }
    }
}
ACT_FN ge vb_pair_buckets_sum(vb_table* t, int r) {
    ge S = bucket_load(t, 9u * (u32)r + 8u), R = S;
    ACT_NOUNROLL for (u32 d = 7; d >= 1; d--) {
        S = ge_add_cached_u<true>(S, ge_to_cached(bucket_load(t, 9u * (u32)r + d)), 0u, true);
        R = ge_add_cached_u<true>(R, ge_to_cached(S), 0u, true);
    }
    return R;
}
#endif

// s * P for a secret s
ACT_NOINLINE void vb_mul_ct_(ge* out, const ge* P, const sc* s) {
    vb_table t;
    vb_table_build(&t, *P);
    sc b = sc_bias<4>(*s);
    ge acc = ge_identity();
    ACT_NOUNROLL for (int i = 63; i >= 0; i--) {
        if (i != 63) {
            acc = ge_dbl(acc, false); acc = ge_dbl(acc, false); acc = ge_dbl(acc, false); acc = ge_dbl(acc, true);
        }
        acc = ge_add_cached(acc, vb_lookup_ct(&t, sc_digit<4>(b, i)));
    }
    *out = acc;
}

// s1 * P and s2 * P for two SECRET scalars on one base (the signing tail: A = X_A * (e+x)^-1 and Y_A = A * alpha =
// X_A * (alpha (e+x)^-1)): the doubling chain of the base is shared as in the range kernel -- 192 + 2 x 60 doublings instead
// of 2 x 252 -- and every lookup scans its whole table (no secret-dependent address or branch).
#ifndef ACT_SIGN_SPLIT
#define ACT_SIGN_SPLIT 4
#endif
ACT_NOINLINE void vb_mul2_ct_(ge* out1, ge* out2, const ge* P, const sc* s1, const sc* s2) {
    const int M = ACT_SIGN_SPLIT, WIN = 64 / M;
    vb_table t[M];
    vb_split_tables<M>(*P, t);
    ACT_NOUNROLL for (int w = 0; w < 2; w++) {
        sc b = sc_bias<4>(w ? *s2 : *s1);
        ge a = ge_identity();
        ACT_NOUNROLL for (int i = WIN - 1; i >= 0; i--) {
            if (i != WIN - 1) {
                ACT_NOUNROLL for (int d = 0; d < 4; d++) a = ge_dbl_u(a, d == 3);
            }
            ACT_NOUNROLL for (int k = 0; k < M; k++) a = ge_add_cached_u(a, vb_lookup_ct(&t[k], sc_digit<4>(b, k * WIN + i)), 0u, k + 1 < M || i == 0);
        }
        if (w) *out2 = a; else *out1 = a;
    }
}

// engine set-up: reduce the stored secret mod l (Scalar::from_bytes_mod_order semantics for the key) and precompute W/2
ACT_FN void ctx_finalize_thread(act_ctx* C) {
    C->x = sc_from_words(C->x.v);
    vb_table t;
    vb_table_build(&t, C->W);
    sc one = sc_from_u32(1);
    C->W_half = vb_mul(&t, sc_half(one), false);     // W is public
}

// ---- single-chunk transcripts ---------------------------------------------------------------------------
struct tr_small { u32 buf[128]; u32 len; };  // up to 512 bytes

ACT_FN void tr_init(tr_small* t, const act_ctx* C, int which) {
    ACT_NOUNROLL for (int i = 0; i < 128; i++) t->buf[i] = (i < 48) ? C->prefix[which][i] : 0u;
    t->len = C->prefix_len[which];
}
ACT_FN void tr_put_word(tr_small* t, u32 w) {
    u32 sh = (t->len & 3u) * 8u, idx = t->len >> 2;
    t->buf[idx] |= w << sh;
    if (sh) t->buf[idx + 1] |= w >> (32u - sh);
    t->len += 4;
}
// Transcript::update with a 32-byte payload: u64be(32) || payload  (src/transcript.rs:95-98)
ACT_FN void tr_add32(tr_small* t, const u32* w) {
    tr_put_word(t, 0u);
    tr_put_word(t, 0x20000000u);
    ACT_NOUNROLL for (int i = 0; i < 8; i++) tr_put_word(t, w[i]);
}
ACT_FN sc tr_challenge(tr_small* t) {
    u32 o[16];
    b3_hash_single_chunk(t->buf, t->len, o);
    return sc_from_wide(o);
}

// =============================================================================================================
// BBS signing tail shared by issue and refund (src/lib.rs:643-662 and :846-868)
// =============================================================================================================
// encode(2 * P_i) for four points with ONE field inversion (double-and-encode, ge25519.cuh): the signing tail produces
// A, X_G, Y_A, Y_G as halves (every scalar involved is known to the signer and gets halved), which replaces four inverse
// square roots (4 x 254 squarings) by one inversion.  Branch-free: the points depend on the issuer's secrets.
ACT_NOINLINE void encode4_doubled_(u32* out /* 4 x 8 words */, const ge* pts /* 4 */) {
    fe prefix[4], ts[4];
    fe acc = fe_one();
    ACT_NOUNROLL for (int i = 0; i < 4; i++) {
        ge_dbl_enc s = ge_dbl_enc_prepare(pts[i]);
        fe t = fe_mul(s.eg, s.fh);
        t = fe_select(t, fe_one(), fe_is_zero(t));
        prefix[i] = acc; ts[i] = t;
        acc = fe_mul(acc, t);
    }
    fe inv = fe_invert(acc);
    ACT_NOUNROLL for (int i = 3; i >= 0; i--) {
        ge_dbl_enc s = ge_dbl_enc_prepare(pts[i]);
        u32 zero = fe_is_zero(fe_mul(s.eg, s.fh));
        fe inv_i = fe_mul(inv, prefix[i]);
        inv = fe_mul(inv, ts[i]);
        u32 w[8];
        ge_dbl_enc_finish(w, s, inv_i);
        u32 m = 0u - (zero ^ 1u);                                  // 2P in the identity coset encodes as 32 zero bytes
        ACT_UNROLL for (int k = 0; k < 8; k++) out[8 * i + k] = w[k] & m;
    }
}
// Overwrites a secret-derived local object once it is dead.  The volatile stores cannot be elided, so whichever home the
// compiler gave the object (registers or its local-memory slot) holds zeros afterwards; spill slots the compiler created on
// its own are covered by scrub_local_kernel (act_engine.cu), which the engine runs when it is destroyed.
template <typename T>
ACT_FN void secret_wipe(T* obj) {
    volatile u32* q = reinterpret_cast<volatile u32*>(obj);
    ACT_UNROLL for (unsigned i = 0; i < sizeof(T) / 4; i++) q[i] = 0u;
}
// X_A given; rnd = 32 words (e_wide || alpha_wide).  kind = ACT_TR_RESPOND (c, e, points) or ACT_TR_REFUND (e, points).
// Writes A (8 words), e, gamma, z.
ACT_NOINLINE void bbs_sign_(const act_ctx* C, const ge* X_A, const u32* rnd, int kind, const sc* c,
                            u32* A_enc, sc* e_out, sc* gamma_out, sc* z_out) {
    sc e = sc_from_wide(rnd);
    sc ex = sc_add(e, C->x);
    sc inv = sc_half(sc_invert(ex));
    ge P[4];                                                         // halves of A, X_G, Y_A, Y_G
    sc alpha = sc_from_wide(rnd + 16);
    sc ainv = sc_mul(alpha, inv);
    // A = X_A * (e+x)^-1 and Y_A = A * alpha = X_A * (alpha (e+x)^-1)   [secret scalars, one base: shared doubling chain]
    vb_mul2_ct_(&P[0], &P[2], X_A, &inv, &ainv);
    P[1] = fb_accumulate(C->W_half, C->fb[ACT_BASE_G], sc_half(e), false);   // X_G = G*e + W     [e is public output]
    sc ah = sc_half(alpha);
    P[3] = fb_accumulate_ct(ge_identity(), C->ct_g, ah);             // Y_G = G * alpha           [secret scalar]
    u32 enc[32];
    encode4_doubled_(enc, P);
    tr_small tr;
    tr_init(&tr, C, kind);
    if (kind == ACT_TR_RESPOND) tr_add32(&tr, c->v);
    tr_add32(&tr, e.v);
    u32 w[8];
    ACT_UNROLL for (int k = 0; k < 8; k++) A_enc[k] = enc[k];
    tr_add32(&tr, A_enc);
    ristretto_encode_(w, X_A); tr_add32(&tr, w);
    tr_add32(&tr, enc + 8); tr_add32(&tr, enc + 16); tr_add32(&tr, enc + 24);
    sc gamma = tr_challenge(&tr);
    *e_out = e; *gamma_out = gamma;
    *z_out = sc_add(sc_mul(gamma, ex), alpha);                   // z = gamma*(x+e) + alpha
    // ZeroizeOnDrop parity (the reference zeroises its secret-bearing values, src/lib.rs:160,571,1160): everything derived from
    // x or alpha that is not an output is overwritten before the thread leaves
    secret_wipe(&ex); secret_wipe(&inv); secret_wipe(&alpha); secret_wipe(&ainv); secret_wipe(&ah);
    secret_wipe(&P[2]); secret_wipe(&P[3]);                      // halves of Y_A = A*alpha and Y_G = G*alpha
}

// =============================================================================================================
// issue (src/lib.rs:621-663).  req: n x 32 words (K, gamma, k_bar, r_bar); cs: n x 8; rnd: n x 32;
// resp: n x 40 words (A, e, gamma, z, c); status: n bytes.
// =============================================================================================================
// mode ACT_MODE_FULL: verify, then sign with rnd[i] (the batch contract: request i owns 128 RNG bytes).
// mode ACT_MODE_VERIFY: verify only (status[i]; nothing else is written).
// mode ACT_MODE_SIGN: status[i] is given (by a VERIFY pass); accepted requests are signed with the RNG bytes at
//      rnd + 32 * rnd_index[i] -- the position a sequential loop over ONE shared RNG would have reached (the reference
//      draws e, alpha only after a request verifies, src/lib.rs:638-643).
#ifndef ACT_ISSUE_PUB
#define ACT_ISSUE_PUB 1
#endif
#define ACT_MODE_FULL 0
#define ACT_MODE_VERIFY 1
#define ACT_MODE_SIGN 2
ACT_FN void issue_thread(const act_ctx* C, size_t i, const u32* req, const u32* cs, const u32* rnd, u32* resp, u8* status,
                         int mode = ACT_MODE_FULL, const u32* rnd_index = nullptr) {
    const u32* rq = req + 32 * i;
    u32* out = resp + 40 * i;
    u32 kw[8];
    load8(kw, rq);
    ge K;
    u32 valid = ristretto_decode_(&K, kw);
    u32 st = ACT_ST_OK;
    if (!valid) st = ACT_ST_DECODE_INVALID_POINT;
    if (mode == ACT_MODE_SIGN) st = status[i];
    else {
    sc gamma = load_scalar(rq + 8), k_bar = load_scalar(rq + 16), r_bar = load_scalar(rq + 24);
    // K1 = h2*k_bar + h3*r_bar - K*gamma                                                     (:629-630)
    vb_table tk;
    vb_table_build(&tk, K);
#if ACT_ISSUE_PUB
    ge K1 = vb_mul_pub(&tk, gamma, true);     // K and gamma are public: variable-time forms, T only on the last addition
#else
    ge K1 = vb_mul(&tk, gamma, true);
#endif
    K1 = fb_accumulate(K1, C->fb[ACT_BASE_H2], k_bar, false);
    K1 = fb_accumulate(K1, C->fb[ACT_BASE_H3], r_bar, false);
    {
        tr_small tr;
        u32 w[8];
        tr_init(&tr, C, ACT_TR_REQUEST);                                                  // (:633-635)
        tr_add32(&tr, kw);  // canonical decode => compress(K) == wire bytes
        ristretto_encode_(w, &K1); tr_add32(&tr, w);
        sc g2 = tr_challenge(&tr);
        if (st == ACT_ST_OK && !sc_eq(g2, gamma)) st = ACT_ST_INVALID_ISSUANCE_REQUEST_PROOF;   // (:638-640)
    }
    }
    if (mode == ACT_MODE_VERIFY) { status[i] = (u8)st; return; }
    if (st != ACT_ST_OK) {
        ACT_NOUNROLL for (int k = 0; k < 5; k++) store8_zero(out + 8 * k);
        status[i] = (u8)st;
        return;
    }
    sc c = load_scalar(cs + 8 * i);
    // X_A = G + h1*c + K                                                                      (:644)
    ge X_A = ge_add(K, ge_basepoint());
    X_A = fb_accumulate(X_A, C->fb[ACT_BASE_H1], c, false);
    u32 A_enc[8];
    sc e, g, z;
    u32 r[32];
    const u32* rsrc = rnd + 32 * (rnd_index ? (size_t)rnd_index[i] : i);
    ACT_NOUNROLL for (int k = 0; k < 4; k++) load8(r + 8 * k, rsrc + 8 * k);
    bbs_sign_(C, &X_A, r, ACT_TR_RESPOND, &c, A_enc, &e, &g, &z);
    secret_wipe(&r);
    store8(out, A_enc); store_scalar(out + 8, e); store_scalar(out + 16, g); store_scalar(out + 24, z); store_scalar(out + 32, c);
    status[i] = ACT_ST_OK;
}

// =============================================================================================================
// PreIssuance::to_credit_token verification (src/lib.rs:528-562).  K: n x 8 words, resp: n x 40 words.
// All inputs are public to the verifier.
// =============================================================================================================
// Y_A = A*z - X_A*gamma, Y_G = G*z - X_G*gamma, then the challenge over (scalars..., A, X_A, X_G, Y_A, Y_G)
ACT_NOINLINE u32 dleq_check_(const act_ctx* C, int kind, const sc* c, const sc* e, const sc* gamma, const sc* z,
                             const u32* A_words, const ge* A, const ge* X_A) {
    ge X_G = fb_accumulate(C->W, C->fb[ACT_BASE_G], *e, false);
    vb_table t[2];
    vb_table_build(&t[0], *A);
    vb_table_build(&t[1], *X_A);
    sc ss[2] = {*z, *gamma};
    bool ng[2] = {false, true};
    ge Y_A = vb_mul_multi<2>(t, ss, ng);
    // Y_G = G*z - X_G*gamma with X_G = G*e + W  =  G*(z - e*gamma) - W*gamma: both bases are fixed per engine, so the
    // variable-base multiplication of the reference's formula becomes two table walks
    ge Y_G = fb_accumulate(ge_identity(), C->fb[ACT_BASE_G], sc_sub(*z, sc_mul(*e, *gamma)), false);
    Y_G = fb_accumulate(Y_G, C->fb[ACT_BASE_W], *gamma, true);
    tr_small tr;
    u32 w[8];
    tr_init(&tr, C, kind);
    if (kind == ACT_TR_RESPOND) tr_add32(&tr, c->v);
    tr_add32(&tr, e->v);
    tr_add32(&tr, A_words);
    ristretto_encode_(w, X_A); tr_add32(&tr, w);
    ristretto_encode_(w, &X_G); tr_add32(&tr, w);
    ristretto_encode_(w, &Y_A); tr_add32(&tr, w);
    ristretto_encode_(w, &Y_G); tr_add32(&tr, w);
    sc g2 = tr_challenge(&tr);
    return sc_eq(g2, *gamma);
}
ACT_FN void issuance_check_thread(const act_ctx* C, size_t i, const u32* Kin, const u32* resp, u8* status) {
    const u32* rs = resp + 40 * i;
    ge K, A;
    u32 aw[8];
    load8(aw, rs);
    u32 valid = load_point(&K, Kin + 8 * i) & ristretto_decode_(&A, aw);
    sc e = load_scalar(rs + 8), gamma = load_scalar(rs + 16), z = load_scalar(rs + 24), c = load_scalar(rs + 32);
    ge X_A = ge_add(K, ge_basepoint());                                                   // (:536)
    X_A = fb_accumulate(X_A, C->fb[ACT_BASE_H1], c, false);
    u32 ok = dleq_check_(C, ACT_TR_RESPOND, &c, &e, &gamma, &z, aw, &A, &X_A);            // (:537-552)
    status[i] = (u8)(!valid ? ACT_ST_DECODE_INVALID_POINT : (ok ? ACT_ST_OK : ACT_ST_INVALID_ISSUANCE_RESPONSE_PROOF));
}

// =============================================================================================================
// spend verification, stage 1: the 256 range-proof commitments (src/lib.rs:800-817).
// One thread per (proof, j).  Writes items 5+j (com_j bytes), 133+2j, 134+2j (C'_j0, C'_j1) and the
// affine-Niels form of com_j for the K' Horner chain in stage 2.
// =============================================================================================================
ACT_FN void spend_range_thread(const act_ctx* C, size_t p, int j, const u32* proofs, u32* items, u32* com_niels, u32* flags,
                               vb_table* tabs /* ACT_RANGE_SPLIT tables private to this thread */, u32* cpts /* n x 256 x 32 words */) {
    const u32* pf = proofs + (size_t)ACT_PROOF_WORDS * p;
    u32* it = items + (size_t)ACT_ITEM_WORDS * p;
    u32 cw[8];
    load8(cw, pf + 8 * (4 + j));
    ge P;
    u32 valid = ristretto_decode_(&P, cw);
    if (!valid) ACT_ATOMIC_OR(&flags[p], ACT_FLAG_BAD_POINT);
    store8(it + 8 * (5 + j), cw);
    {
        ge_niels n = ge_affine_to_niels(P.X, P.Y);
        u32* cn = com_niels + ((size_t)ACT_L * p + j) * 24;
        store_fe(cn, n.ypx); store_fe(cn + 8, n.ymx); store_fe(cn + 16, n.xy2d);
    }
    // Every scalar is HALVED: this stage produces C'/2 and the encode stage emits encode(2 * C'/2) with one batched
    // inversion per 16 points instead of one inverse square root per point.
#if ACT_RANGE_BUCKETS
    {
        sc g0 = load_scalar(pf + 8 * (140 + j));
        sc g1 = sc_sub(load_scalar(pf + 8 * 132), g0);
        vb_pair_buckets_fill(P, sc_half(g0), sc_half(g1), tabs);
    }
#else
    vb_split_tables<ACT_RANGE_SPLIT, true>(P, tabs);   // com_j is public
#endif
    u32* cp = cpts + ((size_t)2 * ACT_L * p + 2 * j) * 32;
    ACT_NOUNROLL for (int b = 0; b < 2; b++) {
        // b = 0: C'_j0 = [h2*w00 +] h3*z_j0 - com_j*gamma0_j                                 (:806-807,814-815)
        // b = 1: C'_j1 = [h2*w01 +] h3*z_j1 + h1*gamma01_j - com_j*gamma01_j                 (:808-809,816)
        //        [..] for j = 0 only, added by spend_head_thread
        //        (the reference's base com_j - H1 is never formed: -(com_j - h1)*g = h1*g - com_j*g)
        // Scalars are re-derived from the proof bytes where they are used: nothing but the accumulator stays live.
#if ACT_RANGE_BUCKETS
        ge Q = vb_pair_buckets_sum(tabs, b);
#else
        sc gb = load_scalar(pf + 8 * (140 + j));
        if (b) gb = sc_sub(load_scalar(pf + 8 * 132), gb);                                  // gamma01[j] (:801,811)
        gb = sc_half(gb);
        ge Q = vb_mul_split_neg<ACT_RANGE_SPLIT>(tabs, gb);
#endif
        // (the h2 terms exist for j = 0 only: one lane of one warp in four would run 40 additions alone, so stage 2 -- a thread
        // per proof -- adds them to the stored halves instead, spend_head_thread)
        ACT_NOUNROLL for (int t = 0; t < 2; t++) {
            int tab;
            sc s;
            if (t == 0) { tab = ACT_BASE_H3; s = load_scalar(pf + 8 * (268 + 2 * j + b)); }
            else { if (!b) continue; tab = ACT_BASE_H1; s = sc_sub(load_scalar(pf + 8 * 132), load_scalar(pf + 8 * (140 + j))); }
            Q = fb_accumulate(Q, C->fb[tab], sc_half(s), false);
        }
        store_fe(cp + 32 * b, Q.X); store_fe(cp + 32 * b + 8, Q.Y); store_fe(cp + 32 * b + 16, Q.Z); store_fe(cp + 32 * b + 24, Q.T);
    }
}

// =============================================================================================================
// spend verification, stage 1b: encode the 256 half-commitments of a proof.  One thread per ACT_ENC_BATCH (64)
// consecutive points: Montgomery-batched inversion, then the square-root-free double-and-encode.
// Writes items 133 .. 388.
// =============================================================================================================
// points per thread = points per field inversion.  Measured at 131 072 proofs (profiles/r02j_variants_enc_sign.txt): 16 -> 13.73 ms,
// 32 -> 12.23 ms, 64 -> 11.81 ms in the encode kernel.
#ifndef ACT_ENC_BATCH
#define ACT_ENC_BATCH 64
#endif
// pts = points per proof in cpts (256 for the verifier: items 133..388; 384 for the prover: items 5..388), item0 = first item
ACT_FN void spend_encode_thread(const act_ctx* C, size_t p, int part, const u32* cpts, u32* items, int pts = 2 * ACT_L, int item0 = 133) {
    (void)C;
    const u32* src = cpts + ((size_t)pts * p + (size_t)part * ACT_ENC_BATCH) * 32;
    u32* dst = items + (size_t)ACT_ITEM_WORDS * p + 8 * (item0 + part * ACT_ENC_BATCH);
    fe prefix[ACT_ENC_BATCH];
    fe acc = fe_one();
    ACT_NOUNROLL for (int i = 0; i < ACT_ENC_BATCH; i++) {
        ge P;
        load_fe(&P.X, src + 32 * i); load_fe(&P.Y, src + 32 * i + 8); load_fe(&P.Z, src + 32 * i + 16); load_fe(&P.T, src + 32 * i + 24);
        ge_dbl_enc s = ge_dbl_enc_prepare(P);
        fe t = fe_mul(s.eg, s.fh);
        t = fe_select(t, fe_one(), fe_is_zero(t));
        prefix[i] = acc;            // product of t_0 .. t_{i-1}
        acc = fe_mul(acc, t);
    }
    fe inv = fe_invert(acc);
    ACT_NOUNROLL for (int i = ACT_ENC_BATCH - 1; i >= 0; i--) {
        ge P;
        load_fe(&P.X, src + 32 * i); load_fe(&P.Y, src + 32 * i + 8); load_fe(&P.Z, src + 32 * i + 16); load_fe(&P.T, src + 32 * i + 24);
        ge_dbl_enc s = ge_dbl_enc_prepare(P);
        fe t = fe_mul(s.eg, s.fh);
        u32 zero = fe_is_zero(t);
        t = fe_select(t, fe_one(), zero);
        fe inv_i = fe_mul(inv, prefix[i]);
        inv = fe_mul(inv, t);
        u32 w[8];
        ge_dbl_enc_finish(w, s, inv_i);
        ACT_UNROLL for (int k = 0; k < 8; k++) w[k] = zero ? 0u : w[k];   // 2P in the identity coset
        store8(dst + 8 * i, w);
    }
}

// =============================================================================================================
// spend verification, stage 2: one thread per proof.  A-bar (secret x), A1, A2, K' (Horner), C
// (src/lib.rs:787-799, 819-829).  Writes items 0..4 and 389, K' for the signing tail; completes C'_00, C'_01 in cpts.
// KEYED: the secret of the A1 term is the x of slots[key_ids[p]] (ACT_KEY_SLOTS entries, null = empty slot) instead of C's.
// An empty or out-of-range id raises ACT_FLAG_NO_KEY and the proof runs on with C's x, so that every proof takes the same
// path; its result is discarded.  The key id is public: the load it selects depends on public data only.
// =============================================================================================================
template <bool KEYED = false>
ACT_FN void spend_head_thread(const act_ctx* C, size_t p, const u32* proofs, u32* items, const u32* com_niels, u32* kprime, u32* flags,
                              u32* cpts /* halves of stage 1: the two of j = 0 get their h2 terms here, BEFORE the encode stage */,
                              const u8* key_ids = nullptr, const act_ctx* const* slots = nullptr) {
    const u32* pf = proofs + (size_t)ACT_PROOF_WORDS * p;
    u32* it = items + (size_t)ACT_ITEM_WORDS * p;
    ACT_NOUNROLL for (int b = 0; b < 2; b++) {   // C'_00 += h2*w00, C'_01 += h2*w01 (as halves)            (:806,808)
        u32* cp = cpts + ((size_t)2 * ACT_L * p + b) * 32;
        ge Q;
        load8_rw(Q.X.v, cp); load8_rw(Q.Y.v, cp + 8); load8_rw(Q.Z.v, cp + 16); load8_rw(Q.T.v, cp + 24);
        Q = fb_accumulate(Q, C->fb[ACT_BASE_H2], sc_half(load_scalar(pf + 8 * (138 + b))), false);
        store_fe(cp, Q.X); store_fe(cp + 8, Q.Y); store_fe(cp + 16, Q.Z); store_fe(cp + 24, Q.T);
    }
    u32 aw[8], bw[8];
    load8(aw, pf + 16); load8(bw, pf + 24);
    ge Ap, Bb;
    u32 valid = ristretto_decode_(&Ap, aw) & ristretto_decode_(&Bb, bw);
    u32 fl = 0;
    if (!valid) fl |= ACT_FLAG_BAD_POINT;
    if (ristretto_is_identity(Ap)) fl |= ACT_FLAG_IDENTITY;                                // (:787-789)
    const act_ctx* K = C;   // whose secret the A1 term uses
    if (KEYED) {
        u32 id = key_ids[p];
        const act_ctx* named = id < ACT_KEY_SLOTS ? slots[id] : nullptr;
        if (named) K = named;
        else fl |= ACT_FLAG_NO_KEY;
    }
    if (fl) ACT_ATOMIC_OR(&flags[p], fl);
    sc k = load_scalar(pf), s = load_scalar(pf + 8), gamma = load_scalar(pf + 8 * 132);
    sc e_bar = load_scalar(pf + 8 * 133), r2_bar = load_scalar(pf + 8 * 134), r3_bar = load_scalar(pf + 8 * 135);
    sc c_bar = load_scalar(pf + 8 * 136), r_bar = load_scalar(pf + 8 * 137);
    sc k_bar = load_scalar(pf + 8 * 524), s_bar = load_scalar(pf + 8 * 525);
    store_scalar(it, k);               // transcript.add_scalar(&k): reduced bytes          (:832)
    store8(it + 8, aw); store8(it + 16, bw);
    vb_table t[2];
    {
        // A1 = A'*e_bar + B*r2_bar - Abar*gamma with Abar = A'*x                          (:791,793-795)
        //    = A'*(e_bar - x*gamma) + B*r2_bar: Abar is never formed (it is not hashed); the scalar on A' depends on the
        //    secret x, so that term scans its table in full, the B term (public scalar) indexes directly.  One doubling chain.
        vb_table_build(&t[0], Ap); vb_table_build(&t[1], Bb);
        sc sa = sc_bias<4>(sc_sub(e_bar, sc_mul(K->x, gamma))), sb = sc_bias<4>(r2_bar);
        ge A1 = ge_identity();
        ACT_NOUNROLL for (int i = 63; i >= 0; i--) {
            if (i != 63) {
                A1 = ge_dbl(A1, false); A1 = ge_dbl(A1, false); A1 = ge_dbl(A1, false); A1 = ge_dbl(A1, true);
            }
            A1 = ge_add_cached(A1, vb_lookup_ct(&t[0], sc_digit<4>(sa, i)));
            A1 = ge_add_cached_u(A1, vb_lookup(&t[1], sc_digit<4>(sb, i), false), 0u, i == 0);   // a doubling follows: no T until the last window
        }
        store_point(it + 24, A1);
    }
    {
        // A2 = B*r3_bar + h1*c_bar + h3*r_bar - (G + h2*k)*gamma                          (:792,796-799)
        ge A2 = vb_mul_pub(&t[1], r3_bar, false);
        A2 = fb_accumulate(A2, C->fb[ACT_BASE_H1], c_bar, false);
        A2 = fb_accumulate(A2, C->fb[ACT_BASE_H3], r_bar, false);
        A2 = fb_accumulate(A2, C->fb[ACT_BASE_G], gamma, true);
        A2 = fb_accumulate(A2, C->fb[ACT_BASE_H2], sc_mul(k, gamma), true);
        store_point(it + 32, A2);
    }
    // K' = sum 2^i com_i by Horner from the top (the reference does 128 scalar mults, :819-824)
    ge Kp = ge_identity();
    const ge_niels* cn = reinterpret_cast<const ge_niels*>(com_niels) + (size_t)ACT_L * p;
    ACT_NOUNROLL for (int i = ACT_L - 1; i >= 0; i--) {
        Kp = ge_dbl(Kp, true);
        Kp = ge_add_niels(Kp, load_niels(cn + i));
    }
    {
        u32* kp = kprime + 32 * p;
        store_fe(kp, Kp.X); store_fe(kp + 8, Kp.Y); store_fe(kp + 16, Kp.Z); store_fe(kp + 24, Kp.T);
    }
    {
        // C = h1*(-c_bar) + h2*k_bar + h3*s_bar - (h1*s + K')*gamma                       (:825-829)
        vb_table_build(&t[0], Kp);
        ge Cc = vb_mul_pub(&t[0], gamma, true);
        Cc = fb_accumulate(Cc, C->fb[ACT_BASE_H1], sc_add(c_bar, sc_mul(s, gamma)), true);
        Cc = fb_accumulate(Cc, C->fb[ACT_BASE_H2], k_bar, false);
        Cc = fb_accumulate(Cc, C->fb[ACT_BASE_H3], s_bar, false);
        store_point(it + 8 * 389, Cc);
    }
}

// =============================================================================================================
// spend verification, stage 3: BLAKE3 over the 15 784-byte transcript.  One thread per (proof, chunk)
// produces the chunk chaining value; one thread per proof folds the 16 CVs and compares with gamma.
// =============================================================================================================
ACT_FN u32 spend_tr_word(const act_ctx* C, const u32* it, u32 g) {
    if (g < 46u) return C->prefix[ACT_TR_SPEND][g];
    u32 q = g - 46u;
    if (q >= 10u * ACT_ITEMS) return 0u;
    u32 item = q / 10u, o = q - item * 10u;
    if (o == 0u) return 0u;
    if (o == 1u) return 0x20000000u;
    return it[item * 8u + o - 2u];
}
ACT_FN void spend_chunk_thread(const act_ctx* C, size_t p, int c, const u32* items, u32* cvs) {
    const u32* it = items + (size_t)ACT_ITEM_WORDS * p;
    u32 cv[8], m[16], o[16];
    ACT_UNROLL for (int i = 0; i < 8; i++) cv[i] = B3_IV_[i];
    u32 nbytes = (c == ACT_SPEND_CHUNKS - 1) ? (ACT_SPEND_BYTES - 1024u * (ACT_SPEND_CHUNKS - 1)) : 1024u;
    u32 nblocks = (nbytes + 63u) / 64u;
    ACT_NOUNROLL for (u32 b = 0; b < nblocks; b++) {
        ACT_UNROLL for (int i = 0; i < 16; i++) m[i] = spend_tr_word(C, it, (u32)c * 256u + b * 16u + i);
        u32 flags = (b == 0 ? B3_CHUNK_START : 0u), blen = 64;
        if (b == nblocks - 1) { flags |= B3_CHUNK_END; blen = nbytes - 64u * b; }
        b3_compress(cv, m, (u32)c, 0, blen, flags, o);
        ACT_UNROLL for (int i = 0; i < 8; i++) cv[i] = o[i];
    }
    store8(cvs + ((size_t)ACT_SPEND_CHUNKS * p + c) * 8, cv);
}
// Root of the 16-chunk BLAKE3 tree (a perfect binary tree: 8 + 4 + 2 parents, then the root with its XOF block 0) from the
// chunk CVs an EARLIER kernel wrote.  The CVs are read once through the read-only path and folded in the thread's own
// storage: nothing is written back to `cvs`, so no load in this kernel ever follows a store to the same address.
ACT_FN void spend_fold_root(const u32* cvs16, u32* o /* 16 words */) {
    u32 cv[ACT_SPEND_CHUNKS * 8];
    ACT_NOUNROLL for (int k = 0; k < ACT_SPEND_CHUNKS; k++) load8(cv + 8 * k, cvs16 + 8 * k);
    ACT_NOUNROLL for (int width = ACT_SPEND_CHUNKS; width > 2; width >>= 1) {
        ACT_NOUNROLL for (int k = 0; k < width / 2; k++) {
            b3_compress(B3_IV_, cv + 16 * k, 0, 0, 64, B3_PARENT, o);
            ACT_UNROLL for (int i = 0; i < 8; i++) cv[8 * k + i] = o[i];
        }
    }
    b3_compress(B3_IV_, cv, 0, 0, 64, B3_PARENT | B3_ROOT, o);
}
// folds the CVs, derives the challenge, sets the final status of the verification
ACT_FN void spend_finish_thread(const act_ctx* C, size_t p, const u32* proofs, const u32* cvs, const u32* flags, u8* status) {
    (void)C;
    u32 o[16];
    spend_fold_root(cvs + (size_t)ACT_SPEND_CHUNKS * p * 8, o);
    sc g2 = sc_from_wide(o);
    sc gamma = load_scalar(proofs + (size_t)ACT_PROOF_WORDS * p + 8 * 132);
    u32 fl = flags[p];
    u32 st = ACT_ST_OK;
    if (fl & ACT_FLAG_BAD_POINT) st = ACT_ST_DECODE_INVALID_POINT;
    else if (fl & ACT_FLAG_IDENTITY) st = ACT_ST_IDENTITY_POINT;
    else if ((fl & ACT_FLAG_NO_KEY) || !sc_eq(g2, gamma)) st = ACT_ST_INVALID_CLIENT_SPEND_PROOF;   // (:842-844); no key: as a failed check
    status[p] = (u8)st;
}

// =============================================================================================================
// refund signing tail (src/lib.rs:846-868).  One thread per proof; rejected proofs get zero output.
// refunds: n x 32 words (A*, e*, gamma, z); nullifiers: n x 8 words (reduced k).
// =============================================================================================================
ACT_FN void refund_sign_thread(const act_ctx* C, size_t p, const u32* proofs, const u32* rnd, const u32* kprime,
                               const u8* status, u32* refunds, u32* nullifiers, const u32* rnd_index = nullptr, const u32* kwords = nullptr) {
    u32* out = refunds + 32 * p;
    if (status[p] != ACT_ST_OK) {
        ACT_NOUNROLL for (int k = 0; k < 4; k++) store8_zero(out + 8 * k);
        if (nullifiers) store8_zero(nullifiers + 8 * p);
        return;
    }
    ge Kp;
    const u32* kp = kprime + 32 * p;
    load_fe(&Kp.X, kp); load_fe(&Kp.Y, kp + 8); load_fe(&Kp.Z, kp + 16); load_fe(&Kp.T, kp + 24);
    ge X_A = ge_add(Kp, ge_basepoint());                                                   // (:848)
    u32 r[32];
    const u32* rsrc = rnd + 32 * (rnd_index ? (size_t)rnd_index[p] : p);   // sequential-RNG mode: see issue_thread
    ACT_NOUNROLL for (int k = 0; k < 4; k++) load8(r + 8 * k, rsrc + 8 * k);
    u32 A_enc[8];
    sc e, g, z, dummy = sc_zero();
    bbs_sign_(C, &X_A, r, ACT_TR_REFUND, &dummy, A_enc, &e, &g, &z);
    secret_wipe(&r);
    store8(out, A_enc); store_scalar(out + 8, e); store_scalar(out + 16, g); store_scalar(out + 24, z);
    // nullifier() = k (:720-722); kwords: the k fields alone (n x 8 words) when the proofs are no longer resident;
    // nullifiers == nullptr: the verification pass already delivered them (act_batch_spend_verify)
    if (nullifiers) store_scalar(nullifiers + 8 * p, kwords ? load_scalar(kwords + 8 * p) : load_scalar(proofs + (size_t)ACT_PROOF_WORDS * p));
}

// =============================================================================================================
// PreRefund::to_credit_token verification (src/lib.rs:1217-1253).  com: n x 128 x 8 words, refund: n x 32 words.
// =============================================================================================================
ACT_FN void refund_check_thread(const act_ctx* C, size_t i, const u32* com, const u32* refund, u8* status) {
    const u32* rf = refund + 32 * i;
    u32 aw[8];
    load8(aw, rf);
    ge A;
    u32 valid = ristretto_decode_(&A, aw);
    sc e = load_scalar(rf + 8), gamma = load_scalar(rf + 16), z = load_scalar(rf + 24);
    ge Kp = ge_identity();
    ACT_NOUNROLL for (int j = ACT_L - 1; j >= 0; j--) {                                    // (:1224-1230) Horner
        ge P;
        valid &= load_point(&P, com + ((size_t)ACT_L * i + j) * 8);
        Kp = ge_dbl(Kp, true);
        Kp = ge_add_niels(Kp, ge_affine_to_niels(P.X, P.Y));
    }
    ge X_A = ge_add(Kp, ge_basepoint());
    sc dummy = sc_zero();
    u32 ok = dleq_check_(C, ACT_TR_REFUND, &dummy, &e, &gamma, &z, aw, &A, &X_A);          // (:1232-1243)
    status[i] = (u8)(!valid ? ACT_ST_DECODE_INVALID_POINT : (ok ? ACT_ST_OK : ACT_ST_INVALID_REFUND_PROOF));
}

// =============================================================================================================
// engine set-up: fixed-base tables and Params::new
// =============================================================================================================
// entry (win, k) of the radix-2^W table of B: k * 2^(W*win) * B as affine Niels (k = 0: identity)
template <int W, int ENT>
ACT_FN void build_table_thread(const ge* B, int win, ge_niels* tab) {
    ge P = *B;
    ACT_NOUNROLL for (int i = 0; i < W * win; i++) P = ge_dbl(P, true);
    ge_cached Pc = ge_to_cached(P);
    ge Q = P;
    ge_niels* row = tab + (size_t)win * ENT;
    row[0] = ge_niels_identity();
    ACT_NOUNROLL for (int k = 1; k < ENT; k++) {
        row[k] = ge_to_niels(Q);
        Q = ge_add_cached(Q, Pc);
    }
}
// The wide-window tables: thread (win, part) writes entries part*N+1 .. part*N+N (N = ACT_FB_PART, or all of them for
// narrow windows) of window `win`, converting to affine with one field inversion per ACT_FB_BATCH points (Montgomery's
// trick).  Part 0 also writes the identity entry 0.
ACT_FN void build_fb_table_thread(const ge* B, u32 bits, int win, int part, ge_niels* tab) {
    const u32 ent = fb_ent_of(bits);
    const int N = (int)((ent - 1) / fb_parts_of(bits));
    ge P = *B;
    ACT_NOUNROLL for (int i = 0; i < (int)bits * win; i++) P = ge_dbl(P, true);
    ge_cached Pc = ge_to_cached(P);
    ge_niels* row = tab + (size_t)win * ent;
    if (part == 0) row[0] = ge_niels_identity();
    // Q = (part * N) * P : N is a power of two
    ge Q = ge_identity();
    if (part > 0) {
        ge S = P;
        ACT_NOUNROLL for (int n = N; n > 1; n >>= 1) S = ge_dbl(S, true);
        ge_cached Sc = ge_to_cached(S);
        ACT_NOUNROLL for (int k = 0; k < part; k++) Q = ge_add_cached(Q, Sc);
    }
    ACT_NOUNROLL for (int k0 = 0; k0 < N; k0 += ACT_FB_BATCH) {
        fe xs[ACT_FB_BATCH], ys[ACT_FB_BATCH], zs[ACT_FB_BATCH], prefix[ACT_FB_BATCH];
        fe acc = fe_one();
        ACT_NOUNROLL for (int i = 0; i < ACT_FB_BATCH; i++) {
            Q = ge_add_cached(Q, Pc);
            xs[i] = Q.X; ys[i] = Q.Y; zs[i] = Q.Z;
            prefix[i] = acc;
            acc = fe_mul(acc, Q.Z);
        }
        fe inv = fe_invert(acc);
        ACT_NOUNROLL for (int i = ACT_FB_BATCH - 1; i >= 0; i--) {
            fe zi = fe_mul(inv, prefix[i]);
            inv = fe_mul(inv, zs[i]);
            row[(size_t)part * N + k0 + i + 1] = ge_affine_to_niels(fe_mul(xs[i], zi), fe_mul(ys[i], zi));
        }
    }
}
// Params::new (src/lib.rs:291-354).  dom: the "ACT-v1:..." separator as bytes (dlen <= 800).
// out: 3 x 8 words = enc(H1), enc(H2), enc(H3).
ACT_FN void params_derive_thread(const u8* dom, u32 dlen, u32* out) {
    u32 buf[256];
    u8* bb = reinterpret_cast<u8*>(buf);
    u32 o[16], seed[8];
    ACT_NOUNROLL for (int i = 0; i < 256; i++) buf[i] = 0;
    ACT_NOUNROLL for (int i = 0; i < 8; i++) bb[i] = (i < 4) ? 0 : (u8)(dlen >> (8 * (7 - i)));
    ACT_NOUNROLL for (u32 i = 0; i < dlen; i++) bb[8 + i] = dom[i];
    b3_hash_single_chunk(buf, 8 + dlen, o);
    ACT_UNROLL for (int i = 0; i < 8; i++) seed[i] = o[i];
    ACT_NOUNROLL for (u32 ctr = 0; ctr < 3; ctr++) {
        u32 n = 8 + dlen;
        ACT_NOUNROLL for (int i = 0; i < 8; i++) bb[n + i] = (i == 7) ? 32 : 0;
        n += 8;
        ACT_NOUNROLL for (int i = 0; i < 32; i++) bb[n + i] = (u8)(seed[i >> 2] >> (8 * (i & 3)));
        n += 32;
        ACT_NOUNROLL for (int i = 0; i < 8; i++) bb[n + i] = (i == 7) ? 4 : 0;
        n += 8;
        bb[n] = (u8)ctr; bb[n + 1] = 0; bb[n + 2] = 0; bb[n + 3] = 0;
        n += 4;
        b3_hash_single_chunk(buf, n, o);
        ge H = ristretto_from_uniform(o);
        ristretto_encode_(out + 8 * ctr, &H);
    }
}
