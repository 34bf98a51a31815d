/* act_oracle_keys.c -- TEST-ONLY: the CPU oracle (oracle/act_oracle.c, included whole) plus the refund of an issuer that holds
 * several keys: a spend proof is verified under the key its token was issued with and refunded under the current key.  A
 * separate library, so that the oracle the CPU baseline times stays as it is. */
#include "../../oracle/act_oracle.c"

/* the signing half of act_refund (src/lib.rs:846-868) under `key`, for a proof that has verified */
static void refund_sign(const act_params *P, const act_key *key, const spend_proof *sp, const u8 *rnd, refund_t *out) {
    ge t1, k_prime, x_a, a, x_g, y_a, y_g;
    sc e, alpha, ex, inv, z, gamma;
    ge_identity(&k_prime);                                                               /* :819-824 */
    for (int i = 0; i < ACT_L; i++) { sc p2; sc_pow2(&p2, i); ge_scalarmult(&t1, &sp->com[i], &p2); ge_add(&k_prime, &k_prime, &t1); }
    scalar_random(&e, &rnd);                                                             /* :846 */
    ge_add(&x_a, &GE_BASE, &k_prime);                                                    /* :848 */
    sc_add(&ex, &e, &key->x); sc_invert(&inv, &ex); ge_scalarmult(&a, &x_a, &inv);       /* :849 */
    ge_scalarmult(&t1, &GE_BASE, &e); ge_add(&x_g, &t1, &key->w);                        /* :851 */
    scalar_random(&alpha, &rnd);                                                         /* :852 */
    ge_scalarmult(&y_a, &a, &alpha); ge_scalarmult(&y_g, &GE_BASE, &alpha);              /* :853-854 */
    transcript tr;
    tr_new(&tr, P, "refund");                                                            /* :856-859 */
    tr_add_scalar(&tr, &e);
    tr_add_element(&tr, &a); tr_add_element(&tr, &x_a); tr_add_element(&tr, &x_g);
    tr_add_element(&tr, &y_a); tr_add_element(&tr, &y_g);
    tr_challenge(&gamma, &tr);
    sc_mul(&z, &gamma, &ex); sc_add(&z, &z, &alpha);                                     /* :861 */
    out->A = a; out->e = e; out->gamma = gamma; out->z = z;
}

/* act_o_refund with the proof verified under verify_ctx's key and the refund signed under sign_ctx's key (both contexts of the
 * same Params).  verify_ctx == NULL stands for a key id that names no key: status 7 after the decode and identity checks. */
EXPORT int act_o_refund_keyed(const act_o_ctx *verify_ctx, const act_o_ctx *sign_ctx, const u8 *proof, const u8 rnd[128], u8 refund[128],
                              u8 nullifier[32]) {
    oracle_init();
    spend_proof *sp = (spend_proof *)malloc(sizeof *sp); refund_t rf;
    memset(refund, 0, 128); memset(nullifier, 0, 32);
    if (!proof_unpack(sp, proof)) { free(sp); return ST_DECODE_INVALID_POINT; }
    int st;
    if (ge_is_identity_ristretto(&sp->a_prime)) st = ST_IDENTITY_POINT;
    else if (!verify_ctx) st = ST_INVALID_CLIENT_SPEND_PROOF;
    else st = act_refund(&verify_ctx->P, &verify_ctx->key, sp, rnd, &rf);   /* its refund is discarded: only the verdict counts */
    if (st == ST_OK) {
        refund_sign(&sign_ctx->P, &sign_ctx->key, sp, rnd, &rf);
        ristretto_encode(refund, &rf.A); sc_tobytes(refund + 32, &rf.e); sc_tobytes(refund + 64, &rf.gamma);
        sc_tobytes(refund + 96, &rf.z); sc_tobytes(nullifier, &sp->k);
    }
    free(sp);
    return st;
}
