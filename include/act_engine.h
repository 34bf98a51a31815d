/*
 * act_engine.h -- C ABI of the B200 batch engine for the issuer side of anonymous-credit-tokens.
 *
 * The reference crate (Rust, /root/reference) has no FFI boundary of its own: the hot path sits
 * behind its public methods.  Each entry point below is what a `-sys` crate would bind in order
 * to offer `batch_issue` / `batch_verify_spend_and_refund` over slices (see INTEGRATION.md):
 *
 *   act_params_derive                  = Params::new                          src/lib.rs:291-354
 *   act_batch_issue[_dev]              = n x PrivateKey::issue                src/lib.rs:621-663
 *   act_batch_verify_spend_and_refund  = n x PrivateKey::refund               src/lib.rs:781-869
 *                                        (+ SpendProof::nullifier             src/lib.rs:720-722)
 *   act_batch_issuance_check[_dev]     = n x PreIssuance::to_credit_token     src/lib.rs:528-562 (verification half)
 *   act_batch_refund_check[_dev]       = n x PreRefund::to_credit_token       src/lib.rs:1217-1253 (verification half)
 *   act_pack_* / act_encode_*          = from_cbor / to_cbor                  src/cbor.rs:94-465
 *   act_batch_issue_verify + _sign,
 *   act_batch_spend_verify + act_batch_refund_sign
 *                                      = the same calls split where the reference draws from its RNG
 *                                        (after verification: src/lib.rs:638-643, 842-846), for hosts that own ONE RNG
 *   act_engine_create_multi            = one handle over several GPUs; host-buffer calls shard by request (SURVEY.md 8b, 8e)
 *   act_batch_verify_spend_and_refund_screened
 *                                      = refund() behind the caller's nullifier check (examples/act.rs:60-77) for a slice
 *   act_nullifier_store_*, act_batch_verify_spend_and_refund_recorded
 *                                      = that check against a nullifier database resident on the GPU, recorded as it goes
 *
 * Records hold WIRE bytes: points are 32-byte compressed ristretto255 encodings (validated on the
 * device exactly like CompressedRistretto::decompress, src/cbor.rs:62-77) and scalars are 32-byte
 * little-endian values reduced mod l on the device (Scalar::from_bytes_mod_order, src/cbor.rs:80-91).
 *
 *   IssuanceRequest  128 B : K | gamma | k_bar | r_bar                       (src/lib.rs:376-385)
 *   IssuanceResponse 160 B : A | e | gamma | z | c                           (src/lib.rs:572-583)
 *   SpendProof     16832 B : k | s | A' | B_bar | com[128] | gamma | e_bar | r2_bar | r3_bar | c_bar |
 *                            r_bar | w00 | w01 | gamma0[128] | z[128][2] | k_bar | s_bar   (src/lib.rs:673-708)
 *   Refund           128 B : A* | e* | gamma | z                             (src/lib.rs:1161-1170)
 *   rnd              128 B : the 64 bytes Scalar::random would draw for e, then the 64 for alpha
 *                            (src/lib.rs:643,649 / :846,852); ignored for rejected requests.
 *
 * Per-request outcome in status[i]:
 *   0        Ok
 *   1..9     1 + discriminant of the reference's `Error` (src/lib.rs:102-112):
 *            1 InvalidIssuanceRequestProof, 2 InvalidIssuanceResponseProof, 3 DoubleSpendError,
 *            4 InvalidRefundProof, 5 InvalidRefundResponseProof, 6 IdentityPointError,
 *            7 InvalidClientSpendProof, 8 AmountTooBigError, 9 ScalarOutOfRangeError
 *   0x81     a point failed to decode  (CborError::InvalidValue("invalid Ristretto point"))
 *   0x82     CBOR structure error      (CborError::InvalidStructure)   -- only from act_pack_*
 *   0x83     CBOR parse error          (CborError::Ciborium)           -- only from act_pack_*
 * Outputs of rejected requests are zero-filled.
 *
 * Return value of every function: 0 on success, negative on a whole-call failure (bad argument,
 * CUDA error); act_last_error() describes it.  There is no CPU fallback: without a usable CUDA
 * device every compute entry point fails.
 *
 * Threading: one engine may be used from one host thread at a time (a `_dev` call on a caller's stream is ordered against the
 * engine's previous pipeline by an event, so calls from different streams do not race on the engine's scratch).  Engines are
 * independent.
 * The caller owns every buffer.  Host-buffer entry points copy H2D/D2H internally (pinned buffers
 * from act_host_alloc make those copies asynchronous); `_dev` entry points take device pointers
 * (16-byte aligned) and a CUDA stream (cudaStream_t cast to void*, NULL = the engine's stream) and
 * are asynchronous with respect to the host.
 */
#ifndef ACT_ENGINE_H
#define ACT_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACT_REQUEST_BYTES 128
#define ACT_RESPONSE_BYTES 160
#define ACT_PROOF_BYTES 16832
#define ACT_REFUND_BYTES 128
#define ACT_RND_BYTES 128
#define ACT_COM_BYTES 4096

typedef struct act_engine act_engine;

#if defined(__GNUC__)
#define ACT_API __attribute__((visibility("default")))
#else
#define ACT_API
#endif

ACT_API const char* act_last_error(void);
ACT_API int act_device_count(void);

/* Params::new: H1 | H2 | H3 encodings (96 bytes).  Runs on `device`. */
ACT_API int act_params_derive(int device, const char* org, const char* service, const char* deployment, const char* version,
                      uint8_t h[96]);

/* Engine for one (Params, PrivateKey) pair on one GPU.  h = H1|H2|H3 encodings, sk_x = secret scalar
 * (reduced mod l), pk_w = encoding of W = G*x.  Fails if any point does not decode or if pk_w is not G*sk_x. */
ACT_API int act_engine_create(act_engine** out, int device, const uint8_t h[96], const uint8_t sk_x[32], const uint8_t pk_w[32]);
/* Multi-device engine: one replica of (tables, x, W) per listed GPU of this box (SURVEY.md 8b: `devices[], n_devices`).
 * Every HOST-buffer entry point below accepts it and shards the batch over the replicas -- replica g takes the contiguous
 * range (sizes differ by at most one request), each replica is driven by its own host thread, there is no cross-GPU arithmetic and the
 * outputs land in the caller's buffers exactly as a single-device call would leave them.  Device-buffer (`_dev`) entry
 * points take one replica: act_engine_replica(e, g).  A single-device engine is its own replica 0.  (A device listed twice
 * gets two replicas: no use in production, but a one-GPU box can exercise the sharded path that way.) */
ACT_API int act_engine_create_multi(act_engine** out, const int* devices, int n_devices, const uint8_t h[96], const uint8_t sk_x[32],
                                    const uint8_t pk_w[32]);
ACT_API int act_engine_replica_count(const act_engine* e);
ACT_API act_engine* act_engine_replica(act_engine* e, int i);
/* Zeroises the device and host copies of the secret, every staging copy of signer randomness and the local memory of the
 * signing kernels, then frees everything (replicas included). */
ACT_API void act_engine_destroy(act_engine* e);
ACT_API int act_engine_device(const act_engine* e);
/* Proofs per chunk of the spend pipeline (default 65536; also read from the environment variable ACT_SPEND_CHUNK at creation).
 * Batches are processed chunk by chunk over two streams; scratch memory is about 57 KB per proof of one chunk, twice. */
ACT_API int act_engine_set_spend_chunk(act_engine* e, size_t proofs);
/* PrivateKey::public: W = G*x for a given secret (convenience for key set-up). */
ACT_API int act_public_key(int device, const uint8_t sk_x[32], uint8_t pk_w[32]);

/* Pinned host memory helpers. */
ACT_API void* act_host_alloc(size_t bytes);
ACT_API void act_host_free(void* p);

/* ---- host-buffer entry points (synchronous) ---- */
ACT_API int act_batch_issue(act_engine* e, size_t n, const uint8_t* req /* n*128 */, const uint8_t* c /* n*32 */,
                    const uint8_t* rnd /* n*128 */, uint8_t* resp /* n*160 */, uint8_t* status /* n */);
ACT_API int act_batch_verify_spend_and_refund(act_engine* e, size_t n, const uint8_t* proofs /* n*16832 */,
                                      const uint8_t* rnd /* n*128 */, uint8_t* refunds /* n*128 */,
                                      uint8_t* nullifiers /* n*32 */, uint8_t* status /* n */);
ACT_API int act_batch_issuance_check(act_engine* e, size_t n, const uint8_t* K /* n*32 */, const uint8_t* resp /* n*160 */,
                             uint8_t* status /* n */);
ACT_API int act_batch_refund_check(act_engine* e, size_t n, const uint8_t* com /* n*4096 */, const uint8_t* refund /* n*128 */,
                           uint8_t* status /* n */);

/* ---- device-buffer entry points (asynchronous on `stream`) ---- */
ACT_API int act_batch_issue_dev(act_engine* e, size_t n, const void* req, const void* c, const void* rnd, void* resp,
                        void* status, void* stream);
ACT_API int act_batch_verify_spend_and_refund_dev(act_engine* e, size_t n, const void* proofs, const void* rnd, void* refunds,
                                          void* nullifiers, void* status, void* stream);
ACT_API int act_batch_issuance_check_dev(act_engine* e, size_t n, const void* K, const void* resp, void* status, void* stream);
ACT_API int act_batch_refund_check_dev(act_engine* e, size_t n, const void* com, const void* refund, void* status, void* stream);

/* Number of kernel launches issued by this engine since creation (for bench accounting). */
ACT_API uint64_t act_engine_launch_count(const act_engine* e);

/* Optional per-kernel device timing: when enabled every launch is bracketed by CUDA events on its stream.
 * act_engine_get_timing sums and clears them per kernel kind: 0 spend_range, 1 spend_head, 2 spend_chunk (hash),
 * 3 spend_finish, 4 refund_sign, 5 issue, 6 issuance_check, 7 refund_check, 8 spend_encode. */
ACT_API int act_engine_set_timing(act_engine* e, int enable);
ACT_API int act_engine_get_timing(act_engine* e, double ms[9], uint64_t count[9]);
/* Measured integer-multiply roofline of the device: sustained 32x32+64->64 multiply-adds per second. */
ACT_API int act_measure_int_mul_peak(int device, double* limb_macs_per_s);

/* Device self-test of the arithmetic layers against built-in known answers; 0 = pass. */
ACT_API int act_selftest(int device);

/* ---- CBOR front doors (host only; src/cbor.rs) ----
 * act_pack_*: decode n CBOR items (items[i], lens[i]) into fixed records; status[i] = 0, 0x82 or 0x83.
 * Point validity is NOT checked here (it is checked on the device and reported as 0x81).
 * act_encode_*: write the canonical CBOR encoding of a record; returns the encoded length. */
ACT_API int act_pack_issuance_requests_cbor(size_t n, const uint8_t* const* items, const size_t* lens, uint8_t* req, uint8_t* status);
ACT_API int act_pack_spend_proofs_cbor(size_t n, const uint8_t* const* items, const size_t* lens, uint8_t* proofs, uint8_t* status);
ACT_API int act_pack_issuance_responses_cbor(size_t n, const uint8_t* const* items, const size_t* lens, uint8_t* resp, uint8_t* status);
ACT_API int act_pack_refunds_cbor(size_t n, const uint8_t* const* items, const size_t* lens, uint8_t* refunds, uint8_t* status);
#define ACT_CBOR_REQUEST_BYTES 141
#define ACT_CBOR_RESPONSE_BYTES 176
#define ACT_CBOR_PROOF_BYTES 18036
#define ACT_CBOR_REFUND_BYTES 141
ACT_API size_t act_encode_issuance_request_cbor(const uint8_t req[128], uint8_t out[141]);
ACT_API size_t act_encode_issuance_response_cbor(const uint8_t resp[160], uint8_t out[176]);
ACT_API size_t act_encode_spend_proof_cbor(const uint8_t* proof /* 16832 */, uint8_t* out /* 18036 */);
ACT_API size_t act_encode_refund_cbor(const uint8_t refund[128], uint8_t out[141]);

/* ---- rows either side of the hot path (SURVEY.md 8f) ----
 *
 * Replay screen over a batch: what the reference leaves to the caller's nullifier database (src/lib.rs:741-745,
 * examples/act.rs:65-69; semantics of NullifierDb in src/tests.rs:28-50 applied in slice order).  Among accepted
 * proofs (status 0) the first occurrence of a nullifier keeps 0; every later one, and every nullifier present in
 * seen[n_seen*32], becomes 3 (DoubleSpendError).  Other statuses are copied.  Refund outputs are not touched. */
ACT_API int act_flag_replays_dev(act_engine* e, size_t n, const void* status, const void* nullifiers, size_t n_seen, const void* seen,
                                 void* status_out, void* stream);
ACT_API int act_flag_replays(act_engine* e, size_t n, const uint8_t* status, const uint8_t* nullifiers, size_t n_seen, const uint8_t* seen,
                             uint8_t* status_out);
/* Canonical-CBOR fast path on the device.  kind: 0 IssuanceRequest (141 B <-> 128 B), 1 IssuanceResponse (176 <-> 160),
 * 2 SpendProof (18036 <-> 16832), 3 Refund (141 <-> 128).  Items are fixed-size and contiguous.  Unpack accepts exactly
 * the encoding the reference's to_cbor produces (src/cbor.rs:96-103,153-161,216-268,413-420): status 0, or 0xFF =
 * "not the canonical skeleton" -> hand that item to act_pack_*_cbor (the lenient host parser). */
#define ACT_KIND_REQUEST 0
#define ACT_KIND_RESPONSE 1
#define ACT_KIND_PROOF 2
#define ACT_KIND_REFUND 3
#define ACT_STATUS_NOT_CANONICAL 0xFF
ACT_API int act_unpack_cbor_dev(act_engine* e, int kind, size_t n, const void* cbor, void* records, void* status, void* stream);
ACT_API int act_encode_cbor_dev(act_engine* e, int kind, size_t n, const void* records, void* cbor, void* stream);
ACT_API int act_unpack_cbor(act_engine* e, int kind, size_t n, const uint8_t* cbor, uint8_t* records, uint8_t* status);
ACT_API int act_encode_cbor(act_engine* e, int kind, size_t n, const uint8_t* records, uint8_t* cbor);

/* Sequential-RNG contract: outputs identical to a loop of PrivateKey::issue / PrivateKey::refund calls over ONE shared RNG.
 * The reference draws e and alpha (64 bytes each) only after a request verifies (src/lib.rs:638-643, 842-846), so
 * request i uses the 128 bytes at offset 128 * (number of accepted requests before i) of rnd_stream.  *consumed
 * (optional) receives the number of stream bytes used; the call fails if the stream is shorter than that.
 * Host buffers; two passes (verify, then sign) with one host-side scan of the accept bits in between. */
ACT_API int act_batch_issue_seq(act_engine* e, size_t n, const uint8_t* req, const uint8_t* c, const uint8_t* rnd_stream, size_t rnd_stream_len,
                                uint8_t* resp, uint8_t* status, size_t* consumed);
ACT_API int act_batch_verify_spend_and_refund_seq(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* rnd_stream, size_t rnd_stream_len,
                                                   uint8_t* refunds, uint8_t* nullifiers, uint8_t* status, size_t* consumed);

/* Two-pass forms: what a host that owns ONE RNG needs in order to behave exactly like a loop over the reference's calls (an
 * `impl CryptoRngCore` taken by value, src/lib.rs:626,785, from which e and alpha are drawn only after a request verifies):
 * verify, count the accepted requests, draw 128 bytes for each of them in slice order, sign.
 *   act_batch_issue_verify : status[i] = 0 / 1 / 0x81; nothing else is written
 *   act_batch_issue_sign   : status is the verify pass's; rnd = 128 bytes per ACCEPTED request, in slice order (rnd_len >= that);
 *                            resp as act_batch_issue (zero-filled for rejected requests)
 *   act_batch_spend_verify : status, nullifiers (reduced k; zero when rejected) and kprime[n*128] -- K' = sum 2^j com_j in extended
 *                            coordinates (public: a function of the proof), the only state the signing pass needs
 *   act_batch_refund_sign  : refunds as act_batch_verify_spend_and_refund
 * The `_seq` calls above are these two passes around a count of the accept bits. */
ACT_API int act_batch_issue_verify(act_engine* e, size_t n, const uint8_t* req, uint8_t* status);
ACT_API int act_batch_issue_sign(act_engine* e, size_t n, const uint8_t* req, const uint8_t* c, const uint8_t* status, const uint8_t* rnd, size_t rnd_len,
                                 uint8_t* resp);
ACT_API int act_batch_spend_verify(act_engine* e, size_t n, const uint8_t* proofs, uint8_t* nullifiers, uint8_t* status, uint8_t* kprime /* n*128 */);
ACT_API int act_batch_refund_sign(act_engine* e, size_t n, const uint8_t* kprime, const uint8_t* status, const uint8_t* rnd, size_t rnd_len,
                                  uint8_t* refunds);

/* The issuer's whole batch step in one call (what examples/act.rs:60-77 does per request: nullifier check, then refund): verify +
 * refund on every replica, gather of status + nullifiers (33 B per proof) to replica 0 over NVLink (cudaMemcpyPeerAsync), replay
 * screen there against the batch itself and `seen`.  A replayed proof gets status 3 (DoubleSpendError) and no refund (zero-filled);
 * its nullifier is kept.  Single-device engines take the same call (no gather). */
ACT_API int act_batch_verify_spend_and_refund_screened(act_engine* e, size_t n, const uint8_t* proofs, const uint8_t* rnd, size_t n_seen,
                                                       const uint8_t* seen, uint8_t* refunds, uint8_t* nullifiers, uint8_t* status);

/* ---- device-resident nullifier store: the set of nullifiers already spent (the reference's NullifierDb, src/lib.rs:741-745,
 * examples/act.rs:60-77), kept in the memory of one GPU between calls.  It holds no key material and is independent of any engine.
 * Members are 32-byte nullifiers reduced mod l (what the engine emits); a screen whose status-0 keys include one that is not
 * reduced fails as a whole.
 *
 * Screen semantics: those of act_flag_replays with the store in place of `seen`: among status-0 entries, one whose nullifier is in
 * the store or occurred at an earlier status-0 index of the batch gets 3 (DoubleSpendError); other statuses are copied.  With
 * record != 0 every nullifier whose output status is 0 is then inserted.  A recording call that fails (bad argument, wrong
 * device, non-reduced key, failure to grow) leaves the store unchanged.  A store may be used from one host thread at a time;
 * calls on different streams are ordered by an event. */
typedef struct act_nullifier_store act_nullifier_store;
/* capacity = nullifiers to size for up front; the store grows on its own (on-device rehash) when a recording call needs it */
ACT_API int    act_nullifier_store_create(act_nullifier_store** out, int device, size_t capacity);
/* frees everything and wipes the slot PRF key */
ACT_API void   act_nullifier_store_destroy(act_nullifier_store* s);
ACT_API int    act_nullifier_store_device(const act_nullifier_store* s);
ACT_API size_t act_nullifier_store_size(const act_nullifier_store* s);     /* synchronises */
/* the screen against store + batch; record != 0 inserts the survivors.  Bulk import = status all zero, record = 1
   (status_out[i] == 0 <=> newly inserted).  The _dev form takes device memory of the store's device (nullifiers 16-byte aligned;
   status_out may equal status) and a stream (NULL = the store's own); it waits once on that stream for a 16-byte read-back (the
   key check and the exact size, which decides growth) and is asynchronous after it. */
ACT_API int act_nullifier_store_screen_dev(act_nullifier_store* s, size_t n, const void* status, const void* nullifiers,
                                           void* status_out, int record, void* stream);
ACT_API int act_nullifier_store_screen(act_nullifier_store* s, size_t n, const uint8_t* status, const uint8_t* nullifiers,
                                       uint8_t* status_out, int record);
/* every member, 32 B each, order unspecified (for checkpoints); *count = size; fails if cap (in keys) < size */
ACT_API int act_nullifier_store_export(act_nullifier_store* s, uint8_t* out, size_t cap, size_t* count);
/* the issuer's step with the store: _screened with the store in place of `seen`, survivors recorded.
   Replays get status 3 and a zero-filled refund, as in _screened.  The store must be on the device of replica 0. */
ACT_API int act_batch_verify_spend_and_refund_recorded(act_engine* e, act_nullifier_store* s, size_t n, const uint8_t* proofs,
                                                       const uint8_t* rnd, uint8_t* refunds, uint8_t* nullifiers, uint8_t* status);

/* Client-side batch generators (SURVEY.md 8f-1), bit-exact with the reference's prover for the same RNG bytes but NOT
 * constant time: they exist to synthesise full-size batches of valid, unique fixtures on the device.
 *   act_batch_request      = n x PreIssuance::request          src/lib.rs:463-487
 *       pre  n*64  : r | k  (the PreIssuance scalars, reduced mod l on the device)
 *       rnd  n*128 : the 64 bytes Scalar::random draws for k', then the 64 for r'   (:468-469)
 *       req  n*128 : IssuanceRequest records
 *   act_batch_prove_spend  = n x CreditToken::prove_spend      src/lib.rs:972-1152
 *       tokens n*160 : A | e | k | r | c  (CreditToken);  charges n*32 : s
 *       rnd    n*33536 : the 524 x 64 bytes the prover draws, in the reference's order (:978-984, 998-999, 1010-1023,
 *                1057-1058); or NULL, then scalar t of proof i is the wide reduction of output block t of
 *                BLAKE3-XOF(seed[32] || u64le(first_index + i))
 *       proofs n*16832 : SpendProof records;  prerefunds n*96 : k* | r* | m  (PreRefund, :1124-1128)
 *       status n : 0, or 0x81 when the token's A does not decode (outputs zero-filled)
 *   Precondition as in the reference (:931-934): 2^128 > c >= s, otherwise the proof is produced but does not verify. */
#define ACT_TOKEN_BYTES 160
#define ACT_PREREFUND_BYTES 96
#define ACT_PROVE_RND_BYTES 33536
ACT_API int act_batch_request_dev(act_engine* e, size_t n, const void* pre, const void* rnd, void* req, void* stream);
ACT_API int act_batch_request(act_engine* e, size_t n, const uint8_t* pre, const uint8_t* rnd, uint8_t* req);
ACT_API int act_batch_prove_spend_dev(act_engine* e, size_t n, const void* tokens, const void* charges, const void* rnd, const uint8_t seed[32],
                                      uint64_t first_index, void* proofs, void* prerefunds, void* status, void* stream);
ACT_API int act_batch_prove_spend(act_engine* e, size_t n, const uint8_t* tokens, const uint8_t* charges, const uint8_t* rnd, const uint8_t seed[32],
                                  uint64_t first_index, uint8_t* proofs, uint8_t* prerefunds, uint8_t* status);

#ifdef __cplusplus
}
#endif
#endif /* ACT_ENGINE_H */
