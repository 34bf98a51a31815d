//! Raw bindings to `include/act_engine.h`.  Record layouts, status codes and ownership rules are documented there.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct act_engine {
    _private: [u8; 0],
}

#[repr(C)]
pub struct act_nullifier_store {
    _private: [u8; 0],
}

pub const ACT_REQUEST_BYTES: usize = 128;
pub const ACT_RESPONSE_BYTES: usize = 160;
pub const ACT_PROOF_BYTES: usize = 16832;
pub const ACT_REFUND_BYTES: usize = 128;
pub const ACT_RND_BYTES: usize = 128;
pub const ACT_COM_BYTES: usize = 4096;
pub const ACT_TOKEN_BYTES: usize = 160;
pub const ACT_PREREFUND_BYTES: usize = 96;
pub const ACT_PROVE_RND_BYTES: usize = 33536;
pub const ACT_CBOR_REQUEST_BYTES: usize = 141;
pub const ACT_CBOR_RESPONSE_BYTES: usize = 176;
pub const ACT_CBOR_PROOF_BYTES: usize = 18036;
pub const ACT_CBOR_REFUND_BYTES: usize = 141;
pub const ACT_KIND_REQUEST: c_int = 0;
pub const ACT_KIND_RESPONSE: c_int = 1;
pub const ACT_KIND_PROOF: c_int = 2;
pub const ACT_KIND_REFUND: c_int = 3;
pub const ACT_STATUS_NOT_CANONICAL: u8 = 0xFF;

extern "C" {
    pub fn act_last_error() -> *const c_char;
    pub fn act_device_count() -> c_int;
    pub fn act_params_derive(device: c_int, org: *const c_char, service: *const c_char, deployment: *const c_char,
                             version: *const c_char, h: *mut u8) -> c_int;
    pub fn act_engine_create(out: *mut *mut act_engine, device: c_int, h: *const u8, sk_x: *const u8, pk_w: *const u8) -> c_int;
    pub fn act_engine_create_multi(out: *mut *mut act_engine, devices: *const c_int, n_devices: c_int, h: *const u8, sk_x: *const u8,
                                   pk_w: *const u8) -> c_int;
    pub fn act_engine_replica_count(e: *const act_engine) -> c_int;
    pub fn act_engine_replica(e: *mut act_engine, i: c_int) -> *mut act_engine;
    pub fn act_engine_set_spend_chunk(e: *mut act_engine, proofs: usize) -> c_int;
    pub fn act_engine_destroy(e: *mut act_engine);
    pub fn act_engine_device(e: *const act_engine) -> c_int;
    pub fn act_public_key(device: c_int, sk_x: *const u8, pk_w: *mut u8) -> c_int;
    pub fn act_host_alloc(bytes: usize) -> *mut c_void;
    pub fn act_host_free(p: *mut c_void);

    pub fn act_batch_issue(e: *mut act_engine, n: usize, req: *const u8, c: *const u8, rnd: *const u8, resp: *mut u8, status: *mut u8) -> c_int;
    pub fn act_batch_verify_spend_and_refund(e: *mut act_engine, n: usize, proofs: *const u8, rnd: *const u8, refunds: *mut u8,
                                             nullifiers: *mut u8, status: *mut u8) -> c_int;
    pub fn act_batch_issuance_check(e: *mut act_engine, n: usize, k: *const u8, resp: *const u8, status: *mut u8) -> c_int;
    pub fn act_batch_refund_check(e: *mut act_engine, n: usize, com: *const u8, refund: *const u8, status: *mut u8) -> c_int;
    pub fn act_batch_issue_seq(e: *mut act_engine, n: usize, req: *const u8, c: *const u8, rnd_stream: *const u8, rnd_stream_len: usize,
                               resp: *mut u8, status: *mut u8, consumed: *mut usize) -> c_int;
    pub fn act_batch_verify_spend_and_refund_seq(e: *mut act_engine, n: usize, proofs: *const u8, rnd_stream: *const u8,
                                                 rnd_stream_len: usize, refunds: *mut u8, nullifiers: *mut u8, status: *mut u8,
                                                 consumed: *mut usize) -> c_int;

    // two-pass forms: verify, then sign with 128 bytes of randomness per ACCEPTED request in slice order
    pub fn act_batch_issue_verify(e: *mut act_engine, n: usize, req: *const u8, status: *mut u8) -> c_int;
    pub fn act_batch_issue_sign(e: *mut act_engine, n: usize, req: *const u8, c: *const u8, status: *const u8, rnd: *const u8, rnd_len: usize,
                                resp: *mut u8) -> c_int;
    pub fn act_batch_spend_verify(e: *mut act_engine, n: usize, proofs: *const u8, nullifiers: *mut u8, status: *mut u8, kprime: *mut u8) -> c_int;
    pub fn act_batch_refund_sign(e: *mut act_engine, n: usize, kprime: *const u8, status: *const u8, rnd: *const u8, rnd_len: usize,
                                 refunds: *mut u8) -> c_int;
    pub fn act_batch_verify_spend_and_refund_screened(e: *mut act_engine, n: usize, proofs: *const u8, rnd: *const u8, n_seen: usize,
                                                      seen: *const u8, refunds: *mut u8, nullifiers: *mut u8, status: *mut u8) -> c_int;

    pub fn act_batch_issue_dev(e: *mut act_engine, n: usize, req: *const c_void, c: *const c_void, rnd: *const c_void, resp: *mut c_void,
                               status: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn act_batch_verify_spend_and_refund_dev(e: *mut act_engine, n: usize, proofs: *const c_void, rnd: *const c_void,
                                                 refunds: *mut c_void, nullifiers: *mut c_void, status: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn act_batch_issuance_check_dev(e: *mut act_engine, n: usize, k: *const c_void, resp: *const c_void, status: *mut c_void,
                                        stream: *mut c_void) -> c_int;
    pub fn act_batch_refund_check_dev(e: *mut act_engine, n: usize, com: *const c_void, refund: *const c_void, status: *mut c_void,
                                      stream: *mut c_void) -> c_int;

    // the spent set resident on one GPU (NullifierDb kept between calls); independent of any engine
    pub fn act_nullifier_store_create(out: *mut *mut act_nullifier_store, device: c_int, capacity: usize) -> c_int;
    pub fn act_nullifier_store_destroy(s: *mut act_nullifier_store);
    pub fn act_nullifier_store_device(s: *const act_nullifier_store) -> c_int;
    pub fn act_nullifier_store_size(s: *const act_nullifier_store) -> usize;
    pub fn act_nullifier_store_screen_dev(s: *mut act_nullifier_store, n: usize, status: *const c_void, nullifiers: *const c_void,
                                          status_out: *mut c_void, record: c_int, stream: *mut c_void) -> c_int;
    pub fn act_nullifier_store_screen(s: *mut act_nullifier_store, n: usize, status: *const u8, nullifiers: *const u8, status_out: *mut u8,
                                      record: c_int) -> c_int;
    pub fn act_nullifier_store_export(s: *mut act_nullifier_store, out: *mut u8, cap: usize, count: *mut usize) -> c_int;
    // the issuer's step with the store in place of `seen`; survivors are recorded (store on the device of replica 0)
    pub fn act_batch_verify_spend_and_refund_recorded(e: *mut act_engine, s: *mut act_nullifier_store, n: usize, proofs: *const u8,
                                                      rnd: *const u8, refunds: *mut u8, nullifiers: *mut u8, status: *mut u8) -> c_int;
    pub fn act_flag_replays(e: *mut act_engine, n: usize, status: *const u8, nullifiers: *const u8, n_seen: usize, seen: *const u8,
                            status_out: *mut u8) -> c_int;
    pub fn act_flag_replays_dev(e: *mut act_engine, n: usize, status: *const c_void, nullifiers: *const c_void, n_seen: usize,
                                seen: *const c_void, status_out: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn act_unpack_cbor(e: *mut act_engine, kind: c_int, n: usize, cbor: *const u8, records: *mut u8, status: *mut u8) -> c_int;
    pub fn act_encode_cbor(e: *mut act_engine, kind: c_int, n: usize, records: *const u8, cbor: *mut u8) -> c_int;
    pub fn act_unpack_cbor_dev(e: *mut act_engine, kind: c_int, n: usize, cbor: *const c_void, records: *mut c_void, status: *mut c_void,
                               stream: *mut c_void) -> c_int;
    pub fn act_encode_cbor_dev(e: *mut act_engine, kind: c_int, n: usize, records: *const c_void, cbor: *mut c_void, stream: *mut c_void) -> c_int;

    pub fn act_batch_request(e: *mut act_engine, n: usize, pre: *const u8, rnd: *const u8, req: *mut u8) -> c_int;
    pub fn act_batch_prove_spend(e: *mut act_engine, n: usize, tokens: *const u8, charges: *const u8, rnd: *const u8, seed: *const u8,
                                 first_index: u64, proofs: *mut u8, prerefunds: *mut u8, status: *mut u8) -> c_int;
    pub fn act_batch_request_dev(e: *mut act_engine, n: usize, pre: *const c_void, rnd: *const c_void, req: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn act_batch_prove_spend_dev(e: *mut act_engine, n: usize, tokens: *const c_void, charges: *const c_void, rnd: *const c_void,
                                     seed: *const u8, first_index: u64, proofs: *mut c_void, prerefunds: *mut c_void, status: *mut c_void,
                                     stream: *mut c_void) -> c_int;

    pub fn act_pack_issuance_requests_cbor(n: usize, items: *const *const u8, lens: *const usize, req: *mut u8, status: *mut u8) -> c_int;
    pub fn act_pack_spend_proofs_cbor(n: usize, items: *const *const u8, lens: *const usize, proofs: *mut u8, status: *mut u8) -> c_int;
    pub fn act_pack_issuance_responses_cbor(n: usize, items: *const *const u8, lens: *const usize, resp: *mut u8, status: *mut u8) -> c_int;
    pub fn act_pack_refunds_cbor(n: usize, items: *const *const u8, lens: *const usize, refunds: *mut u8, status: *mut u8) -> c_int;
    pub fn act_encode_issuance_request_cbor(req: *const u8, out: *mut u8) -> usize;
    pub fn act_encode_issuance_response_cbor(resp: *const u8, out: *mut u8) -> usize;
    pub fn act_encode_spend_proof_cbor(proof: *const u8, out: *mut u8) -> usize;
    pub fn act_encode_refund_cbor(refund: *const u8, out: *mut u8) -> usize;

    pub fn act_engine_launch_count(e: *const act_engine) -> u64;
    pub fn act_engine_set_timing(e: *mut act_engine, enable: c_int) -> c_int;
    pub fn act_engine_get_timing(e: *mut act_engine, ms: *mut f64, count: *mut u64) -> c_int;
    pub fn act_measure_int_mul_peak(device: c_int, limb_macs_per_s: *mut f64) -> c_int;
    pub fn act_selftest(device: c_int) -> c_int;
}
