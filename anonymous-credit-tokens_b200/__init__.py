"""anonymous-credit-tokens_b200 -- B200-native batch engine for the issuer side of Anonymous Credit Tokens.

Host-side mirror of the reference crate's interface for the hot path (names and argument meaning
follow /root/reference src/lib.rs): `Params.new`, `PrivateKey`, and the batch forms of
`PrivateKey::issue` (:621-663), `PrivateKey::refund` (:781-869), `PreIssuance::to_credit_token`
(:528-562) and `PreRefund::to_credit_token` (:1217-1253), all running as CUDA kernels behind the C
ABI of include/act_engine.h (libact_b200.so, loaded with ctypes).

There is no CPU fallback: importing works anywhere, but every compute call requires the CUDA
library and a GPU and raises otherwise.

The package directory name contains a hyphen, so import it with
    importlib.import_module("anonymous-credit-tokens_b200")
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libact_b200.so")

REQUEST_BYTES = 128
RESPONSE_BYTES = 160
PROOF_BYTES = 16832
REFUND_BYTES = 128
RND_BYTES = 128
COM_BYTES = 4096
L = 128
KIND_REQUEST, KIND_RESPONSE, KIND_PROOF, KIND_REFUND = 0, 1, 2, 3
CBOR_BYTES = {0: 141, 1: 176, 2: 18036, 3: 141}
RECORD_BYTES = {0: 128, 1: 160, 2: 16832, 3: 128}
NOT_CANONICAL = 0xFF
TOKEN_BYTES = 160
PREREFUND_BYTES = 96
PROVE_RND_BYTES = 524 * 64
KEY_SLOTS = 16

# status codes (include/act_engine.h; 1 + discriminant of the reference's `Error`, src/lib.rs:102-112)
OK = 0
INVALID_ISSUANCE_REQUEST_PROOF = 1
INVALID_ISSUANCE_RESPONSE_PROOF = 2
DOUBLE_SPEND_ERROR = 3
INVALID_REFUND_PROOF = 4
INVALID_REFUND_RESPONSE_PROOF = 5
IDENTITY_POINT_ERROR = 6
INVALID_CLIENT_SPEND_PROOF = 7
AMOUNT_TOO_BIG_ERROR = 8
SCALAR_OUT_OF_RANGE_ERROR = 9
DECODE_INVALID_POINT = 0x81
DECODE_BAD_STRUCTURE = 0x82
DECODE_PARSE_ERROR = 0x83

ERROR_NAMES = {
    0: "Ok", 1: "InvalidIssuanceRequestProof", 2: "InvalidIssuanceResponseProof", 3: "DoubleSpendError",
    4: "InvalidRefundProof", 5: "InvalidRefundResponseProof", 6: "IdentityPointError",
    7: "InvalidClientSpendProof", 8: "AmountTooBigError", 9: "ScalarOutOfRangeError",
    0x81: "CborError::InvalidValue(invalid Ristretto point)", 0x82: "CborError::InvalidStructure",
    0x83: "CborError::Ciborium",
}

EXPORTED_SYMBOLS = [
    "act_last_error", "act_device_count", "act_params_derive", "act_engine_create", "act_engine_destroy",
    "act_engine_device", "act_public_key", "act_host_alloc", "act_host_free", "act_batch_issue",
    "act_batch_verify_spend_and_refund", "act_batch_issuance_check", "act_batch_refund_check",
    "act_batch_issue_dev", "act_batch_verify_spend_and_refund_dev", "act_batch_issuance_check_dev",
    "act_batch_refund_check_dev", "act_engine_launch_count", "act_selftest", "act_engine_set_timing",
    "act_engine_get_timing", "act_measure_int_mul_peak",
    "act_pack_issuance_requests_cbor", "act_pack_spend_proofs_cbor", "act_pack_issuance_responses_cbor",
    "act_pack_refunds_cbor", "act_encode_issuance_request_cbor", "act_encode_issuance_response_cbor",
    "act_encode_spend_proof_cbor", "act_encode_refund_cbor",
    "act_flag_replays", "act_flag_replays_dev", "act_unpack_cbor", "act_unpack_cbor_dev", "act_encode_cbor", "act_encode_cbor_dev",
    "act_batch_request", "act_batch_request_dev", "act_batch_prove_spend", "act_batch_prove_spend_dev",
    "act_batch_issue_seq", "act_batch_verify_spend_and_refund_seq", "act_engine_set_spend_chunk",
    "act_engine_create_multi", "act_engine_replica_count", "act_engine_replica",
    "act_batch_issue_verify", "act_batch_issue_sign", "act_batch_spend_verify", "act_batch_refund_sign",
    "act_batch_verify_spend_and_refund_screened",
    "act_nullifier_store_create", "act_nullifier_store_destroy", "act_nullifier_store_device", "act_nullifier_store_size",
    "act_nullifier_store_screen_dev", "act_nullifier_store_screen", "act_nullifier_store_export",
    "act_batch_verify_spend_and_refund_recorded",
    "act_engine_set_key", "act_engine_clear_key", "act_engine_select_key", "act_engine_selected_key", "act_engine_key_slots",
    "act_batch_verify_spend_and_refund_keyed_dev", "act_batch_verify_spend_and_refund_keyed", "act_batch_spend_verify_keyed",
]


class ActError(RuntimeError):
    pass


_lib = None


def load_library():
    """dlopen libact_b200.so and declare the C ABI.  Raises if the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ActError(f"{LIB_PATH} is missing: build it with __graft_entry__.build() (nvcc, sm_100a). "
                       "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, cp, sz, i32, u64 = C.c_void_p, C.c_char_p, C.c_size_t, C.c_int, C.c_uint64
    lib.act_last_error.restype = cp
    lib.act_device_count.restype = i32
    lib.act_params_derive.argtypes = [i32, cp, cp, cp, cp, vp]; lib.act_params_derive.restype = i32
    lib.act_engine_create.argtypes = [C.POINTER(vp), i32, vp, vp, vp]; lib.act_engine_create.restype = i32
    lib.act_engine_destroy.argtypes = [vp]; lib.act_engine_destroy.restype = None
    lib.act_engine_device.argtypes = [vp]; lib.act_engine_device.restype = i32
    lib.act_engine_set_spend_chunk.argtypes = [vp, sz]; lib.act_engine_set_spend_chunk.restype = i32
    lib.act_public_key.argtypes = [i32, vp, vp]; lib.act_public_key.restype = i32
    lib.act_host_alloc.argtypes = [sz]; lib.act_host_alloc.restype = vp
    lib.act_host_free.argtypes = [vp]; lib.act_host_free.restype = None
    lib.act_batch_issue.argtypes = [vp, sz, vp, vp, vp, vp, vp]; lib.act_batch_issue.restype = i32
    lib.act_batch_verify_spend_and_refund.argtypes = [vp, sz, vp, vp, vp, vp, vp]; lib.act_batch_verify_spend_and_refund.restype = i32
    lib.act_batch_issuance_check.argtypes = [vp, sz, vp, vp, vp]; lib.act_batch_issuance_check.restype = i32
    lib.act_batch_refund_check.argtypes = [vp, sz, vp, vp, vp]; lib.act_batch_refund_check.restype = i32
    lib.act_batch_issue_dev.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp]; lib.act_batch_issue_dev.restype = i32
    lib.act_batch_verify_spend_and_refund_dev.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp]; lib.act_batch_verify_spend_and_refund_dev.restype = i32
    lib.act_batch_issuance_check_dev.argtypes = [vp, sz, vp, vp, vp, vp]; lib.act_batch_issuance_check_dev.restype = i32
    lib.act_batch_refund_check_dev.argtypes = [vp, sz, vp, vp, vp, vp]; lib.act_batch_refund_check_dev.restype = i32
    lib.act_engine_launch_count.argtypes = [vp]; lib.act_engine_launch_count.restype = u64
    lib.act_selftest.argtypes = [i32]; lib.act_selftest.restype = i32
    lib.act_engine_set_timing.argtypes = [vp, i32]; lib.act_engine_set_timing.restype = i32
    lib.act_engine_get_timing.argtypes = [vp, vp, vp]; lib.act_engine_get_timing.restype = i32
    lib.act_measure_int_mul_peak.argtypes = [i32, vp]; lib.act_measure_int_mul_peak.restype = i32
    for name in ("act_pack_issuance_requests_cbor", "act_pack_spend_proofs_cbor", "act_pack_issuance_responses_cbor", "act_pack_refunds_cbor"):
        f = getattr(lib, name); f.argtypes = [sz, vp, vp, vp, vp]; f.restype = i32
    for name in ("act_encode_issuance_request_cbor", "act_encode_issuance_response_cbor", "act_encode_spend_proof_cbor", "act_encode_refund_cbor"):
        f = getattr(lib, name); f.argtypes = [vp, vp]; f.restype = sz
    lib.act_flag_replays_dev.argtypes = [vp, sz, vp, vp, sz, vp, vp, vp]; lib.act_flag_replays_dev.restype = i32
    lib.act_flag_replays.argtypes = [vp, sz, vp, vp, sz, vp, vp]; lib.act_flag_replays.restype = i32
    lib.act_unpack_cbor_dev.argtypes = [vp, i32, sz, vp, vp, vp, vp]; lib.act_unpack_cbor_dev.restype = i32
    lib.act_encode_cbor_dev.argtypes = [vp, i32, sz, vp, vp, vp]; lib.act_encode_cbor_dev.restype = i32
    lib.act_unpack_cbor.argtypes = [vp, i32, sz, vp, vp, vp]; lib.act_unpack_cbor.restype = i32
    lib.act_encode_cbor.argtypes = [vp, i32, sz, vp, vp]; lib.act_encode_cbor.restype = i32
    lib.act_batch_request_dev.argtypes = [vp, sz, vp, vp, vp, vp]; lib.act_batch_request_dev.restype = i32
    lib.act_batch_request.argtypes = [vp, sz, vp, vp, vp]; lib.act_batch_request.restype = i32
    lib.act_batch_prove_spend_dev.argtypes = [vp, sz, vp, vp, vp, vp, u64, vp, vp, vp, vp]; lib.act_batch_prove_spend_dev.restype = i32
    lib.act_batch_prove_spend.argtypes = [vp, sz, vp, vp, vp, vp, u64, vp, vp, vp]; lib.act_batch_prove_spend.restype = i32
    lib.act_batch_issue_seq.argtypes = [vp, sz, vp, vp, vp, sz, vp, vp, vp]; lib.act_batch_issue_seq.restype = i32
    lib.act_batch_verify_spend_and_refund_seq.argtypes = [vp, sz, vp, vp, sz, vp, vp, vp, vp]; lib.act_batch_verify_spend_and_refund_seq.restype = i32
    lib.act_engine_create_multi.argtypes = [C.POINTER(vp), vp, i32, vp, vp, vp]; lib.act_engine_create_multi.restype = i32
    lib.act_engine_replica_count.argtypes = [vp]; lib.act_engine_replica_count.restype = i32
    lib.act_engine_replica.argtypes = [vp, i32]; lib.act_engine_replica.restype = vp
    lib.act_batch_issue_verify.argtypes = [vp, sz, vp, vp]; lib.act_batch_issue_verify.restype = i32
    lib.act_batch_issue_sign.argtypes = [vp, sz, vp, vp, vp, vp, sz, vp]; lib.act_batch_issue_sign.restype = i32
    lib.act_batch_spend_verify.argtypes = [vp, sz, vp, vp, vp, vp]; lib.act_batch_spend_verify.restype = i32
    lib.act_batch_refund_sign.argtypes = [vp, sz, vp, vp, vp, sz, vp]; lib.act_batch_refund_sign.restype = i32
    lib.act_batch_verify_spend_and_refund_screened.argtypes = [vp, sz, vp, vp, sz, vp, vp, vp, vp]; lib.act_batch_verify_spend_and_refund_screened.restype = i32
    lib.act_nullifier_store_create.argtypes = [C.POINTER(vp), i32, sz]; lib.act_nullifier_store_create.restype = i32
    lib.act_nullifier_store_destroy.argtypes = [vp]; lib.act_nullifier_store_destroy.restype = None
    lib.act_nullifier_store_device.argtypes = [vp]; lib.act_nullifier_store_device.restype = i32
    lib.act_nullifier_store_size.argtypes = [vp]; lib.act_nullifier_store_size.restype = sz
    lib.act_nullifier_store_screen_dev.argtypes = [vp, sz, vp, vp, vp, i32, vp]; lib.act_nullifier_store_screen_dev.restype = i32
    lib.act_nullifier_store_screen.argtypes = [vp, sz, vp, vp, vp, i32]; lib.act_nullifier_store_screen.restype = i32
    lib.act_nullifier_store_export.argtypes = [vp, vp, sz, C.POINTER(sz)]; lib.act_nullifier_store_export.restype = i32
    lib.act_batch_verify_spend_and_refund_recorded.argtypes = [vp, vp, sz, vp, vp, vp, vp, vp]; lib.act_batch_verify_spend_and_refund_recorded.restype = i32
    lib.act_engine_set_key.argtypes = [vp, i32, vp, vp]; lib.act_engine_set_key.restype = i32
    lib.act_engine_clear_key.argtypes = [vp, i32]; lib.act_engine_clear_key.restype = i32
    lib.act_engine_select_key.argtypes = [vp, i32]; lib.act_engine_select_key.restype = i32
    lib.act_engine_selected_key.argtypes = [vp]; lib.act_engine_selected_key.restype = i32
    lib.act_engine_key_slots.argtypes = [vp]; lib.act_engine_key_slots.restype = C.c_uint32
    lib.act_batch_verify_spend_and_refund_keyed_dev.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp, vp]
    lib.act_batch_verify_spend_and_refund_keyed_dev.restype = i32
    lib.act_batch_verify_spend_and_refund_keyed.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp, vp]; lib.act_batch_verify_spend_and_refund_keyed.restype = i32
    lib.act_batch_spend_verify_keyed.argtypes = [vp, sz, vp, vp, vp, vp, vp]; lib.act_batch_spend_verify_keyed.restype = i32
    _lib = lib
    return lib


def _check(rc, what):
    if rc != 0:
        raise ActError(f"{what} failed ({rc}): {load_library().act_last_error().decode()}")


def _u8(a, nbytes=None, name="buffer"):
    if isinstance(a, (bytes, bytearray, memoryview)):
        a = np.frombuffer(bytes(a), dtype=np.uint8)
    a = np.ascontiguousarray(a, dtype=np.uint8).reshape(-1)
    if nbytes is not None and a.size != nbytes:
        raise ValueError(f"{name}: expected {nbytes} bytes, got {a.size}")
    return a


def device_count():
    return load_library().act_device_count()


def selftest(device=0):
    """Device self-test of the PTX field arithmetic against built-in known answers."""
    _check(load_library().act_selftest(device), "act_selftest")


KERNEL_KINDS = ["spend_range", "spend_head", "spend_chunk_hash", "spend_finish", "refund_sign", "issue",
                "issuance_check", "refund_check", "spend_encode"]


def measure_int_mul_peak(device=0):
    """Measured integer-multiply roofline: sustained 32x32+64->64 multiply-adds per second (IMAD.WIDE.U32)."""
    v = C.c_double(0)
    _check(load_library().act_measure_int_mul_peak(device, C.addressof(v)), "act_measure_int_mul_peak")
    return v.value


class Params:
    """System parameters H1, H2, H3 (reference `Params`, src/lib.rs:222-229), held as their 96 encoded bytes."""

    def __init__(self, h):
        self.h = bytes(h)
        if len(self.h) != 96:
            raise ValueError("Params: need 96 bytes (H1|H2|H3)")

    @staticmethod
    def new(organization, service, deployment_id, version, device=0):
        """`Params::new` (src/lib.rs:291-315), computed on the GPU."""
        out = np.zeros(96, np.uint8)
        _check(load_library().act_params_derive(device, organization.encode(), service.encode(), deployment_id.encode(),
                                                version.encode(), out.ctypes.data), "act_params_derive")
        return Params(out.tobytes())


class PrivateKey:
    """Issuer key (reference `PrivateKey`, src/lib.rs:160-167): secret scalar x and public W = G*x (encoded).

    This Python mirror exists for the tests and the bench: it keeps `x` in an immutable `bytes` object, which cannot be
    zeroised (the reference's PrivateKey is ZeroizeOnDrop).  A production host holds the key in memory it controls and passes a
    pointer to act_engine_create, which wipes its own staging copy; the device copy is zeroised by act_engine_destroy."""

    def __init__(self, x, w):
        self.x, self.w = bytes(x), bytes(w)
        if len(self.x) != 32 or len(self.w) != 32:
            raise ValueError("PrivateKey: x and w are 32 bytes each")

    @staticmethod
    def from_secret(x, device=0):
        w = np.zeros(32, np.uint8)
        xb = _u8(x, 32, "x")
        _check(load_library().act_public_key(device, xb.ctypes.data, w.ctypes.data), "act_public_key")
        return PrivateKey(xb.tobytes(), w.tobytes())

    def public(self):
        return self.w


class Engine:
    """One (Params, PrivateKey) pair resident on one GPU; batch forms of the reference's issuer-side calls."""

    def __init__(self, params, key, device=0, devices=None):
        """device: one GPU; devices=[...]: a multi-device engine (act_engine_create_multi) whose host-buffer calls shard the
        batch contiguously over one replica per listed GPU."""
        self.lib = load_library()
        self._h = C.c_void_p()
        hb, xb, wb = _u8(params.h, 96), _u8(key.x, 32), _u8(key.w, 32)
        if devices is not None:
            devs = (C.c_int * len(devices))(*devices)
            self.device = devices[0]
            _check(self.lib.act_engine_create_multi(C.byref(self._h), C.cast(devs, C.c_void_p), len(devices), hb.ctypes.data, xb.ctypes.data, wb.ctypes.data),
                   "act_engine_create_multi")
        else:
            self.device = device
            _check(self.lib.act_engine_create(C.byref(self._h), device, hb.ctypes.data, xb.ctypes.data, wb.ctypes.data), "act_engine_create")

    @property
    def replica_count(self):
        return int(self.lib.act_engine_replica_count(self._h))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.act_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def launch_count(self):
        return int(self.lib.act_engine_launch_count(self._h))

    def set_spend_chunk(self, proofs):
        """Proofs per chunk of the spend pipeline (default 65536)."""
        _check(self.lib.act_engine_set_spend_chunk(self._h, proofs), "act_engine_set_spend_chunk")

    def set_timing(self, enable=True):
        _check(self.lib.act_engine_set_timing(self._h, 1 if enable else 0), "act_engine_set_timing")

    def get_timing(self):
        """{kernel kind: (total device ms, launches)} since the last call (synchronises)."""
        ms = (C.c_double * 9)(); cnt = (C.c_uint64 * 9)()
        _check(self.lib.act_engine_get_timing(self._h, C.addressof(ms), C.addressof(cnt)), "act_engine_get_timing")
        return {k: (ms[i], int(cnt[i])) for i, k in enumerate(KERNEL_KINDS)}

    # ---- host buffers (numpy uint8) ----
    def batch_issue(self, requests, cs, rnd):
        """n x PrivateKey::issue.  requests n*128 (K|gamma|k_bar|r_bar), cs n*32, rnd n*128 (e_wide|alpha_wide).
        Returns (responses n*160, status n)."""
        req = _u8(requests); n = req.size // REQUEST_BYTES
        c, r = _u8(cs, n * 32, "cs"), _u8(rnd, n * RND_BYTES, "rnd")
        resp = np.zeros(n * RESPONSE_BYTES, np.uint8); st = np.zeros(n, np.uint8)
        _check(self.lib.act_batch_issue(self._h, n, req.ctypes.data, c.ctypes.data, r.ctypes.data, resp.ctypes.data, st.ctypes.data), "act_batch_issue")
        return resp, st

    def batch_verify_spend_and_refund(self, proofs, rnd, out=None):
        """n x (spend-proof verification + PrivateKey::refund).  proofs n*16832, rnd n*128.
        Returns (refunds n*128, nullifiers n*32, status n)."""
        pf = _u8(proofs); n = pf.size // PROOF_BYTES
        r = _u8(rnd, n * RND_BYTES, "rnd")
        if out is None:
            ref = np.zeros(n * REFUND_BYTES, np.uint8); nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8)
        else:
            ref, nul, st = out
        _check(self.lib.act_batch_verify_spend_and_refund(self._h, n, pf.ctypes.data, r.ctypes.data, ref.ctypes.data, nul.ctypes.data, st.ctypes.data),
               "act_batch_verify_spend_and_refund")
        return ref, nul, st

    def batch_issuance_check(self, big_k, responses):
        """n x verification half of PreIssuance::to_credit_token.  big_k n*32 (request K), responses n*160."""
        k = _u8(big_k); n = k.size // 32
        rs = _u8(responses, n * RESPONSE_BYTES, "responses")
        st = np.zeros(n, np.uint8)
        _check(self.lib.act_batch_issuance_check(self._h, n, k.ctypes.data, rs.ctypes.data, st.ctypes.data), "act_batch_issuance_check")
        return st

    def batch_refund_check(self, com, refunds):
        """n x verification half of PreRefund::to_credit_token.  com n*4096 (the proof's com[128]), refunds n*128."""
        rf = _u8(refunds); n = rf.size // REFUND_BYTES
        cm = _u8(com, n * COM_BYTES, "com")
        st = np.zeros(n, np.uint8)
        _check(self.lib.act_batch_refund_check(self._h, n, cm.ctypes.data, rf.ctypes.data, st.ctypes.data), "act_batch_refund_check")
        return st

    # ---- sequential-RNG contract: same outputs as a loop of issue()/refund() calls sharing one RNG ----
    def batch_issue_seq(self, requests, cs, rnd_stream):
        """Request i uses rnd_stream[128*a_i : 128*a_i+128], a_i = accepted requests before i (the reference draws
        randomness only after a request verifies).  Returns (responses, status, bytes consumed)."""
        req = _u8(requests); n = req.size // REQUEST_BYTES
        c = _u8(cs, n * 32, "cs"); r = _u8(rnd_stream)
        resp = np.zeros(n * RESPONSE_BYTES, np.uint8); st = np.zeros(n, np.uint8); used = C.c_size_t(0)
        _check(self.lib.act_batch_issue_seq(self._h, n, req.ctypes.data, c.ctypes.data, r.ctypes.data if r.size else None, r.size,
                                            resp.ctypes.data, st.ctypes.data, C.addressof(used)), "act_batch_issue_seq")
        return resp, st, int(used.value)

    def batch_verify_spend_and_refund_seq(self, proofs, rnd_stream):
        pf = _u8(proofs); n = pf.size // PROOF_BYTES
        r = _u8(rnd_stream)
        ref = np.zeros(n * REFUND_BYTES, np.uint8); nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8); used = C.c_size_t(0)
        _check(self.lib.act_batch_verify_spend_and_refund_seq(self._h, n, pf.ctypes.data, r.ctypes.data if r.size else None, r.size,
                                                              ref.ctypes.data, nul.ctypes.data, st.ctypes.data, C.addressof(used)),
               "act_batch_verify_spend_and_refund_seq")
        return ref, nul, st, int(used.value)

    # ---- two-pass forms (verify, then sign with randomness for the accepted requests only) ----
    def batch_issue_verify(self, requests):
        req = _u8(requests); n = req.size // REQUEST_BYTES
        st = np.zeros(n, np.uint8)
        _check(self.lib.act_batch_issue_verify(self._h, n, req.ctypes.data, st.ctypes.data), "act_batch_issue_verify")
        return st

    def batch_issue_sign(self, requests, cs, status, rnd):
        """rnd: 128 bytes per accepted request (status 0), in slice order."""
        req = _u8(requests); n = req.size // REQUEST_BYTES
        c, st, r = _u8(cs, n * 32, "cs"), _u8(status, n, "status"), _u8(rnd)
        resp = np.zeros(n * RESPONSE_BYTES, np.uint8)
        _check(self.lib.act_batch_issue_sign(self._h, n, req.ctypes.data, c.ctypes.data, st.ctypes.data, r.ctypes.data if r.size else None, r.size, resp.ctypes.data),
               "act_batch_issue_sign")
        return resp

    def batch_spend_verify(self, proofs):
        """-> (nullifiers n*32, status n, kprime n*128): the verification half of batch_verify_spend_and_refund."""
        pf = _u8(proofs); n = pf.size // PROOF_BYTES
        nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8); kp = np.zeros(n * 128, np.uint8)
        _check(self.lib.act_batch_spend_verify(self._h, n, pf.ctypes.data, nul.ctypes.data, st.ctypes.data, kp.ctypes.data), "act_batch_spend_verify")
        return nul, st, kp

    def batch_refund_sign(self, kprime, status, rnd):
        st = _u8(status); n = st.size
        kp, r = _u8(kprime, n * 128, "kprime"), _u8(rnd)
        ref = np.zeros(n * REFUND_BYTES, np.uint8)
        _check(self.lib.act_batch_refund_sign(self._h, n, kp.ctypes.data, st.ctypes.data, r.ctypes.data if r.size else None, r.size, ref.ctypes.data),
               "act_batch_refund_sign")
        return ref

    def batch_verify_spend_and_refund_screened(self, proofs, rnd, seen=None, out=None):
        """verify + refund + replay screen (status 3 = DoubleSpendError, no refund) in one call; on a multi-device engine the
        status + nullifier gather to replica 0 runs over NVLink.  Returns (refunds, nullifiers, status)."""
        pf = _u8(proofs); n = pf.size // PROOF_BYTES
        r = _u8(rnd, n * RND_BYTES, "rnd")
        sn = _u8(seen) if seen is not None and len(seen) else np.zeros(0, np.uint8)
        if out is None:
            ref = np.zeros(n * REFUND_BYTES, np.uint8); nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8)
        else:
            ref, nul, st = out
        _check(self.lib.act_batch_verify_spend_and_refund_screened(self._h, n, pf.ctypes.data, r.ctypes.data, sn.size // 32, sn.ctypes.data if sn.size else None,
                                                                   ref.ctypes.data, nul.ctypes.data, st.ctypes.data), "act_batch_verify_spend_and_refund_screened")
        return ref, nul, st

    def batch_verify_spend_and_refund_recorded(self, proofs, rnd, store, out=None):
        """batch_verify_spend_and_refund_screened with a NullifierStore in place of `seen`: replays of the batch or of anything in
        the store get status 3 and no refund, and the nullifiers of the accepted proofs are recorded in the store.  The store must
        be on the device of replica 0.  Returns (refunds, nullifiers, status)."""
        pf = _u8(proofs); n = pf.size // PROOF_BYTES
        r = _u8(rnd, n * RND_BYTES, "rnd")
        if out is None:
            ref = np.zeros(n * REFUND_BYTES, np.uint8); nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8)
        else:
            ref, nul, st = out
        _check(self.lib.act_batch_verify_spend_and_refund_recorded(self._h, store._h, n, pf.ctypes.data, r.ctypes.data, ref.ctypes.data, nul.ctypes.data,
                                                                   st.ctypes.data), "act_batch_verify_spend_and_refund_recorded")
        return ref, nul, st

    # ---- issuer key slots (key rotation) ----
    def set_key(self, slot, key):
        """Installs or replaces the PrivateKey of a slot (0 .. KEY_SLOTS-1); fails, leaving the slot as it was, if key.w != G*key.x."""
        xb, wb = _u8(key.x, 32, "x"), _u8(key.w, 32, "w")
        _check(self.lib.act_engine_set_key(self._h, slot, xb.ctypes.data, wb.ctypes.data), "act_engine_set_key")

    def clear_key(self, slot):
        """Wipes the slot's secret and frees its tables; the selected slot cannot be cleared."""
        _check(self.lib.act_engine_clear_key(self._h, slot), "act_engine_clear_key")

    def select_key(self, slot):
        """The key every single-key call (issue, refund signing, verification, client-side checks) uses from now on."""
        _check(self.lib.act_engine_select_key(self._h, slot), "act_engine_select_key")

    @property
    def selected_key(self):
        return int(self.lib.act_engine_selected_key(self._h))

    @property
    def key_slots(self):
        """The slots that hold a key, ascending."""
        m = int(self.lib.act_engine_key_slots(self._h))
        return [s for s in range(KEY_SLOTS) if m >> s & 1]

    def batch_verify_spend_and_refund_keyed(self, proofs, key_ids, rnd, stores=None, out=None):
        """Proof i is verified under the key of slot key_ids[i] and refunded under the selected key; an empty or out-of-range slot
        gives status 7.  stores: None (no screen), or a NullifierStore per slot that holds a key (a sequence indexed by slot, or a
        dict {slot: store}; slots may share one): each store screens and records the proofs of its slots, as the _recorded call
        does for one.  Returns (refunds, nullifiers, status)."""
        pf = _u8(proofs); n = pf.size // PROOF_BYTES
        ids, r = _u8(key_ids, n, "key_ids"), _u8(rnd, n * RND_BYTES, "rnd")
        if out is None:
            ref = np.zeros(n * REFUND_BYTES, np.uint8); nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8)
        else:
            ref, nul, st = out
        table = None
        if stores is not None:
            items = stores.items() if isinstance(stores, dict) else enumerate(stores)
            table = (C.c_void_p * KEY_SLOTS)()
            for slot, store in items:
                if store is not None:
                    table[slot] = store._h.value
        _check(self.lib.act_batch_verify_spend_and_refund_keyed(self._h, n, pf.ctypes.data, ids.ctypes.data, r.ctypes.data,
                                                                C.cast(table, C.c_void_p) if table is not None else None,
                                                                ref.ctypes.data, nul.ctypes.data, st.ctypes.data),
               "act_batch_verify_spend_and_refund_keyed")
        return ref, nul, st

    def batch_spend_verify_keyed(self, proofs, key_ids):
        """-> (nullifiers, status, kprime): the verification pass of the keyed call; sign with batch_refund_sign (selected key)."""
        pf = _u8(proofs); n = pf.size // PROOF_BYTES
        ids = _u8(key_ids, n, "key_ids")
        nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8); kp = np.zeros(n * 128, np.uint8)
        _check(self.lib.act_batch_spend_verify_keyed(self._h, n, pf.ctypes.data, ids.ctypes.data, nul.ctypes.data, st.ctypes.data, kp.ctypes.data),
               "act_batch_spend_verify_keyed")
        return nul, st, kp

    def batch_verify_spend_and_refund_keyed_dev(self, n, proofs, key_ids, rnd, refunds, nullifiers, status, stream=0):
        _check(self.lib.act_batch_verify_spend_and_refund_keyed_dev(self._h, n, proofs, key_ids, rnd, refunds, nullifiers, status, stream),
               "act_batch_verify_spend_and_refund_keyed_dev")

    def batch_verify_spend_and_refund_screened_ptr(self, n, proofs, rnd, n_seen, seen, refunds, nullifiers, status):
        _check(self.lib.act_batch_verify_spend_and_refund_screened(self._h, n, proofs, rnd, n_seen, seen, refunds, nullifiers, status),
               "act_batch_verify_spend_and_refund_screened")

    # ---- client-side batch generators (fixture grade, not constant time) ----
    def batch_request(self, pre, rnd):
        """n x PreIssuance::request (src/lib.rs:463-487).  pre n*64 (r|k), rnd n*128 (k'_wide|r'_wide) -> requests n*128."""
        p = _u8(pre); n = p.size // 64
        r = _u8(rnd, n * RND_BYTES, "rnd")
        req = np.zeros(n * REQUEST_BYTES, np.uint8)
        _check(self.lib.act_batch_request(self._h, n, p.ctypes.data, r.ctypes.data, req.ctypes.data), "act_batch_request")
        return req

    def batch_prove_spend(self, tokens, charges, rnd=None, seed=None, first_index=0):
        """n x CreditToken::prove_spend (src/lib.rs:972-1152).  tokens n*160 (A|e|k|r|c), charges n*32; rnd n*33536 explicit
        RNG bytes in the reference's order, or seed (32 bytes) for the BLAKE3-XOF derived stream.
        Returns (proofs n*16832, prerefunds n*96 (k*|r*|m), status n)."""
        tk = _u8(tokens); n = tk.size // TOKEN_BYTES
        ch = _u8(charges, n * 32, "charges")
        r = _u8(rnd, n * PROVE_RND_BYTES, "rnd") if rnd is not None else None
        sd = _u8(seed, 32, "seed") if seed is not None else None
        proofs = np.zeros(n * PROOF_BYTES, np.uint8); pr = np.zeros(n * PREREFUND_BYTES, np.uint8); st = np.zeros(n, np.uint8)
        _check(self.lib.act_batch_prove_spend(self._h, n, tk.ctypes.data, ch.ctypes.data, r.ctypes.data if r is not None else None,
                                              sd.ctypes.data if sd is not None else None, first_index, proofs.ctypes.data, pr.ctypes.data, st.ctypes.data),
               "act_batch_prove_spend")
        return proofs, pr, st

    def batch_request_dev(self, n, pre, rnd, req, stream=0):
        _check(self.lib.act_batch_request_dev(self._h, n, pre, rnd, req, stream), "act_batch_request_dev")

    def batch_prove_spend_dev(self, n, tokens, charges, rnd, seed, first_index, proofs, prerefunds, status, stream=0):
        sd = _u8(seed, 32, "seed") if seed is not None else None
        _check(self.lib.act_batch_prove_spend_dev(self._h, n, tokens, charges, rnd, sd.ctypes.data if sd is not None else None, first_index,
                                                  proofs, prerefunds, status, stream), "act_batch_prove_spend_dev")

    # ---- rows either side of the hot path ----
    def flag_replays(self, status, nullifiers, seen=None):
        """Batch replay screen (the caller's NullifierDb, src/tests.rs:28-50, in slice order): accepted proofs whose
        nullifier occurred earlier in the batch or in `seen` (k*32 bytes) get status 3 (DoubleSpendError)."""
        st = _u8(status); n = st.size
        nul = _u8(nullifiers, n * 32, "nullifiers")
        sn = _u8(seen) if seen is not None and len(seen) else np.zeros(0, np.uint8)
        out = np.zeros(n, np.uint8)
        _check(self.lib.act_flag_replays(self._h, n, st.ctypes.data, nul.ctypes.data, sn.size // 32, sn.ctypes.data if sn.size else None, out.ctypes.data),
               "act_flag_replays")
        return out

    def flag_replays_dev(self, n, status, nullifiers, n_seen, seen, status_out, stream=0):
        _check(self.lib.act_flag_replays_dev(self._h, n, status, nullifiers, n_seen, seen, status_out, stream), "act_flag_replays_dev")

    def unpack_cbor(self, kind, cbor):
        """Canonical-CBOR fast path: fixed-size items -> (records, status); status 0xFF = not the canonical skeleton."""
        c = _u8(cbor); n = c.size // CBOR_BYTES[kind]
        rec = np.zeros(n * RECORD_BYTES[kind], np.uint8); st = np.zeros(n, np.uint8)
        _check(self.lib.act_unpack_cbor(self._h, kind, n, c.ctypes.data, rec.ctypes.data, st.ctypes.data), "act_unpack_cbor")
        return rec, st

    def encode_cbor(self, kind, records):
        r = _u8(records); n = r.size // RECORD_BYTES[kind]
        out = np.zeros(n * CBOR_BYTES[kind], np.uint8)
        _check(self.lib.act_encode_cbor(self._h, kind, n, r.ctypes.data, out.ctypes.data), "act_encode_cbor")
        return out

    def unpack_cbor_dev(self, kind, n, cbor, records, status, stream=0):
        _check(self.lib.act_unpack_cbor_dev(self._h, kind, n, cbor, records, status, stream), "act_unpack_cbor_dev")

    def encode_cbor_dev(self, kind, n, records, cbor, stream=0):
        _check(self.lib.act_encode_cbor_dev(self._h, kind, n, records, cbor, stream), "act_encode_cbor_dev")

    # ---- raw pointers (pinned host memory or torch tensors); nothing is allocated here ----
    def batch_issue_ptr(self, n, req, cs, rnd, resp, status):
        _check(self.lib.act_batch_issue(self._h, n, req, cs, rnd, resp, status), "act_batch_issue")

    def batch_verify_spend_and_refund_ptr(self, n, proofs, rnd, refunds, nullifiers, status):
        _check(self.lib.act_batch_verify_spend_and_refund(self._h, n, proofs, rnd, refunds, nullifiers, status), "act_batch_verify_spend_and_refund")

    def batch_issue_dev(self, n, req, cs, rnd, resp, status, stream=0):
        _check(self.lib.act_batch_issue_dev(self._h, n, req, cs, rnd, resp, status, stream), "act_batch_issue_dev")

    def batch_verify_spend_and_refund_dev(self, n, proofs, rnd, refunds, nullifiers, status, stream=0):
        _check(self.lib.act_batch_verify_spend_and_refund_dev(self._h, n, proofs, rnd, refunds, nullifiers, status, stream),
               "act_batch_verify_spend_and_refund_dev")

    def batch_issuance_check_dev(self, n, big_k, resp, status, stream=0):
        _check(self.lib.act_batch_issuance_check_dev(self._h, n, big_k, resp, status, stream), "act_batch_issuance_check_dev")

    def batch_refund_check_dev(self, n, com, refund, status, stream=0):
        _check(self.lib.act_batch_refund_check_dev(self._h, n, com, refund, status, stream), "act_batch_refund_check_dev")


class NullifierStore:
    """The set of nullifiers already spent (the caller's NullifierDb of the reference, src/lib.rs:741-745), resident on one GPU
    and kept between calls.  Independent of any engine; grows on its own.  Members are 32-byte nullifiers reduced mod l."""

    def __init__(self, device=0, capacity=1 << 20):
        self.lib = load_library()
        self._h = C.c_void_p()
        self.device = device
        _check(self.lib.act_nullifier_store_create(C.byref(self._h), device, capacity), "act_nullifier_store_create")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.act_nullifier_store_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def size(self):
        """Exact number of members (synchronises)."""
        return int(self.lib.act_nullifier_store_size(self._h))

    def screen(self, status, nullifiers, record=True):
        """Status-0 entries whose nullifier is in the store or earlier in the batch get 3 (DoubleSpendError); other statuses are
        copied.  record: insert the nullifiers whose output status is 0.  Returns the new status array."""
        st = _u8(status); n = st.size
        nul = _u8(nullifiers, n * 32, "nullifiers")
        out = np.zeros(n, np.uint8)
        _check(self.lib.act_nullifier_store_screen(self._h, n, st.ctypes.data, nul.ctypes.data, out.ctypes.data, 1 if record else 0),
               "act_nullifier_store_screen")
        return out

    def screen_dev(self, n, status, nullifiers, status_out, record=True, stream=0):
        """Device pointers on the store's device (nullifiers 16-byte aligned); stream 0 = the store's own stream."""
        _check(self.lib.act_nullifier_store_screen_dev(self._h, n, status, nullifiers, status_out, 1 if record else 0, stream),
               "act_nullifier_store_screen_dev")

    def export(self):
        """Every member as uint8[size*32], order unspecified."""
        cap = self.size
        out = np.zeros(max(cap, 1) * 32, np.uint8)
        cnt = C.c_size_t(0)
        _check(self.lib.act_nullifier_store_export(self._h, out.ctypes.data, cap, C.byref(cnt)), "act_nullifier_store_export")
        return out[:cnt.value * 32]


# ---- CBOR wire formats (host; src/cbor.rs) ----
def _pack(fn_name, items, rec_bytes):
    lib = load_library()
    n = len(items)
    bufs = [np.frombuffer(bytes(it), dtype=np.uint8) if len(it) else np.zeros(1, np.uint8) for it in items]
    ptrs = (C.c_void_p * max(n, 1))(*[b.ctypes.data for b in bufs])
    lens = (C.c_size_t * max(n, 1))(*[len(it) for it in items])
    rec = np.zeros(n * rec_bytes, np.uint8); st = np.zeros(n, np.uint8)
    rc = getattr(lib, fn_name)(n, C.cast(ptrs, C.c_void_p), C.cast(lens, C.c_void_p), rec.ctypes.data, st.ctypes.data)
    if rc != 0:
        raise ActError(f"{fn_name} failed ({rc})")
    return rec, st


def pack_issuance_requests_cbor(items):
    """`IssuanceRequest::from_cbor` (src/cbor.rs:118-147) for each item -> (records n*128, status n)."""
    return _pack("act_pack_issuance_requests_cbor", items, REQUEST_BYTES)


def pack_spend_proofs_cbor(items):
    """`SpendProof::from_cbor` (src/cbor.rs:276-408) for each item -> (records n*16832, status n)."""
    return _pack("act_pack_spend_proofs_cbor", items, PROOF_BYTES)


def pack_issuance_responses_cbor(items):
    return _pack("act_pack_issuance_responses_cbor", items, RESPONSE_BYTES)


def pack_refunds_cbor(items):
    return _pack("act_pack_refunds_cbor", items, REFUND_BYTES)


def _encode(fn_name, rec, rec_bytes, out_bytes):
    lib = load_library()
    r = _u8(rec, rec_bytes)
    out = np.zeros(out_bytes, np.uint8)
    n = getattr(lib, fn_name)(r.ctypes.data, out.ctypes.data)
    return out[:n].tobytes()


def encode_issuance_request_cbor(rec):
    return _encode("act_encode_issuance_request_cbor", rec, REQUEST_BYTES, 141)


def encode_issuance_response_cbor(rec):
    """`IssuanceResponse::to_cbor` (src/cbor.rs:162-174)."""
    return _encode("act_encode_issuance_response_cbor", rec, RESPONSE_BYTES, 176)


def encode_spend_proof_cbor(rec):
    return _encode("act_encode_spend_proof_cbor", rec, PROOF_BYTES, 18036)


def encode_refund_cbor(rec):
    """`Refund::to_cbor` (src/cbor.rs:421-432)."""
    return _encode("act_encode_refund_cbor", rec, REFUND_BYTES, 141)
