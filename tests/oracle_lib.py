"""ctypes binding of the CPU oracle (oracle/libact_oracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Nothing under anonymous-credit-tokens_b200/ imports it.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
_SO = os.path.join(ORACLE_DIR, "libact_oracle.so")

PROOF_BYTES = 526 * 32
RND_PROVE = 524 * 64

ST_OK = 0
ST_INVALID_ISSUANCE_REQUEST_PROOF = 1
ST_INVALID_ISSUANCE_RESPONSE_PROOF = 2
ST_DOUBLE_SPEND = 3
ST_INVALID_REFUND_PROOF = 4
ST_IDENTITY_POINT = 6
ST_INVALID_CLIENT_SPEND_PROOF = 7
ST_DECODE_INVALID_POINT = 0x81


def build(force=False):
    src = os.path.join(ORACLE_DIR, "act_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "-s"])
    return _SO


_lib = None


def use_native_build():
    """bench.py's CPU-baseline legs: rebuild the oracle with -march=native on the machine it is timed on (the built .so is
    compiled for a portable x86-64-v2 target, so that one build runs on any host).  The native build goes to a temporary
    directory, removed at exit: the benchmark writes nothing into the tree, which may be read-only.  Falls back silently to
    the portable build."""
    global _SO, _lib
    tmp = tempfile.mkdtemp(prefix="act-oracle-native-")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    native = os.path.join(tmp, "libact_oracle_native.so")
    try:
        subprocess.check_call(["make", "-C", ORACLE_DIR, "-s", "-B", "native", f"NATIVE={native}"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        if os.path.exists(native):
            _SO, _lib = native, None
            return True
    except Exception:
        pass
    return False


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        vp, cp, sz, i32, dbl = C.c_void_p, C.c_char_p, C.c_size_t, C.c_int, C.c_double
        L.act_o_params_derive.argtypes = [cp, cp, cp, cp, vp]; L.act_o_params_derive.restype = i32
        L.act_o_ctx_create.argtypes = [vp, vp, vp]; L.act_o_ctx_create.restype = vp
        L.act_o_ctx_destroy.argtypes = [vp]; L.act_o_ctx_destroy.restype = None
        L.act_o_keygen.argtypes = [vp, vp, vp]; L.act_o_keygen.restype = None
        L.act_o_request.argtypes = [vp, vp, vp, vp]; L.act_o_request.restype = None
        L.act_o_issue.argtypes = [vp, vp, vp, vp, vp]; L.act_o_issue.restype = i32
        L.act_o_issuance_check.argtypes = [vp, vp, vp]; L.act_o_issuance_check.restype = i32
        L.act_o_prove_spend.argtypes = [vp, vp, vp, vp, vp, vp]; L.act_o_prove_spend.restype = i32
        L.act_o_refund.argtypes = [vp, vp, vp, vp, vp]; L.act_o_refund.restype = i32
        L.act_o_refund_check.argtypes = [vp, vp, vp]; L.act_o_refund_check.restype = i32
        L.act_o_ristretto_decode_encode.argtypes = [vp, vp]; L.act_o_ristretto_decode_encode.restype = i32
        L.act_o_ristretto_from_uniform.argtypes = [vp, vp]; L.act_o_ristretto_from_uniform.restype = None
        L.act_o_scalarmult.argtypes = [vp, vp, vp]; L.act_o_scalarmult.restype = i32
        L.act_o_scalarmult_base.argtypes = [vp, vp]; L.act_o_scalarmult_base.restype = None
        L.act_o_point_add.argtypes = [vp, vp, vp]; L.act_o_point_add.restype = i32
        L.act_o_blake3.argtypes = [vp, sz, vp, sz]; L.act_o_blake3.restype = None
        L.act_o_sc_reduce32.argtypes = [vp, vp]; L.act_o_sc_reduce32.restype = None
        L.act_o_sc_reduce64.argtypes = [vp, vp]; L.act_o_sc_reduce64.restype = None
        L.act_o_sc_muladd.argtypes = [vp, vp, vp, vp]; L.act_o_sc_muladd.restype = None
        L.act_o_sc_invert.argtypes = [vp, vp]; L.act_o_sc_invert.restype = None
        L.act_o_transcript_challenge.argtypes = [vp, cp, vp, sz, vp]; L.act_o_transcript_challenge.restype = None
        L.act_o_fe_mul.argtypes = [vp, vp, vp]; L.act_o_fe_mul.restype = None
        L.act_o_fe_invert.argtypes = [vp, vp]; L.act_o_fe_invert.restype = None
        L.act_o_batch_issue.argtypes = [vp, sz, i32, vp, vp, vp, vp, vp]; L.act_o_batch_issue.restype = dbl
        L.act_o_batch_refund.argtypes = [vp, sz, i32, vp, vp, vp, vp, vp]; L.act_o_batch_refund.restype = dbl
        L.act_o_batch_issuance_check.argtypes = [vp, sz, i32, vp, vp, vp]; L.act_o_batch_issuance_check.restype = dbl
        L.act_o_batch_refund_check.argtypes = [vp, sz, i32, vp, vp, vp]; L.act_o_batch_refund_check.restype = dbl
        L.act_o_time_refund_typed.argtypes = [vp, sz, i32, i32, vp, vp, vp]; L.act_o_time_refund_typed.restype = dbl
        L.act_o_time_issue_typed.argtypes = [vp, sz, i32, i32, vp, vp, vp, vp]; L.act_o_time_issue_typed.restype = dbl
        L.act_o_generate.argtypes = [vp, sz, i32, vp, vp, vp, vp, vp, vp, vp, vp]; L.act_o_generate.restype = None
        _lib = L
    return _lib


def _buf(b):
    """bytes/bytearray/np.ndarray -> (keepalive, pointer)."""
    if isinstance(b, np.ndarray):
        assert b.flags["C_CONTIGUOUS"]
        return b, b.ctypes.data
    if isinstance(b, (bytes, bytearray)):
        a = np.frombuffer(bytes(b), dtype=np.uint8)
        return a, a.ctypes.data
    raise TypeError(type(b))


def _out(n):
    a = np.zeros(n, dtype=np.uint8)
    return a, a.ctypes.data


def params_derive(org, svc, dep, ver):
    a, p = _out(96)
    assert lib().act_o_params_derive(org.encode(), svc.encode(), dep.encode(), ver.encode(), p) == 0
    return a.tobytes()


def keygen(rnd64):
    k, kp = _buf(rnd64)
    x, xp = _out(32)
    w, wp = _out(32)
    lib().act_o_keygen(kp, xp, wp)
    return x.tobytes(), w.tobytes()


class Ctx:
    """Issuer context: params (encoded H1||H2||H3) + key (x, W)."""

    def __init__(self, h, x, w):
        self.h, self.x, self.w = bytes(h), bytes(x), bytes(w)
        a, ap = _buf(self.h); b, bp = _buf(self.x); c, cp = _buf(self.w)
        self.p = lib().act_o_ctx_create(ap, bp, cp)
        if not self.p:
            raise ValueError("invalid point in params/key")

    def __del__(self):
        try:
            if self.p:
                lib().act_o_ctx_destroy(self.p)
                self.p = None
        except Exception:
            pass

    def request(self, pre64, rnd128):
        a, ap = _buf(pre64); b, bp = _buf(rnd128); o, op = _out(128)
        lib().act_o_request(self.p, ap, bp, op)
        return o.tobytes()

    def issue(self, req, c32, rnd128):
        a, ap = _buf(req); b, bp = _buf(c32); r, rp = _buf(rnd128); o, op = _out(160)
        st = lib().act_o_issue(self.p, ap, bp, rp, op)
        return st, o.tobytes()

    def issuance_check(self, K, resp):
        a, ap = _buf(K); b, bp = _buf(resp)
        return lib().act_o_issuance_check(self.p, ap, bp)

    def prove_spend(self, token160, s32, rnd):
        assert len(rnd) == RND_PROVE
        a, ap = _buf(token160); b, bp = _buf(s32); r, rp = _buf(rnd)
        o, op = _out(PROOF_BYTES); q, qp = _out(96)
        st = lib().act_o_prove_spend(self.p, ap, bp, rp, op, qp)
        assert st == 0
        return o.tobytes(), q.tobytes()

    def refund(self, proof, rnd128):
        a, ap = _buf(proof); r, rp = _buf(rnd128); o, op = _out(128); n, np_ = _out(32)
        st = lib().act_o_refund(self.p, ap, rp, op, np_)
        return st, o.tobytes(), n.tobytes()

    def refund_check(self, com4096, refund128):
        a, ap = _buf(com4096); b, bp = _buf(refund128)
        return lib().act_o_refund_check(self.p, ap, bp)

    def transcript_challenge(self, label, items):
        a, ap = _buf(items) if len(items) else (None, None)
        o, op = _out(32)
        lib().act_o_transcript_challenge(self.p, label.encode(), ap, len(items) // 32, op)
        return o.tobytes()

    # ---- batches (numpy uint8 arrays) ----
    def batch_issue(self, req, cs, rnd, threads=1):
        n = len(req) // 128
        resp = np.zeros(n * 160, np.uint8); st = np.zeros(n, np.uint8)
        t = lib().act_o_batch_issue(self.p, n, threads, req.ctypes.data, cs.ctypes.data, rnd.ctypes.data, resp.ctypes.data, st.ctypes.data)
        return resp, st, t

    def batch_refund(self, proofs, rnd, threads=1):
        n = len(proofs) // PROOF_BYTES
        ref = np.zeros(n * 128, np.uint8); nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8)
        t = lib().act_o_batch_refund(self.p, n, threads, proofs.ctypes.data, rnd.ctypes.data, ref.ctypes.data, nul.ctypes.data, st.ctypes.data)
        return ref, nul, st, t

    def batch_issuance_check(self, K, resp, threads=1):
        n = len(K) // 32
        st = np.zeros(n, np.uint8)
        t = lib().act_o_batch_issuance_check(self.p, n, threads, K.ctypes.data, resp.ctypes.data, st.ctypes.data)
        return st, t

    def batch_refund_check(self, com, refund, threads=1):
        n = len(refund) // 128
        st = np.zeros(n, np.uint8)
        t = lib().act_o_batch_refund_check(self.p, n, threads, com.ctypes.data, refund.ctypes.data, st.ctypes.data)
        return st, t

    def time_refund_typed(self, proofs, rnd, threads=1, reps=1):
        n = len(proofs) // PROOF_BYTES
        ok = C.c_size_t(0)
        t = lib().act_o_time_refund_typed(self.p, n, threads, reps, proofs.ctypes.data, rnd.ctypes.data, C.addressof(ok))
        return t, ok.value

    def time_issue_typed(self, req, cs, rnd, threads=1, reps=1):
        n = len(req) // 128
        ok = C.c_size_t(0)
        t = lib().act_o_time_issue_typed(self.p, n, threads, reps, req.ctypes.data, cs.ctypes.data, rnd.ctypes.data, C.addressof(ok))
        return t, ok.value

    def generate(self, seeds, credits, charges, threads=1, want_proofs=True):
        """n independent request->issue->(prove_spend) trips.  seeds: (n*64) uint8, credits/charges uint64."""
        n = len(seeds) // 64
        credits = np.ascontiguousarray(credits, dtype=np.uint64); charges = np.ascontiguousarray(charges, dtype=np.uint64)
        req = np.zeros(n * 128, np.uint8); cs = np.zeros(n * 32, np.uint8); resp = np.zeros(n * 160, np.uint8)
        proofs = np.zeros(n * PROOF_BYTES, np.uint8) if want_proofs else None
        pre = np.zeros(n * 96, np.uint8) if want_proofs else None
        lib().act_o_generate(self.p, n, threads, seeds.ctypes.data, credits.ctypes.data, charges.ctypes.data,
                             req.ctypes.data, cs.ctypes.data, resp.ctypes.data,
                             proofs.ctypes.data if want_proofs else None, pre.ctypes.data if want_proofs else None)
        return dict(req=req, cs=cs, resp=resp, proofs=proofs, prerefund=pre)


# ---- primitive helpers ----
def blake3(data, outlen=32):
    a, ap = _buf(data) if len(data) else (None, None)
    o, op = _out(outlen)
    lib().act_o_blake3(ap, len(data), op, outlen)
    return o.tobytes()


def decode_encode(b32):
    a, ap = _buf(b32); o, op = _out(32)
    ok = lib().act_o_ristretto_decode_encode(ap, op)
    return (o.tobytes() if ok else None)


def from_uniform(b64):
    a, ap = _buf(b64); o, op = _out(32)
    lib().act_o_ristretto_from_uniform(ap, op)
    return o.tobytes()


def scalarmult(s32, p32):
    a, ap = _buf(s32); b, bp = _buf(p32); o, op = _out(32)
    ok = lib().act_o_scalarmult(ap, bp, op)
    return o.tobytes() if ok else None


def scalarmult_base(s32):
    a, ap = _buf(s32); o, op = _out(32)
    lib().act_o_scalarmult_base(ap, op)
    return o.tobytes()


def point_add(a32, b32):
    a, ap = _buf(a32); b, bp = _buf(b32); o, op = _out(32)
    ok = lib().act_o_point_add(ap, bp, op)
    return o.tobytes() if ok else None


def sc_reduce32(b):
    a, ap = _buf(b); o, op = _out(32); lib().act_o_sc_reduce32(ap, op); return o.tobytes()


def sc_reduce64(b):
    a, ap = _buf(b); o, op = _out(32); lib().act_o_sc_reduce64(ap, op); return o.tobytes()


def sc_muladd(a_, b_, c_):
    a, ap = _buf(a_); b, bp = _buf(b_); c, cp = _buf(c_); o, op = _out(32)
    lib().act_o_sc_muladd(ap, bp, cp, op); return o.tobytes()


def sc_invert(a_):
    a, ap = _buf(a_); o, op = _out(32); lib().act_o_sc_invert(ap, op); return o.tobytes()


def fe_mul(a_, b_):
    a, ap = _buf(a_); b, bp = _buf(b_); o, op = _out(32); lib().act_o_fe_mul(ap, bp, op); return o.tobytes()


def fe_invert(a_):
    a, ap = _buf(a_); o, op = _out(32); lib().act_o_fe_invert(ap, op); return o.tobytes()
