"""ctypes binding of tests/oracle_keys/libact_oracle_keys.so: the CPU oracle's refund for an issuer with several keys.

TEST INFRASTRUCTURE ONLY.  act_o_refund_keyed(verify, sign, ...) verifies a spend proof under the key of the oracle context
`verify` (None: a key id that names no key) and signs the refund under the key of `sign`; contexts come from oracle_lib.Ctx.
"""
import ctypes as C
import os
import subprocess

import numpy as np

import oracle_lib as O

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_keys")
_SO = os.path.join(_DIR, "libact_oracle_keys.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            subprocess.check_call(["make", "-C", _DIR, "-s"])
        L = C.CDLL(_SO)
        vp = C.c_void_p
        L.act_o_refund_keyed.argtypes = [vp, vp, vp, vp, vp, vp]; L.act_o_refund_keyed.restype = C.c_int
        _lib = L
    return _lib


def refund_keyed(verify, sign, proof, rnd128):
    """-> (status, refund 128 B, nullifier 32 B)"""
    pf = np.frombuffer(bytes(proof), np.uint8); r = np.frombuffer(bytes(rnd128), np.uint8)
    ref = np.zeros(128, np.uint8); nul = np.zeros(32, np.uint8)
    st = lib().act_o_refund_keyed(verify.p if verify is not None else None, sign.p, pf.ctypes.data, r.ctypes.data, ref.ctypes.data, nul.ctypes.data)
    return st, ref.tobytes(), nul.tobytes()


def batch_refund_keyed(slots, selected, proofs, key_ids, rnd):
    """slots: {slot: oracle Ctx}; proof i verified under slots.get(key_ids[i]), signed under `selected` (a Ctx).
    Returns (refunds n*128, nullifiers n*32, status n) like Ctx.batch_refund."""
    n = len(key_ids)
    pf = np.asarray(proofs, np.uint8).reshape(n, O.PROOF_BYTES); r = np.asarray(rnd, np.uint8).reshape(n, 128)
    ref = np.zeros((n, 128), np.uint8); nul = np.zeros((n, 32), np.uint8); st = np.zeros(n, np.uint8)
    for i in range(n):
        s, a, b = refund_keyed(slots.get(int(key_ids[i])), selected, pf[i].tobytes(), r[i].tobytes())
        st[i] = s; ref[i] = np.frombuffer(a, np.uint8); nul[i] = np.frombuffer(b, np.uint8)
    return ref.reshape(-1), nul.reshape(-1), st
