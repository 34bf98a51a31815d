"""ctypes binding of tests/hostsim_keys/libact_hostsim_keys.so: the host build of the device headers with the keyed spend pipeline.

TEST INFRASTRUCTURE ONLY -- checks the key selection of the keyed head stage against the oracle without a GPU.  Contexts are made
by this library (hs_ctx_create of the included host build), so they never cross into another library.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim_keys")
_SO = os.path.join(_DIR, "libact_hostsim_keys.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            subprocess.check_call(["make", "-C", _DIR, "-s"])
        L = C.CDLL(_SO)
        vp, sz = C.c_void_p, C.c_size_t
        L.hs_ctx_create.argtypes = [vp, vp, vp]; L.hs_ctx_create.restype = vp
        L.hs_ctx_destroy.argtypes = [vp]
        L.hs_refund_keyed.argtypes = [vp, vp, sz, vp, vp, vp, vp, vp, vp]
        L.hs_refund_check.argtypes = [vp, sz, vp, vp, vp]
        _lib = L
    return _lib


def _buf(b):
    return np.ascontiguousarray(np.frombuffer(bytes(b), np.uint8) if not isinstance(b, np.ndarray) else b, np.uint8)


class Ctx:
    def __init__(self, h, x, w):
        self._keep = [_buf(h), _buf(x), _buf(w)]
        self.p = lib().hs_ctx_create(*[a.ctypes.data for a in self._keep])
        if not self.p:
            raise ValueError("invalid point")

    def __del__(self):
        try:
            if self.p:
                lib().hs_ctx_destroy(self.p); self.p = None
        except Exception:
            pass

    def refund_check(self, com, refund):
        c, r = _buf(com), _buf(refund)
        n = r.size // 128
        st = np.zeros(n, np.uint8)
        lib().hs_refund_check(self.p, n, c.ctypes.data, r.ctypes.data, st.ctypes.data)
        return st


def refund_keyed(sel, slots, proofs, key_ids, rnd):
    """slots: {slot: Ctx}; proof i verified under slots.get(key_ids[i]) and refunded under `sel`.  -> (refunds, nullifiers, status)"""
    n = len(key_ids)
    table = (C.c_void_p * 16)(*[slots[k].p if k in slots else None for k in range(16)])
    pf, ids, r = _buf(proofs), _buf(key_ids), _buf(rnd)
    ref = np.zeros(n * 128, np.uint8); nul = np.zeros(n * 32, np.uint8); st = np.zeros(n, np.uint8)
    lib().hs_refund_keyed(sel.p, C.cast(table, C.c_void_p), n, pf.ctypes.data, ids.ctypes.data, r.ctypes.data, ref.ctypes.data, nul.ctypes.data,
                          st.ctypes.data)
    return ref, nul, st
