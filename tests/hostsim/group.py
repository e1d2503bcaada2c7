"""ctypes view of tests/hostsim/group_sim.cpp: the entry points built on the inversion-group kernels, on the CPU, with
the group size K (1, 4 or 32) chosen per call (test infrastructure only).  Each backend exposes the Engine's method
names, so the same checks run against it and against the product."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import _HERE, _a, _deps, _p

_SO = os.path.join(_HERE, "_build", "group_sim.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "group_sim.cpp")
        stale = not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in _deps() + [src])
        if stale:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", _SO, src])
        _lib = C.CDLL(_SO)
    return _lib


class Backend:
    """The simulation at inversion-group size k, under the Engine's method names."""

    def __init__(self, k):
        if k not in (1, 4, 32):
            raise ValueError(f"inversion-group size {k} is not one the device uses (1, 4, 32)")
        self.k = int(k)

    def _run(self, name, *args):
        if getattr(lib(), name)(self.k, *args) != 0:
            raise ValueError(f"{name}: K = {self.k} refused")

    def ecdsa_verify(self, pk, dg, sig, flags=0):
        pk, dg, sig = _a(pk, 65), _a(dg, 32), _a(sig, 64)
        n = len(pk); ok = np.zeros(n, np.uint8)
        self._run("gsim_ecdsa_verify", _p(pk), _p(dg), _p(sig), C.c_uint32(flags), C.c_size_t(n), _p(ok))
        return ok

    def ecdsa_recover(self, dg, sig65):
        dg, sig65 = _a(dg, 32), _a(sig65, 65)
        n = len(dg); out = np.zeros((n, 65), np.uint8); st = np.zeros(n, np.uint8)
        self._run("gsim_ecdsa_recover", _p(dg), _p(sig65), C.c_size_t(n), _p(out), _p(st))
        return out, st

    def double_scalar_mult_basepoint_vartime(self, u1, u2, pts):
        u1, u2, pts = _a(u1, 32), _a(u2, 32), _a(pts, 65)
        n = len(u1); out = np.zeros((n, 65), np.uint8); st = np.zeros(n, np.uint8)
        self._run("gsim_double_scalar_mult", _p(u1), _p(u2), _p(pts), C.c_size_t(n), _p(out), _p(st))
        return out, st

    def scalar_base_mult(self, k):
        k = _a(k, 32); n = len(k); out = np.zeros((n, 65), np.uint8); st = np.zeros(n, np.uint8)
        self._run("gsim_scalar_base_mult", _p(k), C.c_size_t(n), _p(out), _p(st))
        return out, st

    def scalar_mult(self, k, pts):
        k, pts = _a(k, 32), _a(pts, 65); n = len(k); out = np.zeros((n, 65), np.uint8); st = np.zeros(n, np.uint8)
        self._run("gsim_scalar_mult", _p(k), _p(pts), C.c_size_t(n), 0, _p(out), _p(st))
        return out, st

    def ecdh(self, k, pts):
        k, pts = _a(k, 32), _a(pts, 65); n = len(k); out = np.zeros((n, 32), np.uint8); st = np.zeros(n, np.uint8)
        self._run("gsim_scalar_mult", _p(k), _p(pts), C.c_size_t(n), 1, _p(out), _p(st))
        return out, st

    def ecdsa_sign_rfc6979(self, priv, digest):
        priv, digest = _a(priv, 32), _a(digest, 32); n = len(priv)
        sig = np.zeros((n, 64), np.uint8); rec = np.zeros(n, np.uint8); st = np.zeros(n, np.uint8)
        self._run("gsim_ecdsa_sign_rfc6979", _p(priv), _p(digest), C.c_size_t(n), _p(sig), _p(rec), _p(st))
        return sig, rec, st

    def schnorr_sign(self, priv, msg, aux):
        priv, aux = _a(priv, 32), _a(aux, 32); n = len(priv)
        msg = np.ascontiguousarray(msg, dtype=np.uint8).reshape(n, -1)
        sig = np.zeros((n, 64), np.uint8); st = np.zeros(n, np.uint8)
        self._run("gsim_schnorr_sign", _p(priv), _p(msg), C.c_size_t(msg.shape[1]), _p(aux), C.c_size_t(n), _p(sig), _p(st))
        return sig, st
