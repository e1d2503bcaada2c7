"""ctypes view of tests/hostsim/ecdsa_batch_sim.cpp: the recoverable ECDSA batch verification on the CPU (test
infrastructure only)."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import _HERE, _a, _deps, _p

_SO = os.path.join(_HERE, "_build", "ecdsa_batch_sim.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "ecdsa_batch_sim.cpp")
        stale = not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in _deps() + [src])
        if stale:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", _SO, src])
        _lib = C.CDLL(_SO)
    return _lib


def _rows(pk, dg, sig):
    pk, dg, sig = _a(pk, 65), _a(dg, 32), _a(sig, 65)
    if not len(pk) == len(dg) == len(sig):
        raise ValueError("length mismatch")
    return pk, dg, sig, len(pk)


def ecdsa_batch_randomizers(pk, dg, sig, chunk):
    """Pass 1 of the batch verification with chunks of `chunk` rows: (seed, a) -- 32 bytes and (n, 32) big-endian rows."""
    pk, dg, sig, n = _rows(pk, dg, sig)
    seed = np.zeros(32, np.uint8); a = np.zeros((n, 32), np.uint8)
    lib().sim_ecdsa_batch_randomizers(_p(pk), _p(dg), _p(sig), C.c_size_t(n), C.c_size_t(chunk), _p(seed), _p(a))
    return seed.tobytes(), a


def ecdsa_batch_rows(pk, dg, sig, flags=0, chunk=1 << 19, k=0):
    """What s256_debug_ecdsa_batch_rows returns, and the verdict: (seed, k (n, 2, 32), pts (n, 2, 64), sum, rejected, ok)."""
    pk, dg, sig, n = _rows(pk, dg, sig)
    seed, ks, pts, ssum = np.zeros(32, np.uint8), np.zeros((n, 2, 32), np.uint8), np.zeros((n, 2, 64), np.uint8), np.zeros(32, np.uint8)
    rej, ok = C.c_uint8(0), C.c_uint8(0)
    lib().sim_ecdsa_batch(_p(pk), _p(dg), _p(sig), C.c_uint32(flags), C.c_size_t(n), C.c_size_t(chunk), int(k), _p(seed),
                          _p(ks), _p(pts), _p(ssum), C.byref(rej), C.byref(ok))
    return seed.tobytes(), ks, pts, ssum.tobytes(), bool(rej.value), bool(ok.value)


def ecdsa_batch_verify(pk, dg, sig, flags=0, chunk=1 << 19, k=0):
    """The batch verdict (bool) as s256_ecdsa_recoverable_batch_verify computes it, with chunks of `chunk` rows and
    inversion groups of k rows (0: the device's choice for the chunk size)."""
    pk, dg, sig, n = _rows(pk, dg, sig)
    ok = C.c_uint8(0)
    lib().sim_ecdsa_batch(_p(pk), _p(dg), _p(sig), C.c_uint32(flags), C.c_size_t(n), C.c_size_t(chunk), int(k), None, None,
                          None, None, None, C.byref(ok))
    return bool(ok.value)
