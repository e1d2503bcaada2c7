"""ctypes view of tests/hostsim/batch_sim.cpp: the BIP-340 batch verification on the CPU (test infrastructure only)."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import _HERE, _a, _deps, _p

_SO = os.path.join(_HERE, "_build", "batch_sim.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "batch_sim.cpp")
        stale = not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in _deps() + [src])
        if stale:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", _SO, src])
        _lib = C.CDLL(_SO)
    return _lib


def _rows(pkx, msg, sig):
    pkx, sig = _a(pkx, 32), _a(sig, 64)
    n = len(pkx)
    m = np.ascontiguousarray(msg, dtype=np.uint8)
    return pkx, m.reshape(n, m.size // n if n else 0), sig, n


def schnorr_batch_randomizers(pkx, msg, sig, chunk):
    """Pass 1 of the batch verification with chunks of `chunk` rows: (seed, a) -- 32 bytes and (n, 32) big-endian rows."""
    pkx, msg, sig, n = _rows(pkx, msg, sig)
    seed = np.zeros(32, np.uint8); a = np.zeros((n, 32), np.uint8)
    lib().sim_schnorr_batch_randomizers(_p(pkx), _p(msg), C.c_size_t(msg.shape[1]), _p(sig), C.c_size_t(n), C.c_size_t(chunk),
                                        _p(seed), _p(a))
    return seed.tobytes(), a


def schnorr_batch_verify(pkx, msg, sig, chunk=1 << 19):
    """The batch verdict (bool) as s256_schnorr_batch_verify computes it, with chunks of `chunk` rows."""
    pkx, msg, sig, n = _rows(pkx, msg, sig)
    ok = C.c_uint8(0)
    lib().sim_schnorr_batch_verify(_p(pkx), _p(msg), C.c_size_t(msg.shape[1]), _p(sig), C.c_size_t(n), C.c_size_t(chunk),
                                   C.byref(ok))
    return bool(ok.value)
