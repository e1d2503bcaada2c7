"""ctypes view of tests/hostsim/varlen_sim.cpp: the BIP-340 entry points over messages of different lengths on the CPU
(test infrastructure only).  `msg` is (flat uint8 array, uint64 offsets of n + 1), row i = flat[offsets[i]:offsets[i + 1]]."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import _HERE, _a, _deps, _p

_SO = os.path.join(_HERE, "_build", "varlen_sim.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "varlen_sim.cpp")
        deps = _deps() + [src, os.path.join(_HERE, "batch_sim.cpp")]
        stale = not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps)
        if stale:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", _SO, src])
        _lib = C.CDLL(_SO)
    return _lib


def _flat(msg):
    flat, offs = msg
    flat = np.ascontiguousarray(flat, dtype=np.uint8)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    if flat.size == 0:
        flat = np.zeros(1, np.uint8)  # a valid pointer for an all-empty batch
    return flat, offs


def schnorr_verify(pkx, msg, sig):
    pkx, sig = _a(pkx, 32), _a(sig, 64)
    flat, offs = _flat(msg)
    n = len(pkx); ok = np.zeros(n, np.uint8)
    lib().sim_schnorr_verify_varlen(_p(pkx), _p(flat), _p(offs), _p(sig), C.c_size_t(n), _p(ok))
    return ok


def schnorr_sign(priv, msg, aux):
    priv, aux = _a(priv, 32), _a(aux, 32)
    flat, offs = _flat(msg)
    n = len(priv); sig = np.zeros((n, 64), np.uint8); st = np.zeros(n, np.uint8)
    lib().sim_schnorr_sign_varlen(_p(priv), _p(flat), _p(offs), _p(aux), C.c_size_t(n), _p(sig), _p(st))
    return sig, st


def schnorr_batch_randomizers(pkx, msg, sig, chunk):
    """Pass 1 of the batch verification with chunks of `chunk` rows: (seed, a) -- 32 bytes and (n, 32) big-endian rows."""
    pkx, sig = _a(pkx, 32), _a(sig, 64)
    flat, offs = _flat(msg)
    n = len(pkx); seed = np.zeros(32, np.uint8); a = np.zeros((n, 32), np.uint8)
    lib().sim_schnorr_batch_randomizers_varlen(_p(pkx), _p(flat), _p(offs), _p(sig), C.c_size_t(n), C.c_size_t(chunk), _p(seed),
                                               _p(a))
    return seed.tobytes(), a


def schnorr_batch_verify(pkx, msg, sig, chunk=1 << 19):
    """The batch verdict (bool) as s256_schnorr_batch_verify_varlen computes it, with chunks of `chunk` rows."""
    pkx, sig = _a(pkx, 32), _a(sig, 64)
    flat, offs = _flat(msg)
    n = len(pkx); ok = C.c_uint8(0)
    lib().sim_schnorr_batch_verify_varlen(_p(pkx), _p(flat), _p(offs), _p(sig), C.c_size_t(n), C.c_size_t(chunk), C.byref(ok))
    return bool(ok.value)
