"""ctypes view of tests/hostsim/der_sim.cpp: the device DER parser on the CPU (test infrastructure only).  Rows are
(flat uint8 array, uint64 offsets of n + 1), row i = flat[offsets[i]:offsets[i + 1]]."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import _HERE, _deps, _p

_SO = os.path.join(_HERE, "_build", "der_sim.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "der_sim.cpp")
        deps = _deps() + [src]
        stale = not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps)
        if stale:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", _SO, src])
        _lib = C.CDLL(_SO)
    return _lib


def _flat(rows):
    flat, offs = rows
    flat = np.ascontiguousarray(flat, dtype=np.uint8)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    if flat.size == 0:
        flat = np.zeros(1, np.uint8)  # a valid pointer for an all-empty batch
    return flat, offs


def parse_der(rows, bip66=False):
    """k_parse_der: (sig64 rows, ok).  bip66=True: rows carry the sighash byte (bitcoin.VerifyASN1's parse)."""
    flat, offs = _flat(rows)
    n = len(offs) - 1
    sig = np.zeros((n, 64), np.uint8); ok = np.zeros(n, np.uint8)
    lib().sim_parse_der(_p(flat), _p(offs), C.c_size_t(n), int(bip66), _p(sig), _p(ok))
    return sig, ok


def check_bip66(rows):
    """k_check_bip66: ok bytes of IsValidSignatureEncodingBIP0066."""
    flat, offs = _flat(rows)
    n = len(offs) - 1
    ok = np.zeros(n, np.uint8)
    lib().sim_check_bip66(_p(flat), _p(offs), C.c_size_t(n), _p(ok))
    return ok
