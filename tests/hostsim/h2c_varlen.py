"""ctypes view of tests/hostsim/h2c_varlen_sim.cpp: hash-to-curve over messages of different lengths on the CPU (test
infrastructure only).  `msg` is (flat uint8 array, uint64 offsets of n + 1), row i = flat[offsets[i]:offsets[i + 1]]."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

from . import _HERE, _deps, _p

_SO = os.path.join(_HERE, "_build", "h2c_varlen_sim.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "h2c_varlen_sim.cpp")
        deps = _deps() + [src]
        stale = not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps)
        if stale:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", _SO, src])
        _lib = C.CDLL(_SO)
    return _lib


def hash_to_curve(dst, msg, random_oracle=True):
    """(out65 (n, 65), status (n,)) as s256_hash_to_curve_varlen_dev computes them."""
    dst = bytes(dst)
    if len(dst) > 255:  # the library pre-hashes oversize DSTs on the host
        dst = hashlib.sha256(b"H2C-OVERSIZE-DST-" + dst).digest()
    flat, offs = msg
    flat = np.ascontiguousarray(flat, dtype=np.uint8)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    if flat.size == 0:
        flat = np.zeros(1, np.uint8)  # a valid pointer for an all-empty batch
    n = len(offs) - 1
    out = np.zeros((n, 65), np.uint8)
    st = np.zeros(n, np.uint8)
    lib().sim_hash_to_curve_varlen(dst, C.c_size_t(len(dst)), _p(flat), _p(offs), C.c_size_t(n), int(random_oracle), _p(out),
                                   _p(st))
    return out, st
