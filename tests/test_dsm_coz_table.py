"""The per-key table of the verification ladder (kernels.cuh: item_dsm_table, a co-Z chain scaled to one common
denominator).  On the CPU the table phase runs through the host simulation and every row is checked against Python
integers: row k must be (x(kP) Z^2, y(kP) Z^3) for one non-zero Z, the Z_all the ladder leaves the isomorphic curve
with.  On the GPU, keys at the edges of the field go through the whole ladder against the oracle."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import parity_suites as ps

P, N = ps.P, ps.N
GX = 0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798
GY = 0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostsim", "dsm_table.cpp")
_SO = os.path.join(_HERE, "hostsim", "_build", "dsm_table.so")
_CSRC = os.path.join(os.path.dirname(_HERE), "secp256k1-voi_b200", "csrc")


def _lib():
    deps = [_SRC] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC) if f.endswith(".cuh")]
    if not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", _SO, _SRC])
    return C.CDLL(_SO)


def _add(a, b):
    """Affine addition on secp256k1 over Python integers; None is the identity."""
    if a is None:
        return b
    if b is None:
        return a
    (x1, y1), (x2, y2) = a, b
    if x1 == x2:
        if (y1 + y2) % P == 0:
            return None
        lam = 3 * x1 * x1 * pow(2 * y1, -1, P) % P
    else:
        lam = (y2 - y1) * pow(x2 - x1, -1, P) % P
    x3 = (lam * lam - x1 - x2) % P
    return x3, (lam * (x1 - x3) - y1) % P


def _mul(k, pt):
    acc = None
    for bit in bin(k % N)[2:]:
        acc = _add(acc, acc)
        if bit == "1":
            acc = _add(acc, pt)
    return acc


def _sec1(pt):
    return b"\x04" + pt[0].to_bytes(32, "big") + pt[1].to_bytes(32, "big")


def _edge_keys():
    """Points whose x or y lies just below p (and their negatives), found by search, with both signs."""
    out = []
    t = 1
    while len([q for q in out if q[0] > P - 2**16]) < 6:  # x = p - t with x^3 + 7 a square (p = 3 mod 4)
        x = P - t
        rhs = (x * x * x + 7) % P
        y = pow(rhs, (P + 1) // 4, P)
        if y * y % P == rhs:
            out += [(x, y), (x, P - y)]
        t += 1
    t = 1
    while len([q for q in out if q[1] > P - 2**16]) < 3:  # y = p - t: x = cube root of t^2 - 7 (p = 7 mod 9)
        a = (t * t - 7) % P
        x = pow(a, (P + 2) // 9, P)
        if x * x * x % P == a:
            out += [(x, P - t), (x, t)]
        t += 1
    for q in out:
        assert (q[1] * q[1] - q[0] ** 3 - 7) % P == 0
    return out


def _keys():
    g = (GX, GY)
    rng = random.Random(20261020)
    ks = [g]
    ks += [_mul(j, g) for j in (2, 3, 5, 16, 17, 31)]  # the small-multiples sweep of the parity suites
    ks += [_mul(N - j, g) for j in (1, 2, 15, 16)]
    ks += [_mul(rng.randrange(1, N), g) for _ in range(24)]
    ks += _edge_keys()
    return ks


def test_table_rows_are_multiples_over_one_denominator():
    lib = _lib()
    ts = lib.sim_dsm_table_rows()
    keys = _keys()
    n = len(keys)
    pk = np.frombuffer(b"".join(_sec1(q) for q in keys), np.uint8).copy()
    rows = np.zeros(n * ts * 64, np.uint8)
    zall = np.zeros(n * 32, np.uint8)
    valid = np.zeros(n, np.uint8)
    p_ = lambda a: a.ctypes.data_as(C.c_void_p)
    lib.sim_dsm_table(p_(pk), C.c_size_t(n), p_(rows), p_(zall), p_(valid))
    assert valid.all()
    for i, key in enumerate(keys):
        z = int.from_bytes(zall[32 * i:32 * i + 32].tobytes(), "big")
        assert 0 < z < P, i
        z2, z3 = z * z % P, z * z * z % P
        m = None
        for k in range(1, ts + 1):
            m = _add(m, key)
            off = (i * ts + k - 1) * 64
            x = int.from_bytes(rows[off:off + 32].tobytes(), "big")
            y = int.from_bytes(rows[off + 32:off + 64].tobytes(), "big")
            assert (x, y) == (m[0] * z2 % P, m[1] * z3 % P), (i, k)


def _check_ladder(run, oracle):
    """Every key with random scalars, then with small ones (u2 picks single table rows, including the last)."""
    keys = _keys()
    rng = random.Random(7)
    small = [(0, 1), (1, 16), (2, 17), (0, 15)]
    u1 = [rng.randrange(N) for _ in keys] + [small[j % 4][0] for j in range(len(keys))]
    u2 = [rng.randrange(N) for _ in keys] + [small[j % 4][1] for j in range(len(keys))]
    pts = np.frombuffer(b"".join(_sec1(q) for q in keys + keys), np.uint8).reshape(-1, 65).copy()
    U1, U2 = ps.rows([ps.b32(x) for x in u1], 32), ps.rows([ps.b32(x) for x in u2], 32)
    got, st = run(U1, U2, pts)
    exp, est = oracle.batch_double_scalar_mult(U1, U2, pts)
    assert np.array_equal(st, est)
    assert np.array_equal(got, exp)


def test_edge_keys_through_the_simulated_ladder(oracle):
    import hostsim as hs
    _check_ladder(hs.double_scalar_mult, oracle)


@pytest.mark.gpu
def test_edge_keys_through_the_ladder(engine, oracle):
    _check_ladder(engine.double_scalar_mult_basepoint_vartime, oracle)
