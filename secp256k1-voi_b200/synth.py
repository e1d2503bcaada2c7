"""Deterministic synthetic workloads (SURVEY.md section 8d).

One byte stream usable identically from any language:
    D(tag, i) = SHA-256(tag || LE64(seed) || LE64(i)),  seed = 20261017.
Host-side integer bookkeeping only (Python ints + hashlib); every curve
operation needed to *make* a workload (d*G, k*G) goes through the `base_mult`
callable the caller supplies -- the engine itself in bench.py, the oracle in
tests -- so this module has no arithmetic of its own to get wrong twice.
"""
import hashlib
import struct

import numpy as np

SEED = 20261017
N = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
P = 2**256 - 2**32 - 977


def D(tag, i, seed=SEED):
    return hashlib.sha256(tag + struct.pack("<QQ", seed, i)).digest()


def _stream_ints(tag, start, n, seed):
    return [int.from_bytes(D(tag, start + i, seed), "big") for i in range(n)]


def _nonzero_mod_n(x):
    return x % (N - 1) + 1


def _be32_rows(ints):
    return np.frombuffer(b"".join(x.to_bytes(32, "big") for x in ints), dtype=np.uint8).reshape(-1, 32).copy()


def batch_inverse_mod_n(xs):
    """Montgomery's trick over Python ints (all xs non-zero mod n)."""
    pre, run = [], 1
    for x in xs:
        pre.append(run)
        run = run * x % N
    inv = pow(run, -1, N)
    out = [0] * len(xs)
    for i in range(len(xs) - 1, -1, -1):
        out[i] = inv * pre[i] % N
        inv = inv * xs[i] % N
    return out


def tagged_hash(tag, data):
    t = hashlib.sha256(tag).digest()
    return hashlib.sha256(t + t + data).digest()


def _ecdsa_signatures(n, base_mult, start, seed):
    """d_i = D("key", i) mod n != 0, Q_i = d_i*G, z_i = D("msg", i), k_i = D("nonce", i) mod n != 0, r = x(k*G) mod n,
    s = (z + r*d)/k, low-s normalised for even i only -> (pk65, digest32, sig64, recovery ids) as uint8 arrays; the
    recovery id is the parity of y(kG), + 2 when x(kG) >= n, and flips with the sign of s."""
    d = [_nonzero_mod_n(x) for x in _stream_ints(b"key", start, n, seed)]
    k = [_nonzero_mod_n(x) for x in _stream_ints(b"nonce", start, n, seed)]
    zb = [D(b"msg", start + i, seed) for i in range(n)]
    pk, st = base_mult(_be32_rows(d))
    assert bool((np.asarray(st) == 1).all())
    kg, st = base_mult(_be32_rows(k))
    assert bool((np.asarray(st) == 1).all())
    pk = np.array(pk, dtype=np.uint8).reshape(n, 65)
    kg = np.asarray(kg, dtype=np.uint8).reshape(n, 65)
    kinv = batch_inverse_mod_n(k)
    sig = np.zeros((n, 64), np.uint8)
    recid = np.zeros(n, np.uint8)
    digest = np.frombuffer(b"".join(zb), np.uint8).reshape(n, 32).copy()
    for i in range(n):
        gi = start + i
        x = int.from_bytes(kg[i, 1:33].tobytes(), "big")
        r = x % N
        z = int.from_bytes(zb[i], "big") % N
        s = kinv[i] * (z + r * d[i]) % N
        v = (kg[i, 64] & 1) | (2 if x >= N else 0)
        if gi % 2 == 0 and s > N // 2:
            s = N - s
            v ^= 1
        assert r != 0 and s != 0
        sig[i, :32] = np.frombuffer(r.to_bytes(32, "big"), np.uint8)
        sig[i, 32:] = np.frombuffer(s.to_bytes(32, "big"), np.uint8)
        recid[i] = v
    return pk, digest, sig, recid


def ecdsa_batch(n, base_mult, start=0, seed=SEED, corrupt_every=16):
    """Config 2: returns dict(pk65, digest32, sig64, expected) as uint8 arrays.

    d_i = D("key", i) mod n != 0, Q_i = d_i*G, z_i = D("msg", i),
    k_i = D("nonce", i) mod n != 0, r = x(k*G) mod n, s = (z + r*d)/k,
    low-s normalised for even i only; every `corrupt_every`-th item corrupted,
    cycling: one bit of r / of s / of z flipped, Q replaced by Q_{i-1}.
    `expected` is by construction (valid unless corrupted)."""
    pk, digest, sig, _ = _ecdsa_signatures(n, base_mult, start, seed)
    expected = np.ones(n, np.uint8)
    if corrupt_every:
        pk_orig = pk.copy()
        for i in range(n):
            gi = start + i
            if gi % corrupt_every != corrupt_every - 1:
                continue
            kind = (gi // corrupt_every) % 4
            bit = gi % 250
            if kind == 0:
                sig[i, 31 - bit // 8] ^= 1 << (bit % 8)
            elif kind == 1:
                sig[i, 63 - bit // 8] ^= 1 << (bit % 8)
            elif kind == 2:
                digest[i, 31 - bit // 8] ^= 1 << (bit % 8)
            else:
                if i == 0:
                    sig[i, 40] ^= 1
                else:
                    pk[i] = pk_orig[i - 1]
            expected[i] = 0
    return {"pk65": pk, "digest32": digest, "sig64": sig, "expected": expected}


def ecdsa_recoverable_batch(n, base_mult, start=0, seed=SEED, corrupt_every=16):
    """The signatures of ecdsa_batch as recoverable r||s||v rows (secec EncodingCompactRecoverable): returns
    dict(pk65, digest32, sig65, expected).  v is the parity of y(kG) (+ 2 when x(kG) >= n), flipped where s was low-s
    normalised (even i), so every uncorrupted row recovers its key; odd rows keep a high s about half the time and fail
    under S256_FLAG_REJECT_MALLEABLE.  Every `corrupt_every`-th row is corrupted, cycling: one bit of r / of s / of z
    flipped, Q replaced by Q_{i-1}, v ^= 1."""
    pk, digest, sig, recid = _ecdsa_signatures(n, base_mult, start, seed)
    sig65 = np.concatenate([sig, recid.reshape(n, 1)], axis=1)
    expected = np.ones(n, np.uint8)
    if corrupt_every:
        pk_orig = pk.copy()
        for i in range(n):
            gi = start + i
            if gi % corrupt_every != corrupt_every - 1:
                continue
            kind = (gi // corrupt_every) % 5
            bit = gi % 250
            if kind == 0:
                sig65[i, 31 - bit // 8] ^= 1 << (bit % 8)
            elif kind == 1:
                sig65[i, 63 - bit // 8] ^= 1 << (bit % 8)
            elif kind == 2:
                digest[i, 31 - bit // 8] ^= 1 << (bit % 8)
            elif kind == 3 and i > 0:
                pk[i] = pk_orig[i - 1]
            else:
                sig65[i, 64] ^= 1
            expected[i] = 0
    return {"pk65": pk, "digest32": digest, "sig65": sig65, "expected": expected}


def schnorr_batch(n, base_mult, start=0, seed=SEED, corrupt_every=16):
    """Config 3: BIP-340 signatures over 32-byte messages with aux = D("aux", i);
    pk = x(Q_i) so that verification performs lift_x.  Same corruption cycle
    (r, s, msg, pk)."""
    dd = [_nonzero_mod_n(x) for x in _stream_ints(b"key", start, n, seed)]
    msgs = [D(b"msg", start + i, seed) for i in range(n)]
    aux = [D(b"aux", start + i, seed) for i in range(n)]
    pk, st = base_mult(_be32_rows(dd))
    pk = np.asarray(pk, dtype=np.uint8).reshape(n, 65)
    d, px, kprime = [], [], []
    for i in range(n):
        di = dd[i] if pk[i, 64] % 2 == 0 else N - dd[i]
        d.append(di)
        pxi = pk[i, 1:33].tobytes()
        px.append(pxi)
        t = (di ^ int.from_bytes(tagged_hash(b"BIP0340/aux", aux[i]), "big")).to_bytes(32, "big")
        kp = int.from_bytes(tagged_hash(b"BIP0340/nonce", t + pxi + msgs[i]), "big") % N
        assert kp != 0
        kprime.append(kp)
    R, st = base_mult(_be32_rows(kprime))
    R = np.asarray(R, dtype=np.uint8).reshape(n, 65)
    sig = np.zeros((n, 64), np.uint8)
    for i in range(n):
        kk = kprime[i] if R[i, 64] % 2 == 0 else N - kprime[i]
        rx = R[i, 1:33].tobytes()
        e = int.from_bytes(tagged_hash(b"BIP0340/challenge", rx + px[i] + msgs[i]), "big") % N
        s = (kk + e * d[i]) % N
        sig[i, :32] = np.frombuffer(rx, np.uint8)
        sig[i, 32:] = np.frombuffer(s.to_bytes(32, "big"), np.uint8)
    pkx = np.frombuffer(b"".join(px), np.uint8).reshape(n, 32).copy()
    msg = np.frombuffer(b"".join(msgs), np.uint8).reshape(n, 32).copy()
    expected = np.ones(n, np.uint8)
    if corrupt_every:
        pkx_orig = pkx.copy()
        for i in range(n):
            gi = start + i
            if gi % corrupt_every != corrupt_every - 1:
                continue
            kind = (gi // corrupt_every) % 4
            bit = gi % 250
            if kind == 0:
                sig[i, 31 - bit // 8] ^= 1 << (bit % 8)
            elif kind == 1:
                sig[i, 63 - bit // 8] ^= 1 << (bit % 8)
            elif kind == 2:
                msg[i, 31 - bit // 8] ^= 1 << (bit % 8)
            else:
                if i == 0:
                    sig[i, 40] ^= 1
                else:
                    pkx[i] = pkx_orig[i - 1]
            expected[i] = 0
    return {"pkx32": pkx, "msg": msg, "sig64": sig, "expected": expected}


def base_mult_scalars(n, start=0, seed=SEED):
    """Config 1: k_i = D("sbm", i) (reduced by the engine like NewScalarFromBytes),
    indices 0-7 forced to 0, 1, 2, n-1, n, 2^128, floor(n/2), floor(n/2)+1."""
    ks = [D(b"sbm", start + i, seed) for i in range(n)]
    forced = [0, 1, 2, N - 1, N, 2**128, N // 2, N // 2 + 1]
    for j, v in enumerate(forced):
        if start <= j < start + n:
            ks[j - start] = v.to_bytes(32, "big")
    return np.frombuffer(b"".join(ks), np.uint8).reshape(n, 32).copy()


def ecdh_batch(n, base_mult, start=0, seed=SEED):
    """Config 4: scalars D("ecdh", i) mod n != 0 against points Q_i = d_i*G;
    closed form: result = (k_i * d_i mod n) * G."""
    d = [_nonzero_mod_n(x) for x in _stream_ints(b"key", start, n, seed)]
    k = [_nonzero_mod_n(x) for x in _stream_ints(b"ecdh", start, n, seed)]
    pts, st = base_mult(_be32_rows(d))
    prod = [a * b % N for a, b in zip(d, k)]
    return {"k32": _be32_rows(k), "pt65": np.asarray(pts, np.uint8).reshape(n, 65), "closed_form_scalar": _be32_rows(prod)}


def msm_batch(n, base_mult, start=0, seed=SEED):
    """Config 5: s_i = D("msm", i) mod n, P_i = Q_i; the sum equals
    (sum s_i * d_i mod n) * G."""
    d = [_nonzero_mod_n(x) for x in _stream_ints(b"key", start, n, seed)]
    s = [x % N for x in _stream_ints(b"msm", start, n, seed)]
    pts, st = base_mult(_be32_rows(d))
    total = sum(a * b for a, b in zip(d, s)) % N
    return {"k32": _be32_rows(s), "pt65": np.asarray(pts, np.uint8).reshape(n, 65),
            "closed_form_scalar": total.to_bytes(32, "big"), "key_sum": sum(d) % N}
