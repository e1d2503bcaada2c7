"""BIP-340 on the device against a plain Python reference: the rows of the batch equation the kernels of
s256_schnorr_batch_verify build (seed, a_i, a_i e_i, -R_i, -P_i, sum a_i s_i) at the CTA and chunk edges, randomizers
that must not repeat or cancel across CTAs and chunks, and the byte-stream hashing of messages whose length is not 32
(challenge, nonce, batch leaf, expand_message_xmd) across the SHA-256 padding boundaries.

The reference is Python integers and hashlib.  The CPU tests pin it to the BIP-340 and RFC 9380 vectors and to the host
simulation, so that a GPU failure here points at the device build and not at the reference."""
import hashlib

import numpy as np
import pytest

from conftest import load_golden
from hostsim import batch as batch_sim
import hostsim as hs
from test_schnorr_batch import ref_seed_and_randomizers

P = 2 ** 256 - 2 ** 32 - 977
N = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
G = (0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798,
     0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8)
TPB = 128  # S256_TPB: rows per CTA of k_batch_prepare; k_batch_tree folds 2 * TPB nodes per CTA

# message lengths: 0..130 covers every residue of the 128 + L (challenge, nonce) and 96 + L (batch leaf) byte streams
# mod 64; the rest are the padding edges one and two blocks further out, and a long message
SWEEP_LENGTHS = list(range(131)) + [183, 184, 191, 192, 247, 248, 1000]
XMD_DSTS = (1, 21, 22, 29, 30, 255, 256)  # 256: hashed to 32 bytes first (RFC 9380 section 5.3.3)
XMD_OUT = (1, 31, 32, 33, 48, 64, 95, 96)


# ---- reference: Python integers and hashlib ----------------------------------------------------------------------
def _jadd_affine(p, q):
    """Jacobian p + affine q (None: the identity)."""
    if q is None:
        return p
    if p is None:
        return (q[0], q[1], 1)
    X1, Y1, Z1 = p
    x2, y2 = q
    Z1Z1 = Z1 * Z1 % P
    U2, S2 = x2 * Z1Z1 % P, y2 * Z1 * Z1Z1 % P
    H, r = (U2 - X1) % P, (S2 - Y1) % P
    if H == 0:
        return _jdbl(p) if r == 0 else None
    HH = H * H % P
    HHH = H * HH % P
    V = X1 * HH % P
    X3 = (r * r - HHH - 2 * V) % P
    return X3, (r * (V - X3) - Y1 * HHH) % P, Z1 * H % P


def _jdbl(p):
    if p is None or p[1] == 0:
        return None
    X, Y, Z = p
    YY = Y * Y % P
    S = 4 * X * YY % P
    M = 3 * X * X % P
    X3 = (M * M - 2 * S) % P
    return X3, (M * (S - X3) - 8 * YY * YY) % P, 2 * Y * Z % P


def _affine(p):
    if p is None:
        return None
    zi = pow(p[2], P - 2, P)
    return p[0] * zi * zi % P, p[1] * zi * zi * zi % P


_G_POW2 = [G]
for _ in range(255):
    _G_POW2.append(_affine(_jdbl((_G_POW2[-1][0], _G_POW2[-1][1], 1))))


def point_mul(k, Q=None):
    """k Q for an affine point Q (default G), affine; None for the identity."""
    k %= N
    acc = None
    if Q is None:
        for i in range(k.bit_length()):
            if k >> i & 1:
                acc = _jadd_affine(acc, _G_POW2[i])
        return _affine(acc)
    for i in reversed(range(k.bit_length())):
        acc = _jdbl(acc)
        if k >> i & 1:
            acc = _jadd_affine(acc, Q)
    return _affine(acc)


def point_neg(Q):
    return Q[0], (P - Q[1]) % P


def point_add(a, b):
    return _affine(_jadd_affine(None if a is None else (a[0], a[1], 1), b))


def lift_x(x):
    """BIP-340 lift_x: the point with x-coordinate x and even y, or None."""
    if x >= P:
        return None
    c = (x * x * x + 7) % P
    y = pow(c, (P + 1) // 4, P)
    if y * y % P != c:
        return None
    return x, y if y % 2 == 0 else P - y


def tagged_hash(tag, data):
    t = hashlib.sha256(tag).digest()
    return hashlib.sha256(t + t + data).digest()


def challenge(r32, px32, msg):
    return int.from_bytes(tagged_hash(b"BIP0340/challenge", bytes(r32) + bytes(px32) + bytes(msg)), "big") % N


def ref_sign(d32, msg, aux32):
    """BIP-340 Sign; None for a secret key outside [1, n)."""
    d0 = int.from_bytes(bytes(d32), "big")
    if not 0 < d0 < N:
        return None
    Pt = point_mul(d0)
    d = d0 if Pt[1] % 2 == 0 else N - d0
    px = Pt[0].to_bytes(32, "big")
    t = (d ^ int.from_bytes(tagged_hash(b"BIP0340/aux", bytes(aux32)), "big")).to_bytes(32, "big")
    k0 = int.from_bytes(tagged_hash(b"BIP0340/nonce", t + px + bytes(msg)), "big") % N
    if k0 == 0:
        return None
    R = point_mul(k0)
    k = k0 if R[1] % 2 == 0 else N - k0
    rx = R[0].to_bytes(32, "big")
    return rx + ((k + challenge(rx, px, msg) * d) % N).to_bytes(32, "big")


def ref_verify(px32, msg, sig64):
    sig64 = bytes(sig64)
    Pt = lift_x(int.from_bytes(bytes(px32), "big"))
    r, s = int.from_bytes(sig64[:32], "big"), int.from_bytes(sig64[32:], "big")
    if Pt is None or r >= P or s >= N:
        return False
    e = challenge(sig64[:32], px32, msg)
    R = point_add(point_mul(s), point_mul(N - e, Pt) if e else None)
    return R is not None and R[1] % 2 == 0 and R[0] == r


def ref_expand_xmd(msg, dst, length):
    """expand_message_xmd with SHA-256 (RFC 9380 section 5.3.1), oversize DSTs hashed first (section 5.3.3)."""
    dst = bytes(dst)
    if len(dst) > 255:
        dst = hashlib.sha256(b"H2C-OVERSIZE-DST-" + dst).digest()
    dst_prime = dst + bytes([len(dst)])
    ell = (length + 31) // 32
    b0 = hashlib.sha256(bytes(64) + bytes(msg) + length.to_bytes(2, "big") + b"\x00" + dst_prime).digest()
    bi = hashlib.sha256(b0 + b"\x01" + dst_prime).digest()
    out = bi
    for i in range(2, ell + 1):
        bi = hashlib.sha256(bytes(x ^ y for x, y in zip(b0, bi)) + bytes([i]) + dst_prime).digest()
        out += bi
    return out[:length]


def ref_batch_rows(pkx, msg, sig, points_at=None):
    """The batch equation by definition: (seed, a, ae, negR, negP, sum a_i s_i mod n, rejected), with negR / negP only at
    the rows in points_at (all rows if None) and None at a rejected row.  Rows outside points_at are taken as not
    rejected, so use it for batches of valid rows only."""
    n = len(pkx)
    seed, a = ref_seed_and_randomizers(pkx, msg, sig)
    sample = set(range(n)) if points_at is None else set(points_at)
    ae, negR, negP = [0] * n, {}, {}
    total, rejected = 0, False
    for i in range(n):
        sg = sig[i].tobytes()
        r, s = int.from_bytes(sg[:32], "big"), int.from_bytes(sg[32:], "big")
        if i in sample:
            R, Pt = lift_x(r), lift_x(int.from_bytes(pkx[i].tobytes(), "big"))
            if R is None or Pt is None or s >= N:
                rejected = True
                negR[i] = negP[i] = None
                a[i] = 0
                continue
            negR[i], negP[i] = point_neg(R), point_neg(Pt)
        ae[i] = a[i] * challenge(sg[:32], pkx[i].tobytes(), msg[i].tobytes()) % N
        total += a[i] * s
    return seed, a, ae, negR, negP, total % N, rejected


def _be(x):
    return int.from_bytes(x.tobytes(), "big")


def _pt(row64):
    return _be(row64[:32]), _be(row64[32:])


def check_batch_rows(got, pkx, msg, sig, points_at=None):
    """Every field of Engine.debug_schnorr_batch_rows against ref_batch_rows."""
    seed, k, pts, ssum, rejected = got
    want_seed, a, ae, negR, negP, total, want_rej = ref_batch_rows(pkx, msg, sig, points_at)
    assert seed == want_seed
    assert _be(k[0, 0]) == (1 if a[0] else 0)
    bad = [i for i in range(len(pkx)) if (_be(k[i, 0]), _be(k[i, 1])) != (a[i], ae[i])]
    assert not bad, f"{len(bad)} rows differ in a_i or a_i e_i, first {bad[:8]}"
    for i in negR:
        if negR[i] is None:
            assert _pt(pts[i, 0]) == G and _pt(pts[i, 1]) == G, i
        else:
            assert _pt(pts[i, 0]) == negR[i] and _pt(pts[i, 1]) == negP[i], i
    assert int.from_bytes(ssum, "big") == total
    assert rejected == want_rej


# ---- rows ------------------------------------------------------------------------------------------------------------
def det_bytes(label, i, width):
    out = b""
    ctr = 0
    while len(out) < width:
        out += hashlib.sha256(b"%s/%d/%d" % (label, i, ctr)).digest()
        ctr += 1
    return out[:width]


def sweep_rows(L, count=8):
    """count signed rows with L-byte messages: (priv, msg, aux, pkx, sig) as numpy arrays, signed by the reference."""
    priv = np.zeros((count, 32), np.uint8)
    msg = np.zeros((count, L), np.uint8)
    aux = np.zeros((count, 32), np.uint8)
    pkx = np.zeros((count, 32), np.uint8)
    sig = np.zeros((count, 64), np.uint8)
    for j in range(count):
        d = int.from_bytes(det_bytes(b"key", 1000 * L + j, 32), "big") % (N - 1) + 1
        priv[j] = np.frombuffer(d.to_bytes(32, "big"), np.uint8)
        msg[j] = np.frombuffer(det_bytes(b"msg", 1000 * L + j, L), np.uint8)
        aux[j] = np.frombuffer(det_bytes(b"aux", 1000 * L + j, 32), np.uint8)
        pkx[j] = np.frombuffer(point_mul(d)[0].to_bytes(32, "big"), np.uint8)
        sig[j] = np.frombuffer(ref_sign(priv[j].tobytes(), msg[j].tobytes(), aux[j].tobytes()), np.uint8)
    return priv, msg, aux, pkx, sig


def corrupt_two(msg, sig):
    """Rows 2 and 5 made invalid (a message bit, or an s bit when there is no message; an r bit)."""
    msg, sig = msg.copy(), sig.copy()
    if msg.shape[1]:
        msg[2, msg.shape[1] // 2] ^= 0x10
    else:
        sig[2, 50] ^= 0x10
    sig[5, 7] ^= 0x01
    return msg, sig


_SWEEP = {}


def sweep(L):
    if L not in _SWEEP:
        _SWEEP[L] = sweep_rows(L)
    return _SWEEP[L]


def with_cancelling_pair(rows, i, j, delta=1):
    """s_i + delta and s_j - delta: the unweighted sum of the two equations still holds, the batch must fail."""
    pkx, msg, sig = (x.copy() for x in rows)
    for row, d in ((i, delta), (j, -delta)):
        s = (int.from_bytes(sig[row, 32:].tobytes(), "big") + d) % N
        sig[row, 32:] = np.frombuffer(s.to_bytes(32, "big"), np.uint8)
    return pkx, msg, sig


def nonresidue_x():
    """The smallest x with x^3 + 7 not a square: an x-coordinate of no curve point."""
    x = 0
    while lift_x(x) is not None:
        x += 1
    return x


def reject_row(pkx, sig, i, kind):
    x_bad = nonresidue_x()
    if kind == "s>=n":
        s = N + int.from_bytes(sig[i, 32:36].tobytes(), "big") % 1000
        sig[i, 32:] = np.frombuffer(s.to_bytes(32, "big"), np.uint8)
    elif kind == "r>=p":  # r - p lifts, so only the range check rejects it
        t = 0
        while lift_x(t) is None:
            t += 1
        sig[i, :32] = np.frombuffer((P + t).to_bytes(32, "big"), np.uint8)
    elif kind == "r-not-x":
        sig[i, :32] = np.frombuffer(x_bad.to_bytes(32, "big"), np.uint8)
    else:  # the key does not lift
        pkx[i] = np.frombuffer(x_bad.to_bytes(32, "big"), np.uint8)


REJECT_KINDS = ("s>=n", "r>=p", "r-not-x", "pk-not-x")


# ---- CPU: the reference against the vectors and the host simulation -----------------------------------------------------
def test_reference_matches_bip340_vectors():
    rows = load_golden("bip340.json")["rows"]
    H = bytes.fromhex
    for r in rows:
        assert ref_verify(H(r["pk"]), H(r["msg"]), H(r["sig"])) == r["valid"], r["index"]
        if r["sk"]:
            assert ref_sign(H(r["sk"]), H(r["msg"]), H(r["aux"])) == H(r["sig"]), r["index"]
            assert point_mul(int(r["sk"], 16))[0] == int(r["pk"], 16)
    assert sum(r["valid"] for r in rows) >= 5 and sum(not r["valid"] for r in rows) >= 10


def test_reference_matches_expander_vectors():
    doc = load_golden("h2c.json")
    seen = 0
    for e in doc["expand"]:
        for tc in e["tests"]:
            assert ref_expand_xmd(tc["msg"].encode(), e["dst"].encode(), tc["len"]).hex() == tc["uniform_bytes"]
            seen += 1
    assert seen >= 10


def test_reference_point_arithmetic():
    """lift_x / negation / multiplication agree with each other and with the group order."""
    assert point_mul(N - 1) == point_neg(G) and point_mul(N) is None and point_mul(2) == point_add(G, G)
    x_bad = nonresidue_x()
    assert lift_x(x_bad) is None and lift_x(P) is None and lift_x(G[0]) == G  # G has an even y
    Q = point_mul(0xDEADBEEF)
    assert point_mul(5, Q) == point_mul(5 * 0xDEADBEEF)


def test_hostsim_sign_verify_batch_across_message_lengths():
    """The shared C++ logic (host build) over the whole length sweep: signatures bit-exact with the reference, per-row
    verdicts with two corrupted rows, the batch verdict, and the batch challenges inside the batch equation."""
    for L in SWEEP_LENGTHS:
        priv, msg, aux, pkx, sig = sweep(L)
        got, st = hs.schnorr_sign(priv, msg, aux)
        assert (st == 1).all() and np.array_equal(got, sig), L
        bmsg, bsig = corrupt_two(msg, sig)
        want = [ref_verify(pkx[j], bmsg[j], bsig[j]) for j in range(8)]
        assert want == [j not in (2, 5) for j in range(8)], L
        assert hs.schnorr_verify(pkx, bmsg, bsig).tolist() == [int(w) for w in want], L
        assert hs.schnorr_verify(pkx, msg, sig).all(), L
        assert batch_sim.schnorr_batch_verify(pkx, msg, sig), L
        assert not batch_sim.schnorr_batch_verify(pkx, bmsg, bsig), L
        seed, a = batch_sim.schnorr_batch_randomizers(pkx, msg, sig, chunk=4)
        want_seed, want_a = ref_seed_and_randomizers(pkx, msg, sig)
        assert seed == want_seed and [_be(a[j]) for j in range(8)] == want_a, L


def test_hostsim_expand_xmd_sweep():
    for D in XMD_DSTS:
        dst = det_bytes(b"dst", D, D)
        for L in range(71):
            m = np.frombuffer(det_bytes(b"xmd", 100 * D + L, L), np.uint8).reshape(1, L)
            for out_len in XMD_OUT:
                got = hs.expand_message_xmd(dst, m, out_len)
                assert got[0].tobytes() == ref_expand_xmd(m[0].tobytes(), dst, out_len), (D, L, out_len)


def cancel_pairs(C, n):
    """(i, j) pairs whose equal randomizers would let a cancelling pair through, for chunks of C rows and n rows."""
    pairs = {(0, 1), (0, 2), (0, n - 1), (127, 128), (1, 129), (200, 328), (C - 1, C), (3, 3 + C), (0, C)}
    return sorted((i, j) for i, j in pairs if j < n)


@pytest.fixture(scope="module")
def valid_rows_4200(oracle):
    import parity_suites as ps
    w = ps.synth.schnorr_batch(4200, ps.oracle_base_mult(oracle), corrupt_every=0)
    return w["pkx32"], w["msg"], w["sig64"]


@pytest.mark.parametrize("C", [1, 2048])
def test_hostsim_cancelling_pairs_are_rejected(valid_rows_4200, C):
    n = 300 if C == 1 else 4200
    rows = tuple(x[:n] for x in valid_rows_4200)
    assert batch_sim.schnorr_batch_verify(*rows, chunk=C)
    for i, j in cancel_pairs(C, n):
        assert not batch_sim.schnorr_batch_verify(*with_cancelling_pair(rows, i, j), chunk=C), (C, i, j)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
_POOLS = {}


def signed_pool(engine, L, n):
    """n rows with L-byte messages signed on the device (the prepared-row tests check every row against the reference
    from these bytes, so they do not rely on the signer)."""
    have = _POOLS.get(L)
    if have is None or len(have[0]) < n:
        rng = np.random.default_rng(7000 + L)
        priv = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        priv[:, 0] &= 0x7F
        priv[:, 31] |= 1
        msg = rng.integers(0, 256, (n, L), dtype=np.uint8)
        aux = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        pub, pst = engine.scalar_base_mult(priv)
        sig, sst = engine.schnorr_sign(priv, msg, aux)
        assert (pst == 1).all() and (sst == 1).all()
        _POOLS[L] = have = (pub[:, 1:33].copy(), msg.copy(), sig.copy())
    return tuple(x[:n] for x in have)


ROW_COUNTS = [1, 2, 3, 127, 128, 129, 255, 256, 257, 511, 513, 65535, 65536, 65537]
MSG_LENS = [0, 31, 32, 33, 100]


@pytest.mark.gpu
@pytest.mark.parametrize("n", ROW_COUNTS)
def test_gpu_prepared_rows_match_reference(engine, n):
    """Resident path (one chunk): CTA edges of k_batch_prepare and k_batch_tree, and 2^16 + 1 rows, where a chunk
    needs a third k_batch_tree launch."""
    L = MSG_LENS[ROW_COUNTS.index(n) % len(MSG_LENS)]
    rows = signed_pool(engine, L, n)
    check_batch_rows(engine.debug_schnorr_batch_rows(*rows), *rows)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [(1 << 19) - 1, (1 << 19) + 1])
def test_gpu_prepared_rows_around_the_default_chunk(engine, n):
    """2^19 - 1 rows: three tree launches in one chunk; 2^19 + 1: a second chunk of one row."""
    rows = signed_pool(engine, 33, n)
    edges = {0, 1, 127, 128, 255, 256, n - 2, n - 1, (1 << 19) - 1} | set(range(0, n, 997))
    check_batch_rows(engine.debug_schnorr_batch_rows(*rows), *rows, points_at=sorted(e for e in edges if e < n))


@pytest.mark.gpu
def test_gpu_prepared_rows_full_size(engine):
    """2^20 rows, two chunks on the default engine: the seed, every a_i and a_i e_i, the sum, and a strided sample of
    the points."""
    n = 1 << 20
    rows = signed_pool(engine, 32, n)
    got = engine.debug_schnorr_batch_rows(*rows)
    check_batch_rows(got, *rows, points_at=list(range(0, n, 4093)) + [(1 << 19) - 1, 1 << 19, n - 1])


@pytest.mark.gpu
@pytest.mark.parametrize("max_batch", [2, 3, 4, 1024, 4096])
@pytest.mark.parametrize("L", MSG_LENS)
def test_gpu_prepared_rows_do_not_depend_on_the_chunk_size(engine, s256, max_batch, L):
    """Chunks of C = 1, 1, 2, 512, 2048 rows: the same seed and a_i as the default engine, every row by definition."""
    C = 1
    while 4 * C <= max_batch:
        C *= 2
    n = 300 if C <= 2 else 3 * C + 77
    rows = signed_pool(engine, L, n)
    want = engine.debug_schnorr_batch_rows(*rows)
    small = s256.Engine(max_batch=max_batch)
    try:
        got = small.debug_schnorr_batch_rows(*rows)
    finally:
        small.close()
    assert got[0] == want[0]
    assert np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2]) and got[3] == want[3]
    check_batch_rows(got, *rows)


@pytest.mark.gpu
@pytest.mark.parametrize("max_batch", [0, 4096])
def test_gpu_rejected_rows(engine, s256, max_batch):
    """Each kind of rejected row at the first and last row, a CTA edge and a chunk edge: G with scalar 0 and the flag,
    every other row untouched.  The kinds rotate so that each appears at each position."""
    eng = s256.Engine(max_batch=max_batch) if max_batch else engine
    try:
        C = 2048 if max_batch else 1 << 19
        n = 2 * 2048 + 100
        base = signed_pool(engine, 31, n)
        positions = sorted({0, 127, 128, min(C - 1, n - 1), min(C, n - 1), n - 1})
        for rot in range(len(REJECT_KINDS)):
            pkx, msg, sig = (x.copy() for x in base)
            for q, i in enumerate(positions):
                reject_row(pkx, sig, i, REJECT_KINDS[(q + rot) % len(REJECT_KINDS)])
            got = eng.debug_schnorr_batch_rows(pkx, msg, sig)
            assert got[4]
            check_batch_rows(got, pkx, msg, sig)
            for i in positions:
                assert not got[1][i].any()
            assert not eng.schnorr_batch_verify(pkx, msg, sig)
    finally:
        if max_batch:
            eng.close()


def _cuda(a, off=0):
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(a).reshape(-1))
    buf = torch.zeros(flat.numel() + off, dtype=torch.uint8, device="cuda")
    buf[off:] = flat.cuda()
    return buf[off:]


@pytest.mark.gpu
@pytest.mark.parametrize("max_batch", [0, 2, 4096])
def test_gpu_cancelling_pairs_are_rejected(engine, s256, max_batch):
    """Pairs that cancel when their randomizers are equal: with a_0 = 1, inside and across the CTAs of k_batch_prepare,
    and across chunks (C = 1 and C = 2048), through the host form and the _dev form."""
    eng = s256.Engine(max_batch=max_batch) if max_batch else engine
    try:
        C = 1 if max_batch == 2 else 2048 if max_batch else 1 << 19
        n = 300 if C == 1 else 4200
        rows = signed_pool(engine, 32, n)
        assert eng.schnorr_batch_verify(*rows)
        for i, j in cancel_pairs(C, n):
            bad = with_cancelling_pair(rows, i, j)
            assert not eng.schnorr_batch_verify(*bad), (C, i, j)
            assert eng.schnorr_batch_verify(*(_cuda(x) for x in bad)).item() == 0, (C, i, j)
    finally:
        if max_batch:
            eng.close()


@pytest.mark.gpu
def test_gpu_sign_verify_batch_across_message_lengths(engine):
    for L in SWEEP_LENGTHS:
        priv, msg, aux, pkx, sig = sweep(L)
        got, st = engine.schnorr_sign(priv, msg, aux)
        assert (st == 1).all() and np.array_equal(got, sig), L
        bmsg, bsig = corrupt_two(msg, sig)
        assert engine.schnorr_verify(pkx, msg, sig).all(), L
        assert engine.schnorr_verify(pkx, bmsg, bsig).tolist() == [int(j not in (2, 5)) for j in range(8)], L
        assert engine.schnorr_batch_verify(pkx, msg, sig), L
        assert not engine.schnorr_batch_verify(pkx, bmsg, bsig), L
        check_batch_rows(engine.debug_schnorr_batch_rows(pkx, msg, sig), pkx, msg, sig)


@pytest.mark.gpu
@pytest.mark.parametrize("off", [1, 3])
def test_gpu_dev_forms_misaligned_messages(engine, off):
    import torch
    for L in (31, 33, 55, 56, 63, 64):
        priv, msg, aux, pkx, sig = sweep(L)
        bmsg, bsig = corrupt_two(msg, sig)
        d_sig, d_st = engine.schnorr_sign(_cuda(priv, off), _cuda(msg, off), _cuda(aux, off))
        ok = engine.schnorr_verify(_cuda(pkx, off), _cuda(bmsg, off), _cuda(bsig, off))
        good = engine.schnorr_batch_verify(_cuda(pkx, off), _cuda(msg, off), _cuda(sig, off))
        bad = engine.schnorr_batch_verify(_cuda(pkx, off), _cuda(bmsg, off), _cuda(bsig, off))
        torch.cuda.synchronize()
        assert (d_st.cpu().numpy() == 1).all() and np.array_equal(d_sig.cpu().numpy(), sig), (L, off)
        assert ok.cpu().numpy().tolist() == [int(j not in (2, 5)) for j in range(8)], (L, off)
        assert good.item() == 1 and bad.item() == 0, (L, off)


@pytest.mark.gpu
def test_gpu_expand_xmd_and_hash_to_curve_sweep(engine, oracle):
    for D in XMD_DSTS:
        dst = det_bytes(b"dst", D, D)
        for L in range(71):
            m = np.stack([np.frombuffer(det_bytes(b"xmd", 100 * D + L + 7919 * r, L), np.uint8) for r in range(2)])
            for out_len in XMD_OUT:
                got = engine.expand_message_xmd(dst, m, out_len)
                for r in range(2):
                    assert got[r].tobytes() == ref_expand_xmd(m[r].tobytes(), dst, out_len), (D, L, out_len, r)
            if L in (0, 1, 23, 24, 55, 56, 63, 64, 70):
                for ro in (True, False):
                    out, st = engine.hash_to_curve(dst, m, ro)
                    for r in range(2):
                        want, wst = oracle.hash_to_curve(dst, m[r].tobytes(), ro)
                        assert out[r].tobytes() == bytes(want) and st[r] == wst, (D, L, ro, r)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [100, 33])
def test_gpu_host_pipeline_other_message_lengths(s256, oracle, L):
    """Sign and verify from host memory with L-byte messages through a pipelined chunk of 2^18 rows (sub-chunk cuts at
    6/64, 24/64, 44/64 when signing, 1/8 when verifying) and a second chunk of 5000 rows."""
    cap = 1 << 18
    eng = s256.Engine(device=0, max_batch=cap)
    try:
        n = cap + 5000
        cut = lambda f: (cap * f // 64 + 127) & ~127  # noqa: E731  (ctx.h pipelined)
        cuts = [0, cut(6), cut(8), cut(24), cut(44), cap, n]
        sample = sorted({min(max(c + d, 0), n - 1) for c in cuts for d in (-2, -1, 0, 1, 127, 128)})
        rng = np.random.default_rng(L)
        priv = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        priv[:, 0] &= 0x7F
        priv[:, 31] |= 1
        msg = rng.integers(0, 256, (n, L), dtype=np.uint8)
        aux = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        sig, st = eng.schnorr_sign(priv, msg, aux)
        assert (st == 1).all()
        sig = sig.copy()
        for i in sample:
            want, wst = oracle.schnorr_sign(priv[i].tobytes(), msg[i].tobytes(), aux[i].tobytes())
            assert sig[i].tobytes() == bytes(want), i
        pub, _ = eng.scalar_base_mult(priv)
        pkx = pub[:, 1:33].copy()
        bad = np.zeros(n, bool)
        bad[15::16] = True
        bsig = sig.copy()
        bsig[bad, 40] ^= 0x04
        ok = eng.schnorr_verify(pkx, msg, bsig)
        assert np.array_equal(ok, (~bad).astype(np.uint8))
        assert oracle.batch_schnorr_verify(pkx[sample], msg[sample], bsig[sample]).tolist() == ok[sample].tolist()
    finally:
        eng.close()
