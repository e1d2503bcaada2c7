"""Recoverable ECDSA batch verification (s256_ecdsa_recoverable_batch_verify): the randomizer definition against
hashlib, the batch verdict of the host simulation against the per-row oracle (recover, then compare the key), the rows
of the batch equation against a plain Python reference, and the same through the C ABI on the GPU."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from hostsim import ecdsa_batch as sim
import parity_suites as ps

P = 2 ** 256 - 2 ** 32 - 977
N = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
G = (0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798,
     0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8)
TPB = 128  # rows per CTA of k_ecdsa_batch_points; threads per CTA of k_ecdsa_batch_prepare
EDGE_FLAGS = ("EdgeCaseShamirMultiplication", "PointDuplication", "ArithmeticError", "SmallRandS", "SpecialCaseHash",
              "EdgeCasePublicKey")


def b32(x):
    return np.frombuffer(int(x).to_bytes(32, "big"), np.uint8)


def be(a):
    return int.from_bytes(bytes(a), "big")


# ---- reference: hashlib and Python integers (DESIGN.md section 8, item 6) ------------------------------------------
def ref_seed_and_randomizers(pk, dg, sig):
    n = len(pk)
    nodes = [hashlib.sha256(bytes(pk[i]) + bytes(dg[i]) + bytes(sig[i])).digest() for i in range(n)]
    while len(nodes) > 1:
        nodes = [hashlib.sha256(nodes[j] + nodes[j + 1]).digest() if j + 1 < len(nodes) else nodes[j]
                 for j in range(0, len(nodes), 2)]
    th = hashlib.sha256(b"S256/ECDSA/batch").digest()
    seed = hashlib.sha256(th + th + nodes[0] + n.to_bytes(8, "big")).digest()
    a = [1] + [int.from_bytes(hashlib.sha256(seed + i.to_bytes(8, "big")).digest()[:16], "big") or 1 for i in range(1, n)]
    return seed, a


def ref_row(pk, dg, sig, flags):
    """(accepted by the rejection rules, -R, Q, u1, u2) of one row; the points as (x, y) integers."""
    r, s, v = be(sig[:32]), be(sig[32:64]), int(sig[64])
    ok = 0 < r < N and 0 < s < N and v < 4 and not (flags & 1 and s > N // 2)
    x = r + (N if v & 2 else 0)
    rhs = (x ** 3 + 7) % P
    y = pow(rhs, (P + 1) // 4, P)
    ok = ok and x < P and y * y % P == rhs
    if y & 1 != v & 1:
        y = P - y
    X, Y = be(pk[1:33]), be(pk[33:65])
    ok = ok and pk[0] == 4 and X < P and Y < P and (Y * Y - X ** 3 - 7) % P == 0
    if not ok:
        return False, G, G, 0, 0
    w = pow(s, -1, N)
    return True, (x, (P - y) % P), (X, Y), be(dg) % N * w % N, r * w % N


def ref_rows(pk, dg, sig, flags=0, rows=None):
    """What s256_debug_ecdsa_batch_rows returns: (seed, k (n, 2, 32), pts (n, 2, 64), sum, rejected).  With `rows`, k and
    pts are filled at those rows only (the seed and the sum always cover the whole batch)."""
    n = len(pk)
    seed, a = ref_seed_and_randomizers(pk, dg, sig)
    k, pts = np.zeros((n, 2, 32), np.uint8), np.zeros((n, 2, 64), np.uint8)
    want = set(range(n)) if rows is None else set(rows)
    total, rejected = 0, False
    for i in range(n):
        ok_i, mR, Q, u1, u2 = ref_row(pk[i], dg[i], sig[i], flags)
        if i in want:
            if ok_i:
                k[i, 0], k[i, 1] = b32(a[i]), b32(a[i] * u2 % N)
            for j, (x, y) in enumerate((mR, Q)):
                pts[i, j, :32], pts[i, j, 32:] = b32(x), b32(y)
        rejected |= not ok_i
        if ok_i:
            total += a[i] * u1
    return seed, k, pts, (total % N).to_bytes(32, "big"), rejected


def expected(oracle, pk, dg, sig, flags=0):
    """Every row recovers its key (oracle), and with flags = 1 has s <= n/2."""
    q, st = oracle.batch_ecdsa_recover(dg, sig)
    ok = (st == 1) & (q == pk).all(axis=1)
    if flags & 1:
        ok &= np.array([be(sig[i, 32:64]) <= N // 2 for i in range(len(sig))])
    return bool(ok.all())


# ---- cases ---------------------------------------------------------------------------------------------------------
_BATCHES = {}


def valid_batch(base_mult, n):
    key = (id(base_mult), n)
    if key not in _BATCHES:
        w = ps.synth.ecdsa_recoverable_batch(n, base_mult, corrupt_every=0)
        _BATCHES[key] = (w["pk65"], w["digest32"], w["sig65"])
    return tuple(x.copy() for x in _BATCHES[key])


CORRUPTIONS = ("r", "s", "digest", "v^1", "v^2", "v=4", "v=27", "v=255", "r=0", "s=n", "pk-neighbour", "pk-02",
               "pk-off-curve")


def corrupt(batch, kind, pos):
    pk, dg, sig = batch
    if kind == "r":
        sig[pos, 31] ^= 1
    elif kind == "s":
        sig[pos, 63] ^= 1
    elif kind == "digest":
        dg[pos, 0] ^= 1
    elif kind == "v^1":
        sig[pos, 64] ^= 1
    elif kind == "v^2":
        sig[pos, 64] ^= 2
    elif kind.startswith("v="):
        sig[pos, 64] = int(kind[2:])
    elif kind == "r=0":
        sig[pos, :32] = 0
    elif kind == "s=n":
        sig[pos, 32:64] = b32(N)
    elif kind == "pk-neighbour":
        pk[pos] = pk[(pos + 1) % len(pk)]
    elif kind == "pk-02":
        pk[pos, 0] = 2
    else:
        pk[pos, 64] ^= 1
    return pk, dg, sig


def high_s_batch(base_mult):
    """A valid batch whose row 16 has a high s (and the matching v): passes with flags 0, fails with flags 1."""
    pk, dg, sig = valid_batch(base_mult, 33)
    s = be(sig[16, 32:64])
    if s <= N // 2:
        sig[16, 32:64] = b32(N - s)
        sig[16, 64] ^= 1
    return pk, dg, sig


def one_key_batch(oracle, n=64):
    d = (0x1234567890ABCDEF).to_bytes(32, "big")
    pk, _ = oracle.scalar_base_mult(d)
    dg = np.stack([np.frombuffer(hashlib.sha256(b"one key %d" % i).digest(), np.uint8) for i in range(n)])
    sig = np.zeros((n, 65), np.uint8)
    for i in range(n):
        s64, rec, st = oracle.ecdsa_sign_rfc6979(d, dg[i].tobytes())
        assert st == 1
        sig[i, :64], sig[i, 64] = np.frombuffer(s64, np.uint8), rec
    return np.tile(np.frombuffer(pk, np.uint8), (n, 1)), dg, sig


def high_x_rows(oracle, n=8):
    """Valid rows with v in {2, 3}: x in [n, p) on the curve, r = x - n, s and e chosen, Q = the key they recover."""
    rows, t = [], 1
    while len(rows) < n:
        x = N + t
        t += 1
        if pow((x ** 3 + 7) % P, (P - 1) // 2, P) != 1:
            continue
        v = 2 + len(rows) % 2
        s = be(hashlib.sha256(b"high x s %d" % t).digest()) % N
        e = hashlib.sha256(b"high x e %d" % t).digest()
        sig = (x - N).to_bytes(32, "big") + s.to_bytes(32, "big") + bytes([v])
        q, st = oracle.ecdsa_recover(e, sig)
        assert st == 1
        rows.append((q, e, sig))
    return tuple(np.stack([np.frombuffer(r[j], np.uint8) for r in rows]) for j in range(3))


def cancelling_pair(base_mult, delta=12345):
    """Digests e_1 + delta s_1 and e_2 - delta s_2: D_1 = delta G = -D_2, so the unweighted sum of the rows holds."""
    pk, dg, sig = valid_batch(base_mult, 2)
    for i, sign in ((0, 1), (1, -1)):
        dg[i] = b32((be(dg[i]) + sign * delta * be(sig[i, 32:64])) % N)
    return pk, dg, sig


def wycheproof_cases():
    """(name, pk65, digest32, r||s, edge-flagged) of every Wycheproof ECDSA case"""
    H = bytes.fromhex
    return [(f"wycheproof-{c['tcId']}", np.frombuffer(H(c["pk"]), np.uint8), np.frombuffer(H(c["digest"])[:32], np.uint8),
             np.frombuffer(H(c["r"]) + H(c["s"]), np.uint8), any(f in EDGE_FLAGS for f in c["flags"]))
            for c in load_golden("wycheproof_ecdsa.json")["cases"]]


def at_row_2(base, pk, dg, sig64, v):
    bpk, bdg, bsig = (x.copy() for x in base)
    bpk[2], bdg[2], bsig[2, :64], bsig[2, 64] = pk, dg, sig64, v
    return bpk, bdg, bsig


def verdict_cases(oracle, base_mult):
    """(name, pk, dg, sig, flags) over everything the CPU and the GPU tests check (the Wycheproof pairs apart)."""
    cases = [(f"valid-{n}",) + valid_batch(base_mult, n) + (0,) for n in (1, 2, 31, 32, 33, 200)]
    for kind in CORRUPTIONS:
        for pos in (0, 16, 32):
            cases.append((f"{kind}@{pos}",) + corrupt(valid_batch(base_mult, 33), kind, pos) + (0,))
    cases += [("high-s-flags0",) + high_s_batch(base_mult) + (0,), ("high-s-flags1",) + high_s_batch(base_mult) + (1,)]
    pk, dg, sig = valid_batch(base_mult, 1)
    cases.append(("repeated-64", np.tile(pk, (64, 1)), np.tile(dg, (64, 1)), np.tile(sig, (64, 1)), 0))
    cases.append(("one-key-64",) + one_key_batch(oracle) + (0,))
    cases.append(("one-key-64-flags1",) + one_key_batch(oracle) + (1,))
    hx = high_x_rows(oracle)
    cases.append(("v23-8",) + hx + (0,))
    pk, dg, sig = valid_batch(base_mult, 33)
    pk[[3, 20]], dg[[3, 20]], sig[[3, 20]] = hx[0][:2], hx[1][:2], hx[2][:2]
    cases.append(("v23-in-33", pk, dg, sig, 0))
    pk, dg, sig = (x.copy() for x in hx)
    sig[5, 64] ^= 2
    cases.append(("v23-v^2", pk, dg, sig, 0))
    cases.append(("cancelling-pair",) + cancelling_pair(base_mult) + (0,))
    return cases


@pytest.fixture(scope="module")
def cases(oracle):
    return verdict_cases(oracle, ps.oracle_base_mult(oracle))


# ---- CPU: randomizers ----------------------------------------------------------------------------------------------
def random_rows(n, seed):
    rng = np.random.default_rng(seed)
    return tuple(rng.integers(0, 256, (n, w), dtype=np.uint8) for w in (65, 32, 65))


@pytest.mark.parametrize("n", [1, 2, 3, 5, 8, 33, 1000])
def test_randomizers_match_hashlib(n):
    rows = random_rows(n, n)
    want_seed, want_a = ref_seed_and_randomizers(*rows)
    seed, a = sim.ecdsa_batch_randomizers(*rows, chunk=1 << 19)
    assert seed == want_seed
    assert [be(a[i]) for i in range(n)] == want_a


@pytest.mark.parametrize("n", [1, 2, 3, 5, 8, 33, 1000])
def test_randomizers_do_not_depend_on_the_chunk_size(n):
    rows = random_rows(n, 7 * n)
    seed0, a0 = sim.ecdsa_batch_randomizers(*rows, chunk=1 << 19)
    chunk = 1
    while chunk <= n:
        seed, a = sim.ecdsa_batch_randomizers(*rows, chunk=chunk)
        assert seed == seed0, chunk
        assert np.array_equal(a, a0), chunk
        chunk *= 2


def test_seed_differs_from_the_bip340_seed():
    """The same leaf bytes under the two tags: only the tag tells the seeds apart."""
    pk, dg, sig = random_rows(33, 5)
    seed, _ = ref_seed_and_randomizers(pk, dg, sig)
    th = hashlib.sha256(b"S256/BIP0340/batch").digest()
    nodes = [hashlib.sha256(bytes(pk[i]) + bytes(dg[i]) + bytes(sig[i])).digest() for i in range(33)]
    while len(nodes) > 1:
        nodes = [hashlib.sha256(nodes[j] + nodes[j + 1]).digest() if j + 1 < len(nodes) else nodes[j]
                 for j in range(0, len(nodes), 2)]
    assert seed != hashlib.sha256(th + th + nodes[0] + (33).to_bytes(8, "big")).digest()
    assert sim.ecdsa_batch_randomizers(pk, dg, sig, chunk=1 << 19)[0] == seed


# ---- CPU: verdicts of the host simulation -------------------------------------------------------------------------
def test_hostsim_verdict_matches_oracle(oracle, cases):
    seen = {True: 0, False: 0}
    for name, pk, dg, sig, flags in cases:
        want = expected(oracle, pk, dg, sig, flags)
        assert sim.ecdsa_batch_verify(pk, dg, sig, flags) == want, name
        seen[want] += 1
    assert seen[True] >= 10 and seen[False] >= 40
    names = {c[0]: c for c in cases}
    assert expected(oracle, *names["high-s-flags0"][1:]) and not expected(oracle, *names["high-s-flags1"][1:])
    assert expected(oracle, *names["v23-8"][1:]) and expected(oracle, *names["v23-in-33"][1:])


def test_cancelling_pair_fools_the_unweighted_sum(oracle):
    """(u1_1 + u1_2) G + u2_1 Q_1 + u2_2 Q_2 - R_1 - R_2 = O, each row fails alone, the batch fails."""
    pk, dg, sig = cancelling_pair(ps.oracle_base_mult(oracle))
    ks, pts, u1 = [], [], 0
    for i in range(2):
        ok, mR, Q, a, b = ref_row(pk[i], dg[i], sig[i], 0)
        assert ok
        u1 += a
        ks += [b32(b).tobytes(), b32(1).tobytes()]
        pts += [bytes(pk[i]), b"\x04" + b32(mR[0]).tobytes() + b32(mR[1]).tobytes()]
    out, st = oracle.msm(b32(u1 % N).tobytes() + b"".join(ks), b"\x04" + b32(G[0]).tobytes() + b32(G[1]).tobytes() + b"".join(pts))
    assert st == 2  # the identity
    assert not expected(oracle, pk[:1], dg[:1], sig[:1]) and not expected(oracle, pk[1:], dg[1:], sig[1:])
    assert not sim.ecdsa_batch_verify(pk, dg, sig)


@pytest.fixture(scope="module")
def wycheproof_pairs(oracle):
    """(name, batch, want) for every (edge-flagged Wycheproof case, v) at row 2 of a valid 5-row batch"""
    base = valid_batch(ps.oracle_base_mult(oracle), 5)
    out = []
    for name, pk, dg, sig64, edge in wycheproof_cases():
        if not edge:
            continue
        for v in range(4):
            b = at_row_2(base, pk, dg, sig64, v)
            out.append((f"{name}-v{v}", b, expected(oracle, b[0][2:3], b[1][2:3], b[2][2:3])))
    return out


def test_hostsim_wycheproof_pairs(wycheproof_pairs):
    assert len(wycheproof_pairs) == 4 * 399
    assert sum(w for _, _, w in wycheproof_pairs) >= 300
    for name, b, want in wycheproof_pairs:
        assert sim.ecdsa_batch_verify(*b, chunk=8) == want, name


def test_hostsim_chunked_verdict(oracle):
    pk, dg, sig = valid_batch(ps.oracle_base_mult(oracle), 33)
    for chunk in (1, 4, 16, 32):
        assert sim.ecdsa_batch_verify(pk, dg, sig, chunk=chunk), chunk
        bad = corrupt((pk.copy(), dg.copy(), sig.copy()), "s", 32)
        assert not sim.ecdsa_batch_verify(*bad, chunk=chunk), chunk


@pytest.mark.parametrize("k", [1, 4, 32])
def test_hostsim_rows_match_reference(oracle, k):
    """The simulated kernels' rows against the Python reference, with inversion groups of k rows at n = 70 (partial and
    empty groups) and rejected rows at group edges."""
    pk, dg, sig = valid_batch(ps.oracle_base_mult(oracle), 200)
    pk, dg, sig = pk[:70].copy(), dg[:70].copy(), sig[:70].copy()
    stride = (70 + k - 1) // k
    for pos, kind in ((0, "r=0"), (stride - 1, "s=n"), (min(stride, 69), "v=4"), (69, "pk-off-curve")):
        corrupt((pk, dg, sig), kind, pos)
    for flags in (0, 1):
        got = sim.ecdsa_batch_rows(pk, dg, sig, flags, chunk=32, k=k)
        want = ref_rows(pk, dg, sig, flags)
        assert got[0] == want[0]
        assert np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2])
        assert got[3] == want[3] and got[4] == want[4] is True and got[5] is False


MIRROR_SRC = os.path.join(ROOT, "tests", "cpp", "ecdsa_batch_mirror.cpp")
MIRROR_EXE = os.path.join(ROOT, "tests", "cpp", "_build", "ecdsa_batch_mirror")


def build_mirror(s256):
    s256.load_library()
    libdir = os.path.dirname(s256.library_path())
    os.makedirs(os.path.dirname(MIRROR_EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-o", MIRROR_EXE, MIRROR_SRC, "-L", libdir, "-lsecp256k1_b200",
                           f"-Wl,-rpath,{libdir}"])
    return MIRROR_EXE


def test_mirror_compiles_and_links(s256):
    assert os.path.exists(build_mirror(s256))


# ---- GPU: the same through the C ABI -------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_verdict_matches_oracle(engine, oracle, cases):
    for name, pk, dg, sig, flags in cases:
        assert engine.ecdsa_recoverable_batch_verify(pk, dg, sig, flags) == expected(oracle, pk, dg, sig, flags), name


@pytest.mark.gpu
def test_gpu_wycheproof_every_case_and_recovery_id(engine, oracle):
    base = valid_batch(ps.oracle_base_mult(oracle), 5)
    seen = 0
    for name, pk, dg, sig64, _ in wycheproof_cases():
        for v in range(4):
            b = at_row_2(base, pk, dg, sig64, v)
            want = expected(oracle, b[0][2:3], b[1][2:3], b[2][2:3])
            assert engine.ecdsa_recoverable_batch_verify(*b) == want, (name, v)
            seen += 1
    assert seen == 4 * 432


@pytest.mark.gpu
def test_gpu_empty_batch_and_misuse(engine, s256):
    assert engine.ecdsa_recoverable_batch_verify(np.zeros((0, 65), np.uint8), np.zeros((0, 32), np.uint8),
                                                 np.zeros((0, 65), np.uint8))
    lib, ctx = engine._lib, engine._ctx
    buf = (C.c_uint8 * 65)()
    ok = C.c_uint8(7)
    f, one = C.c_uint32(0), C.c_size_t(1)
    assert lib.s256_ecdsa_recoverable_batch_verify(ctx, None, buf, buf, f, one, C.byref(ok)) == -3
    assert lib.s256_ecdsa_recoverable_batch_verify(ctx, buf, None, buf, f, one, C.byref(ok)) == -3
    assert lib.s256_ecdsa_recoverable_batch_verify(ctx, buf, buf, None, f, one, C.byref(ok)) == -3
    assert lib.s256_ecdsa_recoverable_batch_verify(ctx, buf, buf, buf, f, one, None) == -3
    assert lib.s256_ecdsa_recoverable_batch_verify(None, buf, buf, buf, f, one, C.byref(ok)) == -3
    assert lib.s256_ecdsa_recoverable_batch_verify_dev(ctx, None, None, None, f, one, None, None) == -3
    assert lib.s256_ecdsa_recoverable_batch_verify_dev(None, buf, buf, buf, f, one, C.byref(ok), None) == -3
    assert lib.s256_debug_ecdsa_batch_rows(ctx, buf, buf, buf, f, C.c_size_t(0), buf, buf, buf, buf, C.byref(ok)) == -3
    assert ok.value == 7
    tiny = s256.Engine(max_batch=1)
    try:
        assert tiny._lib.s256_ecdsa_recoverable_batch_verify(tiny._ctx, buf, buf, buf, f, one, C.byref(ok)) == -3
        assert ok.value == 7
    finally:
        tiny.close()
    with pytest.raises(ValueError):
        engine.ecdsa_recoverable_batch_verify(np.zeros((3, 65), np.uint8), np.zeros((3, 32), np.uint8),
                                              np.zeros((2, 65), np.uint8))
    import torch
    d = torch.zeros(0, dtype=torch.uint8, device="cuda")
    assert engine.ecdsa_recoverable_batch_verify(d, d, d).item() == 1


@pytest.mark.gpu
def test_gpu_dev_form_matches_host_form(engine, oracle, cases):
    import torch

    def at_offset(a, off):  # a device copy starting `off` bytes into a larger buffer
        flat = torch.from_numpy(np.ascontiguousarray(a).reshape(-1))
        buf = torch.zeros(flat.numel() + off, dtype=torch.uint8, device="cuda")
        buf[off:] = flat.cuda()
        return buf[off:]

    for off in (0, 1, 3):
        for name, pk, dg, sig, flags in cases[::3]:
            got = engine.ecdsa_recoverable_batch_verify(at_offset(pk, off), at_offset(dg, off), at_offset(sig, off), flags)
            assert bool(got.item()) == engine.ecdsa_recoverable_batch_verify(pk, dg, sig, flags), (name, off)


@pytest.mark.gpu
def test_gpu_chunked_equals_default_engine(engine, s256, oracle):
    small = s256.Engine(max_batch=4096)  # chunks of 2048 rows
    try:
        n = 3 * 2048 + 5
        rows = valid_batch(engine.scalar_base_mult, n)
        assert small.ecdsa_recoverable_batch_verify(*rows) and engine.ecdsa_recoverable_batch_verify(*rows)
        for pos in (0, 2047, 2048, 4095, 4096, 6143, 6144, n - 1):
            bad = corrupt(tuple(x.copy() for x in rows), "s", pos)
            got = small.ecdsa_recoverable_batch_verify(*bad)
            assert got == engine.ecdsa_recoverable_batch_verify(*bad) == expected(oracle, *[x[pos:pos + 1] for x in bad]) == False, pos
    finally:
        small.close()


@pytest.mark.gpu
def test_gpu_full_size(engine):
    import torch
    pk, dg, sig = valid_batch(engine.scalar_base_mult, 1 << 20)
    assert engine.ecdsa_recoverable_batch_verify(pk, dg, sig)
    bad = sig.copy()
    bad[777_777, 40] ^= 4
    assert not engine.ecdsa_recoverable_batch_verify(pk, dg, bad)
    d = [torch.from_numpy(x).cuda() for x in (pk, dg, sig)]
    assert engine.ecdsa_recoverable_batch_verify(*d).item() == 1
    d[2] = torch.from_numpy(bad).cuda()
    assert engine.ecdsa_recoverable_batch_verify(*d).item() == 0


@pytest.mark.gpu
def test_gpu_side_stream_after_other_dev_call(engine, oracle):
    """A batch verification on a side stream right after a _dev call of another entry point on the same context."""
    import torch
    pk, dg, sig = valid_batch(ps.oracle_base_mult(oracle), 200)
    d_pk, d_dg, d_sig = (torch.from_numpy(x).cuda() for x in (pk, dg, sig))
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for _ in range(3):
        q, st = engine.ecdsa_recover(d_dg, d_sig)
        with torch.cuda.stream(side):
            ok = engine.ecdsa_recoverable_batch_verify(d_pk, d_dg, d_sig)
        side.synchronize()
        assert ok.item() == 1
        torch.cuda.synchronize()
        assert bool((st == 1).all()) and bool((q == d_pk).all())


def _check_rows(eng, pk, dg, sig, flags, rows=None):
    got = eng.debug_ecdsa_batch_rows(pk, dg, sig, flags)
    want = ref_rows(pk, dg, sig, flags, rows)
    sel = slice(None) if rows is None else sorted(set(rows))
    assert got[0] == want[0]
    assert got[3] == want[3] and got[4] == want[4]
    for j in (1, 2):
        bad = np.nonzero((got[j][sel] != want[j][sel]).any(axis=(1, 2)))[0]
        assert len(bad) == 0, (j, np.arange(len(pk))[sel][bad][:5].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 257])
def test_gpu_rows_at_cta_edges(engine, oracle, n):
    pk, dg, sig = valid_batch(ps.oracle_base_mult(oracle), 257)
    pk, dg, sig = pk[:n].copy(), dg[:n].copy(), sig[:n].copy()
    if n > 2:
        corrupt((pk, dg, sig), "r=0", n - 2)
    for flags in (0, 1):
        _check_rows(engine, pk, dg, sig, flags)


def group_edges(c, k):
    """Rows at the edges of the K-row inversion groups of a chunk of c rows (thread t holds rows t + m * stride)."""
    stride = (c + k - 1) // k
    rows = set()
    for m in range(k):
        for t in (0, 1, TPB - 1, TPB, stride - 2, stride - 1):
            if 0 <= t < stride and t + m * stride < c:
                rows.add(t + m * stride)
    return sorted(rows | {c - 1})


@pytest.mark.gpu
@pytest.mark.parametrize("n,k", [(65541, 4), ((1 << 19) + 3, 32)])
def test_gpu_rows_at_inversion_group_edges(engine, n, k):
    """Chunks of 65536 + 5 rows (K = 4) and 2^19 + 3 rows (one chunk of 2^19, K = 32, and one of 3, K = 1) with rejected
    rows planted at group edges: every edge row, its group neighbours and the sum must match the reference."""
    pk, dg, sig = valid_batch(engine.scalar_base_mult, n)
    c = min(n, 1 << 19)
    edges = group_edges(c, k)
    stride = (c + k - 1) // k
    for j, pos in enumerate([0, stride - 1, stride, 2 * stride + 1, c - 1]):
        corrupt((pk, dg, sig), ("r=0", "s=n", "v=4", "pk-off-curve", "r=0")[j], pos)
    _check_rows(engine, pk, dg, sig, 0, rows=edges + list(range(c, n)))


@pytest.mark.gpu
def test_gpu_rows_at_chunk_edges(engine, s256, oracle):
    small = s256.Engine(max_batch=4096)  # chunks of 2048 rows
    try:
        n = 2 * 2048 + 130
        pk, dg, sig = valid_batch(engine.scalar_base_mult, n)
        corrupt((pk, dg, sig), "s=n", 2048)
        _check_rows(small, pk, dg, sig, 0)
        pk, dg, sig = valid_batch(engine.scalar_base_mult, n)
        got_small, got_big = small.debug_ecdsa_batch_rows(pk, dg, sig), engine.debug_ecdsa_batch_rows(pk, dg, sig)
        assert got_small[0] == got_big[0] and got_small[3] == got_big[3]
        assert np.array_equal(got_small[1], got_big[1]) and np.array_equal(got_small[2], got_big[2])
    finally:
        small.close()


@pytest.mark.gpu
def test_gpu_mirror_accepts_valid_and_rejects_corrupted(s256, oracle):
    exe = build_mirror(s256)
    pk, dg, sig = one_key_batch(oracle, 8)
    args = [x for i in range(8) for x in (pk[i].tobytes().hex(), dg[i].tobytes().hex(), sig[i].tobytes().hex())]
    r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "ecdsa batch mirror ok" in r.stdout
