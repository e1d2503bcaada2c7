"""BIP-340 over messages of different lengths in one call (s256_schnorr_verify_varlen, s256_schnorr_batch_verify_varlen,
s256_schnorr_sign_varlen): the kernels' item functions with the offsets accessor on the CPU against the oracle and
hashlib, then the same cases through the C ABI on the GPU, host and device forms, against the uniform entry points."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from hostsim import batch as batch_sim
from hostsim import varlen as vsim

N = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
P = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEFFFFFC2F
EDGE_LENS = [0, 1, 31, 32, 33, 55, 56, 63, 64, 65, 119, 120, 127, 128, 129, 1000]


def ragged(msgs):
    offs = np.zeros(len(msgs) + 1, np.uint64)
    offs[1:] = np.cumsum([len(m) for m in msgs]) if msgs else []
    return np.frombuffer(b"".join(bytes(m) for m in msgs), np.uint8).copy(), offs


def tagged(tag, data):
    t = hashlib.sha256(tag).digest()
    return hashlib.sha256(t + t + data).digest()


# ---- the randomizer definition (DESIGN.md section 8), restated with hashlib ------------------------------------------
def ref_seed_and_randomizers(pkx, msgs, sig):
    n = len(pkx)
    nodes = [hashlib.sha256(bytes(pkx[i]) + bytes(sig[i]) + bytes(msgs[i])).digest() for i in range(n)]
    while len(nodes) > 1:
        nodes = [hashlib.sha256(nodes[j] + nodes[j + 1]).digest() if j + 1 < len(nodes) else nodes[j]
                 for j in range(0, len(nodes), 2)]
    th = hashlib.sha256(b"S256/BIP0340/batch").digest()
    seed = hashlib.sha256(th + th + nodes[0] + n.to_bytes(8, "big")).digest()
    a = [1] + [int.from_bytes(hashlib.sha256(seed + i.to_bytes(8, "big")).digest()[:16], "big") or 1 for i in range(1, n)]
    return seed, a


def mixed_lens(n, seed):
    rng = np.random.default_rng(seed)
    return [EDGE_LENS[i] if i < len(EDGE_LENS) else int(rng.integers(0, 301)) for i in range(n)]


def signed_rows(oracle, lens, seed, keys=None):
    """(pkx (n, 32), msgs list of bytes, sig (n, 64), priv (n, 32), aux (n, 32)): valid BIP-340 rows from the oracle."""
    rng = np.random.default_rng(seed)
    n = len(lens)
    keys = keys or n
    priv = [((int.from_bytes(rng.bytes(32), "big") % (N - 1)) + 1).to_bytes(32, "big") for _ in range(keys)]
    pub = [bytes(oracle.scalar_base_mult(d)[0])[1:33] for d in priv]
    pkx, msgs, sig, pv, aux = [], [], [], [], []
    for i, ln in enumerate(lens):
        d, m, ax = priv[i % keys], rng.bytes(ln), rng.bytes(32)
        s, st = oracle.schnorr_sign(d, m, ax)
        assert st == 1
        pkx.append(pub[i % keys]); msgs.append(m); sig.append(s); pv.append(d); aux.append(ax)
    rows = lambda xs, w: np.frombuffer(b"".join(xs), np.uint8).reshape(n, w).copy()
    return rows(pkx, 32), msgs, rows(sig, 64), rows(pv, 32), rows(aux, 32)


def corrupt(pkx, msgs, sig, kind, pos):
    pkx, msgs, sig = pkx.copy(), list(msgs), sig.copy()
    if kind == "r":
        sig[pos, 31] ^= 1
    elif kind == "s":
        sig[pos, 63] ^= 1
    elif kind == "msg":
        msgs[pos] = bytes([msgs[pos][0] ^ 1]) + msgs[pos][1:] if msgs[pos] else b"\x00"
    else:
        pkx[pos] = pkx[(pos + 1) % len(pkx)]
    return pkx, msgs, sig


def oracle_ok(oracle, pkx, msgs, sig):
    return np.array([oracle.schnorr_verify(pkx[i].tobytes(), msgs[i], sig[i].tobytes()) for i in range(len(pkx))], np.uint8)


def golden_rows():
    rows = load_golden("bip340.json")["rows"]
    H = bytes.fromhex
    pkx = np.stack([np.frombuffer(H(r["pk"]), np.uint8) for r in rows])
    sig = np.stack([np.frombuffer(H(r["sig"]), np.uint8) for r in rows])
    return rows, pkx, [H(r["msg"]) for r in rows], sig


# ---- CPU: the item functions with the offsets accessor ----------------------------------------------------------------
def test_all_bip340_vectors_in_one_call():
    rows, pkx, msgs, sig = golden_rows()
    assert len(rows) == 19 and {len(m) for m in msgs} == {0, 1, 17, 32, 100}
    ok = vsim.schnorr_verify(pkx, ragged(msgs), sig)
    assert ok.tolist() == [int(r["valid"]) for r in rows]


def test_sign_vectors_in_one_call():
    rows = [r for r in load_golden("bip340.json")["rows"] if r["sk"]]
    assert [r["index"] for r in rows] == [0, 1, 2, 3, 15, 16, 17, 18]
    H = bytes.fromhex
    priv = np.stack([np.frombuffer(H(r["sk"]), np.uint8) for r in rows])
    aux = np.stack([np.frombuffer(H(r["aux"]), np.uint8) for r in rows])
    sig, st = vsim.schnorr_sign(priv, ragged([H(r["msg"]) for r in rows]), aux)
    assert st.tolist() == [1] * len(rows)
    assert [s.tobytes().hex().upper() for s in sig] == [r["sig"].upper() for r in rows]


@pytest.fixture(scope="module")
def mixed(oracle):
    return signed_rows(oracle, mixed_lens(48, 7), 7)


def test_mixed_lengths_match_oracle(oracle, mixed):
    pkx, msgs, sig, priv, aux = mixed
    cases = [(pkx, msgs, sig)]
    for kind, pos in (("r", 3), ("s", 12), ("msg", 20), ("pk", 40), ("msg", 0)):
        cases.append(corrupt(pkx, msgs, sig, kind, pos))
    for p, m, s in cases:
        want = oracle_ok(oracle, p, m, s)
        assert np.array_equal(vsim.schnorr_verify(p, ragged(m), s), want)
    assert oracle_ok(oracle, *cases[0]).all() and not oracle_ok(oracle, *cases[1]).all()
    got, st = vsim.schnorr_sign(priv, ragged(msgs), aux)
    assert st.all() and np.array_equal(got, sig)


@pytest.mark.parametrize("n", [1, 2, 5, 33, 100])
def test_randomizers_match_hashlib_for_every_chunk_size(n):
    rng = np.random.default_rng(n)
    lens = mixed_lens(n, n)
    pkx, sig = rng.integers(0, 256, (n, 32), dtype=np.uint8), rng.integers(0, 256, (n, 64), dtype=np.uint8)
    msgs = [rng.bytes(ln) for ln in lens]
    want_seed, want_a = ref_seed_and_randomizers(pkx, msgs, sig)
    chunk = 1
    while chunk <= 2 * n:
        seed, a = vsim.schnorr_batch_randomizers(pkx, ragged(msgs), sig, chunk)
        assert seed == want_seed, chunk
        assert [int.from_bytes(a[i].tobytes(), "big") for i in range(n)] == want_a, chunk
        chunk *= 2


@pytest.mark.parametrize("msg_len", [0, 1, 32, 100])
def test_equal_lengths_give_the_uniform_seed(msg_len):
    rng = np.random.default_rng(msg_len)
    n = 37
    pkx, msg, sig = (rng.integers(0, 256, (n, 32), dtype=np.uint8), rng.integers(0, 256, (n, msg_len), dtype=np.uint8),
                     rng.integers(0, 256, (n, 64), dtype=np.uint8))
    for chunk in (4, 1 << 19):
        assert vsim.schnorr_batch_randomizers(pkx, ragged(list(msg)), sig, chunk)[0] == \
            batch_sim.schnorr_batch_randomizers(pkx, msg, sig, chunk)[0]


def verdict_cases(oracle, mixed):
    pkx, msgs, sig, _, _ = mixed
    cases = [("valid", pkx, msgs, sig)]
    for kind in ("r", "s", "msg", "pk"):
        for pos in (0, len(pkx) // 2, len(pkx) - 1):
            cases.append((f"{kind}@{pos}",) + corrupt(pkx, msgs, sig, kind, pos))
    p2, m2, s2, _, _ = signed_rows(oracle, [0, 77], 11)
    s1, s2_ = (int.from_bytes(s2[i, 32:].tobytes(), "big") for i in (0, 1))
    s2 = s2.copy()
    s2[0, 32:] = np.frombuffer(((s1 + 1) % N).to_bytes(32, "big"), np.uint8)
    s2[1, 32:] = np.frombuffer(((s2_ - 1) % N).to_bytes(32, "big"), np.uint8)
    cases.append(("cancelling-pair", p2, m2, s2))
    cases.append(("one-key",) + signed_rows(oracle, mixed_lens(24, 5), 5, keys=1)[:3])
    cases.append(("empty-messages",) + signed_rows(oracle, [0] * 9, 9)[:3])
    rows, gp, gm, gs = golden_rows()
    good = [i for i, r in enumerate(rows) if r["valid"]]
    cases.append(("golden-valid", gp[good], [gm[i] for i in good], gs[good]))
    return cases


@pytest.fixture(scope="module")
def cases(oracle, mixed):
    return verdict_cases(oracle, mixed)


def test_batch_verdict_matches_oracle(oracle, cases):
    seen = set()
    for name, pkx, msgs, sig in cases:
        want = bool(oracle_ok(oracle, pkx, msgs, sig).all())
        assert vsim.schnorr_batch_verify(pkx, ragged(msgs), sig) == want, name
        assert vsim.schnorr_batch_verify(pkx, ragged(msgs), sig, chunk=4) == want, name
        seen.add(want)
    assert seen == {True, False}


def decreasing_at(offs, i):
    bad = offs.copy()
    assert bad[i] > 0
    bad[i + 1] = bad[i] - 1
    return bad


def test_decreasing_offsets_make_only_that_row_invalid(mixed):
    """The _dev forms' rule: a row with offsets[i+1] < offsets[i] is invalid and none of its bytes is read."""
    pkx, msgs, sig, priv, aux = mixed
    flat, offs = ragged(msgs)
    bad = decreasing_at(offs, 5)
    ok = vsim.schnorr_verify(pkx, (flat, bad), sig)
    assert ok[5] == 0 and ok[6] == 0 and ok.sum() == len(pkx) - 2  # row 6 now starts one byte early
    assert not vsim.schnorr_batch_verify(pkx, (flat, bad), sig)
    s, st = vsim.schnorr_sign(priv, (flat, bad), aux)
    assert st[5] == 0 and not s[5].any() and st.sum() == len(pkx) - 1


def test_mirror_compiles_and_links(s256):
    assert os.path.exists(build_mirror(s256))


# ---- GPU ---------------------------------------------------------------------------------------------------------------
MIRROR_SRC = os.path.join(ROOT, "tests", "cpp", "schnorr_varlen_mirror.cpp")
MIRROR_EXE = os.path.join(ROOT, "tests", "cpp", "_build", "schnorr_varlen_mirror")


def build_mirror(s256):
    s256.load_library()
    libdir = os.path.dirname(s256.library_path())
    os.makedirs(os.path.dirname(MIRROR_EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-o", MIRROR_EXE, MIRROR_SRC, "-L", libdir, "-lsecp256k1_b200",
                           f"-Wl,-rpath,{libdir}"])
    return MIRROR_EXE


def dev(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def dev_ragged(msgs, off=0):
    """The device form of the rows, the bytes starting `off` bytes into a larger buffer."""
    import torch
    flat, offs = ragged(msgs)
    buf = torch.zeros(flat.size + off + 1, dtype=torch.uint8, device="cuda")
    if flat.size:
        buf[off:off + flat.size] = torch.from_numpy(flat).cuda()
    return buf[off:], torch.from_numpy(offs.astype(np.int64)).cuda()


@pytest.mark.gpu
def test_gpu_bip340_vectors_and_cases_match_oracle(engine, oracle, cases):
    rows, pkx, msgs, sig = golden_rows()
    want = np.array([int(r["valid"]) for r in rows], np.uint8)
    assert np.array_equal(engine.schnorr_verify_varlen(pkx, msgs, sig), want)
    assert np.array_equal(engine.schnorr_verify_varlen(dev(pkx), dev_ragged(msgs), dev(sig)).cpu().numpy(), want)
    for name, p, m, s in cases:
        want = oracle_ok(oracle, p, m, s)
        assert np.array_equal(engine.schnorr_verify_varlen(p, m, s), want), name
        assert np.array_equal(engine.schnorr_verify_varlen(dev(p), dev_ragged(m), dev(s)).cpu().numpy(), want), name
        assert engine.schnorr_batch_verify_varlen(p, m, s) == bool(want.all()), name
        assert engine.schnorr_batch_verify_varlen(dev(p), dev_ragged(m), dev(s)).item() == int(want.all()), name


@pytest.mark.gpu
def test_gpu_sign_vectors_and_mixed(engine, mixed):
    rows = [r for r in load_golden("bip340.json")["rows"] if r["sk"]]
    H = bytes.fromhex
    priv = np.stack([np.frombuffer(H(r["sk"]), np.uint8) for r in rows])
    aux = np.stack([np.frombuffer(H(r["aux"]), np.uint8) for r in rows])
    msgs = [H(r["msg"]) for r in rows]
    sig, st = engine.schnorr_sign_varlen(priv, msgs, aux)
    assert st.all() and [s.tobytes().hex().upper() for s in sig] == [r["sig"].upper() for r in rows]
    pkx, msgs, sig, priv, aux = mixed
    for got, st in (engine.schnorr_sign_varlen(priv, msgs, aux), engine.schnorr_sign_varlen(dev(priv), dev_ragged(msgs, 3), dev(aux))):
        assert np.array_equal(np.asarray(got.cpu() if hasattr(got, "cpu") else got), sig)
        assert np.asarray(st.cpu() if hasattr(st, "cpu") else st).all()


@pytest.mark.gpu
@pytest.mark.parametrize("msg_len", [0, 1, 32, 100])
def test_gpu_equal_lengths_match_uniform_entry_points(engine, oracle, msg_len):
    """Ragged rows that all have length L give byte for byte what the uniform calls give with msg_len = L."""
    pkx, msgs, sig, priv, aux = signed_rows(oracle, [msg_len] * 300, msg_len)
    pkx, msgs, sig = corrupt(pkx, msgs, sig, "s", 130)
    msg = np.frombuffer(b"".join(msgs), np.uint8).reshape(300, msg_len)
    assert np.array_equal(engine.schnorr_verify_varlen(pkx, msgs, sig), engine.schnorr_verify(pkx, msg, sig))
    assert np.array_equal(engine.schnorr_verify_varlen(dev(pkx), dev_ragged(msgs, 1), dev(sig)).cpu(),
                          engine.schnorr_verify(dev(pkx), dev(msg), dev(sig)).cpu())
    for p, s in ((pkx, sig), (pkx[:130], sig[:130])):
        k = len(p)
        assert engine.schnorr_batch_verify_varlen(p, msgs[:k], s) == engine.schnorr_batch_verify(p, msg[:k], s) == (k == 130)
        assert engine.schnorr_batch_verify_varlen(dev(p), dev_ragged(msgs[:k]), dev(s)).item() == (k == 130)
    got = engine.schnorr_sign_varlen(priv, msgs, aux)
    want = engine.schnorr_sign(priv, msg, aux)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and want[1].all()
    gd = engine.schnorr_sign_varlen(dev(priv), dev_ragged(msgs, 5), dev(aux))
    assert np.array_equal(gd[0].cpu().numpy(), want[0]) and np.array_equal(gd[1].cpu().numpy(), want[1])
    a, b = engine.debug_schnorr_batch_rows_varlen(pkx, msgs, sig), engine.debug_schnorr_batch_rows(pkx, msg, sig)
    assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and a[3] == b[3] and a[4] == b[4]


def lift_x(x):
    c = (pow(x, 3, P) + 7) % P
    y = pow(c, (P + 1) // 4, P)
    assert y * y % P == c
    return y if y % 2 == 0 else P - y


@pytest.mark.gpu
def test_gpu_debug_rows_match_python_reference_across_chunks(s256, oracle):
    """seed, a_i, a_i e_i, -R_i, -P_i and sum a_i s_i at the CTA (128 rows) and chunk (128 rows at max_batch 512) edges:
    the chunks cut through the ragged byte ranges."""
    small = s256.Engine(max_batch=512)
    try:
        n = 3 * 128 + 5
        pkx, msgs, sig, _, _ = signed_rows(oracle, mixed_lens(n, 21), 21, keys=17)
        seed, k, pts, ssum, rej = small.debug_schnorr_batch_rows_varlen(pkx, msgs, sig)
        want_seed, a = ref_seed_and_randomizers(pkx, msgs, sig)
        assert seed == want_seed and not rej
        total = 0
        for i in sorted({0, 1, 126, 127, 128, 129, 255, 256, 383, 384, n - 1} | set(range(0, n, 37))):
            r, px, s = sig[i, :32].tobytes(), pkx[i].tobytes(), int.from_bytes(sig[i, 32:].tobytes(), "big")
            e = int.from_bytes(tagged(b"BIP0340/challenge", r + px + msgs[i]), "big") % N
            assert int.from_bytes(k[i, 0].tobytes(), "big") == a[i], i
            assert int.from_bytes(k[i, 1].tobytes(), "big") == a[i] * e % N, i
            for j, x in ((0, int.from_bytes(r, "big")), (1, int.from_bytes(px, "big"))):
                assert pts[i, j].tobytes() == x.to_bytes(32, "big") + (P - lift_x(x)).to_bytes(32, "big"), (i, j)
        for i in range(n):
            total += a[i] * int.from_bytes(sig[i, 32:].tobytes(), "big")
        assert ssum == (total % N).to_bytes(32, "big")
        assert small.schnorr_batch_verify_varlen(pkx, msgs, sig)
        assert small.schnorr_verify_varlen(pkx, msgs, sig).all()
        bad = corrupt(pkx, msgs, sig, "msg", 300)
        assert not small.schnorr_batch_verify_varlen(*bad)
        assert small.schnorr_verify_varlen(*bad).tolist() == [int(i != 300) for i in range(n)]
    finally:
        small.close()


@pytest.mark.gpu
def test_gpu_one_mib_message_among_short_ones(engine, oracle):
    lens = [0, 33, 1 << 20] + [int(x) for x in np.random.default_rng(3).integers(0, 100, 61)]
    pkx, msgs, sig, priv, aux = signed_rows(oracle, lens, 3, keys=4)
    assert engine.schnorr_verify_varlen(pkx, msgs, sig).all()
    assert engine.schnorr_verify_varlen(dev(pkx), dev_ragged(msgs, 7), dev(sig)).cpu().numpy().all()
    assert engine.schnorr_batch_verify_varlen(pkx, msgs, sig)
    got, st = engine.schnorr_sign_varlen(priv, msgs, aux)
    assert st.all() and np.array_equal(got, sig)
    assert not engine.schnorr_batch_verify_varlen(*corrupt(pkx, msgs, sig, "msg", 2))


@pytest.mark.gpu
def test_gpu_dev_decreasing_offsets(engine, mixed):
    import torch
    pkx, msgs, sig, priv, aux = mixed
    flat, offs = ragged(msgs)
    bad = torch.from_numpy(decreasing_at(offs, 5).astype(np.int64)).cuda()
    dflat = dev(flat)
    ok = engine.schnorr_verify_varlen(dev(pkx), (dflat, bad), dev(sig)).cpu().numpy()
    assert ok[5] == 0 and ok[6] == 0 and ok.sum() == len(pkx) - 2
    assert engine.schnorr_batch_verify_varlen(dev(pkx), (dflat, bad), dev(sig)).item() == 0
    s, st = engine.schnorr_sign_varlen(dev(priv), (dflat, bad), dev(aux))
    s, st = s.cpu().numpy(), st.cpu().numpy()
    assert st[5] == 0 and not s[5].any() and st.sum() == len(pkx) - 1
    keep = [i for i in range(len(pkx)) if i not in (5, 6)]
    assert np.array_equal(s[keep], sig[keep])
    # the host forms refuse the same offsets before enqueueing anything
    lib, ctx = engine._lib, engine._ctx
    hp = lambda a: a.ctypes.data_as(C.c_void_p)
    hbad, out = decreasing_at(offs, 5), np.full(len(pkx), 7, np.uint8)
    okb = C.c_uint8(7)
    n = C.c_size_t(len(pkx))
    assert lib.s256_schnorr_verify_varlen(ctx, hp(pkx), hp(flat), hp(hbad), hp(sig), n, hp(out)) == -3
    assert lib.s256_schnorr_batch_verify_varlen(ctx, hp(pkx), hp(flat), hp(hbad), hp(sig), n, C.byref(okb)) == -3
    sg = np.zeros((len(pkx), 64), np.uint8)
    assert lib.s256_schnorr_sign_varlen(ctx, hp(priv), hp(flat), hp(hbad), hp(aux), n, hp(sg), hp(out)) == -3
    assert (out == 7).all() and okb.value == 7


@pytest.mark.gpu
def test_gpu_empty_null_and_side_stream(engine, mixed):
    import torch
    lib, ctx = engine._lib, engine._ctx
    z = np.zeros((0, 32), np.uint8)
    assert engine.schnorr_verify_varlen(z, [], np.zeros((0, 64), np.uint8)).size == 0
    assert engine.schnorr_batch_verify_varlen(z, [], np.zeros((0, 64), np.uint8))
    assert engine.schnorr_sign_varlen(z, [], z)[1].size == 0
    d0, o0 = torch.zeros(0, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda")
    assert engine.schnorr_batch_verify_varlen(d0, (d0, o0), d0).item() == 1
    buf = (C.c_uint8 * 128)()
    offs = (C.c_size_t * 2)(0, 32)
    one, okb = C.c_size_t(1), C.c_uint8(7)
    for f in (lib.s256_schnorr_verify_varlen, lib.s256_schnorr_batch_verify_varlen):
        assert f(ctx, None, buf, offs, buf, one, buf) == -3
        assert f(ctx, buf, None, offs, buf, one, buf) == -3  # a non-empty row needs bytes
        assert f(ctx, buf, buf, None, buf, one, buf) == -3
        assert f(ctx, buf, buf, offs, None, one, buf) == -3
        assert f(ctx, buf, buf, offs, buf, one, None) == -3
        assert f(None, buf, buf, offs, buf, one, buf) == -3
    assert lib.s256_schnorr_sign_varlen(ctx, buf, buf, None, buf, one, buf, buf) == -3
    assert lib.s256_schnorr_verify_varlen_dev(ctx, None, None, None, None, one, None, None) == -3
    assert lib.s256_schnorr_batch_verify_varlen_dev(ctx, None, None, None, None, one, None, None) == -3
    assert lib.s256_schnorr_sign_varlen_dev(ctx, None, None, None, None, one, None, None, None) == -3
    assert lib.s256_debug_schnorr_batch_rows_varlen(ctx, buf, buf, offs, buf, C.c_size_t(0), buf, buf, buf, buf, buf) == -3
    empty = (C.c_size_t * 2)(5, 5)  # one empty row: msg may be NULL on the host
    assert lib.s256_schnorr_verify_varlen(ctx, buf, None, empty, buf, one, buf) == 0
    pkx, msgs, sig, _, _ = mixed
    d_pkx, d_msg, d_sig = dev(pkx), dev_ragged(msgs, 1), dev(sig)
    k = torch.from_numpy(np.frombuffer(hashlib.sha256(b"k").digest() * 4096, np.uint8).copy()).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for _ in range(3):
        engine.scalar_base_mult(k)
        ok_items = engine.schnorr_verify_varlen(d_pkx, d_msg, d_sig)
        with torch.cuda.stream(side):
            ok = engine.schnorr_batch_verify_varlen(d_pkx, d_msg, d_sig)
        side.synchronize()
        assert ok.item() == 1
        torch.cuda.synchronize()
        assert bool(ok_items.all())


@pytest.mark.gpu
def test_gpu_full_size_round_trip(engine):
    import torch
    n = 1 << 20
    rng = np.random.default_rng(20)
    lens = rng.integers(0, 301, n)
    lens[:len(EDGE_LENS)] = EDGE_LENS
    offs = np.zeros(n + 1, np.uint64)
    np.cumsum(lens, out=offs[1:])
    flat = rng.integers(0, 256, int(offs[-1]), dtype=np.uint8)
    priv = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    priv[:, 0] &= 0x7F  # below n
    priv[:, 31] |= 1    # not zero
    aux = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    msgs = [flat[offs[i]:offs[i + 1]] for i in range(n)]
    sig, st = engine.schnorr_sign_varlen(priv, msgs, aux)
    sig = np.array(sig)
    assert st.all()
    pub, pst = engine.scalar_base_mult(priv)
    pkx = np.ascontiguousarray(np.asarray(pub)[:, 1:33])
    d_msg = (dev(flat), torch.from_numpy(offs.astype(np.int64)).cuda())
    d_sig, dst = engine.schnorr_sign_varlen(dev(priv), d_msg, dev(aux))
    assert np.array_equal(d_sig.cpu().numpy(), sig)
    assert engine.schnorr_verify_varlen(pkx, msgs, sig).all()
    assert engine.schnorr_verify_varlen(dev(pkx), d_msg, dev(sig)).cpu().numpy().all()
    assert engine.schnorr_batch_verify_varlen(pkx, msgs, sig)
    assert engine.schnorr_batch_verify_varlen(dev(pkx), d_msg, dev(sig)).item() == 1
    bad = sig.copy()
    bad[654_321, 40] ^= 4
    ok = engine.schnorr_verify_varlen(pkx, msgs, bad)
    assert ok.sum() == n - 1 and ok[654_321] == 0
    assert not engine.schnorr_batch_verify_varlen(pkx, msgs, bad)
    assert engine.schnorr_batch_verify_varlen(dev(pkx), d_msg, dev(bad)).item() == 0


@pytest.mark.gpu
def test_gpu_mirror(s256):
    exe = build_mirror(s256)
    rows = [r for r in load_golden("bip340.json")["rows"] if r["valid"]]
    args = [x for r in rows for x in (r["pk"], r["msg"] or "-", r["sig"])]
    r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "varlen mirror ok" in r.stdout
