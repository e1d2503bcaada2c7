"""BIP-340 batch verification (s256_schnorr_batch_verify): the randomizer definition against hashlib, the batch verdict
of the host simulation against the per-row oracle, and the same cases through the C ABI on the GPU."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from hostsim import batch as batch_sim
import parity_suites as ps

N = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141


# ---- reference of the randomizer definition (DESIGN.md, batch verification) -----------------------------------
def ref_seed_and_randomizers(pkx, msg, sig):
    n = len(pkx)
    nodes = [hashlib.sha256(bytes(pkx[i]) + bytes(sig[i]) + bytes(msg[i])).digest() for i in range(n)]
    while len(nodes) > 1:
        nodes = [hashlib.sha256(nodes[j] + nodes[j + 1]).digest() if j + 1 < len(nodes) else nodes[j]
                 for j in range(0, len(nodes), 2)]
    th = hashlib.sha256(b"S256/BIP0340/batch").digest()
    seed = hashlib.sha256(th + th + nodes[0] + n.to_bytes(8, "big")).digest()
    a = [1] + [int.from_bytes(hashlib.sha256(seed + i.to_bytes(8, "big")).digest()[:16], "big") or 1 for i in range(1, n)]
    return seed, a


def random_rows(n, msg_len, seed):
    rng = np.random.default_rng(seed)
    return (rng.integers(0, 256, (n, 32), dtype=np.uint8), rng.integers(0, 256, (n, msg_len), dtype=np.uint8),
            rng.integers(0, 256, (n, 64), dtype=np.uint8))


@pytest.mark.parametrize("msg_len", [0, 32, 100])
@pytest.mark.parametrize("n", [1, 2, 3, 5, 8, 33, 1000])
def test_randomizers_match_hashlib(n, msg_len):
    pkx, msg, sig = random_rows(n, msg_len, 1000 * n + msg_len)
    want_seed, want_a = ref_seed_and_randomizers(pkx, msg, sig)
    seed, a = batch_sim.schnorr_batch_randomizers(pkx, msg, sig, chunk=1 << 19)
    assert seed == want_seed
    assert [int.from_bytes(a[i].tobytes(), "big") for i in range(n)] == want_a


@pytest.mark.parametrize("n", [1, 3, 33, 1000])
def test_randomizers_do_not_depend_on_the_chunk_size(n):
    pkx, msg, sig = random_rows(n, 32, n)
    seed0, a0 = batch_sim.schnorr_batch_randomizers(pkx, msg, sig, chunk=1 << 19)
    chunk = 1
    while chunk <= n:
        seed, a = batch_sim.schnorr_batch_randomizers(pkx, msg, sig, chunk=chunk)
        assert seed == seed0, chunk
        assert np.array_equal(a, a0), chunk
        chunk *= 2


# ---- verdict cases ----------------------------------------------------------------------------------------------
_BATCHES = {}


def valid_batch(oracle, n):
    if n not in _BATCHES:
        w = ps.synth.schnorr_batch(n, ps.oracle_base_mult(oracle), corrupt_every=0)
        _BATCHES[n] = (w["pkx32"], w["msg"], w["sig64"])
    return tuple(x.copy() for x in _BATCHES[n])


def corrupt(batch, kind, pos):
    pkx, msg, sig = batch
    if kind == "r":
        sig[pos, 31] ^= 1
    elif kind == "s":
        sig[pos, 63] ^= 1
    elif kind == "msg":
        msg[pos, 0] ^= 1
    else:
        pkx[pos] = pkx[(pos + 1) % len(pkx)]
    return pkx, msg, sig


def cancelling_pair(oracle):
    """Two valid signatures with s1 + 1 and s2 - 1: the plain (unweighted) sum of the two equations still holds."""
    pkx, msg, sig = valid_batch(oracle, 2)
    s1, s2 = (int.from_bytes(sig[i, 32:].tobytes(), "big") for i in (0, 1))
    sig[0, 32:] = np.frombuffer(((s1 + 1) % N).to_bytes(32, "big"), np.uint8)
    sig[1, 32:] = np.frombuffer(((s2 - 1) % N).to_bytes(32, "big"), np.uint8)
    return pkx, msg, sig


def one_key_batch(oracle, n=64):
    d = (0x1234567890ABCDEF).to_bytes(32, "big")
    pk, _ = oracle.scalar_base_mult(d)
    pkx = np.frombuffer(bytes(pk)[1:33], np.uint8)
    rows = [(hashlib.sha256(b"one key %d" % i).digest(), hashlib.sha256(b"aux %d" % i).digest()) for i in range(n)]
    sig = np.stack([np.frombuffer(oracle.schnorr_sign(d, m, a)[0], np.uint8) for m, a in rows])
    msg = np.stack([np.frombuffer(m, np.uint8) for m, _ in rows])
    return np.tile(pkx, (n, 1)), msg, sig


def golden_cases():
    """(name, pkx, msg, sig): the valid rows batched by message length, and each invalid row inside a valid batch."""
    rows = load_golden("bip340.json")["rows"]
    H = bytes.fromhex
    out = []
    for ml in sorted({len(H(r["msg"])) for r in rows if r["valid"] and r["pk"]}):
        g = [r for r in rows if r["valid"] and len(H(r["msg"])) == ml]
        out.append((f"valid-msglen{ml}", np.stack([np.frombuffer(H(r["pk"]), np.uint8) for r in g]),
                    np.stack([np.frombuffer(H(r["msg"]), np.uint8) for r in g]).reshape(len(g), ml),
                    np.stack([np.frombuffer(H(r["sig"]), np.uint8) for r in g])))
    return out, [r for r in rows if not r["valid"]]


def verdict_cases(oracle):
    """(name, pkx, msg, sig) over everything the CPU and the GPU tests check."""
    cases = []
    for n in (1, 2, 31, 32, 33, 200):
        cases.append((f"valid-{n}",) + valid_batch(oracle, n))
    for kind in ("r", "s", "msg", "pk"):
        for pos in (0, 16, 32):
            cases.append((f"{kind}@{pos}",) + corrupt(valid_batch(oracle, 33), kind, pos))
    good, bad = golden_cases()
    cases += good
    for r in bad:
        pkx, msg, sig = valid_batch(oracle, 5)
        pkx[2] = np.frombuffer(bytes.fromhex(r["pk"]), np.uint8)
        msg[2] = np.frombuffer(bytes.fromhex(r["msg"]), np.uint8)
        sig[2] = np.frombuffer(bytes.fromhex(r["sig"]), np.uint8)
        cases.append((f"golden-invalid-{r['index']}", pkx, msg, sig))
    cases.append(("one-key-64",) + one_key_batch(oracle))
    pkx, msg, sig = valid_batch(oracle, 1)
    cases.append(("repeated-64", np.tile(pkx, (64, 1)), np.tile(msg, (64, 1)), np.tile(sig, (64, 1))))
    cases.append(("cancelling-pair",) + cancelling_pair(oracle))
    return cases


@pytest.fixture(scope="module")
def cases(oracle):
    return verdict_cases(oracle)


def expected(oracle, pkx, msg, sig):
    return bool(np.all(oracle.batch_schnorr_verify(pkx, msg, sig)))


def test_hostsim_verdict_matches_oracle(oracle, cases):
    seen_true = seen_false = 0
    for name, pkx, msg, sig in cases:
        want = expected(oracle, pkx, msg, sig)
        assert batch_sim.schnorr_batch_verify(pkx, msg, sig) == want, name
        seen_true += want
        seen_false += not want
    assert seen_true >= 8 and seen_false >= 20


def test_cancelling_pair_fools_the_unweighted_sum(oracle):
    """The pair passes the check without randomizers (sum s_i) G == sum R_i + sum e_i P_i, and each row fails alone."""
    pkx, msg, sig = cancelling_pair(oracle)
    assert not oracle.batch_schnorr_verify(pkx, msg, sig).any()
    tag = hashlib.sha256(b"BIP0340/challenge").digest()
    ks, pts = [], []
    ssum = 0
    for i in range(2):
        pt, st = oracle.point_decode(b"\x02" + sig[i, :32].tobytes())
        ks.append((1).to_bytes(32, "big")); pts.append(bytes(pt))
        pp, st = oracle.point_decode(b"\x02" + pkx[i].tobytes())
        e = int.from_bytes(hashlib.sha256(tag + tag + sig[i, :32].tobytes() + pkx[i].tobytes() + msg[i].tobytes()).digest(), "big") % N
        ks.append(e.to_bytes(32, "big")); pts.append(bytes(pp))
        ssum += int.from_bytes(sig[i, 32:].tobytes(), "big")
    lhs, _ = oracle.scalar_base_mult((ssum % N).to_bytes(32, "big"))
    rhs, _ = oracle.msm(b"".join(ks), b"".join(pts))
    assert bytes(lhs) == bytes(rhs)
    assert not batch_sim.schnorr_batch_verify(pkx, msg, sig)


def test_hostsim_chunked_verdict(oracle):
    pkx, msg, sig = valid_batch(oracle, 33)
    for chunk in (1, 4, 16, 32):
        assert batch_sim.schnorr_batch_verify(pkx, msg, sig, chunk=chunk), chunk
        assert not batch_sim.schnorr_batch_verify(*corrupt((pkx.copy(), msg.copy(), sig.copy()), "s", 32), chunk=chunk), chunk


MIRROR_SRC = os.path.join(ROOT, "tests", "cpp", "schnorr_batch_mirror.cpp")
MIRROR_EXE = os.path.join(ROOT, "tests", "cpp", "_build", "schnorr_batch_mirror")


def build_mirror(s256):
    s256.load_library()
    libdir = os.path.dirname(s256.library_path())
    os.makedirs(os.path.dirname(MIRROR_EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-o", MIRROR_EXE, MIRROR_SRC, "-L", libdir, "-lsecp256k1_b200",
                           f"-Wl,-rpath,{libdir}"])
    return MIRROR_EXE


def test_mirror_compiles_and_links(s256):
    assert os.path.exists(build_mirror(s256))


# ---- GPU: the same cases through the C ABI ------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_verdict_matches_oracle(engine, oracle, cases):
    for name, pkx, msg, sig in cases:
        assert engine.schnorr_batch_verify(pkx, msg, sig) == expected(oracle, pkx, msg, sig), name


@pytest.mark.gpu
def test_gpu_empty_batch_and_misuse(engine, s256):
    assert engine.schnorr_batch_verify(np.zeros((0, 32), np.uint8), np.zeros((0, 32), np.uint8), np.zeros((0, 64), np.uint8))
    lib, ctx = engine._lib, engine._ctx
    buf = (C.c_uint8 * 64)()
    ok = C.c_uint8(7)
    assert lib.s256_schnorr_batch_verify(ctx, None, buf, C.c_size_t(32), buf, C.c_size_t(1), C.byref(ok)) == -3
    assert lib.s256_schnorr_batch_verify(ctx, buf, None, C.c_size_t(32), buf, C.c_size_t(1), C.byref(ok)) == -3
    assert lib.s256_schnorr_batch_verify(ctx, buf, buf, C.c_size_t(32), None, C.c_size_t(1), C.byref(ok)) == -3
    assert lib.s256_schnorr_batch_verify(ctx, buf, buf, C.c_size_t(32), buf, C.c_size_t(1), None) == -3
    assert lib.s256_schnorr_batch_verify_dev(ctx, None, None, C.c_size_t(32), None, C.c_size_t(1), None, None) == -3
    assert lib.s256_schnorr_batch_verify(None, buf, buf, C.c_size_t(32), buf, C.c_size_t(1), C.byref(ok)) == -3
    assert ok.value == 7
    with pytest.raises(ValueError):
        engine.schnorr_batch_verify(np.zeros((3, 32), np.uint8), np.zeros((3, 32), np.uint8), np.zeros((2, 64), np.uint8))
    import torch
    d = torch.zeros(0, dtype=torch.uint8, device="cuda")
    assert engine.schnorr_batch_verify(d, d, d).item() == 1


@pytest.mark.gpu
def test_gpu_dev_form_matches_host_form(engine, oracle, cases):
    import torch

    def at_offset(a, off):  # a device copy starting `off` bytes into a larger buffer
        flat = torch.from_numpy(np.ascontiguousarray(a).reshape(-1))
        buf = torch.zeros(flat.numel() + off, dtype=torch.uint8, device="cuda")
        buf[off:] = flat.cuda()
        return buf[off:]

    for off in (0, 1, 3):
        for name, pkx, msg, sig in cases[::3]:
            got = engine.schnorr_batch_verify(at_offset(pkx, off), at_offset(msg, off), at_offset(sig, off))
            assert bool(got.item()) == engine.schnorr_batch_verify(pkx, msg, sig), (name, off)


@pytest.mark.gpu
def test_gpu_chunked_equals_default_engine(engine, s256, oracle):
    small = s256.Engine(max_batch=4096)  # chunks of 2048 rows
    try:
        n = 3 * 2048 + 5
        w = ps.synth.schnorr_batch(n, engine.scalar_base_mult, corrupt_every=0)
        rows = (w["pkx32"], w["msg"], w["sig64"])
        assert small.schnorr_batch_verify(*rows) and engine.schnorr_batch_verify(*rows)
        for pos in (5, 3000, n - 1):
            bad = corrupt(tuple(x.copy() for x in rows), "s", pos)
            got = small.schnorr_batch_verify(*bad)
            assert got == engine.schnorr_batch_verify(*bad) == expected(oracle, *[x[pos:pos + 1] for x in bad]) == False, pos
    finally:
        small.close()


@pytest.fixture(scope="module")
def full_batch(engine):
    w = ps.synth.schnorr_batch(1 << 20, engine.scalar_base_mult, corrupt_every=0)
    return w["pkx32"], w["msg"], w["sig64"]


@pytest.mark.gpu
def test_gpu_full_size(engine, full_batch):
    import torch
    pkx, msg, sig = full_batch
    assert bool(engine.schnorr_verify(pkx, msg, sig).all())
    assert engine.schnorr_batch_verify(pkx, msg, sig)
    bad = sig.copy()
    bad[777_777, 40] ^= 4
    assert not engine.schnorr_batch_verify(pkx, msg, bad)
    d = [torch.from_numpy(x).cuda() for x in (pkx, msg, bad)]
    assert engine.schnorr_batch_verify(*d).item() == 0


@pytest.mark.gpu
def test_gpu_side_stream_after_other_dev_call(engine, oracle):
    """A batch verification on a side stream right after a _dev call of another entry point on the same context."""
    import torch
    pkx, msg, sig = valid_batch(oracle, 200)
    d_pkx, d_msg, d_sig = (torch.from_numpy(x).cuda() for x in (pkx, msg, sig))
    k = torch.from_numpy(ps.synth.base_mult_scalars(1 << 16)).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for _ in range(3):
        out, st = engine.scalar_base_mult(k)
        ok_items = engine.schnorr_verify(d_pkx, d_msg, d_sig)
        with torch.cuda.stream(side):
            ok = engine.schnorr_batch_verify(d_pkx, d_msg, d_sig)
        side.synchronize()
        assert ok.item() == 1
        torch.cuda.synchronize()
        assert bool(ok_items.all())


@pytest.mark.gpu
def test_gpu_mirror_accepts_valid_and_rejects_corrupted(s256):
    exe = build_mirror(s256)
    rows = [r for r in load_golden("bip340.json")["rows"] if r["valid"] and len(r["msg"]) == 64]
    args = [x for r in rows for x in (r["pk"], r["msg"], r["sig"])]
    r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "batch mirror ok" in r.stdout
