"""Strict-DER and BIP-66 signature parsing on the device (csrc/der.cuh): the parser against the host codecs, which the
Wycheproof and BIP-66 vectors pin (test_codecs.py), on those vectors and on a seeded mutation corpus; then the
device-resident and host forms of Verify(EncodingASN1) / bitcoin.VerifyASN1 against the route of host parse, compact
verification and AND."""
import ctypes as C
import random

import numpy as np
import pytest

from conftest import load_golden
from hostsim import der as sim

H = bytes.fromhex
N = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
ERR_ARG = -3


def ragged(rows):
    offs = np.zeros(len(rows) + 1, np.uint64)
    np.cumsum([len(r) for r in rows], out=offs[1:])
    return np.frombuffer(b"".join(rows), np.uint8), offs


def _uint(v, pad=b""):
    """DER INTEGER content of v >= 0 (minimal), behind `pad`"""
    b = v.to_bytes(max(1, (v.bit_length() + 7) // 8), "big")
    if b[0] & 0x80:
        b = b"\x00" + b
    return pad + b


def _tlv(tag, body, form=0):
    """form 0: short length; 1-5: long form with that many octets (1 octet below 128 and leading zeros are not
    minimal, which is the point)"""
    n = len(body)
    if form == 0:
        return bytes([tag, n & 0xFF]) + body
    form = max(form, (n.bit_length() + 7) // 8)
    return bytes([tag, 0x80 | form]) + n.to_bytes(form, "big") + body


def _sig(r, s, rf=0, sf=0, qf=0, rpad=b"", spad=b""):
    return _tlv(0x30, _tlv(0x02, _uint(r, rpad), rf) + _tlv(0x02, _uint(s, spad), sf), qf)


def corpus(seed=66, size=120_000):
    """DER signatures and their mutations: bit flips, byte insertions and deletions, truncations, length bytes off by
    one, long-form lengths 0x81-0x85 (minimal and not), high-tag-number tags, leading 0x00 / 0xff on the integers,
    r or s in {0, 1, n - 1, n, 33 bytes}, random rows of 0-80 bytes and rows far longer than 73 bytes."""
    rng = random.Random(seed)
    edge = [0, 1, 0x7F, 0x80, 0xFF, 0x100, N // 2, N // 2 + 1, N - 1, N, N + 1, 2**256 - 1, 2**256, 2**263 + 5]

    def value():
        k = rng.random()
        if k < 0.25:
            return rng.choice(edge)
        if k < 0.35:
            return rng.getrandbits(rng.randrange(1, 260))
        return rng.randrange(1, N)

    base = [_sig(rng.randrange(1, N), rng.randrange(1, N)) for _ in range(2000)]
    base += [_sig(value(), value()) for _ in range(2000)]
    rows = list(base)

    def mutate(b):
        b = bytearray(b)
        k = rng.randrange(12)
        if k == 0:  # bit flips
            for _ in range(rng.randrange(1, 4)):
                if b:
                    i = rng.randrange(len(b))
                    b[i] ^= 1 << rng.randrange(8)
        elif k == 1:  # insertion
            b.insert(rng.randrange(len(b) + 1), rng.choice([0, 0x02, 0x30, 0x80, 0xFF, rng.randrange(256)]))
        elif k == 2 and b:  # deletion
            del b[rng.randrange(len(b))]
        elif k == 3:  # truncation
            b = b[:rng.randrange(len(b) + 1)]
        elif k == 4:  # a length byte off by one
            pos = [1, 3] + ([5 + b[3]] if len(b) > 3 and 5 + b[3] < len(b) else [])
            i = rng.choice(pos)
            if i < len(b):
                b[i] = (b[i] + rng.choice([-1, 1])) & 0xFF
        elif k == 5:  # long-form lengths
            return _sig(value(), value(), rf=rng.choice([0, 0, 1, 2, 3, 4, 5]), sf=rng.choice([0, 0, 1, 2, 5]),
                        qf=rng.choice([0, 1, 1, 2, 3, 4, 5]))
        elif k == 6:  # high-tag-number or other tags
            i = rng.choice([0, 2, 4 + b[3] if len(b) > 3 else 2])
            if i < len(b):
                b[i] = rng.choice([0x1F, 0x3F, 0x5F, 0x9F, 0xFF, 0x31, 0x10, 0x22, 0x03, rng.randrange(256)])
        elif k == 7:  # leading 0x00 / 0xff on an integer
            pad = rng.choice([b"\x00", b"\xff", b"\x00\x00", b"\x00\x80"])
            return _sig(value(), value(), rpad=pad) if rng.random() < 0.5 else _sig(value(), value(), spad=pad)
        elif k == 8:  # r or s at the edges, and 33-byte values
            big = [0, 1, N - 1, N, N + 1, 2**256 + 1, 2**263]
            r = rng.choice(big) if rng.random() < 0.6 else value()
            s = rng.choice(big) if rng.random() < 0.6 else value()
            return _sig(r, s)
        elif k == 9:  # random rows of 0-80 bytes, some of them with a DER-like start
            m = rng.randrange(81)
            b = bytearray(rng.randrange(256) for _ in range(m))
            if m > 2 and rng.random() < 0.5:
                b[0], b[1] = 0x30, (m - 2 + rng.choice([-1, 0, 0, 1])) & 0xFF
        elif k == 10:  # rows far longer than 73 bytes
            m = rng.choice([74, 75, 80, 100, 127, 128, 200, 300, 1000, 5000])
            head = _sig(rng.randrange(1, N), rng.randrange(1, N))
            if rng.random() < 0.5:
                return head + bytes(rng.randrange(256) for _ in range(m - len(head)))
            r = rng.getrandbits(8 * (m // 2 - 6))
            return _sig(r, rng.randrange(1, N), qf=rng.choice([0, 1, 2]))
        else:  # trailing bytes
            b += bytes(rng.randrange(256) for _ in range(rng.randrange(1, 4)))
        return bytes(b)

    while len(rows) < size:
        rows.append(mutate(rng.choice(base)))
    return rows


def with_sighash(rows, seed=7):
    rng = random.Random(seed)
    return [r + bytes([rng.randrange(256)]) for r in rows]


def reference_parse(s256, rows):
    return s256.parse_asn1_signatures(rows)


def reference_bip66_parse(s256, rows):
    """bitcoin.VerifyASN1's parse: IsValidSignatureEncodingBIP0066 on the row, then the strict parse without its last
    byte; a rejected row gives a zeroed r||s"""
    bip = s256.is_valid_signature_encoding_bip0066(rows)
    sig, ok = s256.parse_asn1_signatures([r[:-1] for r in rows])
    ok = ok & bip
    sig[ok == 0] = 0
    return sig, ok, bip


@pytest.fixture(scope="module")
def mutations():
    return corpus()


def vector_rows():
    der = [H(c["sig"]) for c in load_golden("wycheproof_ecdsa_der.json")["cases"]]
    doc = load_golden("bip66.json")
    b66 = [H(v["der"]) for v in doc["valid"] + doc["invalid"]]
    assert len(der) == 996 and len(b66) == 25
    return der, b66


# --------------------------------------------------------------------------------------------------------------------
# CPU: the host simulation of der.cuh against the host codecs
# --------------------------------------------------------------------------------------------------------------------

def _check_sim(s256, rows):
    sig, ok = sim.parse_der(ragged(rows))
    esig, strict_ok = reference_parse(s256, rows)
    assert np.array_equal(ok, strict_ok) and np.array_equal(sig, esig)
    hrows = with_sighash(rows)
    sig, ok = sim.parse_der(ragged(hrows), bip66=True)
    esig, eok, bip = reference_bip66_parse(s256, hrows)
    assert np.array_equal(ok, eok) and np.array_equal(sig, esig)
    assert np.array_equal(sim.check_bip66(ragged(hrows)), bip)
    # BIP-66 on the rows as they are (the vectors' own sighash bytes, odd shapes)
    assert np.array_equal(sim.check_bip66(ragged(rows)), s256.is_valid_signature_encoding_bip0066(rows))
    return strict_ok, eok


def test_sim_matches_host_codecs_on_vectors(s256):
    der, b66 = vector_rows()
    ok, _ = _check_sim(s256, der)
    assert int(ok.sum()) == 432
    _check_sim(s256, b66)
    doc = load_golden("bip66.json")
    rows = [H(v["der"]) + bytes([69]) for v in doc["valid"] + doc["invalid"]]
    assert sim.check_bip66(ragged(rows)).tolist() == [1] * 9 + [0] * 16


def test_sim_matches_host_codecs_on_mutations(s256, mutations):
    ok, bip_ok = _check_sim(s256, mutations)
    # the corpus reaches both verdicts in volume
    assert 5_000 < int(ok.sum()) < len(mutations) - 50_000


def test_rows_longer_than_73_bytes_are_rejected(s256, mutations):
    rows = [r for r in mutations if len(r) > 73]
    rows += [_sig(2**500, 1, qf=2), b"\x30" * 74, bytes(100)]
    assert len(rows) > 1000
    hrows = with_sighash(rows)
    for rr, bip66 in ((rows, False), (hrows, True)):
        sig, ok = sim.parse_der(ragged(rr), bip66=bip66)
        assert not ok.any() and not sig.any()
    assert not sim.check_bip66(ragged(hrows)).any()
    assert not s256.parse_asn1_signatures(rows)[1].any()
    assert not s256.is_valid_signature_encoding_bip0066(hrows).any()


def decreasing_rows():
    """flat = 8 junk bytes + a valid signature A; offsets 8, 16, 8, 16: rows 0 and 2 are A, row 1 decreases"""
    a = _sig(5, 7)
    assert len(a) == 8
    flat = np.frombuffer(bytes(range(8)) + a, np.uint8)
    return flat, np.array([8, 16, 8, 16], np.uint64)


def test_sim_decreasing_offsets_make_only_that_row_invalid():
    flat, offs = decreasing_rows()
    sig, ok = sim.parse_der((flat, offs))
    assert ok.tolist() == [1, 0, 1] and not sig[1].any() and sig[0, 31] == 5 and sig[2, 63] == 7
    hflat = np.concatenate([flat, [1]]).astype(np.uint8)
    hoffs = np.array([8, 17, 8, 17], np.uint64)
    assert sim.parse_der((hflat, hoffs), bip66=True)[1].tolist() == [1, 0, 1]
    assert sim.check_bip66((hflat, hoffs)).tolist() == [1, 0, 1]


# --------------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------------

def dev_rows(rows, lead=5, shift=3):
    """rows on the device at a misaligned address (data_ptr % 16 == shift), offsets starting at `lead`"""
    import torch
    flat, offs = ragged(rows)
    buf = torch.zeros(shift + lead + len(flat), dtype=torch.uint8, device="cuda")
    buf[shift + lead:] = torch.from_numpy(flat.copy()).cuda()
    d = buf[shift:]
    assert d.data_ptr() % 16 == shift
    return d, torch.from_numpy((offs + lead).astype(np.int64)).cuda()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def wycheproof():
    der = load_golden("wycheproof_ecdsa_der.json")["cases"]
    pk = np.frombuffer(b"".join(H(c["pk"]) for c in der), np.uint8).reshape(-1, 65)
    dg = np.frombuffer(b"".join(H(c["digest"])[:32] for c in der), np.uint8).reshape(-1, 32)
    return der, pk, dg, [H(c["sig"]) for c in der]


@pytest.mark.gpu
def test_gpu_parse_matches_host_codecs(engine, s256, mutations):
    import torch
    der, b66 = vector_rows()
    for rows in (der, b66, mutations):
        esig, eok = reference_parse(s256, rows)
        sig, ok = engine.parse_asn1_signatures_dev(dev_rows(rows))
        assert np.array_equal(ok.cpu().numpy(), eok) and np.array_equal(sig.cpu().numpy(), esig)
        bip = s256.is_valid_signature_encoding_bip0066(rows)
        assert np.array_equal(engine.is_valid_signature_encoding_bip0066_dev(dev_rows(rows, 1, 7)).cpu().numpy(), bip)
        hrows = with_sighash(rows)
        assert np.array_equal(engine.is_valid_signature_encoding_bip0066_dev(dev_rows(hrows)).cpu().numpy(),
                              s256.is_valid_signature_encoding_bip0066(hrows))
    # outputs at misaligned addresses (byte stores) give the same bytes
    rows = mutations[:5000]
    d, o = dev_rows(rows, 0, 1)
    n = len(rows)
    out = torch.full((64 * n + 3,), 0xAA, dtype=torch.uint8, device="cuda")
    okb = torch.full((n + 1,), 0xAA, dtype=torch.uint8, device="cuda")
    lib, ctx = engine._lib, engine._ctx
    assert lib.s256_parse_asn1_signatures_dev(ctx, C.c_void_p(d.data_ptr()), C.c_void_p(o.data_ptr()), C.c_size_t(n),
                                              C.c_void_p(out.data_ptr() + 3), C.c_void_p(okb.data_ptr() + 1),
                                              engine._stream()) == 0
    esig, eok = reference_parse(s256, rows)
    got = out.cpu().numpy()
    assert got[:3].tolist() == [0xAA] * 3 and np.array_equal(got[3:].reshape(n, 64), esig)
    assert okb[0].item() == 0xAA and np.array_equal(okb[1:].cpu().numpy(), eok)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, 1])
def test_gpu_verify_asn1_wycheproof(engine, oracle, s256, flags):
    der, pk, dg, rows = wycheproof()
    sig, ok = s256.parse_asn1_signatures(rows)
    exp = ok & oracle.batch_ecdsa_verify(pk, dg, sig, flags)
    if flags == 0:
        assert np.array_equal(exp, np.array([c["valid"] for c in der], np.uint8))
    host = engine.ecdsa_verify_asn1(pk, dg, rows, flags)
    devok = engine.ecdsa_verify_asn1(dev(pk), dev(dg), dev_rows(rows), flags).cpu().numpy()
    assert np.array_equal(host, exp) and np.array_equal(devok, exp)


@pytest.mark.gpu
def test_gpu_bitcoin_verify_asn1_wycheproof(engine, oracle, s256):
    der, pk, dg, sigs = wycheproof()
    keep = [i for i, c in enumerate(der) if "sha256" in c["src"]]
    pk, dg = pk[keep], dg[keep]
    plain = [sigs[i] for i in keep]
    rows = [r + b"\x01" for r in plain]
    # the expectation test_codecs.py::test_bitcoin_verify_asn1 assembles
    bip = s256.is_valid_signature_encoding_bip0066(rows)
    sig, ok = s256.parse_asn1_signatures(plain)
    exp = bip & ok & oracle.batch_ecdsa_verify(pk, dg, sig, 1)
    assert 0 < int(exp.sum())
    assert np.array_equal(engine.bitcoin_verify_asn1(pk, dg, rows), exp)
    assert np.array_equal(engine.bitcoin_verify_asn1(dev(pk), dev(dg), dev_rows(rows)).cpu().numpy(), exp)


def mangle(rows, every=7):
    """turns every `every`-th row into invalid DER, cycling through the kinds of damage"""
    out = list(rows)
    for j, i in enumerate(range(3, len(rows), every)):
        r = bytearray(out[i])
        k = j % 5
        if k == 0:
            r = r[:-1]
        elif k == 1:
            r[1] ^= 1
        elif k == 2:
            r[0] = 0x1F
        elif k == 3:
            r = r + b"\x00"
        else:
            r = bytes([0x30, 0x81]) + r[1:]
        out[i] = bytes(r)
    return out


def route_before(engine, s256, pk, dg, rows, bitcoin):
    """host codecs, compact verification, AND"""
    if bitcoin:
        bip = s256.is_valid_signature_encoding_bip0066(rows)
        sig, ok = s256.parse_asn1_signatures([r[:-1] for r in rows])
        return bip & ok & engine.ecdsa_verify(pk, dg, sig, 1)
    sig, ok = s256.parse_asn1_signatures(rows)
    return ok & engine.ecdsa_verify(pk, dg, sig, 0)


@pytest.mark.gpu
def test_gpu_full_size_matches_route_before(engine, s256):
    import torch
    n = 1 << 20
    w = s256.synth.ecdsa_batch(n, engine.scalar_base_mult)
    pk, dg = w["pk65"], w["digest32"]
    rows = mangle(s256.build_asn1_signatures(w["sig64"]))
    exp = route_before(engine, s256, pk, dg, rows, False)
    assert np.array_equal(engine.ecdsa_verify_asn1(pk, dg, rows), exp)
    d_pk, d_dg = dev(pk), dev(dg)
    assert np.array_equal(engine.ecdsa_verify_asn1(d_pk, d_dg, dev_rows(rows)).cpu().numpy(), exp)
    assert 0 < int(exp.sum()) < int(w["expected"].sum())
    hrows = with_sighash(rows)
    hrows[11] = hrows[11][:-1] + b"\x01\x01"  # a trailing byte too many for BIP-66
    exp = route_before(engine, s256, pk, dg, hrows, True)
    assert exp[11] == 0
    assert np.array_equal(engine.bitcoin_verify_asn1(pk, dg, hrows), exp)
    assert np.array_equal(engine.bitcoin_verify_asn1(d_pk, d_dg, dev_rows(hrows)).cpu().numpy(), exp)
    assert 0 < int(exp.sum())
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_gpu_small_max_batch_crosses_chunks(s256, oracle):
    small = s256.Engine(max_batch=384)
    try:
        der, pk, dg, rows = wycheproof()
        sig, ok = s256.parse_asn1_signatures(rows)
        exp = ok & oracle.batch_ecdsa_verify(pk, dg, sig, 0)
        assert np.array_equal(small.ecdsa_verify_asn1(pk, dg, rows), exp)
        assert np.array_equal(small.ecdsa_verify_asn1(dev(pk), dev(dg), dev_rows(rows)).cpu().numpy(), exp)
        hrows = [r + b"\x01" for r in rows]
        bip = s256.is_valid_signature_encoding_bip0066(hrows)
        bexp = bip & ok & oracle.batch_ecdsa_verify(pk, dg, sig, 1)
        assert np.array_equal(small.bitcoin_verify_asn1(pk, dg, hrows), bexp)
        assert np.array_equal(small.bitcoin_verify_asn1(dev(pk), dev(dg), dev_rows(hrows)).cpu().numpy(), bexp)
    finally:
        small.close()


def _valid_batch(engine, s256, n=64):
    w = s256.synth.ecdsa_batch(n, engine.scalar_base_mult, corrupt_every=0)
    for i in range(n):  # low s everywhere, so that the Bitcoin form accepts every row too
        s = int.from_bytes(w["sig64"][i, 32:].tobytes(), "big")
        if s > N // 2:
            w["sig64"][i, 32:] = np.frombuffer((N - s).to_bytes(32, "big"), np.uint8)
    rows = s256.build_asn1_signatures(w["sig64"])
    assert engine.ecdsa_verify_asn1(w["pk65"], w["digest32"], rows).all()
    return w["pk65"], w["digest32"], rows


@pytest.mark.gpu
def test_gpu_decreasing_offsets(engine, s256):
    import torch
    # rows 0 and 2 are the same valid signature, row 1 decreases
    a = s256.build_asn1_signatures(np.frombuffer(bytes(31) + b"\x05" + bytes(31) + b"\x07", np.uint8))[0]
    flat = np.frombuffer(bytes(range(8)) + a, np.uint8)
    offs = np.array([8, 16, 8, 16], np.uint64)
    sig, ok = engine.parse_asn1_signatures_dev((dev(flat), dev(offs.astype(np.int64))))
    assert ok.cpu().tolist() == [1, 0, 1] and not sig[1].any()
    # verification: a real signature in rows 0 and 2, keys and digests to match
    pk1, dg1, rows = _valid_batch(engine, s256, 1)
    sflat = np.frombuffer(bytes(8) + rows[0], np.uint8)
    L = len(rows[0])
    doffs = np.array([8, 8 + L, 8, 8 + L], np.int64)
    pk3, dg3 = np.repeat(pk1, 3, 0), np.repeat(dg1, 3, 0)
    got = engine.ecdsa_verify_asn1(dev(pk3), dev(dg3), (dev(sflat), dev(doffs))).cpu().tolist()
    assert got == [1, 0, 1]
    hflat = np.frombuffer(bytes(8) + rows[0] + b"\x01", np.uint8)
    hoffs = np.array([8, 9 + L, 8, 9 + L], np.int64)
    assert engine.bitcoin_verify_asn1(dev(pk3), dev(dg3), (dev(hflat), dev(hoffs))).cpu().tolist() == [1, 0, 1]
    assert engine.is_valid_signature_encoding_bip0066_dev((dev(hflat), dev(hoffs))).cpu().tolist() == [1, 0, 1]
    torch.cuda.synchronize()
    # the host forms refuse the same offsets before enqueueing anything
    lib, ctx = engine._lib, engine._ctx
    hp = lambda x: x.ctypes.data_as(C.c_void_p)
    out = np.full(3, 7, np.uint8)
    hoffs_u = hoffs.astype(np.uint64)
    before = engine.launch_count
    assert lib.s256_ecdsa_verify_asn1(ctx, hp(pk3), hp(dg3), hp(sflat), hp(doffs.astype(np.uint64)), C.c_uint32(0),
                                      C.c_size_t(3), hp(out)) == ERR_ARG
    assert lib.s256_bitcoin_verify_asn1(ctx, hp(pk3), hp(dg3), hp(hflat), hp(hoffs_u), C.c_size_t(3), hp(out)) == ERR_ARG
    assert engine.launch_count == before and (out == 7).all()


@pytest.mark.gpu
def test_gpu_one_gib_junk_row(engine, s256):
    import torch
    pk, dg, rows = _valid_batch(engine, s256, 64)
    j = 17
    lens = [len(r) for r in rows]
    big = 1 << 30
    flat = np.zeros(sum(lens) - lens[j] + big, np.uint8)  # zero pages: the junk row's bytes are never touched
    offs = np.zeros(65, np.uint64)
    pos = 0
    for i, r in enumerate(rows):
        offs[i] = pos
        if i == j:
            pos += big
        else:
            flat[pos:pos + len(r)] = np.frombuffer(r, np.uint8)
            pos += len(r)
    offs[64] = pos
    exp = np.ones(64, np.uint8)
    exp[j] = 0
    lib, ctx = engine._lib, engine._ctx
    hp = lambda x: x.ctypes.data_as(C.c_void_p)
    out = np.full(64, 7, np.uint8)
    assert lib.s256_ecdsa_verify_asn1(ctx, hp(pk), hp(dg), hp(flat), hp(offs), C.c_uint32(0), C.c_size_t(64), hp(out)) == 0
    assert np.array_equal(out, exp)
    # the same row among sighash-carrying rows: the Bitcoin form
    hrows = [r + b"\x01" for r in rows]
    hflat = np.zeros(sum(len(r) for r in hrows) - len(hrows[j]) + big, np.uint8)
    pos = 0
    for i, r in enumerate(hrows):
        offs[i] = pos
        if i == j:
            pos += big
        else:
            hflat[pos:pos + len(r)] = np.frombuffer(r, np.uint8)
            pos += len(r)
    offs[64] = pos
    out[:] = 7
    assert lib.s256_bitcoin_verify_asn1(ctx, hp(pk), hp(dg), hp(hflat), hp(offs), C.c_size_t(64), hp(out)) == 0
    assert np.array_equal(out, exp)
    # device rows: the long row is rejected without being read
    d_flat = dev(hflat)
    assert np.array_equal(engine.bitcoin_verify_asn1(dev(pk), dev(dg), (d_flat, dev(offs.astype(np.int64)))).cpu().numpy(), exp)
    del d_flat
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_gpu_empty_null_and_side_stream(engine, s256):
    import torch
    lib, ctx = engine._lib, engine._ctx
    z = np.zeros((0, 65), np.uint8)
    assert engine.ecdsa_verify_asn1(z, np.zeros((0, 32), np.uint8), []).size == 0
    assert engine.bitcoin_verify_asn1(z, np.zeros((0, 32), np.uint8), []).size == 0
    zero = C.c_size_t(0)
    assert lib.s256_bitcoin_verify_asn1(ctx, None, None, None, None, zero, None) == 0  # NULL offsets with n == 0
    assert lib.s256_ecdsa_verify_asn1(ctx, None, None, None, None, C.c_uint32(0), zero, None) == 0
    for f in (lib.s256_ecdsa_verify_asn1_dev, ):
        assert f(ctx, None, None, None, None, C.c_uint32(0), zero, None, None) == 0
    assert lib.s256_bitcoin_verify_asn1_dev(ctx, None, None, None, None, zero, None, None) == 0
    assert lib.s256_parse_asn1_signatures_dev(ctx, None, None, zero, None, None, None) == 0
    assert lib.s256_is_valid_signature_encoding_bip0066_dev(ctx, None, None, zero, None, None) == 0
    d0, o0 = torch.zeros(0, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda")
    assert engine.ecdsa_verify_asn1(d0, d0, (d0, o0)).numel() == 0
    buf = (C.c_uint8 * 128)()
    offs = (C.c_size_t * 2)(0, 8)
    one, f0 = C.c_size_t(1), C.c_uint32(0)
    for args in ((None, buf, buf, offs), (buf, None, buf, offs), (buf, buf, None, offs), (buf, buf, buf, None)):
        assert lib.s256_ecdsa_verify_asn1(ctx, *args, f0, one, buf) == ERR_ARG
        assert lib.s256_bitcoin_verify_asn1(ctx, *args, one, buf) == ERR_ARG
        assert lib.s256_ecdsa_verify_asn1_dev(ctx, *args, f0, one, buf, None) == ERR_ARG
        assert lib.s256_bitcoin_verify_asn1_dev(ctx, *args, one, buf, None) == ERR_ARG
    assert lib.s256_ecdsa_verify_asn1(ctx, buf, buf, buf, offs, f0, one, None) == ERR_ARG
    assert lib.s256_ecdsa_verify_asn1(None, buf, buf, buf, offs, f0, one, buf) == ERR_ARG
    assert lib.s256_bitcoin_verify_asn1(None, buf, buf, buf, offs, one, buf) == ERR_ARG
    assert lib.s256_ecdsa_verify_asn1_dev(None, buf, buf, buf, offs, f0, one, buf, None) == ERR_ARG
    assert lib.s256_parse_asn1_signatures_dev(ctx, None, offs, one, buf, buf, None) == ERR_ARG
    assert lib.s256_parse_asn1_signatures_dev(ctx, buf, offs, one, None, buf, None) == ERR_ARG
    assert lib.s256_parse_asn1_signatures_dev(None, buf, offs, one, buf, buf, None) == ERR_ARG
    assert lib.s256_is_valid_signature_encoding_bip0066_dev(ctx, buf, None, one, buf, None) == ERR_ARG
    assert lib.s256_is_valid_signature_encoding_bip0066_dev(ctx, buf, offs, one, None, None) == ERR_ARG
    # a _dev call on a side stream, then calls on the same context
    pk, dg, rows = _valid_batch(engine, s256, 512)
    d_pk, d_dg, d_rows = dev(pk), dev(dg), dev_rows(rows)
    d_h = dev_rows([r + b"\x01" for r in rows])
    k = torch.from_numpy(np.frombuffer(bytes(range(32)) * 4096, np.uint8).copy()).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for _ in range(3):
        with torch.cuda.stream(side):
            ok_side = engine.ecdsa_verify_asn1(d_pk, d_dg, d_rows)
        engine.scalar_base_mult(k)
        ok_main = engine.bitcoin_verify_asn1(d_pk, d_dg, d_h)
        ok_host = engine.ecdsa_verify_asn1(pk, dg, rows)
        side.synchronize()
        torch.cuda.synchronize()
        assert bool(ok_side.all()) and bool(ok_main.all()) and ok_host.all()
