"""Hash to curve (RFC 9380, secp256k1_XMD:SHA-256_SSWU_RO_ / _NU_) over messages of different lengths in one call and
from device memory (s256_hash_to_curve_varlen[_dev], s256_hash_to_curve_dev): the kernel's item function with the
offsets accessor on the CPU against the oracle, then the C ABI on the GPU, host and device forms, against the oracle
and the uniform entry point."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from hostsim import h2c_varlen as hsim

SUITE_DST = b"QUUX-V01-CS02-with-secp256k1_XMD:SHA-256_SSWU_RO_"
EQUAL_LENS = [0, 1, 32, 55, 56, 64, 119, 120, 517]


def ragged(msgs):
    offs = np.zeros(len(msgs) + 1, np.uint64)
    offs[1:] = np.cumsum([len(m) for m in msgs]) if msgs else []
    return np.frombuffer(b"".join(bytes(m) for m in msgs), np.uint8).copy(), offs


def suites():
    return load_golden("h2c.json")["suites"]


def suite_msgs(s):
    return [v["msg"].encode() for v in s["vectors"]]


def suite_points(s):
    return [bytes.fromhex("04" + v["Px"] + v["Py"]) for v in s["vectors"]]


def random_rows(n, seed, hi=600):
    rng = np.random.default_rng(seed)
    return [rng.bytes(int(ln)) for ln in rng.integers(0, hi + 1, n)]


def oracle_rows(oracle, dst, msgs, ro):
    out = np.zeros((len(msgs), 65), np.uint8)
    st = np.zeros(len(msgs), np.uint8)
    for i, m in enumerate(msgs):
        o, s = oracle.hash_to_curve(dst, m, ro)
        out[i] = np.frombuffer(bytes(o), np.uint8)
        st[i] = s
    return out, st


def b0_edge_lengths(dst_len, hi=600):
    """Message lengths around the SHA-256 block edges of expand_message_xmd's b0 input: Z_pad (64) || msg ||
    l_i_b_str (2) || 0x00 || DST || len(DST), padded with at least 9 bytes, fills a whole number of blocks exactly at
    64 + len + 3 + dst_len + 1 + 9 = 0 (mod 64)."""
    lens = set()
    for k in range(1, (64 + hi + 3 + dst_len + 1 + 9) // 64 + 2):
        exact = 64 * k - (64 + 3 + dst_len + 1 + 9)
        lens.update(x for x in (exact - 1, exact, exact + 1) if 0 <= x <= hi)
    return sorted(lens)


def decreasing_at(offs, i):
    bad = offs.copy()
    assert bad[i] > 0
    bad[i + 1] = bad[i] - 1
    return bad


# ---- CPU: the kernel's item function with the offsets accessor --------------------------------------------------------
@pytest.mark.parametrize("s", suites(), ids=lambda s: "RO" if s["random_oracle"] else "NU")
def test_suite_vectors_in_one_call(s):
    msgs = suite_msgs(s)
    assert [len(m) for m in msgs] == [0, 3, 16, 133, 517]
    out, st = hsim.hash_to_curve(s["dst"].encode(), ragged(msgs), s["random_oracle"])
    assert st.tolist() == [1] * 5
    assert [o.tobytes() for o in out] == suite_points(s)


@pytest.mark.parametrize("ro", [True, False])
def test_random_lengths_match_oracle(oracle, ro):
    msgs = random_rows(64, 9 + ro)
    out, st = hsim.hash_to_curve(SUITE_DST, ragged(msgs), ro)
    want, wst = oracle_rows(oracle, SUITE_DST, msgs, ro)
    assert np.array_equal(st, wst) and np.array_equal(out, want)


@pytest.mark.parametrize("dst_len", [1, 49, 200])
def test_b0_block_edges_match_oracle(oracle, dst_len):
    dst = bytes((7 * i + 1) % 256 for i in range(dst_len))
    lens = b0_edge_lengths(dst_len)
    assert len(lens) >= 20
    rng = np.random.default_rng(dst_len)
    msgs = [rng.bytes(ln) for ln in lens]
    for ro in (True, False):
        out, st = hsim.hash_to_curve(dst, ragged(msgs), ro)
        want, wst = oracle_rows(oracle, dst, msgs, ro)
        assert np.array_equal(st, wst) and np.array_equal(out, want), (dst_len, ro)


@pytest.mark.parametrize("dst_len", [1, 255, 256])
def test_dst_lengths_match_oracle(oracle, dst_len):
    """1 and 255 bytes go to the kernel as they are; 256 is hashed on the host first (RFC 9380 section 5.3.3)."""
    dst = bytes((3 * i + 5) % 256 for i in range(dst_len))
    msgs = random_rows(12, dst_len, hi=200)
    for ro in (True, False):
        out, st = hsim.hash_to_curve(dst, ragged(msgs), ro)
        want, wst = oracle_rows(oracle, dst, msgs, ro)
        assert np.array_equal(st, wst) and np.array_equal(out, want), (dst_len, ro)


def test_decreasing_offsets_make_only_that_row_invalid(oracle):
    """The _dev form's rule: a row with offsets[i+1] < offsets[i] reads none of its bytes, gets S256_ST_INVALID and 65
    zero bytes; the other rows are hashed as their offsets say (row 6 now starts one byte early)."""
    msgs = random_rows(24, 4, hi=100)
    msgs[5] = msgs[5] or b"x"
    flat, offs = ragged(msgs)
    bad = decreasing_at(offs, 5)
    out, st = hsim.hash_to_curve(SUITE_DST, (flat, bad), True)
    assert st[5] == 0 and not out[5].any()
    rows = [flat[int(bad[i]):int(bad[i + 1])].tobytes() for i in range(len(msgs)) if i != 5]
    want, wst = oracle_rows(oracle, SUITE_DST, rows, True)
    keep = [i for i in range(len(msgs)) if i != 5]
    assert np.array_equal(out[keep], want) and np.array_equal(st[keep], wst) and wst.all()


def test_mirror_compiles_and_links(s256):
    assert os.path.exists(build_mirror(s256))


# ---- GPU ---------------------------------------------------------------------------------------------------------------
MIRROR_SRC = os.path.join(ROOT, "tests", "cpp", "h2c_varlen_mirror.cpp")
MIRROR_EXE = os.path.join(ROOT, "tests", "cpp", "_build", "h2c_varlen_mirror")


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


def dev_ragged(msgs, off=0, base=0):
    """The device form of the rows: the bytes start `off` bytes into a larger buffer, and the offsets start at `base`
    (relative to the returned flat tensor, whose first `base` bytes belong to no row)."""
    import torch
    flat, offs = ragged(msgs)
    buf = torch.full((flat.size + base + off + 1,), 0xA5, dtype=torch.uint8, device="cuda")
    if flat.size:
        buf[off + base:off + base + flat.size] = torch.from_numpy(flat).cuda()
    return buf[off:], torch.from_numpy(offs.astype(np.int64) + base).cuda()


def host(x):
    return np.asarray(x.cpu() if hasattr(x, "cpu") else x)


@pytest.mark.gpu
def test_gpu_suite_vectors_one_call_per_suite(engine):
    for s in suites():
        msgs, dst, ro = suite_msgs(s), s["dst"].encode(), s["random_oracle"]
        for out, st in (engine.hash_to_curve_varlen(dst, msgs, ro), engine.hash_to_curve_varlen(dst, dev_ragged(msgs, 3), ro)):
            assert host(st).tolist() == [1] * 5
            assert [o.tobytes() for o in host(out)] == suite_points(s)


@pytest.mark.gpu
@pytest.mark.parametrize("L", EQUAL_LENS)
def test_gpu_equal_lengths_match_uniform_call(engine, L):
    """Ragged rows that all have length L give byte for byte what the uniform call gives with msg_len = L."""
    rng = np.random.default_rng(L)
    n = 300
    msg = rng.integers(0, 256, (n, L), dtype=np.uint8)
    msgs = [m.tobytes() for m in msg]
    for ro in (True, False):
        want = engine.hash_to_curve(SUITE_DST, msg, ro)
        want = (np.array(want[0]), np.array(want[1]))
        assert want[1].all()
        for got in (engine.hash_to_curve_varlen(SUITE_DST, msgs, ro), engine.hash_to_curve_varlen(SUITE_DST, dev_ragged(msgs, 1), ro),
                    engine.hash_to_curve(SUITE_DST, dev(msg), ro)):
            assert np.array_equal(host(got[0]), want[0]) and np.array_equal(host(got[1]), want[1]), (L, ro)


@pytest.mark.gpu
def test_gpu_mixed_lengths_match_oracle(engine, oracle):
    msgs = random_rows(3000, 31)
    for ro in (True, False):
        out, st = (np.array(x) for x in engine.hash_to_curve_varlen(SUITE_DST, msgs, ro))
        d_out, d_st = engine.hash_to_curve_varlen(SUITE_DST, dev_ragged(msgs, 2, 9), ro)
        assert np.array_equal(host(d_out), out) and np.array_equal(host(d_st), st)
        sample = sorted(set(np.random.default_rng(ro).integers(0, len(msgs), 96).tolist()) | {0, len(msgs) - 1})
        want, wst = oracle_rows(oracle, SUITE_DST, [msgs[i] for i in sample], ro)
        assert np.array_equal(out[sample], want) and np.array_equal(st[sample], wst)


@pytest.mark.gpu
def test_gpu_one_mib_message_among_short_ones(engine, oracle):
    rng = np.random.default_rng(5)
    msgs = [b"", rng.bytes(33), rng.bytes(1 << 20)] + random_rows(61, 5, hi=100)
    want, wst = oracle_rows(oracle, SUITE_DST, msgs, True)
    for got in (engine.hash_to_curve_varlen(SUITE_DST, msgs), engine.hash_to_curve_varlen(SUITE_DST, dev_ragged(msgs, 7))):
        assert np.array_equal(host(got[0]), want) and np.array_equal(host(got[1]), wst)


@pytest.mark.gpu
def test_gpu_dev_misaligned_inputs_and_outputs(engine, oracle):
    import torch
    lib, ctx = engine._lib, engine._ctx
    msgs = random_rows(200, 17, hi=300)
    want, wst = oracle_rows(oracle, SUITE_DST, msgs, True)
    n = len(msgs)
    for off in (1, 2, 3):
        for base in (0, 5):
            d_msg, d_offs = dev_ragged(msgs, off, base)
            obuf = torch.zeros(65 * n + off, dtype=torch.uint8, device="cuda")
            sbuf = torch.zeros(n + off, dtype=torch.uint8, device="cuda")
            rc = lib.s256_hash_to_curve_varlen_dev(ctx, SUITE_DST, C.c_size_t(len(SUITE_DST)), C.c_void_p(d_msg.data_ptr()),
                                                   C.c_void_p(d_offs.data_ptr()), C.c_size_t(n), 1,
                                                   C.c_void_p(obuf.data_ptr() + off), C.c_void_p(sbuf.data_ptr() + off),
                                                   engine._stream())
            assert rc == 0
            torch.cuda.synchronize()
            assert np.array_equal(obuf[off:].cpu().numpy().reshape(n, 65), want), (off, base)
            assert np.array_equal(sbuf[off:].cpu().numpy(), wst), (off, base)
    # the uniform _dev form on a misaligned message block and output
    msg = np.random.default_rng(18).integers(0, 256, (n, 37), dtype=np.uint8)
    uw, uwst = (np.array(x) for x in engine.hash_to_curve(SUITE_DST, msg, False))
    mbuf = torch.zeros(msg.size + 3, dtype=torch.uint8, device="cuda")
    mbuf[3:] = dev(msg.reshape(-1))
    obuf = torch.zeros(65 * n + 1, dtype=torch.uint8, device="cuda")
    sbuf = torch.zeros(n + 1, dtype=torch.uint8, device="cuda")
    assert lib.s256_hash_to_curve_dev(ctx, SUITE_DST, C.c_size_t(len(SUITE_DST)), C.c_void_p(mbuf.data_ptr() + 3), C.c_size_t(37),
                                      C.c_size_t(n), 0, C.c_void_p(obuf.data_ptr() + 1), C.c_void_p(sbuf.data_ptr() + 1),
                                      engine._stream()) == 0
    torch.cuda.synchronize()
    assert np.array_equal(obuf[1:].cpu().numpy().reshape(n, 65), uw) and np.array_equal(sbuf[1:].cpu().numpy(), uwst)


@pytest.mark.gpu
def test_gpu_decreasing_offsets(engine, oracle):
    import torch
    lib, ctx = engine._lib, engine._ctx
    msgs = random_rows(40, 23, hi=150)
    msgs[5] = msgs[5] or b"y"
    flat, offs = ragged(msgs)
    bad = decreasing_at(offs, 5)
    out, st = engine.hash_to_curve_varlen(SUITE_DST, (dev(flat), torch.from_numpy(bad.astype(np.int64)).cuda()))
    out, st = host(out), host(st)
    assert st[5] == 0 and not out[5].any()
    keep = [i for i in range(len(msgs)) if i != 5]
    rows = [flat[int(bad[i]):int(bad[i + 1])].tobytes() for i in keep]
    want, wst = oracle_rows(oracle, SUITE_DST, rows, True)
    assert np.array_equal(out[keep], want) and np.array_equal(st[keep], wst) and wst.all()
    # the host form refuses the same offsets before enqueueing anything
    hp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    o65, ost = np.full((len(msgs), 65), 7, np.uint8), np.full(len(msgs), 7, np.uint8)
    assert lib.s256_hash_to_curve_varlen(ctx, SUITE_DST, C.c_size_t(len(SUITE_DST)), hp(flat), hp(bad), C.c_size_t(len(msgs)), 1,
                                         hp(o65), hp(ost)) == -3
    assert (o65 == 7).all() and (ost == 7).all()


@pytest.mark.gpu
def test_gpu_empty_null_and_side_stream(engine):
    import torch
    lib, ctx = engine._lib, engine._ctx
    dl = C.c_size_t(len(SUITE_DST))
    out, st = engine.hash_to_curve_varlen(SUITE_DST, [])
    assert out.shape == (0, 65) and st.size == 0
    d0, o0 = torch.zeros(0, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda")
    out, st = engine.hash_to_curve_varlen(SUITE_DST, (d0, o0))
    assert out.shape == (0, 65) and st.numel() == 0
    out, st = engine.hash_to_curve(SUITE_DST, torch.zeros((0, 4), dtype=torch.uint8, device="cuda"))
    assert out.shape == (0, 65)
    buf = (C.c_uint8 * 256)()
    offs = (C.c_size_t * 2)(0, 32)
    one, zero, s = C.c_size_t(1), C.c_size_t(0), engine._stream()
    hv, dv, ud = lib.s256_hash_to_curve_varlen, lib.s256_hash_to_curve_varlen_dev, lib.s256_hash_to_curve_dev
    for args in ((None, SUITE_DST, dl, buf, offs, one, 1, buf, buf), (ctx, None, dl, buf, offs, one, 1, buf, buf),
                 (ctx, SUITE_DST, zero, buf, offs, one, 1, buf, buf), (ctx, SUITE_DST, dl, None, offs, one, 1, buf, buf),
                 (ctx, SUITE_DST, dl, buf, None, one, 1, buf, buf), (ctx, SUITE_DST, dl, buf, offs, one, 1, None, buf),
                 (ctx, SUITE_DST, dl, buf, offs, one, 1, buf, None)):
        assert hv(*args) == -3, args
    assert hv(ctx, SUITE_DST, zero, buf, offs, zero, 1, buf, buf) == -3  # errInvalidDomainSep, even with no rows
    assert dv(ctx, SUITE_DST, zero, None, None, zero, 1, None, None, s) == -3
    assert dv(ctx, None, dl, None, None, zero, 1, None, None, s) == -3
    assert ud(ctx, SUITE_DST, zero, None, zero, zero, 1, None, None, s) == -3
    for i in (3, 4, 7, 8):  # d_msg, d_offsets, d_out65, d_status
        args = [ctx, SUITE_DST, dl, buf, buf, one, 1, buf, buf, s]
        args[i] = None
        assert dv(*args) == -3, i
    assert ud(ctx, SUITE_DST, dl, None, C.c_size_t(4), one, 1, buf, buf, s) == -3
    assert ud(ctx, SUITE_DST, dl, buf, C.c_size_t(4), one, 1, None, buf, s) == -3
    assert ud(ctx, SUITE_DST, dl, buf, C.c_size_t(4), one, 1, buf, None, s) == -3
    assert dv(None, SUITE_DST, dl, buf, buf, one, 1, buf, buf, s) == -3 and ud(None, SUITE_DST, dl, buf, zero, one, 1, buf, buf, s) == -3
    empty = (C.c_size_t * 2)(5, 5)  # one empty row: msg may be NULL on the host
    o65, ost = (C.c_uint8 * 65)(), (C.c_uint8 * 1)()
    assert hv(ctx, SUITE_DST, dl, None, empty, one, 1, o65, ost) == 0 and ost[0] == 1
    assert bytes(o65) == hash_of_empty(engine)
    # a side stream: results read after that stream is synchronised
    msgs = random_rows(4096, 41, hi=200)
    want = np.array(engine.hash_to_curve_varlen(SUITE_DST, msgs)[0])
    d_msg = dev_ragged(msgs, 1)
    k = torch.from_numpy(np.frombuffer(hashlib.sha256(b"k").digest() * 4096, np.uint8).copy()).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for _ in range(3):
        engine.scalar_base_mult(k)
        with torch.cuda.stream(side):
            out, st = engine.hash_to_curve_varlen(SUITE_DST, d_msg)
        side.synchronize()
        assert np.array_equal(out.cpu().numpy(), want) and bool(st.cpu().numpy().all())


def hash_of_empty(engine):
    return np.array(engine.hash_to_curve(SUITE_DST, np.zeros((1, 0), np.uint8))[0]).tobytes()


@pytest.mark.gpu
def test_gpu_small_context_chunks_cut_through_the_batch(s256, engine, oracle):
    """max_batch 512: chunks of 512 rows cut through the ragged byte ranges; and max_batch 2^18 with 2^18 + 5000 rows,
    so that the host form's first chunk runs as four pipeline parts on two streams."""
    for cap, n in ((512, 3 * 512 + 5), (1 << 18, (1 << 18) + 5000)):
        small = s256.Engine(max_batch=cap)
        try:
            msgs = random_rows(n, cap, hi=120)
            want = [x.cpu().numpy() for x in engine.hash_to_curve_varlen(SUITE_DST, dev_ragged(msgs))]
            got_host = small.hash_to_curve_varlen(SUITE_DST, msgs)
            got_dev = small.hash_to_curve_varlen(SUITE_DST, dev_ragged(msgs, 3, 2))
            for got in (got_host, got_dev):
                assert np.array_equal(host(got[0]), want[0]) and np.array_equal(host(got[1]), want[1]), cap
            cuts = [(cap // 64 * c + 127) & ~127 for c in (6, 24, 44)]  # ctx.h pipelined
            edges = sorted({e for c in [512, 1024, cap] + cuts for e in (c - 1, c) if e < n} | {0, n - 1})
            ow, ows = oracle_rows(oracle, SUITE_DST, [msgs[i] for i in edges], True)
            assert np.array_equal(want[0][edges], ow) and np.array_equal(want[1][edges], ows)
        finally:
            small.close()


@pytest.mark.gpu
def test_gpu_full_size_ragged_equals_uniform_and_chains_into_ecdh(engine):
    import torch
    n = 1 << 20
    rng = np.random.default_rng(20)
    msg = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    d_msg = dev(msg)
    offs = torch.arange(0, 32 * (n + 1), 32, dtype=torch.int64, device="cuda")
    for ro in (True, False):
        u_out, u_st = engine.hash_to_curve(SUITE_DST, d_msg, ro)
        r_out, r_st = engine.hash_to_curve_varlen(SUITE_DST, (d_msg.view(-1), offs), ro)
        assert torch.equal(u_out, r_out) and torch.equal(u_st, r_st) and bool((u_st == 1).all())
    # hash ragged items to points and multiply them by one key, on the device, against the host chain
    lens = rng.integers(0, 257, n)
    ho = np.zeros(n + 1, np.uint64)
    np.cumsum(lens, out=ho[1:])
    flat = rng.integers(0, 256, int(ho[-1]), dtype=np.uint8)
    key = np.frombuffer(hashlib.sha256(b"psi key").digest(), np.uint8)
    k = np.ascontiguousarray(np.broadcast_to(key, (n, 32)))
    pts, st = engine.hash_to_curve_varlen(SUITE_DST, (dev(flat), torch.from_numpy(ho.astype(np.int64)).cuda()))
    x_dev, xs_dev = engine.ecdh(dev(k), pts)
    msgs = [flat[ho[i]:ho[i + 1]] for i in range(n)]
    h_pts, h_st = engine.hash_to_curve_varlen(SUITE_DST, msgs)
    h_pts, h_st = np.array(h_pts), np.array(h_st)
    x_host, xs_host = (np.array(a) for a in engine.ecdh(k, h_pts))
    assert np.array_equal(st.cpu().numpy(), h_st) and h_st.all()
    assert np.array_equal(pts.cpu().numpy(), h_pts)
    assert np.array_equal(x_dev.cpu().numpy(), x_host) and np.array_equal(xs_dev.cpu().numpy(), xs_host) and xs_host.all()


@pytest.mark.gpu
def test_gpu_mirror(s256):
    exe = build_mirror(s256)
    s = suites()[0]
    msgs = suite_msgs(s) + [bytes(range(64)), b"\xff" * 200]
    r = subprocess.run([exe, s["dst"]] + [m.hex() or "-" for m in msgs], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "h2c varlen mirror ok" in r.stdout
