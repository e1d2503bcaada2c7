"""The kernel variants that batch size selects, and the device-resident entry points that reach them.

Batch size picks the kernel that runs in two places:
  * the inversion-group size K of the group kernels (Montgomery's trick: K rows share one inversion) --
    k_finish_affine<K> (projective -> affine + encoding behind every entry point that returns a point, an
    x-coordinate or a recovered key), k_ecdsa_scalars<K, RECOVER> and k_sign_finish<K>;
  * the fixed-base kernel: k_base_mult_ct_split<8> up to 8192 rows, split<4> up to 16384, k_base_mult_ct_w7 above.
The host-pointer calls cut a chunk into sub-chunks below 2^19 rows, so K = 32 runs only in the *_dev forms on a chunk
of at least 2^19 rows.  These tests run every *_dev entry point at the sizes where K changes, with invalid rows and rows
whose result is the identity planted at the edges of the inversion groups and warps, and check every row against
closed forms, the host-pointer path (another K on the same rows) and a sample against the oracle.  The host simulation
runs the same planted rows for each K on the CPU."""
import ctypes as C

import numpy as np
import pytest

import hostsim as hs
import parity_suites as ps
from hostsim import group as group_sim

synth = ps.synth
N, P = ps.N, ps.P


# ---------------------------------------------------------------------------
# Layout of the group kernels.  This mirrors ctx.h (inv_k_for) and the strides of api.cu (k_finish_affine,
# k_ecdsa_scalars) and api_sign.cu (k_sign_finish).  If those rules change the tests stay correct, but the planted
# rows no longer land on the edges they were chosen for.
# ---------------------------------------------------------------------------
def inv_k_for(n):
    return 32 if n >= 1 << 19 else (4 if n >= 1 << 16 else 1)


def group_stride(n, k):
    """k_ecdsa_scalars / k_sign_finish: thread t owns rows t + m * stride, m < k."""
    return -(-n // k)


def finish_stride(n, k):
    """k_finish_affine: the same, with the stride rounded up to a multiple of 32 so that a warp's rows are contiguous."""
    return (group_stride(n, k) + 31) // 32 * 32


def layout_rows(n, k, stride):
    """Rows at the edges of the groups and warps of a group kernel over n rows: thread t converts rows t + m * stride
    (m < k, row < n) with one shared inversion, and 32 consecutive threads form a warp.  -> {edge name: sorted rows}."""
    def members(t):
        return [t + m * stride for m in range(k) if t + m * stride < n]

    # groups t < first_partial have all k members, the later ones fewer (or none)
    first_partial = min(max(n - (k - 1) * stride, 0), stride)
    top = min(stride, n) - 1  # the last thread with a row; later ones (stride > n) have empty groups
    live = [t for t in (top, top - 1, first_partial, first_partial + 1) if 0 <= t <= top]
    mid = first_partial // 2
    picks = [min(mid + d, top) for d in range(5)]
    out = {
        "whole group": members(picks[0]),
        "position 0 only": [picks[1]],
        "last position only": [members(picks[2])[-1]],
        "alternating positions": members(picks[3])[::2] + members(picks[4])[1::2],
        "partial groups": sorted({r for t in live for r in (members(t)[0], members(t)[-1])}),
    }
    warps = []
    last_m = (n - 1) // stride
    for m in sorted({0, min(k - 1, last_m), last_m}):
        w_tail = ((n - 1 - m * stride) // 32) if m == last_m else (stride - 1) // 32
        for w in sorted({0, (stride - 1) // 32, w_tail}):
            lo = 32 * w + m * stride
            hi = min(32 * w + 31, stride - 1) + m * stride
            rows_ = [r for r in (lo, hi, min(hi, n - 1)) if lo <= r < n]
            warps += rows_
    out["warp edges"] = sorted(set(warps))
    return {name: sorted(set(r)) for name, r in out.items()}


def plant_positions(n, strides):
    """Ordered, de-duplicated rows from the layouts of every (k, stride) an entry point runs."""
    seen, order = set(), []
    for k, stride in strides:
        for rows_ in layout_rows(n, k, stride).values():
            for r in rows_:
                if r not in seen:
                    seen.add(r)
                    order.append(r)
    return order


def neighbours(rows_, n):
    return sorted({min(max(r + d, 0), n - 1) for r in rows_ for d in (-1, 0, 1)})


# which group kernels (and so which strides) each entry point runs
FINISH, GROUP = "finish", "group"
ENTRY_LAYOUTS = {
    "scalar_base_mult": (FINISH,), "scalar_mult": (FINISH,), "ecdh": (FINISH,), "double_scalar_mult": (FINISH,),
    "recover": (FINISH, GROUP), "verify": (GROUP,), "sign": (FINISH, GROUP), "schnorr_sign": (FINISH,),
}


def entry_strides(entry, n, k=None):
    k = inv_k_for(n) if k is None else k
    return [(k, finish_stride(n, k) if kind == FINISH else group_stride(n, k)) for kind in ENTRY_LAYOUTS[entry]]


# ---------------------------------------------------------------------------
# Inputs: one set of rows at the largest size; every test takes a prefix and plants its own rows
# ---------------------------------------------------------------------------
def ints_rows(ints):
    return synth._be32_rows(ints)


def make_inputs(n, base_mult, sign, tag=b""):
    """Rows for every entry point: keys d and their points, scalars and closed-form scalars, RFC 6979 signatures
    (with recovery ids) from `sign`, BIP-340 messages and aux.  base_mult / sign run the rows through a
    reference (the oracle, or the engine's host-pointer path, which other tests pin to the oracle)."""
    d = [synth._nonzero_mod_n(x) for x in synth._stream_ints(b"key" + tag, 0, n, synth.SEED)]
    k = [synth._nonzero_mod_n(x) for x in synth._stream_ints(b"ecdh" + tag, 0, n, synth.SEED)]
    u1 = [x % N for x in synth._stream_ints(b"u1" + tag, 0, n, synth.SEED)]
    u2 = [x % N for x in synth._stream_ints(b"u2" + tag, 0, n, synth.SEED)]
    w = {"d": d, "priv": ints_rows(d), "k32": ints_rows(k), "u1": ints_rows(u1), "u2": ints_rows(u2),
         "dg": np.frombuffer(b"".join(synth.D(b"msg" + tag, i) for i in range(n)), np.uint8).reshape(n, 32).copy(),
         "aux": np.frombuffer(b"".join(synth.D(b"aux" + tag, i) for i in range(n)), np.uint8).reshape(n, 32).copy(),
         "sbm_k": synth.base_mult_scalars(n, start=8)}   # (rows 0-7 of the stream are forced edge values)
    pk, st = base_mult(w["priv"])
    assert (np.asarray(st) == 1).all()
    w["pk65"] = np.array(pk, np.uint8)
    w["pkx"] = w["pk65"][:, 1:33].copy()
    cf, st = base_mult(ints_rows([a * b % N for a, b in zip(k, d)]))
    w["cf_scalar_mult"] = np.array(cf, np.uint8)
    cf, st = base_mult(ints_rows([(a + b * c) % N for a, b, c in zip(u1, u2, d)]))
    w["cf_dsm"], w["cf_dsm_st"] = np.array(cf, np.uint8), np.array(st, np.uint8)
    sig, rec, st = sign(w["priv"], w["dg"])
    assert (np.asarray(st) == 1).all()
    w["sig64"] = np.array(sig, np.uint8)
    w["sig65"] = np.concatenate([w["sig64"], np.asarray(rec, np.uint8).reshape(-1, 1)], axis=1)
    return w


def identity_recover_rows(count, o):
    """(digest, r||s||v) rows whose recovered key is the identity: R = k G, r = x(R) mod n, s = e / k, v = parity of
    y(R) (x(R) >= n has probability 2^-128): then u1 G + u2 R = (-e / r) G + (e / (k r)) k G = O."""
    ks = [synth._nonzero_mod_n(x) for x in synth._stream_ints(b"identity-k", 0, count, synth.SEED)]
    es = [synth._nonzero_mod_n(x) for x in synth._stream_ints(b"identity-e", 0, count, synth.SEED)]
    R, st = o.batch_scalar_base_mult(ints_rows(ks))
    assert (st == 1).all()
    dg, sig = [], []
    for j in range(count):
        x = int.from_bytes(R[j, 1:33].tobytes(), "big")
        assert x < N
        r, s = x % N, es[j] * pow(ks[j], -1, N) % N
        dg.append(es[j].to_bytes(32, "big"))
        sig.append(r.to_bytes(32, "big") + s.to_bytes(32, "big") + bytes([R[j, 64] & 1]))
    return ps.rows(dg, 32), ps.rows(sig, 65)


# planted kinds per entry point: (name, status the row must come back with).  The first kind of each list is the
# one that lands on the single-row edges (position 0 only, last position only).
KINDS = {
    "scalar_base_mult": [("k = 0", 2), ("k = n", 2)],
    "scalar_mult": [("k = 0", 2), ("k = n", 2), ("bad prefix", 0), ("off the curve", 0), ("x = p", 0)],
    "ecdh": [("k = 0", 2), ("k = n", 2), ("bad prefix", 0), ("off the curve", 0), ("x = p", 0)],
    "double_scalar_mult": [("u1 = u2 = 0", 2), ("u1 = -u2 d", 2), ("u1 G = u2 P", 1), ("bad point", 0)],
    "recover": [("r = 0", 0), ("v >= 4", 0), ("r + n >= p", 0), ("identity", 0)],
    "verify": [("s = 0", 0), ("s >= n", 0), ("r = 0", 0)],
    "sign": [("d = 0", 0), ("d = n", 0), ("d = 2^256 - 1", 0)],
    "schnorr_sign": [("d = 0", 0), ("d = n", 0)],
}
INPUTS = {
    "scalar_base_mult": ("sbm_k",), "scalar_mult": ("k32", "pk65"), "ecdh": ("k32", "pk65"),
    "double_scalar_mult": ("u1", "u2", "pk65"), "recover": ("dg", "sig65"), "verify": ("pk65", "dg", "sig64"),
    "sign": ("priv", "dg"), "schnorr_sign": ("priv", "dg", "aux"),
}


def plant(entry, w, n, positions, ident_rows):
    """Prefix copies of the inputs of `entry` with planted rows at `positions`.  -> (inputs, expected status, planted
    row -> kind name)"""
    ins = [w[name][:n].copy() for name in INPUTS[entry]]
    exp = np.ones(n, np.uint8)
    planted = {}
    kinds = KINDS[entry]
    for j, r in enumerate(positions):
        kind, status = kinds[j % len(kinds)]
        planted[r] = kind
        exp[r] = status
        if entry == "scalar_base_mult":
            ins[0][r] = np.frombuffer(ps.b32(0 if kind == "k = 0" else N), np.uint8)
        elif entry in ("scalar_mult", "ecdh"):
            k, pt = ins
            if kind in ("k = 0", "k = n"):
                k[r] = np.frombuffer(ps.b32(0 if kind == "k = 0" else N), np.uint8)
            elif kind == "bad prefix":
                pt[r, 0] = 0x05
            elif kind == "off the curve":
                pt[r, 64] ^= 1
            else:
                pt[r, 1:33] = np.frombuffer(ps.b32(P), np.uint8)
        elif entry == "double_scalar_mult":
            u1, u2, pt = ins
            if kind == "u1 = u2 = 0":
                u1[r] = 0
                u2[r] = 0
            elif kind == "u1 = -u2 d":
                u1[r] = np.frombuffer(ps.b32(-int.from_bytes(u2[r].tobytes(), "big") * w["d"][r] % N), np.uint8)
            elif kind == "u1 G = u2 P":
                u1[r] = np.frombuffer(ps.b32(int.from_bytes(u2[r].tobytes(), "big") * w["d"][r] % N), np.uint8)
            else:
                pt[r, 33:65] = pt[r, 1:33]
        elif entry == "recover":
            dg, sig = ins
            if kind == "r = 0":
                sig[r, :32] = 0
            elif kind == "v >= 4":
                sig[r, 64] = 4 | (sig[r, 64] & 3)
            elif kind == "r + n >= p":
                sig[r, :32] = np.frombuffer(ps.b32(P - N + r % 1000), np.uint8)
                sig[r, 64] = 2 | (sig[r, 64] & 1)
            else:
                j2 = j % len(ident_rows[0])
                dg[r], sig[r] = ident_rows[0][j2], ident_rows[1][j2]
        elif entry == "verify":
            sig = ins[2]
            if kind == "s = 0":
                sig[r, 32:] = 0
            elif kind == "s >= n":
                sig[r, 32:] = np.frombuffer(ps.b32(N + r % 1000), np.uint8)
            else:
                sig[r, :32] = 0
        else:  # sign, schnorr_sign
            v = {"d = 0": 0, "d = n": N, "d = 2^256 - 1": 2**256 - 1}[kind]
            ins[0][r] = np.frombuffer(ps.b32(v), np.uint8)
    return ins, exp, planted


def call(be, entry, ins):
    """The entry point of an Engine (host arrays or CUDA tensors) or of the host simulation; outputs as numpy."""
    f = {"scalar_base_mult": "scalar_base_mult", "scalar_mult": "scalar_mult", "ecdh": "ecdh",
         "double_scalar_mult": "double_scalar_mult_basepoint_vartime", "recover": "ecdsa_recover",
         "verify": "ecdsa_verify", "sign": "ecdsa_sign_rfc6979", "schnorr_sign": "schnorr_sign"}[entry]
    out = getattr(be, f)(*ins)
    out = out if isinstance(out, tuple) else (out,)
    return tuple(np.array(o.cpu() if hasattr(o, "cpu") else o, np.uint8) for o in out)


def oracle_rows(o, entry, ins, idx):
    sub = [np.ascontiguousarray(a[idx]) for a in ins]
    if entry == "schnorr_sign":
        got = [o.schnorr_sign(p.tobytes(), m.tobytes(), a.tobytes()) for p, m, a in zip(*sub)]
        return (ps.rows([g[0] for g in got], 64).reshape(-1, 64), np.array([g[1] for g in got], np.uint8))
    f = {"scalar_base_mult": o.batch_scalar_base_mult, "scalar_mult": o.batch_scalar_mult, "ecdh": o.batch_ecdh,
         "double_scalar_mult": o.batch_double_scalar_mult, "recover": o.batch_ecdsa_recover,
         "verify": o.batch_ecdsa_verify, "sign": o.batch_ecdsa_sign_rfc6979}[entry]
    out = f(*sub)
    return out if isinstance(out, tuple) else (out,)


def off_curve_rows(out65, st):
    """Status-1 rows that are not 04 || x || y with y^2 = x^3 + 7 (mod p): a wrong inverse from a mixed-up group
    lands off the curve with overwhelming probability."""
    idx = np.nonzero(st == 1)[0]
    raw = np.ascontiguousarray(out65[idx]).tobytes()
    bad = []
    for j, i in enumerate(idx):
        o = 65 * j
        x, y = int.from_bytes(raw[o + 1:o + 33], "big"), int.from_bytes(raw[o + 33:o + 65], "big")
        if raw[o] != 4 or x >= P or y >= P or (y * y - x * x * x - 7) % P:
            bad.append(int(i))
    return bad


def check_status_and_encoding(entry, out, exp, planted):
    """Check 1: the status byte is what the planted row demands, rows that are not status 1 are all zero bytes, and
    every point that comes back is on the curve."""
    st = out[-1]
    wrong = np.nonzero(st != exp)[0]
    assert len(wrong) == 0, [(int(i), planted.get(int(i), "valid"), int(st[i]), int(exp[i])) for i in wrong[:8]]
    if entry == "verify":
        return
    for o in out[:-1]:
        assert not o[st != 1].any(), f"{entry}: a row that is not status 1 has non-zero output bytes"
    if entry in ("scalar_base_mult", "scalar_mult", "double_scalar_mult", "recover"):
        bad = off_curve_rows(out[0], st)
        assert not bad, f"{entry}: status-1 rows off the curve: {bad[:8]}"


def check_closed_form(entry, out, w, n, planted, host_verify=None):
    """Check 2: every row that was not planted against a closed form built from Python integers mod n, whose points
    come from a reference ScalarBaseMult."""
    keep = np.ones(n, bool)
    keep[list(planted)] = False
    if entry == "scalar_mult":
        assert np.array_equal(out[0][keep], w["cf_scalar_mult"][:n][keep])
    elif entry == "ecdh":
        assert np.array_equal(out[0][keep], w["cf_scalar_mult"][:n, 1:33][keep])
    elif entry == "double_scalar_mult":
        assert np.array_equal(out[0][keep], w["cf_dsm"][:n][keep])
        assert np.array_equal(out[1][keep], w["cf_dsm_st"][:n][keep])
    elif entry == "recover":
        assert np.array_equal(out[0][keep], w["pk65"][:n][keep])
    elif entry == "sign":
        assert np.array_equal(out[0][keep], w["sig64"][:n][keep])
        assert np.array_equal(out[1][keep], w["sig65"][:n, 64][keep])
    elif entry == "schnorr_sign":
        ok = host_verify(w["pkx"][:n], w["dg"][:n], out[0])
        assert np.array_equal(np.asarray(ok)[keep], np.ones(int(keep.sum()), np.uint8))


def check_oracle(o, entry, ins, out, idx):
    exp = oracle_rows(o, entry, ins, idx)
    for g, e in zip(out, exp):
        bad = np.nonzero((g[idx] != e).reshape(len(idx), -1).any(axis=1))[0]
        assert len(bad) == 0, f"{entry}: rows differ from the oracle: {[int(idx[b]) for b in bad[:8]]}"


def base_mult_edge_scalars():
    """Scalars at the boundaries of the signed fixed-base recoding, each twice in a row (an even and an odd index):
    every single window digit at +-1, at the largest magnitude 2^(WB-1) and at 2^(WB-1) + 1, runs of carries, the top
    window with its small range, values around n and n/2 -- for the 5-bit windows of the lane-split kernels
    (n <= 16384) and the 6- and 7-bit windows of the throughput kernels."""
    vals = [0, 1, 2, N - 1, N - 2, N, N + 1, 2**256 - 1, N // 2, N // 2 + 1, 2**252, 2**252 - 1, 2**252 + 1, 15 * 2**252,
            2**255, 2**256 - N, 2 * (2**256 - N)]
    for wb in (5, 6, 7):
        nw = (257 + wb - 1) // wb
        for w in range(nw):
            vals += [(1 << (wb * w)) % N, ((1 << (wb - 1)) << (wb * w)) % N, (((1 << (wb - 1)) + 1) << (wb * w)) % N]
        vals += [sum(((1 << (wb - 1)) + 1) << (wb * w) for w in range(nw - 1)) % N,
                 sum(((1 << wb) - 1) << (wb * w) for w in range(nw - 1)) % N, sum(1 << (wb * w) for w in range(nw)) % N]
    return ps.rows([ps.b32(v % 2**256) for v in vals for _ in (0, 1)], 32)


# ---------------------------------------------------------------------------
# CPU: the layout helper, and the host simulation for every K
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 20, 31, 32, 33, 70, 131, 2000, 65535, 65539, 524287, 524321, 1 << 20])
def test_layout_rows_are_at_the_edges(n):
    for k in (1, 4, 32):
        for stride in (group_stride(n, k), finish_stride(n, k)):
            lay = layout_rows(n, k, stride)
            rows_ = [r for v in lay.values() for r in v]
            assert rows_ and all(0 <= r < n for r in rows_)
            # every row lies in exactly one group: t = r mod stride, position r // stride < k
            assert all(r // stride < k for r in rows_)
            assert n - 1 in lay["warp edges"]
            whole = lay["whole group"]
            assert all(b - a == stride for a, b in zip(whole, whole[1:]))
            if n >= k * stride:   # every group is whole
                assert len(whole) == k and len(lay["partial groups"]) <= 4
    assert finish_stride(524321, 32) == 16416 and group_stride(524321, 32) == 16386
    assert [inv_k_for(n) for n in (65535, 65536, 524287, 524288)] == [1, 4, 4, 32]


# n for the host simulation: with K = 1, 4 and 32 these have whole, partial and (for the finish stride) empty groups
HOSTSIM_SIZES = (20, 131, 2000)


@pytest.fixture(scope="module")
def cpu_rows(oracle):
    n = max(HOSTSIM_SIZES)
    w = make_inputs(n, oracle.batch_scalar_base_mult, oracle.batch_ecdsa_sign_rfc6979, tag=b"-hostsim")
    return w, identity_recover_rows(16, oracle)


HOSTSIM_ENTRIES = ("recover", "double_scalar_mult", "scalar_mult", "ecdh", "scalar_base_mult", "sign", "verify")


@pytest.mark.parametrize("k", [1, 4, 32])
@pytest.mark.parametrize("entry", HOSTSIM_ENTRIES)
def test_hostsim_group_kernels_for_every_k(oracle, cpu_rows, entry, k):
    """The group kernels of csrc/kernels.cuh at one K, with planted rows at that K's group and warp edges: every row
    against the oracle, the closed forms and the status the planted row demands."""
    w, ident = cpu_rows
    be = group_sim.Backend(k)
    for n in HOSTSIM_SIZES:
        positions = plant_positions(n, entry_strides(entry, n, k))
        ins, exp, planted = plant(entry, w, n, positions, ident)
        out = call(be, entry, ins)
        check_status_and_encoding(entry, out, exp, planted)
        check_closed_form(entry, out, w, n, planted)
        check_oracle(oracle, entry, ins, out, np.arange(n))


def test_hostsim_schnorr_sign_for_every_k(oracle, cpu_rows):
    w, _ = cpu_rows
    n = 131
    for k in (1, 4, 32):
        ins, exp, planted = plant("schnorr_sign", w, n, plant_positions(n, entry_strides("schnorr_sign", n, k)), None)
        out = call(group_sim.Backend(k), "schnorr_sign", ins)
        check_status_and_encoding("schnorr_sign", out, exp, planted)
        check_closed_form("schnorr_sign", out, w, n, planted, host_verify=hs.schnorr_verify)
        check_oracle(oracle, "schnorr_sign", ins, out, np.arange(n))


def test_hostsim_lane_split_base_mult_edges(oracle):
    """The recoding edges through the lane-split form (T = 8 and T = 4 lanes per scalar, 5-bit windows), which the
    simulation takes for calls of at most 8 rows."""
    ks = base_mult_edge_scalars()
    exp, est = oracle.batch_scalar_base_mult(ks)
    for a in range(0, len(ks), 8):
        got, st = hs.scalar_base_mult(ks[a:a + 8])
        assert np.array_equal(got, exp[a:a + 8]) and np.array_equal(st, est[a:a + 8]), a


def test_hostsim_group_size_must_be_one_the_device_uses():
    for k in (0, 2, 8, 16, 64):
        with pytest.raises(ValueError):
            group_sim.Backend(k)


# ---------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------
GPU_SIZES = (65535, 65539, 524287, 524321, 1 << 20)
CHUNKED_N = (1 << 20) + 40
ORACLE_SPREAD = 2048


def torch_cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def gpu_rows(engine, oracle):
    """Inputs at the largest size, made with the engine's host-pointer path (sub-chunks below 2^19 rows: K <= 4)."""
    w = make_inputs(CHUNKED_N, engine.scalar_base_mult, engine.ecdsa_sign_rfc6979)
    # the references themselves, on a sample against the oracle
    idx = np.arange(0, CHUNKED_N, CHUNKED_N // 512)
    eo, es = oracle.batch_scalar_base_mult(w["priv"][idx])
    assert np.array_equal(w["pk65"][idx], eo)
    so, ro, sto = oracle.batch_ecdsa_sign_rfc6979(w["priv"][idx], w["dg"][idx])
    assert np.array_equal(w["sig64"][idx], so) and np.array_equal(w["sig65"][idx, 64], ro)
    return w, identity_recover_rows(64, oracle)


def dev_call(engine, entry, ins):
    import torch
    out = call(engine, entry, [torch_cuda(a) for a in ins])
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", GPU_SIZES)
@pytest.mark.parametrize("entry", ["scalar_base_mult", "scalar_mult", "ecdh", "double_scalar_mult", "recover", "verify",
                                   "sign", "schnorr_sign"])
def test_dev_entry_point_at_group_size_edges(engine, oracle, gpu_rows, entry, n):
    """One *_dev call over n rows (one chunk, so K = inv_k_for(n)), with planted rows at that K's group and warp edges:
    every row against the status the planted row demands and the closed form, every row against the host-pointer path
    (sub-chunks, another K above 2^18 rows), and the planted rows, their neighbours and a spread sample against the
    oracle."""
    w, ident = gpu_rows
    positions = plant_positions(n, entry_strides(entry, n))
    ins, exp, planted = plant(entry, w, n, positions, ident)
    out = dev_call(engine, entry, ins)
    check_status_and_encoding(entry, out, exp, planted)
    check_closed_form(entry, out, w, n, planted, host_verify=engine.schnorr_verify)
    if entry == "sign":
        keep = np.ones(n, bool)
        keep[positions] = False
        assert engine.ecdsa_verify(w["pk65"][:n][keep], ins[1][keep], out[0][keep]).all()
    host = call(engine, entry, ins)
    for h, d in zip(host, out):
        bad = np.nonzero((h != d).reshape(n, -1).any(axis=1))[0]
        assert len(bad) == 0, f"{entry} n={n}: _dev and host path differ at rows {bad[:8].tolist()}"
    spread = np.linspace(0, n - 1, ORACLE_SPREAD if entry != "schnorr_sign" else 64).astype(np.int64)
    edges = positions if entry != "schnorr_sign" else positions[:64]
    idx = np.unique(np.concatenate([neighbours(edges, n), spread]))
    check_oracle(oracle, entry, ins, out, idx)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["scalar_base_mult", "scalar_mult", "double_scalar_mult", "recover", "sign"])
def test_dev_chunks_of_an_odd_capacity(s256, engine, oracle, gpu_rows, entry):
    """A context of 2^19 + 8 rows cuts 2^20 + 40 rows into chunks of K = 32, K = 32 and K = 1.  The second chunk's
    65-byte rows start at 65 (2^19 + 8) bytes, not 16-byte aligned, so its K = 32 finish must take the per-row store."""
    w, ident = gpu_rows
    n = CHUNKED_N
    cap = (1 << 19) + 8
    edges = [0, cap - 1, cap, cap + 1, 2 * cap - 1, 2 * cap, n - 1]
    positions = [r for r in plant_positions(cap, entry_strides(entry, cap))][:48]
    positions = sorted(set(positions) | {cap + r for r in positions} | set(edges[1:]))
    ins, exp, planted = plant(entry, w, n, positions, ident)
    eng = s256.Engine(device=0, max_batch=cap)
    try:
        out = dev_call(eng, entry, ins)
    finally:
        eng.close()
    check_status_and_encoding(entry, out, exp, planted)
    check_closed_form(entry, out, w, n, planted)
    ref = dev_call(engine, entry, ins)
    for r, d in zip(ref, out):
        assert np.array_equal(r, d)
    idx = np.unique(np.concatenate([neighbours(edges + positions, n), np.linspace(0, n - 1, 512).astype(np.int64)]))
    check_oracle(oracle, entry, ins, out, idx)


# *_dev entry points called through the C ABI with output pointers the Python wrapper would never make
def _abi_args(engine, entry, ins, outs, n, stream):
    p = [C.c_void_p(t.data_ptr()) for t in ins]
    q = [C.c_void_p(t.data_ptr()) for t in outs]
    if entry == "schnorr_sign":
        return "s256_schnorr_sign_dev", [engine._ctx, p[0], p[1], C.c_size_t(32), p[2], C.c_size_t(n), *q, stream]
    name = {"scalar_mult": "s256_scalar_mult_dev", "ecdh": "s256_ecdh_dev",
            "double_scalar_mult": "s256_double_scalar_mult_basepoint_vartime_dev", "recover": "s256_ecdsa_recover_dev",
            "sign": "s256_ecdsa_sign_rfc6979_dev"}[entry]
    return name, [engine._ctx, *p, C.c_size_t(n), *q, stream]


OUT_WIDTHS = {"scalar_mult": (65, 1), "ecdh": (32, 1), "double_scalar_mult": (65, 1), "recover": (65, 1),
              "sign": (64, 1, 1), "schnorr_sign": (64, 1)}


def odd(a, off=1):
    """A contiguous CUDA view of `a` that starts `off` bytes into its allocation."""
    import torch
    a = np.ascontiguousarray(a)
    buf = torch.empty(a.size + off, dtype=torch.uint8, device="cuda")
    v = buf[off:].view(a.shape)
    v.copy_(torch.from_numpy(a))
    assert v.data_ptr() % 16 == off % 16 and v.is_contiguous()
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("n", [700, 524321])
@pytest.mark.parametrize("entry", ["recover", "double_scalar_mult", "scalar_mult", "ecdh", "sign", "schnorr_sign"])
def test_dev_misaligned_inputs_and_outputs(engine, gpu_rows, entry, n):
    """Inputs at offset 1 and outputs at offsets 1 and 8 give the same bytes as 16-byte aligned buffers: the kernels
    use 128-bit accesses only where a row is aligned."""
    import torch
    w, ident = gpu_rows
    ins, _, _ = plant(entry, w, n, plant_positions(n, entry_strides(entry, n)), ident)
    ref = dev_call(engine, entry, ins)
    lib = engine._lib
    for in_off, out_off in ((1, 0), (1, 1), (0, 8), (1, 8)):
        tin = [odd(a, in_off) for a in ins]
        outs = [odd(np.zeros((n, wd), np.uint8), out_off) for wd in OUT_WIDTHS[entry]]
        name, args = _abi_args(engine, entry, tin, outs, n, C.c_void_p(torch.cuda.current_stream().cuda_stream))
        engine._check(getattr(lib, name)(*args), name)
        torch.cuda.synchronize()
        for r, o in zip(ref, outs):
            got = o.cpu().numpy().reshape(r.shape)
            assert np.array_equal(got, r), (entry, n, in_off, out_off)


# ---- the fixed-base kernel by size: split<8> up to 8192 rows, split<4> up to 16384, w7 above ----
BASE_MULT_SIZES = (1, 31, 32, 33, 8191, 8192, 8193, 16383, 16384, 16385)


@pytest.mark.gpu
@pytest.mark.parametrize("n", BASE_MULT_SIZES)
def test_base_mult_kernel_by_size(engine, oracle, n):
    """The 5-, 6- and 7-bit recoding edges first, then random scalars: every row against the oracle, host and _dev."""
    ks = np.concatenate([base_mult_edge_scalars(), synth.base_mult_scalars(n, start=3000)])[:n].copy()
    exp, est = oracle.batch_scalar_base_mult(ks)
    got, st = engine.scalar_base_mult(ks)
    assert np.array_equal(st, est) and np.array_equal(got, exp)
    got, st = dev_call(engine, "scalar_base_mult", [ks])
    assert np.array_equal(st, est) and np.array_equal(got, exp)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [8193, 16384])
def test_signing_with_the_split4_base_mult(engine, oracle, n):
    """R = k G from k_base_mult_ct_split<4>: RFC 6979 against the oracle on every row, BIP-340 on a sample."""
    priv = ints_rows([synth._nonzero_mod_n(x) for x in synth._stream_ints(b"split4-key", 0, n, synth.SEED)])
    dg = synth.base_mult_scalars(n, start=n)
    aux = synth.base_mult_scalars(n, start=2 * n)
    es, er, est = oracle.batch_ecdsa_sign_rfc6979(priv, dg)
    for out in (call(engine, "sign", [priv, dg]), dev_call(engine, "sign", [priv, dg])):
        assert np.array_equal(out[0], es) and np.array_equal(out[1], er) and np.array_equal(out[2], est)
    idx = np.unique(np.concatenate([np.arange(0, 40), np.arange(n - 40, n), np.linspace(0, n - 1, 200).astype(np.int64)]))
    for out in (call(engine, "schnorr_sign", [priv, dg, aux]), dev_call(engine, "schnorr_sign", [priv, dg, aux])):
        assert (out[1] == 1).all()
        check_oracle(oracle, "schnorr_sign", [priv, dg, aux], out, idx)
