"""DER-encoded ECDSA verification (PublicKey.Verify with EncodingASN1, bitcoin.VerifyASN1) on one GPU.

For n in {2^16, 2^20, 2^22} valid low-s signatures (signed on the GPU, encoded with s256_build_asn1_signatures) it times
  device-resident (CUDA events around each call after warm-up):
    s256_ecdsa_verify_dev on the compact r||s rows, s256_ecdsa_verify_asn1_dev and s256_bitcoin_verify_asn1_dev on the
    same signatures in DER (the Bitcoin rows with a sighash byte), and the parse kernel alone
    (s256_parse_asn1_signatures_dev, which also writes the ok bytes);
  from page-locked host buffers (host clock around calls that end in a synchronisation):
    s256_ecdsa_verify on the compact rows, the host forms s256_ecdsa_verify_asn1 and s256_bitcoin_verify_asn1, and the
    route they replace: the host codec s256_parse_asn1_signatures into a fresh pageable buffer, s256_ecdsa_verify on
    its rows and an AND; for Bitcoin first s256_is_valid_signature_encoding_bip0066 and the copy without the sighash
    bytes (the loop the host form ran, compiled with g++ -O2 into a temporary directory).
Reports the median; every call's verdict must be "all valid".  Prints one JSON line with the card's name and power
limit, and writes it to --out.

    python scripts/bench_ecdsa_der.py [--reps 10] [--warmup 2] [--sizes 65536,1048576,4194304]
                                      [--out profiles/r07_ecdsa_der.json]
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# the sighash-stripping copy of the Bitcoin host form before rows were parsed on the device
STRIP_SRC = r"""
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <vector>
extern "C" size_t strip_sighash(const uint8_t *der, const size_t *offsets, size_t n, const uint8_t *bip, uint8_t **out,
                                size_t *off2) {
    static std::vector<uint8_t> der2;
    der2.clear();
    der2.shrink_to_fit();
    der2.reserve(offsets[n] - offsets[0]);
    for (size_t i = 0; i < n; i++) {
        off2[i] = der2.size();
        if (bip[i]) der2.insert(der2.end(), der + offsets[i], der + offsets[i + 1] - 1);
    }
    off2[n] = der2.size();
    if (der2.empty()) der2.push_back(0);
    *out = der2.data();
    return der2.size();
}
"""


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in q.split(",")]
    return name, power


def events_ms(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def host_ms(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t) * 1e3)
    return float(np.median(times))


def strip_lib(tmp):
    src, so = os.path.join(tmp, "strip.cpp"), os.path.join(tmp, "strip.so")
    with open(src, "w") as f:
        f.write(STRIP_SRC)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src])
    lib = C.CDLL(so)
    lib.strip_sighash.restype = C.c_size_t
    return lib


def flatten(rows72, lens, extra=None):
    """(n, 72) rows with lens[i] bytes used (+ one sighash byte per row when extra is given) -> flat bytes, offsets"""
    n = len(lens)
    width = lens.astype(np.int64) + (1 if extra is not None else 0)
    full = np.zeros((n, 73), np.uint8)
    full[:, :72] = rows72
    if extra is not None:
        full[np.arange(n), lens] = extra
    mask = np.arange(73)[None, :] < width[:, None]
    offs = np.zeros(n + 1, np.uint64)
    np.cumsum(width, out=offs[1:])
    return full[mask], offs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sizes", default="65536,1048576,4194304")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_ecdsa_der.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_ecdsa_der: no CUDA device")
    name, power = card()
    s256 = importlib.import_module("secp256k1-voi_b200")
    eng = s256.Engine()
    lib, ctx = eng._lib, eng._ctx
    ptr = lambda a: C.c_void_p(a.ctypes.data)
    dptr = lambda t: C.c_void_p(t.data_ptr())
    rng = np.random.default_rng(2027)
    tmp = tempfile.mkdtemp(prefix="bench_ecdsa_der_")
    strip = strip_lib(tmp)
    result = {"bench": "ecdsa_der", "gpu": name, "power_limit": power, "reps": args.reps, "warmup": args.warmup,
              "timing": "median of CUDA-event times per call (dev); host clock around synchronous calls, page-locked "
                        "inputs (host)", "rows": []}
    for n in [int(x) for x in args.sizes.split(",")]:
        priv = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        priv[:, 0] &= 0x7F
        priv[:, 31] |= 1
        d_priv = torch.from_numpy(priv).cuda()
        d_dg = torch.from_numpy(rng.integers(0, 256, (n, 32), dtype=np.uint8)).cuda()
        d_pk, st = eng.scalar_base_mult(d_priv)
        assert bool(st.eq(1).all().item())
        d_sig, _, st = eng.ecdsa_sign_rfc6979(d_priv, d_dg)
        assert bool(st.eq(1).all().item())
        sig = d_sig.cpu().numpy()
        rows72, lens = np.zeros((n, 72), np.uint8), np.zeros(n, np.uint8)
        assert lib.s256_build_asn1_signatures(ptr(sig), C.c_size_t(n), ptr(rows72), ptr(lens)) == 0
        flat, offs = flatten(rows72, lens)
        hflat, hoffs = flatten(rows72, lens, extra=rng.integers(0, 256, n, dtype=np.uint8))
        d_flat, d_offs = torch.from_numpy(flat).cuda(), torch.from_numpy(offs.astype(np.int64)).cuda()
        d_hflat, d_hoffs = torch.from_numpy(hflat).cuda(), torch.from_numpy(hoffs.astype(np.int64)).cuda()
        # page-locked host copies
        h = {}
        for key, a in (("pk", d_pk.cpu().numpy()), ("dg", d_dg.cpu().numpy()), ("sig", sig), ("flat", flat),
                       ("hflat", hflat)):
            h[key] = eng.pinned_empty(a.shape)
            h[key][:] = a
        for key, a in (("offs", offs), ("hoffs", hoffs)):
            h[key] = eng.pinned_empty(8 * (n + 1)).view(np.uint64)
            h[key][:] = a
        h_ok = eng.pinned_empty(n)
        d_ok = torch.empty(n, dtype=torch.uint8, device="cuda")
        d_sig_out = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
        stream = eng._stream()
        nn, f0 = C.c_size_t(n), C.c_uint32(0)

        def compact_dev():
            return lib.s256_ecdsa_verify_dev(ctx, dptr(d_pk), dptr(d_dg), dptr(d_sig), f0, nn, dptr(d_ok), stream)

        def asn1_dev():
            return lib.s256_ecdsa_verify_asn1_dev(ctx, dptr(d_pk), dptr(d_dg), dptr(d_flat), dptr(d_offs), f0, nn,
                                                  dptr(d_ok), stream)

        def bitcoin_dev():
            return lib.s256_bitcoin_verify_asn1_dev(ctx, dptr(d_pk), dptr(d_dg), dptr(d_hflat), dptr(d_hoffs), nn,
                                                    dptr(d_ok), stream)

        def parse_dev():
            return lib.s256_parse_asn1_signatures_dev(ctx, dptr(d_flat), dptr(d_offs), nn, dptr(d_sig_out), dptr(d_ok),
                                                      stream)

        def compact_host():
            return lib.s256_ecdsa_verify(ctx, ptr(h["pk"]), ptr(h["dg"]), ptr(h["sig"]), f0, nn, ptr(h_ok))

        def asn1_host():
            return lib.s256_ecdsa_verify_asn1(ctx, ptr(h["pk"]), ptr(h["dg"]), ptr(h["flat"]), ptr(h["offs"]), f0, nn,
                                              ptr(h_ok))

        def bitcoin_host():
            return lib.s256_bitcoin_verify_asn1(ctx, ptr(h["pk"]), ptr(h["dg"]), ptr(h["hflat"]), ptr(h["hoffs"]), nn,
                                                ptr(h_ok))

        def before_asn1(der=h["flat"], offsets=h["offs"], flags=f0):
            s64, parsed = np.empty((n, 64), np.uint8), np.empty(n, np.uint8)
            rc = lib.s256_parse_asn1_signatures(ptr(der), ptr(offsets), nn, ptr(s64), ptr(parsed))
            rc |= lib.s256_ecdsa_verify(ctx, ptr(h["pk"]), ptr(h["dg"]), ptr(s64), flags, nn, ptr(h_ok))
            h_ok[:] &= parsed
            return rc

        def before_bitcoin():
            bip = np.empty(n, np.uint8)
            rc = lib.s256_is_valid_signature_encoding_bip0066(ptr(h["hflat"]), ptr(h["hoffs"]), nn, ptr(bip))
            off2 = np.empty(n + 1, np.uint64)
            out = C.c_void_p()
            size = strip.strip_sighash(ptr(h["hflat"]), ptr(h["hoffs"]), nn, ptr(bip), C.byref(out), ptr(off2))
            der2 = np.ctypeslib.as_array((C.c_uint8 * size).from_address(out.value))
            rc |= before_asn1(der2, off2, C.c_uint32(1))
            h_ok[:] &= bip
            return rc

        row = {"n": n, "der_bytes": int(offs[-1])}
        dev_fns = {"compact_dev_ms": compact_dev, "asn1_dev_ms": asn1_dev, "bitcoin_dev_ms": bitcoin_dev,
                   "parse_kernel_dev_ms": parse_dev}
        host_fns = {"compact_host_ms": compact_host, "asn1_host_ms": asn1_host, "bitcoin_host_ms": bitcoin_host,
                    "asn1_host_before_ms": before_asn1, "bitcoin_host_before_ms": before_bitcoin}
        for key, fn in dev_fns.items():
            assert fn() == 0, key
            row[key] = events_ms(fn, args.reps, args.warmup)
            assert bool(d_ok.eq(1).all().item()), key
        for key, fn in host_fns.items():
            assert fn() == 0, key
            row[key] = host_ms(fn, args.reps, args.warmup)
            assert (h_ok == 1).all(), key
        row["asn1_dev_over_compact_dev"] = row["asn1_dev_ms"] / row["compact_dev_ms"]
        row["bitcoin_dev_over_compact_dev"] = row["bitcoin_dev_ms"] / row["compact_dev_ms"]
        row["asn1_host_over_compact_host"] = row["asn1_host_ms"] / row["compact_host_ms"]
        row["asn1_host_speedup_over_before"] = row["asn1_host_before_ms"] / row["asn1_host_ms"]
        row["bitcoin_host_speedup_over_before"] = row["bitcoin_host_before_ms"] / row["bitcoin_host_ms"]
        result["rows"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del d_flat, d_offs, d_hflat, d_hoffs, d_sig, d_sig_out, d_pk, d_dg, d_priv, d_ok
        torch.cuda.empty_cache()
    eng.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
