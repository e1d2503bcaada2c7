"""BIP-340 over messages of different lengths (the *_varlen entry points) on one GPU.

For n in {4096, 2^16, 2^20, 2^22} and three message cases
  (a) every row 32 bytes: the uniform call (msg_len = 32) against the ragged call on the same rows,
  (b) lengths uniform in 0..256,
  (c) lengths uniform in 0..256 with 1 % of the rows at 4 KiB (the straggler case: one thread hashes one row, so a warp
      waits for its longest message),
it times per-item verification and batch verification, device-resident (CUDA events around each call after warm-up)
and from page-locked host buffers (host clock around calls that end in a synchronisation), and reports the median.
The rows are valid BIP-340 signatures (signed on the GPU); every call's verdict must be "all valid".  Prints one JSON
line with the card's name and power limit, and writes it to --out.

    python scripts/bench_schnorr_varlen.py [--reps 10] [--warmup 2] [--sizes 4096,65536,1048576,4194304]
                                           [--out profiles/r06_schnorr_varlen.json]
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


def lengths(case, n, rng):
    if case == "a_32":
        return np.full(n, 32, np.int64)
    lens = rng.integers(0, 257, n)
    if case == "c_1pct_4k":
        lens[rng.random(n) < 0.01] = 4096
    return lens


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sizes", default="4096,65536,1048576,4194304")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_schnorr_varlen.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_schnorr_varlen: no CUDA device")
    name, power = card()
    s256 = importlib.import_module("secp256k1-voi_b200")
    eng = s256.Engine()
    lib, ctx = eng._lib, eng._ctx
    ptr = lambda a: C.c_void_p(a.ctypes.data)
    dptr = lambda t: C.c_void_p(t.data_ptr())
    rng = np.random.default_rng(2026)
    result = {"bench": "schnorr_varlen", "gpu": name, "power_limit": power, "reps": args.reps, "warmup": args.warmup,
              "timing": "median of CUDA-event times per call (dev); host clock around synchronous calls, page-locked "
                        "inputs (host)", "rows": []}
    for n in [int(x) for x in args.sizes.split(",")]:
        priv = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        priv[:, 0] &= 0x7F
        priv[:, 31] |= 1
        d_priv, d_aux = torch.from_numpy(priv).cuda(), torch.from_numpy(rng.integers(0, 256, (n, 32), dtype=np.uint8)).cuda()
        pub, _ = eng.scalar_base_mult(d_priv)
        d_pkx = pub[:, 1:33].contiguous()
        for case in ("a_32", "b_0_256", "c_1pct_4k"):
            lens = lengths(case, n, rng)
            offs = np.zeros(n + 1, np.int64)
            np.cumsum(lens, out=offs[1:])
            d_flat = torch.from_numpy(rng.integers(0, 256, int(offs[-1]), dtype=np.uint8)).cuda()
            d_offs = torch.from_numpy(offs).cuda()
            d_sig, st = eng.schnorr_sign_varlen(d_priv, (d_flat, d_offs), d_aux)
            assert bool(st.all().item())
            # page-locked host copies of the same rows
            h_pkx, h_sig = eng.pinned_empty((n, 32)), eng.pinned_empty((n, 64))
            h_flat = eng.pinned_empty(max(int(offs[-1]), 1))
            h_offs = eng.pinned_empty(8 * (n + 1)).view(np.uint64)
            h_pkx[:] = d_pkx.cpu().numpy()
            h_sig[:] = d_sig.cpu().numpy()
            h_flat[:int(offs[-1])] = d_flat.cpu().numpy()
            h_offs[:] = offs.astype(np.uint64)
            h_ok = eng.pinned_empty(n)
            ok1 = C.c_uint8(0)
            d_ok = torch.empty(n, dtype=torch.uint8, device="cuda")
            d_ok1 = torch.empty(1, dtype=torch.uint8, device="cuda")
            stream = eng._stream()
            nn = C.c_size_t(n)

            def rl_item_dev():
                return lib.s256_schnorr_verify_varlen_dev(ctx, dptr(d_pkx), dptr(d_flat), dptr(d_offs), dptr(d_sig), nn,
                                                          dptr(d_ok), stream)

            def rl_batch_dev():
                return lib.s256_schnorr_batch_verify_varlen_dev(ctx, dptr(d_pkx), dptr(d_flat), dptr(d_offs), dptr(d_sig), nn,
                                                                dptr(d_ok1), stream)

            def rl_item_host():
                return lib.s256_schnorr_verify_varlen(ctx, ptr(h_pkx), ptr(h_flat), ptr(h_offs), ptr(h_sig), nn, ptr(h_ok))

            def rl_batch_host():
                return lib.s256_schnorr_batch_verify_varlen(ctx, ptr(h_pkx), ptr(h_flat), ptr(h_offs), ptr(h_sig), nn,
                                                            C.byref(ok1))

            row = {"n": n, "case": case, "msg_bytes": int(offs[-1])}
            for fn in (rl_item_dev, rl_batch_dev, rl_item_host, rl_batch_host):
                assert fn() == 0
            row["ragged_item_dev_ms"] = events_ms(rl_item_dev, args.reps, args.warmup)
            assert bool(d_ok.all().item())
            row["ragged_batch_dev_ms"] = events_ms(rl_batch_dev, args.reps, args.warmup)
            assert d_ok1.item() == 1
            row["ragged_item_host_ms"] = host_ms(rl_item_host, args.reps, args.warmup)
            assert h_ok.all()
            row["ragged_batch_host_ms"] = host_ms(rl_batch_host, args.reps, args.warmup)
            assert ok1.value == 1
            if case == "a_32":
                ml = C.c_size_t(32)
                row["uniform_item_dev_ms"] = events_ms(
                    lambda: lib.s256_schnorr_verify_dev(ctx, dptr(d_pkx), dptr(d_flat), ml, dptr(d_sig), nn, dptr(d_ok), stream),
                    args.reps, args.warmup)
                assert bool(d_ok.all().item())
                row["uniform_batch_dev_ms"] = events_ms(
                    lambda: lib.s256_schnorr_batch_verify_dev(ctx, dptr(d_pkx), dptr(d_flat), ml, dptr(d_sig), nn, dptr(d_ok1),
                                                              stream), args.reps, args.warmup)
                assert d_ok1.item() == 1
                row["uniform_item_host_ms"] = host_ms(
                    lambda: lib.s256_schnorr_verify(ctx, ptr(h_pkx), ptr(h_flat), ml, ptr(h_sig), nn, ptr(h_ok)),
                    args.reps, args.warmup)
                assert h_ok.all()
                row["uniform_batch_host_ms"] = host_ms(
                    lambda: lib.s256_schnorr_batch_verify(ctx, ptr(h_pkx), ptr(h_flat), ml, ptr(h_sig), nn, C.byref(ok1)),
                    args.reps, args.warmup)
                assert ok1.value == 1
                for k in ("item_dev", "batch_dev", "item_host", "batch_host"):
                    row[f"ragged_over_uniform_{k}"] = row[f"ragged_{k}_ms"] / row[f"uniform_{k}_ms"]
            result["rows"].append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
            del d_flat, d_offs, d_sig
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
