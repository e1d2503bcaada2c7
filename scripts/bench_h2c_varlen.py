"""Hash to curve over device-resident rows and over messages of different lengths (s256_hash_to_curve_dev,
s256_hash_to_curve_varlen[_dev]) on one GPU.

For n in {2^16, 2^20, 2^22}, both suites (random_oracle 1 = hash_to_curve, 0 = encode_to_curve) and three message cases
  (a) every row 32 bytes: the uniform call (msg_len = 32) against the ragged call on the same rows,
  (b) lengths uniform in 0..256,
  (c) lengths uniform in 0..256 with 1 % of the rows at 4 KiB (the straggler case: one thread hashes one row, so a warp
      waits for its longest message),
it times each form device-resident (CUDA events around each call after warm-up) and from page-locked host buffers
(host clock around calls that end in a synchronisation), and reports the median.  Every row's status must be
S256_ST_OK.  Prints one JSON line with the card's name and power limit, and writes it to --out.

    python scripts/bench_h2c_varlen.py [--reps 10] [--warmup 2] [--sizes 65536,1048576,4194304]
                                       [--out profiles/r08_h2c_varlen.json]
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

DST = b"QUUX-V01-CS02-with-secp256k1_XMD:SHA-256_SSWU_RO_"


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
    ap.add_argument("--sizes", default="65536,1048576,4194304")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_h2c_varlen.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_h2c_varlen: no CUDA device")
    name, power = card()
    s256 = importlib.import_module("secp256k1-voi_b200")
    eng = s256.Engine()
    lib, ctx = eng._lib, eng._ctx
    ptr = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    dptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    dl = C.c_size_t(len(DST))
    rng = np.random.default_rng(2026)
    result = {"bench": "h2c_varlen", "gpu": name, "power_limit": power, "reps": args.reps, "warmup": args.warmup, "dst": DST.decode(),
              "timing": "median of CUDA-event times per call (dev); host clock around synchronous calls, page-locked "
                        "inputs and outputs (host)", "rows": []}
    for n in [int(x) for x in args.sizes.split(",")]:
        nn = C.c_size_t(n)
        d_out = torch.empty((n, 65), dtype=torch.uint8, device="cuda")
        d_st = torch.empty(n, dtype=torch.uint8, device="cuda")
        h_out, h_st = eng.pinned_empty((n, 65)), eng.pinned_empty(n)
        for case in ("a_32", "b_0_256", "c_1pct_4k"):
            lens = lengths(case, n, rng)
            offs = np.zeros(n + 1, np.int64)
            np.cumsum(lens, out=offs[1:])
            flat = rng.integers(0, 256, int(offs[-1]), dtype=np.uint8)
            d_flat, d_offs = torch.from_numpy(flat).cuda(), torch.from_numpy(offs).cuda()
            h_flat = eng.pinned_empty(max(int(offs[-1]), 1))
            h_offs = eng.pinned_empty(8 * (n + 1)).view(np.uint64)
            h_flat[:int(offs[-1])] = flat
            h_offs[:] = offs.astype(np.uint64)
            stream = eng._stream()
            for ro in (1, 0):
                def ragged_dev():
                    return lib.s256_hash_to_curve_varlen_dev(ctx, DST, dl, dptr(d_flat), dptr(d_offs), nn, ro, dptr(d_out),
                                                             dptr(d_st), stream)

                def ragged_host():
                    return lib.s256_hash_to_curve_varlen(ctx, DST, dl, ptr(h_flat), ptr(h_offs), nn, ro, ptr(h_out), ptr(h_st))

                forms = {"ragged_dev": ragged_dev, "ragged_host": ragged_host}
                if case == "a_32":
                    ml = C.c_size_t(32)
                    forms["uniform_dev"] = lambda: lib.s256_hash_to_curve_dev(ctx, DST, dl, dptr(d_flat), ml, nn, ro, dptr(d_out),
                                                                              dptr(d_st), stream)
                    forms["uniform_host"] = lambda: lib.s256_hash_to_curve(ctx, DST, dl, ptr(h_flat), ml, nn, ro, ptr(h_out),
                                                                           ptr(h_st))
                row = {"n": n, "case": case, "random_oracle": ro, "msg_bytes": int(offs[-1])}
                for form, fn in forms.items():
                    assert fn() == 0, form
                    timer = events_ms if form.endswith("_dev") else host_ms
                    row[f"{form}_ms"] = timer(fn, args.reps, args.warmup)
                    torch.cuda.synchronize()
                    ok = bool((d_st == 1).all().item()) if form.endswith("_dev") else bool((h_st == 1).all())
                    assert ok, (n, case, ro, form)
                if case == "a_32":
                    row["ragged_over_uniform_dev"] = row["ragged_dev_ms"] / row["uniform_dev_ms"]
                    row["ragged_over_uniform_host"] = row["ragged_host_ms"] / row["uniform_host_ms"]
                    row["uniform_host_over_dev"] = row["uniform_host_ms"] / row["uniform_dev_ms"]
                result["rows"].append(row)
                print(json.dumps(row), file=sys.stderr, flush=True)
            del d_flat, d_offs
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
