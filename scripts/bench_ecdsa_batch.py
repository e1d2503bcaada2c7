"""Recoverable ECDSA batch verification against recover-and-compare on one GPU.

For n in {4096, 2^16, 2^20, 2^22} (2^22 = the 2^20 synthetic batch tiled four times) it times, with CUDA events after
warm-up and on the same device-resident r||s||v rows: s256_ecdsa_recoverable_batch_verify_dev (the batch),
s256_ecdsa_recover_dev followed by an on-device comparison of the recovered keys (the per-item route a caller has
without the batch form), and s256_ecdsa_verify_dev on the r||s rows for reference.  The host-pointer forms of the batch
and of recover-and-compare are timed with a host clock around calls that end in a synchronisation.  One profiled call
per n (a separate run of torch.profiler) splits the batch call's kernel time into pass 1 (leaf hashes, tree, seed), the
per-row preparation, the MSM and the finish.  All verdicts must agree, and a batch with one corrupted s must fail.
Prints one JSON line, with the card's name and power limit.

    python scripts/bench_ecdsa_batch.py [--reps 20] [--warmup 3] [--sizes 4096,65536,1048576,4194304]
"""
import argparse
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
    return float(np.median(times)), float(np.min(times))


def host_ms(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t) * 1e3)
    return float(np.median(times)), float(np.min(times))


GROUPS = (("pass1", ("k_ecdsa_batch_leaves", "k_batch_tree", "k_batch_seed")),
          ("prepare", ("k_ecdsa_batch_points", "k_ecdsa_batch_prepare", "k_batch_fold")),
          ("finish", ("k_base_mult", "k_acc_point", "k_batch_verdict")))


def kernel_split(fn):
    """Kernel time (ms) of one call by stage; everything else the call launches (the MSM) counts as msm."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {"pass1": 0.0, "prepare": 0.0, "msm": 0.0, "finish": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0 or ev.key.startswith(("cudaMemcpy", "Memcpy", "Memset", "cudaMemset")):
            continue
        stage = "msm"
        for g, names in GROUPS:
            if any(k in ev.key for k in names):
                stage = g
        out[stage] += t / 1e3
    return {k: round(v, 4) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sizes", default="4096,65536,1048576,4194304")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_ecdsa_batch: no CUDA device")
    name, power = card()
    s256 = importlib.import_module("secp256k1-voi_b200")
    eng = s256.Engine()
    sizes = [int(x) for x in args.sizes.split(",")]
    base = min(max(sizes), 1 << 20)
    w = s256.synth.ecdsa_recoverable_batch(base, eng.scalar_base_mult, corrupt_every=0)
    rows = (w["pk65"], w["digest32"], w["sig65"])
    result = {"bench": "ecdsa_recoverable_batch_verify", "gpu": name, "power_limit": power, "reps": args.reps,
              "warmup": args.warmup, "timing": "median (min) of CUDA-event times per call; host forms: host clock", "sizes": []}

    def recover_dev(pk, dg, sig):  # recover, then compare the keys on the device
        q, st = eng.ecdsa_recover(dg, sig)
        return ((st == 1) & (q == pk).all(dim=1)).all()

    def recover_host(pk, dg, sig):
        q, st = eng.ecdsa_recover(dg, sig)
        return bool(((st == 1) & (q == pk).all(axis=1)).all())

    for n in sizes:
        if n <= base:
            h = tuple(x[:n].copy() for x in rows)
        else:
            t = (n + base - 1) // base
            h = tuple(np.tile(x, (t, 1))[:n].copy() for x in rows)
        d = tuple(torch.from_numpy(x).cuda() for x in h)
        d64 = d[2][:, :64].contiguous()
        batch_dev = events_ms(lambda: eng.ecdsa_recoverable_batch_verify(*d), args.reps, args.warmup)
        recover_dev_ms = events_ms(lambda: recover_dev(*d), args.reps, args.warmup)
        verify_dev = events_ms(lambda: eng.ecdsa_verify(d[0], d[1], d64), args.reps, args.warmup)
        batch_host = host_ms(lambda: eng.ecdsa_recoverable_batch_verify(*h), args.reps, args.warmup)
        recover_host_ms = host_ms(lambda: recover_host(*h), args.reps, args.warmup)
        split = kernel_split(lambda: eng.ecdsa_recoverable_batch_verify(*d))
        v_recover = bool(recover_dev(*d).item())
        v_verify = bool(eng.ecdsa_verify(d[0], d[1], d64).all().item())
        v_batch = bool(eng.ecdsa_recoverable_batch_verify(*d).item())
        v_host = eng.ecdsa_recoverable_batch_verify(*h)
        v_recover_host = recover_host(*h)
        bad = h[2].copy()
        bad[n // 2, 40] ^= 1
        v_bad = eng.ecdsa_recoverable_batch_verify(h[0], h[1], bad)
        d_bad = torch.from_numpy(bad).cuda()
        v_bad_dev = bool(eng.ecdsa_recoverable_batch_verify(d[0], d[1], d_bad).item())
        v_bad_recover = bool(recover_dev(d[0], d[1], d_bad).item())
        row = {"n": n, "batch_dev_ms": batch_dev[0], "batch_dev_min_ms": batch_dev[1],
               "recover_compare_dev_ms": recover_dev_ms[0], "recover_compare_dev_min_ms": recover_dev_ms[1],
               "verify_dev_ms": verify_dev[0], "batch_host_ms": batch_host[0], "recover_compare_host_ms": recover_host_ms[0],
               "batch_dev_rate_per_s": n / (batch_dev[0] / 1e3), "recover_compare_dev_rate_per_s": n / (recover_dev_ms[0] / 1e3),
               "speedup_dev": recover_dev_ms[0] / batch_dev[0], "batch_kernel_ms": split,
               "verdict_batch": v_batch, "verdict_batch_host": v_host, "verdict_recover_compare": v_recover,
               "verdict_recover_compare_host": v_recover_host, "verdict_verify": v_verify,
               "verdict_corrupted": [v_bad, v_bad_dev, v_bad_recover],
               "agree": v_batch == v_host == v_recover == v_recover_host == v_verify and not (v_bad or v_bad_dev or v_bad_recover)}
        result["sizes"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del d, d64, d_bad
        torch.cuda.empty_cache()
    eng.close()
    print(json.dumps(result))
    if not all(r["agree"] for r in result["sizes"]):
        raise SystemExit("bench_ecdsa_batch: verdicts disagree")


if __name__ == "__main__":
    main()
