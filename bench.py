#!/usr/bin/env python3
"""bench.py -- ECDSA verifies/s at batch 2^20 per GPU (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step returned (the verify result
per row, 0.0 / 1.0) as DIR/ecdsa_verify_ok.npy (float32; one file per rank,
ecdsa_verify_ok_rank<g>.npy, when N > 1).  The inputs depend only on the
arguments, so two builds can be compared output for output.

A step = one pass of the hot path (secec Verify, EncodingCompact) over one
batch of 2^20 synthetic (public key, digest, signature) rows per GPU; rank g
owns the contiguous global slice [g*2^20, (g+1)*2^20) -- independent items, no
data-path collective ("weak" scaling).  Rank 0 prints ONE JSON line:

  value     whole-job verifies/s, inputs resident in HBM, CUDA events on the
            launching stream, barrier + synchronize on both sides, max over ranks
  e2e       same metric through the C ABI with HOST buffers (pinned), the
            host->device copy of the inputs and device->host read of the result
            inside the timed region
  roofline  dominant kernel (u1*G + u2*P ladder) against the integer-multiply
            peak measured live by an IMAD.WIDE.U32 microbenchmark
  cpu_baseline  the CPU oracle (reference-algorithm port) on this box's cores,
            bounded sample
`--impl reference` times the reference's CPU algorithm (the oracle port: the
reference is Go and no Go toolchain exists here) on all host threads.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH_LOG2 = 20
METRIC = "ecdsa_verifies_per_sec"
UNIT = "verifies/s"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def workload_config(n_gpus, batch):
    return {"workload": "ECDSA verify batch 2^20 per GPU (secec.Verify compact, DoubleScalarMultBasepointVartime)",
            "batch_per_gpu": batch, "global_batch": batch * n_gpus, "corrupted_fraction": 1.0 / 16,
            "sharding": "contiguous batch slices, no collective",
            "l2_policy": "inputs (169 MB) plus 2.1 GB of per-item tables exceed the 126 MB L2 every step"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.gpu_index), "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self, t_begin=None, t_end=None):
        """The sampler is started BEFORE the warm-up (nvidia-smi needs ~0.1 s to produce its first line,
        longer with one instance per rank); only samples stamped inside [t_begin, t_end] are kept."""
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if getattr(self, "rows", None) is not None:
            return self.summarise(t_begin, t_end)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        import datetime
        rows = []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = None
            try:
                rows.append((ts, float(c[1]), float(c[2]), float(c[3]), c[5:9]))
            except ValueError:
                continue
        os.unlink(self.f.name)
        self.rows = rows
        return self.summarise(t_begin, t_end)

    def summarise(self, t_begin=None, t_end=None):
        rows = self.rows
        window = "timed region"
        if t_begin is not None:
            inside = [r for r in rows if r[0] is not None and t_begin - 0.02 <= r[0] <= t_end + 0.02]
            if inside:
                rows = inside
            elif rows:  # region shorter than the sampling period, or an unparsed timestamp: nearest samples
                rows, window = rows[-3:], "last samples before the region ended"
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        reasons = set()
        for r in rows:
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": max(r[2] for r in rows),
                "power_w_max": max(r[3] for r in rows), "samples": len(rows), "window": window, "reasons": sorted(reasons)}


def cpu_reference_arm(args):
    """--impl reference: the reference's CPU algorithm for the same path."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    from oracle import oracle as orc
    pkg = importlib.import_module("secp256k1-voi_b200")
    threads = orc.default_threads()
    sample = max(4096, 2048 * threads)  # ~0.3 s of all-thread work per step
    w = pkg.synth.ecdsa_batch(sample, lambda k: orc.batch_scalar_base_mult(k))
    for _ in range(max(1, min(args.warmup, 1))):
        orc.batch_ecdsa_verify(w["pk65"], w["digest32"], w["sig64"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ok = orc.batch_ecdsa_verify(w["pk65"], w["digest32"], w["sig64"])
    dt = time.perf_counter() - t0
    assert np.array_equal(ok, w["expected"])
    value = sample * args.steps / dt
    kind = "port"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (4x64-limb Montgomery)",
            "data": "synthetic", "config": workload_config(args.gpus, 1 << BATCH_LOG2),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                             "sample": f"{sample} items of the same workload per step, {threads} threads; "
                                       "C port of the reference's algorithms (Go toolchain absent)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"ecdsa_verify_ok": ok})
    return 0


_REAL_STDOUT = None


def hbm_peak_gbs():
    """Measured HBM copy bandwidth of this pool's B200s (driver-written MEASURED_PEAKS.json), else the recipe's fallback."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"])
    except (OSError, KeyError, ValueError):
        return 6548.2


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays):
    """Writes each 1-D array as out_dir/<name>.npy in float32.  An array too large for DUMP_BYTES is replaced by a
    fixed, seeded sample of its rows, written with the sampled row numbers (<name>_rows.npy, float64)."""
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a).reshape(-1)
        if a.size * 4 > budget:
            rows = np.sort(np.random.default_rng(0).choice(a.size, budget // 12, replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def emit(line):
    """The one JSON line, on the real stdout."""
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch-log2", type=int, default=BATCH_LOG2)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true",
                    help="only the device-resident headline steps (for the ncu launch list in profiles/): "
                         "no end-to-end leg, no other paths")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly ONE JSON line: libraries that print to the C-level stdout (NCCL's version
    # banner, for one) are sent to stderr for the duration of the run
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return cpu_reference_arm(args)

    import torch
    import torch.distributed as dist

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this engine has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks(x):
        """x of every rank, in rank order (diagnostics: which rank set the max)."""
        if world == 1:
            return [x]
        t = torch.zeros(world, dtype=torch.float64, device="cuda")
        t[rank] = x
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    pkg = importlib.import_module("secp256k1-voi_b200")
    n = 1 << args.batch_log2
    eng = pkg.Engine(device=local, max_batch=n)

    # ---- synthetic inputs: signatures made with the engine's own d*G, k*G ----
    t_gen = time.perf_counter()
    w = pkg.synth.ecdsa_batch(n, eng.scalar_base_mult, start=rank * n)
    t_gen = time.perf_counter() - t_gen
    h_pk = torch.from_numpy(w["pk65"]).pin_memory()
    h_dg = torch.from_numpy(w["digest32"]).pin_memory()
    h_sg = torch.from_numpy(w["sig64"]).pin_memory()
    d_pk, d_dg, d_sg = h_pk.cuda(), h_dg.cuda(), h_sg.cuda()
    expected = w["expected"]

    # ---- device-resident timing ------------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    t_warm = time.perf_counter()
    for _ in range(max(args.warmup, 3)):
        ok = eng.ecdsa_verify(d_pk, d_dg, d_sg)
    torch.cuda.synchronize()
    while time.perf_counter() - t_warm < 0.3:  # at least 0.3 s under load: clocks and power state settled
        ok = eng.ecdsa_verify(d_pk, d_dg, d_sg)
        torch.cuda.synchronize()
    assert np.array_equal(ok.cpu().numpy(), expected), "verify booleans differ from the construction"
    launches0 = eng.launch_count
    eng.profile_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); torch.cuda.synchronize()
    t_begin = time.time()
    e0.record()
    for _ in range(args.steps):
        ok = eng.ecdsa_verify(d_pk, d_dg, d_sg)
    e1.record()
    torch.cuda.synchronize()
    t_end = time.time()
    barrier()
    ms_total = e0.elapsed_time(e1)
    # integer-multiply peak: measured HERE, straight after the timed steps, on the clocks and power state they ran at
    # (round 1 probed before the warm-up, on clocks still ramping, and read 5 % low); best of five
    t_probe = time.time()
    imad_runs = [eng.microbench_imad(8192)[0] for _ in range(5)]
    imad_peak = max(imad_runs)
    t_probe_end = time.time()
    clocks = sampler.stop(t_begin, t_end)
    probe_clocks = sampler.stop(t_probe, t_probe_end)
    dsm_ms, dsm_launches = eng.profile_read()
    eng.profile_enable(False)
    # the ladder additions that really ran (zero digits are skipped): measured on the last step's recoded scalars
    adds_a, adds_b = eng.ladder_add_count(n)
    launches = eng.launch_count - launches0
    per_rank_ms = [v / args.steps for v in all_ranks(ms_total)]
    rank_sm_mhz = all_ranks(clocks["sm_mhz"] if clocks.get("sm_mhz") else 0.0)
    ms_total = max_over_ranks(ms_total)
    ms_per_step = ms_total / args.steps
    value = n * world / (ms_per_step * 1e-3)
    ok_last = ok.cpu().numpy()
    assert np.array_equal(ok_last, expected)

    # ---- end to end through the C ABI with host buffers --------------------------
    np_pk, np_dg, np_sg = h_pk.numpy(), h_dg.numpy(), h_sg.numpy()
    e2e_value = e2e_single = e2e_two = None
    h2d_gbs = None
    if not args.headline_only:
        for _ in range(2):
            ok_h = eng.ecdsa_verify(np_pk, np_dg, np_sg)
        barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ok_h = eng.ecdsa_verify(np_pk, np_dg, np_sg)
        torch.cuda.synchronize()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        barrier()
        assert np.array_equal(ok_h, expected)
        e2e_single = n * world * args.steps / e2e_s
        # Two callers: a second context on a second host thread, the two submitting alternate batches (what a Go
        # service does with two goroutines, or any caller that double-buffers).  Every batch still goes host -> device
        # -> host inside the timed region; the copies of one caller's batch overlap the other caller's ladder, which
        # a single synchronous caller cannot arrange (its next batch is not submitted before the last one returned).
        import threading
        eng2 = pkg.Engine(device=local, max_batch=n)
        h2 = [torch.empty_like(t).pin_memory().copy_(t) for t in (h_pk, h_dg, h_sg)]
        np2 = [t.numpy() for t in h2]
        calls = [(args.steps + 1) // 2, args.steps // 2]
        res2 = [None, None]

        def caller(k, e, bufs, reps):
            torch.cuda.set_device(local)
            for _ in range(reps):
                res2[k] = e.ecdsa_verify(*bufs)

        for e, bufs in ((eng, (np_pk, np_dg, np_sg)), (eng2, np2)):
            e.ecdsa_verify(*bufs)
        barrier(); torch.cuda.synchronize()
        ths = [threading.Thread(target=caller, args=(0, eng, (np_pk, np_dg, np_sg), calls[0])),
               threading.Thread(target=caller, args=(1, eng2, np2, calls[1]))]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        torch.cuda.synchronize()
        e2e2_s = max_over_ranks(time.perf_counter() - t0)
        barrier()
        assert all(r is None or np.array_equal(r, expected) for r in res2)
        e2e_two = n * world * sum(calls) / e2e2_s
        del eng2
        e2e_value = max(e2e_single, e2e_two)
        # what the PCIe link of every rank gives while ALL ranks copy at once (the e2e pipeline needs ~32 GB/s per link to
        # hide the copies under the ladder; on these boxes every GPU reports CPU affinity 0-31 / NUMA node 0, so there is
        # no NUMA placement to choose)
        barrier(); torch.cuda.synchronize()
        ca, cb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ca.record()
        for _ in range(5):
            d_pk.copy_(h_pk, non_blocking=True); d_dg.copy_(h_dg, non_blocking=True); d_sg.copy_(h_sg, non_blocking=True)
        cb.record(); torch.cuda.synchronize()
        h2d_gbs = all_ranks(5 * n * 161 / (ca.elapsed_time(cb) * 1e-3) / 1e9)
        barrier()

    # ---- ScalarBaseMult ops/s (BASELINE configs[0] and at 2^20) -------------------
    sbm = {}
    for nn in (() if args.headline_only else (4096, n)):
        ks = torch.from_numpy(pkg.synth.base_mult_scalars(nn)).cuda()
        for _ in range(3):
            eng.scalar_base_mult(ks)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        reps = 5
        for _ in range(reps):
            eng.scalar_base_mult(ks)
        b.record(); torch.cuda.synchronize()
        sbm[str(nn)] = nn * reps / (a.elapsed_time(b) * 1e-3)

    # ---- the other hot-path entry points at the same batch size (device-resident, rank 0 only) ----
    other = {}
    if rank == 0 and not args.headline_only:
        def timed(fn, reps=3):
            fn(); torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record(); torch.cuda.synchronize()
            return a.elapsed_time(b) / reps
        priv = torch.from_numpy(pkg.synth.base_mult_scalars(n, start=77))
        priv[:, 0] &= 0x7F                                   # every key below n
        d_priv = priv.cuda()
        d_aux = torch.from_numpy(pkg.synth.base_mult_scalars(n, start=78)).cuda()
        pub, _ = eng.scalar_base_mult(d_priv)
        sig, rec, st = eng.ecdsa_sign_rfc6979(d_priv, d_dg)
        sig65 = torch.cat([sig, rec[:, None]], dim=1).contiguous()
        ssig, sst = eng.schnorr_sign(d_priv, d_dg, d_aux)
        pkx = pub[:, 1:33].contiguous()
        assert bool(eng.ecdsa_verify(pub, d_dg, sig).all()) and bool(eng.schnorr_verify(pkx, d_dg, ssig).all())
        q, qst = eng.ecdsa_recover(d_dg, sig65)
        assert bool((qst == 1).all()) and bool((q == pub).all())
        for name, key, fn in (
                ("schnorr_verify", "schnorr_verify", lambda: eng.schnorr_verify(pkx, d_dg, ssig)),
                ("ecdsa_recover", "ecdsa_recover", lambda: eng.ecdsa_recover(d_dg, sig65)),
                ("ecdh", "ecdh", lambda: eng.ecdh(d_priv, pub)),
                ("scalar_mult_ct", "scalar_mult", lambda: eng.scalar_mult(d_priv, pub)),
                ("ecdsa_sign_rfc6979", "ecdsa_sign_rfc6979", lambda: eng.ecdsa_sign_rfc6979(d_priv, d_dg)),
                ("schnorr_sign", "schnorr_sign", lambda: eng.schnorr_sign(d_priv, d_dg, d_aux))):
            ms = timed(fn)
            mac = pkg.mac32_per_item(key)
            other[name] = {"items_per_s": n / (ms * 1e-3), "ms": ms,
                           "frac_of_int_mul_peak": n / (ms * 1e-3) * mac / imad_peak if mac else None}
        # the same calls end to end: pinned host buffers in AND out through the host-pointer entry points
        eng_h = pkg.Engine(device=local, max_batch=n, pinned_outputs=True)
        pin = lambda t_: t_.cpu().pin_memory().numpy()
        h_priv, h_aux, h_pub, h_pkx, h_sig65, h_ssig = pin(d_priv), pin(d_aux), pin(pub), pin(pkx), pin(sig65), pin(ssig)

        def wall(fn, reps=3):
            fn()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            return (time.perf_counter() - t0) / reps * 1e3
        for name, fn in (
                ("schnorr_verify", lambda: eng_h.schnorr_verify(h_pkx, np_dg, h_ssig)),
                ("ecdsa_recover", lambda: eng_h.ecdsa_recover(np_dg, h_sig65)),
                ("ecdh", lambda: eng_h.ecdh(h_priv, h_pub)),
                ("scalar_mult_ct", lambda: eng_h.scalar_mult(h_priv, h_pub)),
                ("ecdsa_sign_rfc6979", lambda: eng_h.ecdsa_sign_rfc6979(h_priv, np_dg)),
                ("schnorr_sign", lambda: eng_h.schnorr_sign(h_priv, np_dg, h_aux))):
            ms = wall(fn)
            other[name]["e2e_items_per_s"] = n / (ms * 1e-3)
            other[name]["e2e_ms"] = ms
        ms = wall(lambda: eng_h.scalar_base_mult(h_priv))
        sbm["1048576_e2e"] = n / (ms * 1e-3)
        eng_h.close()

    # ---- BASELINE configs[4]: Pippenger MSM over n = 2^20 points, SHARDED across the N GPUs (strong scaling) --------
    # every rank reduces its contiguous slice; ONE ncclAllGather of 112 bytes per rank inside s256_msm_sharded[_dev];
    # bit-exact against the closed form (sum s_i d_i) G before it is timed
    msm = None
    if not args.headline_only:
        n_msm = 1 << args.batch_log2
        lo, hi = pkg.parallel.shard_range(n_msm, rank, world)
        if world > 1:
            pkg.parallel.init_comm(eng)
        wm = pkg.synth.msm_batch(hi - lo, eng.scalar_base_mult, start=lo)
        mine = int.from_bytes(wm["closed_form_scalar"], "big")
        if world > 1:
            rows = pkg.parallel.gather_bytes(np.frombuffer(wm["closed_form_scalar"], np.uint8), device="cuda")
            mine = sum(int.from_bytes(r.tobytes(), "big") for r in rows) % pkg.synth.N
        exp_pt, exp_st = eng.scalar_base_mult(np.frombuffer(mine.to_bytes(32, "big"), np.uint8))
        hk = torch.from_numpy(np.ascontiguousarray(wm["k32"])).pin_memory()
        hp = torch.from_numpy(np.ascontiguousarray(wm["pt65"])).pin_memory()
        dk, dp = hk.cuda(), hp.cuda()
        run_dev = (lambda: eng.msm_sharded(dk, dp)) if world > 1 else (lambda: eng.msm(dk, dp))
        run_host = (lambda: eng.msm_sharded(hk.numpy(), hp.numpy())) if world > 1 else (lambda: eng.msm(hk.numpy(), hp.numpy()))
        for _ in range(3):
            mo, mst = run_dev()
        torch.cuda.synchronize()
        assert int(mst.cpu()[0]) == int(exp_st[0]) and np.array_equal(mo.cpu().numpy(), np.asarray(exp_pt)[0]), \
            "sharded MSM differs from the closed form"
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        barrier(); torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            run_dev()
        b.record(); torch.cuda.synchronize()
        msm_ms = max_over_ranks(a.elapsed_time(b)) / reps
        barrier()
        ho, hst = run_host()
        assert hst == int(exp_st[0]) and np.array_equal(np.asarray(ho), np.asarray(exp_pt)[0])
        barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            run_host()
        msm_e2e_ms = max_over_ranks(time.perf_counter() - t0) / reps * 1e3
        barrier()
        c_win, nwin = pkg.msm_plan(hi - lo)
        msm = {"n": n_msm, "n_gpus": world, "scaling": "strong", "ms_per_call": msm_ms, "points_per_s": n_msm / (msm_ms * 1e-3),
               "e2e_ms_per_call": msm_e2e_ms, "e2e_points_per_s": n_msm / (msm_e2e_ms * 1e-3),
               "bit_exact_vs_closed_form": True, "window_bits": c_win, "windows": nwin,
               "collective": ("one ncclAllGather of 112 B per rank inside s256_msm_sharded[_dev] (NCCL dlopen'ed by the C ABI)"
                              if world > 1 else "none (one GPU)"),
               "h2d_bytes_per_call_per_rank": int((hi - lo) * 97), "d2h_bytes_per_call": 66,
               # bucket accumulation only: one mixed addition per point and window with a non-zero digit
               # (2 (hi - lo) virtual points: every scalar is split in two 128-bit halves by the endomorphism)
               "mac32_bucket_accumulation": float(2 * (hi - lo) * nwin * (1 - 2.0 ** -c_win) * pkg.mac32_per_item("msm_mixed_add")),
               "frac_of_int_mul_peak_whole_call": float(2 * (hi - lo) * nwin * (1 - 2.0 ** -c_win) * pkg.mac32_per_item("msm_mixed_add")
                                                        / (msm_ms * 1e-3) / imad_peak)}

    if rank == 0:
        # dominant kernel: executed MAC32 of one k_dsm launch (measured addition count) / its mean duration
        ladder_mac = pkg.load_library().s256_mac32_k_dsm((adds_a + adds_b) / n, adds_b / n)
        mac_item = pkg.mac32_per_item("ecdsa_verify") - pkg.mac32_per_item("k_dsm") + ladder_mac
        achieved = ladder_mac * n / ((dsm_ms / max(dsm_launches, 1)) * 1e-3) if dsm_launches else None
        rcb_mac = 8 * 519 + 7 * 776 + 125 * 519 + ((adds_a + adds_b) / n) * 849 + (adds_b / n) * 73 + 12 * 776
        cpu = None
        if not args.skip_cpu_baseline:
            from oracle import oracle as orc
            threads = orc.default_threads()
            sample = min(n, max(4096, 2048 * threads))
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < 5.0 or reps < 1:
                okc = orc.batch_ecdsa_verify(np_pk[:sample], np_dg[:sample], np_sg[:sample])
                reps += 1
            dt = time.perf_counter() - t0
            assert np.array_equal(okc, expected[:sample])
            cpu = {"value": sample * reps / dt, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"first {sample} items of the same batch x {reps} passes on {threads} threads (~{dt:.0f} s); C port of "
                             "the reference's algorithms (Go toolchain absent; the reference's README quotes ~1.1e4 "
                             "verifies/s per core for its Go code, so this port runs at about half the reference's speed)"}
            # sanity anchor beside the port (BASELINE.md 3.3): OpenSSL's ECDSA_do_verify on the same rows, all threads,
            # keys and signatures parsed outside the timed region
            osl_n = min(sample, 1024 * threads)
            r = orc.openssl_ecdsa_verify(np_pk[:osl_n], np_dg[:osl_n], np_sg[:osl_n], reps=1)
            if r is None:
                cpu["openssl"] = {"unavailable": "libcrypto or its headers are missing on this box"}
            else:
                reps_o = max(1, min(64, int(3.0 / max(r[1], 1e-3))))
                ok_o, secs = orc.openssl_ecdsa_verify(np_pk[:osl_n], np_dg[:osl_n], np_sg[:osl_n], reps=reps_o)
                assert np.array_equal(ok_o, expected[:osl_n]), "OpenSSL disagrees with the construction"
                cpu["openssl"] = {"value": osl_n * reps_o / secs, "unit": UNIT, "cores": threads,
                                  "sample": f"ECDSA_do_verify of the system libcrypto over the first {osl_n} rows x {reps_o} passes on "
                                            f"{threads} threads; keys and signatures parsed outside the timed region"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32 limbs (8x32, IMAD.WIDE.U32 carry chains)", "data": "synthetic",
            "config": workload_config(world, n),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(n * 161), "d2h_bytes_per_step": int(n),
                    "callers": None if e2e_value is None else (2 if e2e_value == e2e_two else 1),
                    "single_caller": e2e_single, "two_callers": e2e_two,
                    "note": "value = the better of one synchronous caller and two callers (two contexts, two host threads, "
                            "alternate batches); every batch crosses PCIe both ways inside the timed region.  Two contexts also "
                            "overlap each other's scalar kernels and kernel tails with a ladder, which the single device-resident "
                            "caller behind `value` cannot, so two_callers may exceed `value` by ~0.5 %",
                    "h2d_gbs_per_rank_all_ranks_copying": h2d_gbs},
            "gpu_launches": int(launches),
            "clocks": dict(clocks, per_rank_sm_mhz=rank_sm_mhz), "per_rank_ms_per_step": per_rank_ms,
            "roofline": {"bound": "int-mul",
                         "bound_note": "32x32->64 multiply issue (IMAD.WIDE.U32, half rate on sm_100); not hbm/tensor: "
                                       "161 B and ~110k multiply-accumulates per verification",
                         "kernel": "k_dsm", "achieved": achieved / 1e12 if achieved else None,
                         "peak": imad_peak / 1e12, "unit": "TMAC32/s",
                         "frac": (achieved / imad_peak) if achieved else None,
                         "frac_vs_nominal": (achieved / 9.3062e12) if achieved else None,
                         "peak_source": "measured live in this process straight AFTER the timed steps (hot clocks), best of 5: "
                                        "s256_microbench_imad (mad.lo.cc/madc.hi.cc chains = IMAD.WIDE.U32[.X], SASS-checked, all "
                                        "SMs); nominal 148 SM x 32 MAC32/clk x 1.965 GHz = 9.306",
                         "peak_runs": [v / 1e12 for v in imad_runs],
                         "peak_probe_clocks": {k: probe_clocks.get(k) for k in ("sm_mhz", "power_w_max", "reasons", "window")},
                         # the highest the same probe has read on this pool, standalone on a cold GPU
                         # (profiles/r01_microbench_int_pipes.json, r01_bench_final_1gpu.json): 8.85
                         "frac_vs_best_probe_on_record": (achieved / 8.85e12) if achieved else None,
                         "ladder_adds_per_item_measured": (adds_a + adds_b) / n,
                         "mac32_per_item_kernel": ladder_mac, "mac32_per_item_whole_verify": mac_item,
                         "kernel_ms": dsm_ms / max(dsm_launches, 1), "kernel_share_of_step": dsm_ms / ms_total if world == 1 else None,
                         "whole_step_frac": value / world * mac_item / imad_peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum of ONE k_dsm launch at 2^20 items, from the
                         # committed capture profiles/r01_ncu_final_dsm.txt (4.752 GB + 1.850 GB); scaled if --batch-log2 differs
                         # The same launch counted with the complete-formula work of rounds 1-2a (doubling 519, addition 849,
                         # mixed 776 MAC32: what this kernel executed before its ladder moved to Jacobian coordinates).  The
                         # result is identical, so this is the rate at which the OLD amount of work is now retired -- quoted
                         # only to compare with the earlier rounds' fractions; `frac` above counts executed work.
                         "mac32_per_item_kernel_complete_formulas": rcb_mac,
                         "frac_if_counted_as_complete_formulas": (rcb_mac * n / ((dsm_ms / max(dsm_launches, 1)) * 1e-3) / imad_peak)
                         if dsm_launches else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum of ONE k_dsm launch at 2^20 items, from the
                         # committed capture profiles/r02b_ncu_dsm.txt (4.155 GB + 2.469 GB); scaled if --batch-log2 differs
                         "traffic": 6.624e9 * n / (1 << 20), "traffic_unit": "bytes per launch",
                         "traffic_note": "ncu --set full, profiles/r02b_ncu_dsm.txt: ~6.3 KB per item (Jacobian multiples and "
                                         "their Z products written and read back, 16 affine rows written, row and comb "
                                         "gathers) = 0.36 TB/s, 5-6 % of the measured HBM copy peak; not the bound",
                         "hbm_frac": (6.624e9 * n / (1 << 20)) / ((dsm_ms / max(dsm_launches, 1)) * 1e-3) / (hbm_peak_gbs() * 1e9),
                         "hbm_peak_gbs": hbm_peak_gbs()},
            "cpu_baseline": cpu,
            "msm": msm,
            "scalar_base_mult_ops_per_sec": sbm,
            "other_paths": other,
            "input_generation_s": t_gen,
        }
        emit(line)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"ecdsa_verify_ok" + (f"_rank{rank}" if world > 1 else ""): ok_last})
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
