"""Builds the C-ABI shared library for sm_100a with nvcc (in-tree, so the .so
travels to the GPU box with the repo snapshot)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
# S256_LIB=<path> selects a prebuilt variant (tuning experiments); it is never rebuilt.
LIB = os.environ.get("S256_LIB") or os.path.join(LIBDIR, "libsecp256k1_b200.so")
SOURCES = ["api.cu", "api_msm.cu", "api_sign.cu", "api_h2c.cu", "kern_ct.cu", "codecs.cpp"]
HEADERS = ["fe.cuh", "sc.cuh", "point.cuh", "sha256.cuh", "kernels.cuh", "microbench.cuh", "launchers.h", "msm.cuh", "fe_sqr_gen.cuh", "ctx.h", "h2c.cuh", "fe_vt.cuh", "coop.cuh", "modinv.cuh", "fe_mul_gen.cuh", "jac.cuh", "batch.cuh"]


def nvcc_cmd(extra=(), out=None):
    return ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
            "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
            "-Xptxas", "-v", *extra,
            "-o", out or LIB] + [os.path.join(CSRC, s) for s in SOURCES]


def is_stale():
    if os.environ.get("S256_LIB"):
        return False
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "secp256k1_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_one(args):
    src, obj, extra = args
    cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v", *extra, "-c", "-o", obj, src]
    p = subprocess.run(cmd, capture_output=True, text=True)
    return p.returncode, p.stdout + p.stderr


def build(force=False, verbose=False, extra=(), out=None):
    """One nvcc per source in parallel (cicc + ptxas dominate), then one link step."""
    if out is None and not force and not is_stale():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(LIBDIR, exist_ok=True)
    target = out or LIB
    objdir = target + ".obj"
    os.makedirs(objdir, exist_ok=True)
    jobs = [(os.path.join(CSRC, s), os.path.join(objdir, s.rsplit(".", 1)[0] + ".o"), tuple(extra)) for s in SOURCES]
    with ThreadPoolExecutor(len(jobs)) as ex:
        results = list(ex.map(_compile_one, jobs))
    log = "".join(r[1] for r in results)
    rc = max(r[0] for r in results)
    if rc == 0:
        link = subprocess.run(["nvcc", "-shared", "-o", target] + [j[1] for j in jobs], capture_output=True, text=True)
        log += link.stdout + link.stderr
        rc = link.returncode

    class _P:  # keep the shape the code below expects
        returncode = rc
    p = _P()
    with open((out or os.path.join(LIBDIR, "build")) + ".log" if out else os.path.join(LIBDIR, "build.log"), "w") as f:
        f.write(log)
    if p.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed building libsecp256k1_b200.so")
    if verbose:
        print(log)
    return out or LIB


if __name__ == "__main__":
    build(force=True, verbose="-v" in sys.argv)
    print(LIB)
