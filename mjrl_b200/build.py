"""Build libmjrl_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

    python -m mjrl_b200.build [--force]
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libmjrl_b200.so")
SOURCES = ["engine.cu", "mlp_h32.cu", "mlp_h64.cu", "mlp_h128.cu", "mlp_h256.cu", "linear_kernel.cu",
           "scan.cu", "vecops.cu", "vf_fit.cu", "fvp_tc.cu", "linear_tc.cu", "vf_fit_tc.cu", "host_perm.cu", "p2p.cu", "ridge.cu",
           "policy_sgd.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "mjrl_b200.h"))
    nvcc = _nvcc()
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (s, r.stdout, r.stderr))
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        logs = list(ex.map(compile_one, jobs))
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    if verbose:
        for l in logs:
            sys.stderr.write(l)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
