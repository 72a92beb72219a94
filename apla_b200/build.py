"""Builds libapla_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m apla_b200.build [--force]

No torch dependency: the library exports plain `extern "C"` symbols (include/apla_b200.h) and is loaded with
ctypes by apla_b200/_lib.py.  Objects are cached per source file under apla_b200/csrc/build/.
"""
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libapla_b200.so")
SOURCES = ["common.cu", "gemm.cu", "gemm2.cu", "attention.cu", "attention_tc.cu", "attention_tc_bwd.cu", "attention_fused.cu", "attention_bwd2.cu", "attention_fwd_sr.cu", "attention_cls.cu", "attention_probs.cu", "rowwise.cu", "head_optim.cu", "dp_allreduce.cu", "ssl.cu", "engine.cu", "block.cu", "capi.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "--use_fast_math",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-DNDEBUG"] + os.environ.get("APLA_NVCC_EXTRA", "").split()


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _digest(paths):
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(os.path.dirname(HERE), "include", "apla_b200.h"))
    return hs


def build(force=False, verbose=False):
    os.makedirs(BUILD, exist_ok=True)
    nvcc = nvcc_path()
    hdr = _headers()
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs, jobs = [], []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(BUILD, s + ".o")
        stamp = obj + ".sha"
        dig = _digest([src] + hdr)
        objs.append(obj)
        if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
            continue
        jobs.append((s, src, obj, stamp, dig))

    def compile_one(job):
        s, src, obj, stamp, dig = job
        cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{r.stdout}\n{r.stderr}")
        with open(os.path.join(BUILD, s + ".ptxas.txt"), "w") as f:
            f.write(r.stderr)
        with open(stamp, "w") as f:
            f.write(dig)
        return s

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for s in ex.map(compile_one, jobs):
                if verbose:
                    print("compiled", s)
    if jobs or not os.path.exists(LIB):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
