"""In-tree build of libb200zk.so (sm_100a only) with plain nvcc.

Objects are cached by source hash under csrc/_build/ so that a rebuild only
recompiles what changed; the shared library lands next to this file and travels
to the GPU box with the repo snapshot.
"""
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(CSRC, "_build")
LIB = os.path.join(HERE, "libb200zk.so")
SOURCES = ["api.cu", "ntt.cu", "msm_g1.cu", "msm_g2.cu", "prove.cu", "r1cs.cu", "hostcheck.cu", "verify.cu", "witness.cu", "setup_host.cu", "setup.cu", "verify_batch.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libb200zk cannot be built (there is no CPU fallback)")
    return exe


def _digest(paths):
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    return h.hexdigest()[:16]


def _headers():
    out = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".hpp", ".inc"))]
    out.append(os.path.join(HERE, "..", "include", "b200zk.h"))
    return out


def build_library(verbose=False, force=False):
    """Compile every translation unit and link libb200zk.so; returns its path."""
    os.makedirs(BUILD, exist_ok=True)
    nvcc = _nvcc()
    hdrs = _headers()
    jobs = []
    objs = []
    for src in SOURCES:
        sp = os.path.join(CSRC, src)
        tag = _digest([sp] + hdrs)
        obj = os.path.join(BUILD, "%s.%s.o" % (src[:-3], tag))
        objs.append(obj)
        if force or not os.path.exists(obj):
            for old in os.listdir(BUILD):
                if old.startswith(src[:-3] + ".") and old.endswith(".o"):
                    os.remove(os.path.join(BUILD, old))
            jobs.append([nvcc] + NVCC_FLAGS + ["-c", sp, "-o", obj])

    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), r.stderr[-4000:]))
        return r

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(run, jobs))
    stamp = os.path.join(BUILD, "link.stamp")
    want = _digest(objs) if all(os.path.exists(o) for o in objs) else ""
    have = open(stamp).read() if os.path.exists(stamp) else ""
    if force or jobs or not os.path.exists(LIB) or want != have:
        run([nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
        with open(stamp, "w") as f:
            f.write(want)
    return LIB


if __name__ == "__main__":
    print(build_library(verbose=True, force="--force" in sys.argv))
