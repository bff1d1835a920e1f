"""Compiles libjvector_b200.so in-tree with nvcc for sm_100a (no GPU needed: nvcc cross-compiles)."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# JV_B200_LIBDIR: where a tuning variant (built with JV_NVCC_EXTRA) goes, next to the product library
LIBDIR = os.environ.get("JV_B200_LIBDIR") or os.path.join(HERE, "lib")
SO = os.path.join(LIBDIR, "libjvector_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CU = ["kernels_batch.cu", "bq_imma.cu", "bq_umma.cu", "search.cu", "sketch.cu", "build.cu", "api.cu"]
CPP = ["legacy_host.cpp", "legacy_simd.cpp", "legacy_avx512.cpp"]
HEADERS = ["common.cuh", "scorers.cuh", "kernels.h", "legacy_avx512.h", os.path.join("..", "..", "include", "jvector_b200.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
# -fmad=false: only explicit fmaf() fuses (NVQ bit tricks and score maps must round like the reference's scalar code)
EXTRA = os.environ.get("JV_NVCC_EXTRA", "").split()
NVFLAGS = EXTRA + ["-O3", "-std=c++17", "-lineinfo", "-fmad=false", "-Xcompiler", "-fPIC,-fvisibility=hidden,-O3", "-Xptxas", "-v"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    objs = []
    for src in CU + CPP:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src + ".o")
        objs.append(o)
        if force or _newer(o, [s] + hdrs):
            if src.endswith(".cu"):
                cmd = [NVCC] + ARCH + NVFLAGS + ["-c", s, "-o", o]
            else:
                # legacy_host.cpp: explicit fmaf only (NVQ bit tricks); legacy_simd.cpp: let the vectoriser fuse (target_clones pick the ISA)
                # legacy_host.cpp: explicit fmaf only (NVQ bit tricks); legacy_simd.cpp: let the vectoriser fuse (target_clones pick the ISA);
                # legacy_avx512.cpp: intrinsics under per-function target attributes, explicit FMAs only
                host = {"legacy_simd.cpp": "-fPIC,-fvisibility=hidden,-O3,-ffp-contract=fast,-fno-math-errno",
                        "legacy_avx512.cpp": "-fPIC,-fvisibility=hidden,-O3,-ffp-contract=off,-fno-math-errno"}.get(src, "-fPIC,-fvisibility=hidden,-O3,-mfma,-ffp-contract=off")
                cmd = [NVCC, "-O3", "-std=c++17", "-Xcompiler", host, "-c", s, "-o", o]
            jobs.append((src, cmd))

    def run(job):
        src, cmd = job
        p = subprocess.run(cmd, capture_output=True, text=True)
        return src, p.returncode, p.stdout + p.stderr

    logs = {}
    if jobs:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            for src, rc, out in ex.map(run, jobs):
                logs[src] = out
                if rc != 0:
                    sys.stderr.write(out)
                    raise RuntimeError("nvcc failed on %s" % src)
                if verbose:
                    sys.stderr.write(out)
        with open(os.path.join(LIBDIR, "ptxas_info.log"), "a") as f:
            for src, out in logs.items():
                f.write("==== %s ====\n%s\n" % (src, out))
    if jobs or force or _newer(SO, objs):
        cmd = [NVCC] + ARCH + ["-shared", "-o", SO] + objs + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"]
        p = subprocess.run(cmd, capture_output=True, text=True)
        if p.returncode != 0:
            sys.stderr.write(p.stdout + p.stderr)
            raise RuntimeError("link failed")
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
