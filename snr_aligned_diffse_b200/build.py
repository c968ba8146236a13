"""Build `libsnrse_b200.so` (all CUDA kernels + the C ABI) for sm_100a with nvcc, in-tree.

    python -m snr_aligned_diffse_b200.build [--force]

nvcc cross-compiles without a GPU.  The library lands next to this file so it travels with the
source tree; objects go to `csrc/build/` (git-ignored).
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libsnrse_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; cannot build the sm_100a library")
    return exe


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _newest_header():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hs.append(os.path.join(os.path.dirname(HERE), "include", "snrse_b200.h"))
    hs.append(os.path.join(os.path.dirname(HERE), "include", "snrse_b200_debug.h"))
    hs.append(os.path.join(os.path.dirname(HERE), "include", "snrse_b200_layers.h"))
    hs.append(os.path.join(os.path.dirname(HERE), "include", "snrse_b200_plans.h"))
    return max(os.path.getmtime(h) for h in hs if os.path.exists(h))


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    hdr = _newest_header()
    jobs = []
    for src in sources():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src[:-3] + ".o")
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hdr):
            jobs.append((s, o))

    def run(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (s, r.stdout, r.stderr))
        return s

    with concurrent.futures.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        for s in ex.map(run, jobs):
            if verbose:
                print("compiled", os.path.basename(s))
    objs = [os.path.join(OBJ, src[:-3] + ".o") for src in sources()]
    if jobs or force or not os.path.exists(LIB):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
