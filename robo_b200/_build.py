"""Builds robo_b200/libgpk.so (sm_100a) with nvcc.  In-tree, so the .so travels to the GPU box."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgpk.so")
SOURCES = ["gpk_api.cu"]
HEADERS = ["gpk_internal.cuh", "gpk_gemm.cuh", "gpk_kernels.cuh", "gpk_diag16.cuh", "gpk_chain.cuh", "gpk_multi.inl", "gpk_ozaki.cuh", "gpk_es.cuh", os.path.join("..", "..", "include", "gpk.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile the CUDA library if it is missing or older than its sources.  nvcc writes to a temporary file that is
    renamed over libgpk.so under an exclusive file lock, so concurrent ranks (torchrun) never load a half-written
    library and only one of them compiles."""
    if not force and not needs_build():
        return LIB
    import fcntl
    with open(LIB + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():          # another process built it while we waited
                return LIB
            tmp = "%s.%d.tmp" % (LIB, os.getpid())
            cmd = [_nvcc()] + NVCC_FLAGS + ["-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            try:
                res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            except OSError as e:
                raise RuntimeError("nvcc could not be started: %s" % e)
            if res.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + res.stdout)
            os.replace(tmp, LIB)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
