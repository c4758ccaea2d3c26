"""Builds libvn_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

No torch headers are involved: the library is plain CUDA runtime + extern "C" and is bound with
ctypes (lib.py).  nvcc cross-compiles without a GPU, so this also runs in the CPU-only container.
"""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libvn_b200.so")
SOURCES = ["vn_env.cu", "vn_rollout.cu", "vn_conv.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math=false",
              "-Xcompiler", "-fPIC,-O3,-Wall", "-shared", "-cudart", "shared"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "vn_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compiles into a temporary file and renames it over libvn_b200.so under an exclusive file lock: ranks of one
    torchrun job that all find the library missing build one after the other (the later ones find it fresh and
    return), and no process can ever CDLL a half-written file."""
    import fcntl
    import tempfile
    with open(os.path.join(PKG, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB
            fd, tmp = tempfile.mkstemp(prefix=".libvn_b200.", suffix=".so.tmp", dir=PKG)
            os.close(fd)
            cmd = [nvcc_path()] + [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + \
                ["-I", os.path.join(ROOT, "include"), "-I", CSRC] + (["-Xptxas", "-v"] if verbose else []) + \
                [os.path.join(CSRC, s) for s in SOURCES] + ["-o", tmp]
            try:
                res = subprocess.run(cmd, capture_output=True, text=True)
                if res.returncode != 0:
                    sys.stderr.write(res.stdout + res.stderr)
                    raise RuntimeError("nvcc failed building libvn_b200.so")
                os.chmod(tmp, 0o755)
                os.replace(tmp, LIB)
            finally:
                if os.path.exists(tmp):
                    os.unlink(tmp)
            if verbose:
                sys.stderr.write(res.stderr)
            return LIB
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
