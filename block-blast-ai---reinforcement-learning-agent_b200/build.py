"""In-tree build of libbbgpu.so (hand-written sm_100a CUDA behind the C ABI of include/bbgpu.h).

nvcc cross-compiles without a GPU; the .so stays next to this file (git-ignored, but it
travels to the GPU box with the gpurun snapshot).
"""
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB = os.path.join(PKG_DIR, "libbbgpu.so")
SOURCES = ["bb_env_kernels.cu", "bb_policy_kernels.cu", "bb_gae_kernels.cu", "bb_bn_kernels.cu", "bb_capi.cu"]
HEADERS = ["bb_rules.cuh", "bb_kernels.h", "bb_piece_table.inc", "bb_sym_table.inc", os.path.join("..", "..", "include", "bbgpu.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--fmad=true", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-Xptxas", "-warn-spills"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _host_compiler_flags():
    # the image's $CC may be a toolchain wrapper; the distro g++ is what nvcc 12.9 expects
    if os.path.exists("/usr/bin/g++"):
        return ["-ccbin", "/usr/bin/g++"]
    return []


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a into libbbgpu.so. Returns the library path."""
    if not force and not needs_build():
        return LIB
    objs = []
    log = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [_nvcc()] + _host_compiler_flags() + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append(r.stderr)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed on " + src)
        objs.append(obj)
    cmd = [_nvcc()] + _host_compiler_flags() + ["-shared", "-o", LIB] + objs + ["-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    with open(os.path.join(CSRC, "ptxas_report.txt"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
