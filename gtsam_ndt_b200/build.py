"""In-tree build recipes: nvcc for the CUDA library (sm_100a only), gcc for the host-only synth helper.

The built .so files live next to this file; they are git-ignored but travel to the GPU box.
"""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB_CUDA = os.path.join(HERE, "libndt2d.so")
LIB_SYNTH = os.path.join(HERE, "libndt2d_synth.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",  # SPEC.md: only explicit fma() fuses
    "-Xcompiler", "-fPIC,-ffp-contract=off,-O2", "-shared", "-Xptxas", "-v",
]


def _stale(out, srcs):
    return (not os.path.exists(out)) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs)


def _host_cc():
    for c in ("/usr/bin/gcc", shutil.which("gcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("gcc not found")


def cuda_sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def build_cuda(force=False, verbose=False):
    srcs = cuda_sources()
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))] + \
        [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE)]
    if not force and not _stale(LIB_CUDA, deps):
        return LIB_CUDA
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libndt2d.so must be prebuilt")
    extra = os.environ.get("NDT2D_NVCC_EXTRA", "").split()   # kernel tuning experiments, e.g. -maxrregcount=96
    cmd = [nvcc, "-ccbin", "/usr/bin/g++"] + NVCC_FLAGS + extra + ["-I", INCLUDE, "-I", CSRC, "-o", LIB_CUDA] + srcs + ["-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log = r.stdout + r.stderr
    with open(os.path.join(HERE, "build_cuda.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-6000:])
    if verbose:
        print(log)
    return LIB_CUDA


def build_variant(name, extra_flags):
    """Kernel tuning experiments: the same sources with extra nvcc flags -> build/variants/libndt2d_<name>.so
    (git-ignored, travels to the GPU box). Select it at run time with NDT2D_LIB=<path>."""
    out_dir = os.path.join(os.path.dirname(HERE), "build", "variants")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, f"libndt2d_{name}.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc, "-ccbin", "/usr/bin/g++"] + NVCC_FLAGS + list(extra_flags) + ["-I", INCLUDE, "-I", CSRC, "-o", out] + cuda_sources() + ["-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(out + ".log", "w") as f:
        f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + (r.stdout + r.stderr)[-6000:])
    return out


def build_synth(force=False):
    src = os.path.join(CSRC, "synth.c")
    if not force and not _stale(LIB_SYNTH, [src]):
        return LIB_SYNTH
    cmd = [_host_cc(), "-O2", "-std=c11", "-fPIC", "-fopenmp", "-shared", "-o", LIB_SYNTH, src, "-lm"]
    subprocess.check_call(cmd)
    return LIB_SYNTH


def build_all(force=False, verbose=False):
    build_synth(force)
    return build_cuda(force, verbose)


if __name__ == "__main__":
    import sys
    build_all(force="--force" in sys.argv, verbose=True)
