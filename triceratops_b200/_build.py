"""Builds csrc/ into the in-tree shared library with nvcc for sm_100a (no JIT cache)."""
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(CSRC, "libtriceratops_b200.so")
HOST_SO_PATH = os.path.join(CSRC, "libtriceratops_host.so")   # prior-draw helpers (host_*.c)
SOURCES = ["tri_cabi.cu"]
HEADERS = ["tri_kernels.cuh", "tri_model.cuh", "tri_sampler.cuh", os.path.join("..", "..", "include", "triceratops_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-shared", "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built")


def needs_build():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build_host(force=False):
    """gcc build of csrc/host_prep.c (OpenMP spline evaluation for the prior-draw preparation)."""
    srcs = [os.path.join(CSRC, "host_prep.c"), os.path.join(CSRC, "host_rng.c"),
            os.path.join(CSRC, "host_blocks.c")]
    if (not force and os.path.exists(HOST_SO_PATH)
            and os.path.getmtime(HOST_SO_PATH) >= max(os.path.getmtime(s) for s in srcs)):
        return HOST_SO_PATH
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    # -O3 for the vectorised MT19937 recurrence of host_rng.c (integer work; the spline code
    # of host_prep.c keeps its operation order: no contraction, no fast-math)
    base = [cc, "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-std=gnu11"]
    for extra in (["-fopenmp"], []):
        if subprocess.run(base + extra + ["-o", HOST_SO_PATH] + srcs).returncode == 0:
            return HOST_SO_PATH
    raise RuntimeError("could not build " + HOST_SO_PATH)


def build(force=False, verbose=False):
    """Compile the CUDA library if sources are newer than the .so; returns its path."""
    build_host(force)
    if not force and not needs_build():
        return SO_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + ["-o", SO_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    env = dict(os.environ)
    # the image exports CC/CXX=/opt/gcc/bin/*; nvcc should use the system host compiler
    if os.path.exists("/usr/bin/g++"):
        cmd += ["-ccbin", "/usr/bin/g++"]
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    log = os.path.join(CSRC, "build.log")
    with open(log, "w") as f:
        f.write(" ".join(cmd) + "\n" + proc.stdout)
    if verbose:
        print(proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout[-4000:])
    return SO_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
