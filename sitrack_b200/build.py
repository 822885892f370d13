"""Build libsitrack_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m sitrack_b200.build [--force]
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libsitrack_b200.so")
SOURCES = ["st_api.cu", "st_advect.cu", "st_locate.cu", "st_geom.cu", "st_ext.cu", "st_deform.cu", "st_deform_scale.cu", "st_deform_grid.cu", "st_disperse.cu"]
HEADERS = ["st_device.cuh", "st_kernels.h", "st_deform.cuh", "st_persist.cuh", "st_pipe.cuh", "st_warp.cuh", "st_cert.cuh", "st_experiments.cuh", os.path.join("..", "..", "include", "sitrack_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # parity-critical expressions use __dmul_rn/__dadd_rn explicitly; this keeps
    # everything else un-contracted too unless it asks for fma() by name
    "-fmad=false",
    "--shared", "-Xcompiler", "-fPIC",
    "-cudart", "shared",
]


def nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """defines/out: experimental A/B builds (`python -m sitrack_b200.build -DNAME=V -o path.so`)."""
    if not force and not stale() and not out:
        return SO
    cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-D" + d for d in defines] + \
          ["-o", out or SO] + [os.path.join(CSRC, f) for f in SOURCES]
    env = dict(os.environ)
    # an env CC/CXX may point at a wrapper; let nvcc use the system g++
    if os.path.exists("/usr/bin/g++"):
        cmd[1:1] = ["-ccbin", "/usr/bin/g++"]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout)
    if r.returncode:
        raise RuntimeError("nvcc failed (%d)" % r.returncode)
    return out or SO


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv if a.startswith("-D")]
    outp = sys.argv[sys.argv.index("-o") + 1] if "-o" in sys.argv else None
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs, out=outp))
