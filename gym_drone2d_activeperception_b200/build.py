"""In-tree build of libdrone2d.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m gym_drone2d_activeperception_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdrone2d.so")
SOURCES = ["drone2d.cu"]
DEPS = ["drone2d.cu", "d2d_state.cuh", "d2d_math.cuh", "d2d_step.cuh", "d2d_plan.cuh", "d2d_plan_host.inl", "d2d_plan_math.cuh", "d2d_rvo.cuh", "d2d_rvo_math.cuh", "d2d_clone.cuh", "d2d_worldgen.cuh", "d2d_worldgen_body.inc", "d2d_episode.cuh", "d2d_render.cuh", "d2d_difficulty.cuh", "d2d_agent_math.cuh",
        "d2d_tan_table.inc", "d2d_sincos_table.inc", os.path.join("..", "..", "include", "drone2d.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false",            # parity: the reference rounds every multiply/add separately; FMAs only where written
    "--shared", "-Xcompiler", "-fPIC",
]


def needs_build():
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS if os.path.exists(os.path.join(CSRC, d)))


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout)
    if verbose:
        print(res.stdout)
    return LIB


def build_variant(name, extra_flags):
    """An A/B build of the same ABI next to the product library (selected at run time with D2D_LIB=<path>), e.g.
    build_variant("psmall40", ["-DD2D_PS_NODES=40", "-DD2D_PS_HASH=128"]): nearly every A* search overflows the
    small-footprint kernel and is redone by d2d_plan_kernel."""
    out = os.path.join(HERE, "libdrone2d_%s.so" % name)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
