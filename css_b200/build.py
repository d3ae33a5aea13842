"""Builds libcss_b200.so in-tree with nvcc for sm_100a (no libtorch link, so it cross-compiles without a GPU).

    python -m css_b200.build            # incremental
    python -m css_b200.build --force
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcss_b200.so")
SOURCES = ["css_api.cu", "css_sim.cu", "css_sim_tc.cu", "css_select.cu", "css_stream.cu", "css_proto.cu", "css_score.cu", "css_grad.cu", "css_atl.cu", "css_ohem.cu", "css_aug.cu", "css_aug_image.cu", "css_comm.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--use_fast_math=false"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "css_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
    cmd = [_nvcc(), *flags, "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
           *([] if not verbose else ["-Xptxas", "-v"]),
           "-o", LIB, *[os.path.join(CSRC, s) for s in SOURCES]]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
