"""Build libacoss_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["api.cu", "k0_onramp.cu", "k1_oti.cu", "k2_exact.cu", "k2_fast.cu", "k3_dp.cu", "k4_knn.cu", "k5_earlyfusion.cu", "k6_simple.cu", "k7_snf.cu"]
HEADERS = ["common.cuh", "k2_fast.cuh", "k2_tc.inl", "../../include/acoss_b200.h"]
OUT = os.path.join(HERE, "libacoss_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(HERE, f)) > t for f in SOURCES + HEADERS + ["build.py"])


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    objs = []
    for src in SOURCES:
        obj = os.path.join(HERE, src.replace(".cu", ".o"))
        cmd = ["nvcc", *NVCC_FLAGS, "-c", os.path.join(HERE, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        subprocess.check_call(cmd)
        objs.append(obj)
    subprocess.check_call(["nvcc", "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT, *objs])
    return OUT


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
