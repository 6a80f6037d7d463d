"""In-tree build of the CUDA library and the CLI (sm_100a only).

    python -m microphaser_b200.build

produces microphaser_b200/_lib/libmicrophaser_gpu.so and microphaser_b200/_lib/microphaser.
nvcc cross-compiles without a GPU; the built files travel to the GPU box with the repo snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "_lib")
LIB = os.path.join(OUT, "libmicrophaser_gpu.so")
CLI = os.path.join(OUT, "microphaser")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVFLAGS = ARCH + ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-missing-field-initializers"]


def _sources():
    out = []
    for root, _, files in os.walk(CSRC):
        for f in files:
            if f.endswith((".cu", ".cuh", ".h", ".hpp", ".cpp")):
                out.append(os.path.join(root, f))
    out.append(os.path.join(HERE, "..", "include", "microphaser_gpu.h"))
    return out


def _stale(target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in _sources())


def build_all(force=False, verbose=False):
    os.makedirs(OUT, exist_ok=True)
    if force or _stale(LIB):
        objs = []
        for src in (os.path.join(CSRC, "kernels", "phase_kernels.cu"), os.path.join(CSRC, "kernels", "replay_kernels.cu"),
                    os.path.join(CSRC, "kernels", "normal_kernels.cu"), os.path.join(CSRC, "kernels", "peptide_kernels.cu"),
                    os.path.join(CSRC, "kernels", "record_kernels.cu"), os.path.join(CSRC, "kernels", "inflate_kernels.cu"),
                    os.path.join(CSRC, "kernels", "block_kernels.cu"),
                    os.path.join(CSRC, "capi.cu")):
            obj = os.path.join(OUT, os.path.basename(src) + ".o")
            cmd = [NVCC] + NVFLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            subprocess.run(cmd, check=True)
            objs.append(obj)
        subprocess.run([NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-lz", "-lpthread", "-cudart", "static"], check=True)
    if force or _stale(CLI):
        subprocess.run(["g++", "-std=c++17", "-O2", "-o", CLI, os.path.join(CSRC, "cli_main.cpp"), "-L" + OUT, "-lmicrophaser_gpu",
                        "-Wl,-rpath,$ORIGIN"], check=True)
    return LIB, CLI


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv, verbose="-v" in sys.argv))
