"""Builds libpolypolish_b200.so (CUDA kernels + C-ABI + host text layer) and the `polypolish` CLI for sm_100a.

nvcc cross-compiles without a GPU; the artefacts land in-tree under build/ (git-ignored, shipped by gpurun)."""
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "polypolish_b200", "csrc")
OUT = os.path.join(ROOT, "build")
LIB = os.path.join(OUT, "libpolypolish_b200.so")
CLI = os.path.join(OUT, "polypolish")

NVCC = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function,-ffp-contract=off",
          "-fmad=false"]   # IEEE double semantics: no FMA contraction anywhere near the vote

LIB_SOURCES = ["polish_kernels.cu", "filter_kernels.cu", "tok_kernels.cu", "fasta.cpp", "sam_pack.cpp", "filter_pack.cpp",
               "host_api.cpp", "synth.cpp", "shard.cpp", "bam.cpp"]
CLI_SOURCES = ["cli_main.cpp"]


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    deps = list(sources) + [os.path.join(CSRC, "pp_internal.h"), os.path.join(CSRC, "nib_utils.h"), os.path.join(CSRC, "pp_ctx.cuh"), os.path.join(CSRC, "polish_dev.cuh"),
                            os.path.join(CSRC, "tok_line.h"), os.path.join(CSRC, "tok_table.h"), os.path.join(CSRC, "filter_dev.h"), os.path.join(CSRC, "tok_strip.h"), os.path.join(CSRC, "bam_rec.h"), os.path.join(ROOT, "include", "pp_abi.h"),
                            os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    os.makedirs(OUT, exist_ok=True)
    objs = []
    for src in LIB_SOURCES:
        sp = os.path.join(CSRC, src)
        if not os.path.exists(sp):
            continue
        obj = os.path.join(OUT, src.rsplit(".", 1)[0] + ".o")
        if force or _stale(obj, [sp]):
            cmd = [NVCC] + ARCH + COMMON + ["-x", "cu", "-c", sp, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
        objs.append(obj)
    if force or _stale(LIB, objs):
        subprocess.check_call([NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-lz", "-lpthread"])
    cli_src = [os.path.join(CSRC, s) for s in CLI_SOURCES if os.path.exists(os.path.join(CSRC, s))]
    if cli_src and (force or _stale(CLI, cli_src + [LIB])):
        subprocess.check_call([NVCC, "-O2", "-std=c++17", "-o", CLI] + cli_src +
                              ["-L" + OUT, "-lpolypolish_b200", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"])
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
