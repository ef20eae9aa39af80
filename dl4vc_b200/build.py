"""Build the C-ABI CUDA library in-tree: dl4vc_b200/libdan_b200.so (sm_100a only).

    python -m dl4vc_b200.build [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libdan_b200.so")
SOURCES = ["dan_capi.cu", "dan_fp32.cu", "dan_bf16.cu", "dan_train.cu", "dan_losses.cu", "dan_feeder.cu", "dan_inflate.cu", "dan_deflate.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--use_fast_math=false",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--expt-relaxed-constexpr", "-Xptxas", "-v"]
NVCC_FLAGS.remove("--use_fast_math=false")


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "dan_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, defines=(), out: str = OUT) -> str:
    """defines / out: development builds beside the product library (e.g. --prof: cycle counters in the conv-stack kernel,
    loaded through DAN_B200_LIB)."""
    if not force and not defines and not _stale():
        return OUT
    nvcc = nvcc_path()
    objs = []
    build_dir = os.path.join(HERE, "build" + ("_" + "_".join(defines).lower() if defines else ""))
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *["-D" + d for d in defines], "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, obj, p in procs:
        text, _ = p.communicate()
        log.append(text)
        if p.returncode != 0:
            sys.stderr.write(text)
            raise RuntimeError(f"nvcc failed on {src}")
        objs.append(obj)
    with open(os.path.join(build_dir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    cmd = [nvcc, "-shared", "-o", out, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-lcuda"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    return out


if __name__ == "__main__":
    if "--define" in sys.argv:      # development: python -m dl4vc_b200.build --define NAME -> libdan_b200_name.so
        d = sys.argv[sys.argv.index("--define") + 1]
        print(build(force=True, verbose="-v" in sys.argv, defines=(d,), out=os.path.join(HERE, "libdan_b200_%s.so" % d.lower())))
    elif "--prof" in sys.argv:
        print(build(force=True, verbose="-v" in sys.argv, defines=("DAN_STK_PROF",), out=os.path.join(HERE, "libdan_b200_prof.so")))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
