"""Build libptts_b200.so in-tree with nvcc for sm_100a (no torch / pybind dependency: pure C ABI).

Usage: python parler_tts_b200/csrc/build.py [--force] [--tag NAME -DMACRO ...]
The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
`--tag NAME` builds a VARIANT (extra nvcc flags after it, e.g. -DPTTS_SOME_EXPERIMENT) into libptts_b200_NAME.so next to the
product library without touching it; load it with PTTS_LIB=<path> (parler_tts_b200/_lib.py).
"""
from __future__ import annotations
import concurrent.futures as cf
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["api.cu", "gemm.cu", "gemm_tc.cu", "attention.cu", "embed.cu", "sample.cu", "dac.cu", "dac_tc.cu", "dac_enc.cu", "step.cu", "step2.cu"]
LIB = os.path.join(HERE, "libptts_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]
if os.environ.get("PTTS_PTXAS_V"):
    FLAGS += ["-Xptxas", "-v"]


def _stamp() -> str:
    h = hashlib.sha256()
    for f in sorted(os.listdir(HERE)) + ["../../include/ptts_b200.h"]:
        p = os.path.join(HERE, f)
        if f.endswith((".cu", ".cuh", ".h", ".py")) and os.path.isfile(p):
            h.update(open(p, "rb").read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = True) -> str:
    stamp_file = os.path.join(HERE, "build", "stamp")
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)

    def cc(src):
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(HERE, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    objs = []
    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        for src, obj, r in ex.map(cc, SOURCES):
            if verbose and (r.stderr.strip() or r.stdout.strip()):
                print(f"--- {src}\n{r.stdout}{r.stderr}", file=sys.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
            objs.append(obj)
    cmd = [NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    open(stamp_file, "w").write(stamp)
    return LIB


def build_variant(tag: str, extra_flags: list[str]) -> str:
    """Compile every source with extra flags into build_<tag>/ and link libptts_b200_<tag>.so (the product .so is untouched)."""
    out_dir = os.path.join(HERE, f"build_{tag}")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(HERE, f"libptts_b200_{tag}.so")

    def cc(src):
        obj = os.path.join(out_dir, src.replace(".cu", ".o"))
        r = subprocess.run([NVCC, *FLAGS, *extra_flags, "-c", os.path.join(HERE, src), "-o", obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        return obj

    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(cc, SOURCES))
    r = subprocess.run([NVCC, "-shared", "-o", lib, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return lib


if __name__ == "__main__":
    if "--tag" in sys.argv:
        i = sys.argv.index("--tag")
        print(build_variant(sys.argv[i + 1], sys.argv[i + 2:]))
    else:
        print(build(force="--force" in sys.argv))
