"""Build libtgn_b200.so (the C-ABI CUDA library) in-tree for sm_100a.

    python -m toothgroupnetwork_b200.build [--force] [--jobs N]

nvcc cross-compiles without a GPU; the resulting ``toothgroupnetwork_b200/_lib/libtgn_b200.so``
is git-ignored but travels to the GPU box with the gpurun snapshot.  sm_100a is the only target.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_lib")
LIB = os.path.join(OUT_DIR, "libtgn_b200.so")
SOURCES = ["lib.cu", "fps.cu", "fps_bucket.cu", "knn.cu", "knn_grid.cu", "crop_knn.cu", "gather.cu", "csr.cu", "ballquery.cu", "ballquery_grid.cu", "sa_mlp.cu", "sa_mlp_tc.cu", "sa_mlp_tc8.cu", "sa_mlp_tcw.cu", "pw_mlp.cu", "pt_layer.cu", "dbscan.cu", "knn_f64.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-I" + os.path.join(ROOT, "include"), "-I" + CSRC,
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libtgn_b200.so cannot be built here")
    return exe


def _newest_source_mtime() -> float:
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "tgn_b200.h")]
    return max(os.path.getmtime(p) for p in paths)


def is_fresh() -> bool:
    return os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_source_mtime()


def build(force: bool = False, jobs: int = 0, verbose: bool = False) -> str:
    if not force and is_fresh():
        return LIB
    nvcc = _nvcc()
    os.makedirs(OUT_DIR, exist_ok=True)
    obj_dir = os.path.join(OUT_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)

    def compile_one(src: str) -> str:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{res.stdout}\n{res.stderr}")
        if verbose:
            sys.stderr.write(res.stderr)
        return obj

    with cf.ThreadPoolExecutor(max_workers=jobs or min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB + ".tmp"] + objs
    res = subprocess.run(link, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    os.replace(LIB + ".tmp", LIB)
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--jobs", type=int, default=0)
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    print(build(force=a.force, jobs=a.jobs, verbose=a.verbose))
