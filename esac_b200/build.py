"""Builds libesac_b200.so (hand-written sm_100a CUDA + the C ABI) in-tree with nvcc.

No torch extension machinery: the library has a plain C ABI (include/esac_b200.h) and is loaded
with ctypes, so the build is four nvcc compiles and one link.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
OBJ = HERE / "_obj"
LIB = HERE / "libesac_b200.so"
SOURCES = ["score.cu", "hyp.cu", "refine.cu", "bwd.cu", "gating.cu", "reproj.cu", "initloss.cu", "capi.cu"]
HEADERS = ["esac_internal.h", "esac_geom.cuh", "esac_rng.cuh", "esac_p3p_fast.cuh", "../../include/esac_b200.h",
           "../../include/esac_b200_testhooks.h"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-ccbin", "/usr/bin/g++", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _digest(paths) -> str:
    """Content hash of the sources (mtimes do not survive the snapshot that carries the tree to the GPU box)."""
    h = hashlib.sha256(" ".join(FLAGS).encode())
    for p in paths:
        h.update(Path(p).name.encode())
        h.update(Path(p).read_bytes())
    return h.hexdigest()


def build_library(force: bool = False, verbose: bool = False) -> Path:
    OBJ.mkdir(exist_ok=True)
    hdrs = [CSRC / h for h in HEADERS]
    stamp = HERE / "libesac_b200.so.srchash"
    want = _digest([CSRC / s for s in SOURCES] + hdrs)
    if not force and LIB.exists() and stamp.exists() and stamp.read_text().strip() == want:
        return LIB

    def compile_one(src: str):
        s = CSRC / src
        o = OBJ / (src + ".o")
        ostamp = OBJ / (src + ".srchash")
        owant = _digest([s] + hdrs)
        if force or not o.exists() or not ostamp.exists() or ostamp.read_text().strip() != owant:
            r = subprocess.run([NVCC] + FLAGS + ["-c", str(s), "-o", str(o)], capture_output=True, text=True)
            (OBJ / (src + ".log")).write_text(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
            ostamp.write_text(owant)
            if verbose:
                print(r.stderr)
        return o

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    r = subprocess.run([NVCC, "-ccbin", "/usr/bin/g++", "-shared", "-o", str(LIB)] + [str(o) for o in objs] + ["-lcudart", "-ldl"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    stamp.write_text(want)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
