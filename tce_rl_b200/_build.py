"""Build libtce_b200.so in-tree with nvcc for sm_100a (no torch headers: the library is a plain C ABI)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtce_b200.so")
SOURCES = ["tce_tables.cu", "tce_traj.cu", "tce_traj_cov.cu", "tce_seglik.cu", "tce_seglik_fused.cu", "tce_gauss.cu", "tce_adv.cu", "tce_proj.cu", "tce_proj_diag.cu", "tce_adam.cu", "tce_epoch.cu", "tce_p2p.cu", "tce_bench.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "tce_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = nvcc_path()
    objs = []
    obj_dir = os.path.join(HERE, "build")
    os.makedirs(obj_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *[f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")], "-c", path, "-o", obj]
        if os.environ.get("TCE_PROFILE"):            # phase-clock stamps + tce_debug_* (scripts/kl_phases*.py); never shipped
            cmd.insert(1, "-DTCE_PROFILE")
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs])   # static cudart (nvcc default)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
