"""Build libssi.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIBDIR = PKG / "lib"
LIB = LIBDIR / "libssi.so"
SOURCES = ["ssi_api.cu", "ssi_multi.cu", "ssi_gemm_tc.cu", "ssi_decoder.cu", "ssi_logpost.cu", "ssi_mh.cu", "ssi_hmc.cu", "ssi_construct.cu", "ssi_gram_tc.cu", "ssi_basis.cu", "ssi_basis_mma.cu", "ssi_gemm.cu", "ssi_grad.cu", "ssi_train.cu", "ssi_tc.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xcompiler", "-Wno-unknown-pragmas",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found; libssi.so cannot be built")


def _stamp() -> str:
    h = hashlib.sha256()
    for f in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "ssi.h", Path(__file__)]):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    LIBDIR.mkdir(exist_ok=True)
    stamp_file = LIBDIR / "libssi.stamp"
    stamp = _stamp()
    if not force and LIB.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = LIBDIR / (src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-Xptxas", "-v" if verbose else "-warn-spills", "-c", str(CSRC / src), "-o", str(obj)]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(f"--- nvcc {src} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed, see output above")
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(LIB), *objs, "-cudart", "static"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    stamp_file.write_text(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
