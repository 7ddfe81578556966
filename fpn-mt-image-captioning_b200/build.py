"""Build libfpnmt.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python build.py [--force]

Objects go to csrc/build/, the library to fpn-mt-image-captioning_b200/libfpnmt.so (git-ignored; it travels to
the GPU box with the gpurun snapshot).
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libfpnmt.so")
SOURCES = ["api.cu", "engine.cu", "igemm.cu", "tgemm.cu", "tgemmw.cu", "xattn.cu", "dstep.cu", "stem.cu", "tensormap.cu", "elementwise.cu", "attention.cu", "beam.cu", "sample.cu", "score.cu", "jpeg.cu", "dlapi.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
         "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _stamp() -> str:
    h = hashlib.sha256()
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(CSRC, f), "rb").read())
    for hdr in ("fpnmt.h", "fpnmt_dlpack.h"):
        h.update(open(os.path.join(HERE, "..", "include", hdr), "rb").read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = True, dbg_stamps: bool = False) -> str:
    global OUT
    bdir = os.path.join(CSRC, "build")
    if dbg_stamps:    # developer build -> libfpnmt_dbg.so: globaltimer timelines inside the kernels (FPNMT_DBG_OP=<op name>);
        FLAGS.append("-DFPNMT_DBG_STAMPS")      # load it by setting fpnmt._lib.LIB_PATH before the first Engine
        OUT = os.path.join(HERE, "libfpnmt_dbg.so")
        bdir = os.path.join(CSRC, "build_dbg")
    os.makedirs(bdir, exist_ok=True)
    stamp_file = os.path.join(bdir, "stamp")
    stamp = _stamp()

    def lib_id() -> str:    # the stamp also pins the library file itself (a copied-over .so must not pass as up to date)
        return hashlib.sha256(open(OUT, "rb").read()).hexdigest()[:16]    # content, not mtime: the file is copied to the GPU box

    if not force and os.path.exists(OUT) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp + " " + lib_id():
        return OUT

    def cc(src):
        obj = os.path.join(bdir, src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(cc, SOURCES))
    cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static",
                                                 "-lnvjpeg_static", "-lculibos", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    open(stamp_file, "w").write(stamp + " " + lib_id())
    if verbose:
        print("built", OUT)
    return OUT


if __name__ == "__main__":
    build(force="--force" in sys.argv, dbg_stamps="--dbg-stamps" in sys.argv)
