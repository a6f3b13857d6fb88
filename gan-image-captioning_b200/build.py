"""In-tree build of libgic_b200.so (nvcc, sm_100a only).  The built library travels to the GPU box
with the repo snapshot; it is rebuilt only when the sources' hash changes."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgic_b200.so")
STAMP = LIB + ".srchash"
SOURCES = ["gemm_f32.cu", "gemm_dispatch.cu", "gemm_tcgen05.cu", "gemm_persistent.cu", "gemm_pair_tcgen05.cu", "attn.cu", "lstm_tcgen05.cu", "bptt_tcgen05.cu", "vocab_sample_tcgen05.cu", "dz_fused_tcgen05.cu", "beam_tcgen05.cu", "decode.cu", "disc.cu", "loss_optim.cu", "allreduce.cu", "capi.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _hash() -> str:
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + ["../../include/gic_b200.h"]
    for f in files:
        p = os.path.join(CSRC, f)
        if os.path.isfile(p):
            h.update(f.encode())
            h.update(open(p, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def up_to_date() -> bool:
    return os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == _hash()


def _compile_one(nvcc, src, verbose):
    """Compile one .cu to build/<name>.o unless its (source + headers + flags) hash is unchanged."""
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    obj = os.path.join(bdir, src.replace(".cu", ".o"))
    h = hashlib.sha256()
    for f in [src] + sorted(x for x in os.listdir(CSRC) if x.endswith((".cuh", ".h"))) + ["../../include/gic_b200.h"]:
        h.update(open(os.path.join(CSRC, f), "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    stamp = obj + ".hash"
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == h.hexdigest() and not verbose:
        return obj, ""
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    cmd = [nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed on %s" % src)
    with open(stamp, "w") as f:
        f.write(h.hexdigest())
    return obj, r.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not verbose and up_to_date():
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libgic_b200.so cannot be built (there is no CPU fallback)")
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        res = list(ex.map(lambda s: _compile_one(nvcc, s, verbose), SOURCES))
    if verbose:
        sys.stderr.write("".join(r[1] for r in res))
    r = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + [o for o, _ in res],
                       cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed linking libgic_b200.so")
    with open(STAMP, "w") as f:
        f.write(_hash())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
