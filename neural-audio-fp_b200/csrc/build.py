"""Build libnafp.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

Staleness is decided by CONTENT, not by mtime: the SHA-256 of every source / header and of the compiler flags is
kept next to the library (`libnafp.so.srchash`).  A snapshot copy of the tree (gpurun) keeps the prebuilt library
only as long as it was built from exactly the sources that travel with it; `build()` says which of the two happened.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["capi.cu", "flat_search.cu", "seq_match.cu", "ivfpq.cu", "ivfpq_lm.cu", "logmel.cu", "encoder.cu", "synth.cu", "mini_search.cu",
           "resample.cu"]
OUT = os.path.join(HERE, "libnafp.so")
HASH = OUT + ".srchash"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
LAST = {"action": None, "compiled": []}      # what the last build() call did (reported by __graft_entry__.build)


def _headers():
    hs = [os.path.join(HERE, f) for f in sorted(os.listdir(HERE)) if f.endswith((".h", ".cuh"))]
    hs.append(os.path.normpath(os.path.join(HERE, "..", "..", "include", "nafp.h")))
    return hs


def _digest(paths):
    h = hashlib.sha256(" ".join(FLAGS).encode())
    for p in paths:
        h.update(os.path.basename(p).encode())
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def source_hash():
    srcs = [os.path.join(HERE, s) for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    return _digest(srcs + _headers())


def build(force=False, verbose=False):
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    want = source_hash()
    have = open(HASH).read().strip() if os.path.exists(HASH) else None
    if not force and os.path.exists(OUT) and have == want:
        LAST.update(action="reused", compiled=[])
        return OUT
    objs, compiled = [], []
    hdr = _headers()
    for s in srcs:
        src = os.path.join(HERE, s)
        obj = os.path.join(HERE, s.replace(".cu", ".o"))
        tag = obj + ".srchash"
        objs.append(obj)
        d = _digest([src] + hdr)
        if force or not os.path.exists(obj) or not os.path.exists(tag) or open(tag).read().strip() != d:
            cmd = [NVCC, *FLAGS, "-c", src, "-o", obj]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {s}")
            with open(tag, "w") as f:
                f.write(d)
            compiled.append(s)
    cmd = [NVCC, "-shared", "-o", OUT, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static",
           "-ldl", "-lrt", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    with open(HASH, "w") as f:
        f.write(want)
    LAST.update(action="compiled", compiled=compiled)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True), LAST)
