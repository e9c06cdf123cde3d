"""Build libdril_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels to the GPU box).

Staleness is decided by CONTENT, not mtime: the SHA-256 of every source / header plus the compiler flags is embedded in the
library (dril_source_hash()); build() recompiles when the embedded hash differs from the tree's and says which happened."""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdril_b200.so")
SOURCES = ["api.cu"]
HEADERS = ["common.cuh", "env.cuh", "mlp.cuh", "mma_tiles.cuh", "rollout.cuh", "rollout_tc.cuh", "rollout_syn.cuh", "rollout_gtc.cuh", "gae.cuh", "update.cuh", "update_tc.cuh", "update_ft.cuh", "update_ftg.cuh", "adr.cuh",
           os.path.join("..", "..", "include", "dril_b200.h")]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "--cudart", "static"]


def source_hash():
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    h.update(" ".join(FLAGS + os.environ.get("DRIL_NVCC_EXTRA", "").split()).encode())
    return h.hexdigest()[:16]


def embedded_hash():
    if not os.path.exists(LIB):
        return None
    # read from the file, not through dlopen: a library loaded here would shadow the rebuilt one in this process
    with open(LIB, "rb") as fh:
        blob = fh.read()
    i = blob.find(b"DRIL_SOURCE_HASH=")
    if i < 0:
        return None
    return blob[i + 17:i + 33].decode(errors="replace")


def build(force=False, verbose=False, quiet=False):
    want, have = source_hash(), embedded_hash()
    if not force and want == have:
        if not quiet:
            sys.stderr.write(f"[dril_b200.build] libdril_b200.so is up to date (source hash {want} == embedded hash): nvcc not run\n")
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + FLAGS + ["-Xptxas", "-v" if verbose else "-O3", f'-DDRIL_SOURCE_HASH="{want}"',
           "-o", LIB] + os.environ.get("DRIL_NVCC_EXTRA", "").split() + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libdril_b200.so")
    if verbose:
        sys.stderr.write(r.stderr)
    if not quiet:
        sys.stderr.write(f"[dril_b200.build] nvcc ran: libdril_b200.so rebuilt for sm_100a (source hash {want}, was {have})\n")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
