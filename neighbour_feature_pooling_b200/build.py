"""Build libnfp_b200.so (hand-written sm_100a kernels + C ABI) in-tree with nvcc.

    python -m neighbour_feature_pooling_b200.build [--force] [--verbose]

The library has no torch / Python dependency: it is plain CUDA behind the C ABI
declared in include/nfp_b200.h.  nvcc cross-compiles without a GPU, and the
built .so travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(REPO_ROOT, "include")
LIB_DIR = os.path.join(PKG_DIR, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libnfp_b200.so")
OBJ_DIR = os.path.join(PKG_DIR, "build")
SOURCES = ["nfp_capi.cu", "nfp_generic.cu", "nfp_stream.cu", "nfp_stream_f32.cu", "nfp_stream_bf16.cu", "nfp_stream_f16.cu",
           "nfp_split_f32.cu", "nfp_split_bf16.cu", "nfp_planar.cu", "nfp_token.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-I", INCLUDE, "-I", CSRC,
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


HASH_PATH = os.path.join(LIB_DIR, "libnfp_b200.so.srchash")


def source_hash() -> str:
    """sha256 over the contents of every source the library is built from (and the flags): the built .so is reused only
    when this matches the hash recorded beside it -- a stale library shipped with newer sources is rebuilt, whatever
    the file times say."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS[:6]).encode())
    for path in sorted([os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "nfp_b200.h")]):
        h.update(os.path.basename(path).encode())
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH) or not os.path.exists(HASH_PATH):
        return True
    with open(HASH_PATH) as f:
        return f.read().strip() != source_hash()


def build(force: bool = False, verbose: bool = False, variant: str = "", defines=()) -> str:
    """variant / defines: an experimental build `lib/libnfp_b200.<variant>.so` compiled with extra -D flags
    (selected at run time with NFPB200_LIB=<path>); the default build is what ships."""
    lib_path, obj_dir = LIB_PATH, OBJ_DIR
    if variant:
        lib_path = os.path.join(LIB_DIR, f"libnfp_b200.{variant}.so")
        obj_dir = os.path.join(OBJ_DIR, variant)
    elif not force and not needs_build():
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(obj_dir, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    flags = [*NVCC_FLAGS, *[f"-D{d}" for d in defines]]

    def compile_one(src):
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc, *flags, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj + ".ptxas.log", "w") as f:
            f.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = lib_path + ".tmp"
    r = subprocess.run([nvcc, "-shared", "--cudart", "static", "-o", tmp, *objs], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, lib_path)
    if not variant:
        with open(HASH_PATH, "w") as f:
            f.write(source_hash() + "\n")
    return lib_path


if __name__ == "__main__":
    variant = sys.argv[sys.argv.index("--variant") + 1] if "--variant" in sys.argv else ""
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, variant=variant,
                 defines=[a[2:] for a in sys.argv if a.startswith("-D")])
    print(path)
