"""Builds libdebigulator_b200.so in-tree with nvcc for sm_100a (and nothing else).

    python -m debigulator_b200.build

nvcc cross-compiles without a GPU; the built .so is git-ignored but travels
with the working tree.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdebigulator_b200.so")
SOURCES = ["dbg_api.cu", "scalar_api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    # the library exports `inflate`; keep internal calls away from zlib's symbol
    "-Xlinker", "-Bsymbolic",
]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libdebigulator_b200.so")


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    inc = os.path.join(os.path.dirname(HERE), "include")
    deps += [os.path.join(inc, f) for f in os.listdir(inc)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    extra = os.environ.get("DBG_BUILD_DEFS", "").split()  # experiments: e.g. -DDBG_BUILD_INFLATE_CTAS=5
    cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        sys.stderr.write(r.stderr)
    return LIB


STBGEN = os.path.join(HERE, "tools", "libstbgen.so")
CORPUS_TOOLS = os.path.join(HERE, "tools", "libcorpus_tools.so")
REF_SRC = "/root/reference/src"


def build_corpus_tools():
    """The corpus's own single-block fixed-Huffman encoder (tools/fixed_deflate.c). Returns the library path."""
    src = os.path.join(HERE, "tools", "fixed_deflate.c")
    if not os.path.exists(CORPUS_TOOLS) or os.path.getmtime(src) > os.path.getmtime(CORPUS_TOOLS):
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", src, "-o", CORPUS_TOOLS])
    return CORPUS_TOOLS


def build_tools():
    """Corpus tooling (not product code): the corpus's own encoder, and the synthetic-PNG writer compiled against the
    reference's vendored stb_write.h where it lies. Returns the stb library path, or None when neither the reference
    tree nor a prebuilt library is there."""
    build_corpus_tools()
    src = os.path.join(HERE, "tools", "stb_gen.c")
    if os.path.isdir(REF_SRC):
        if not os.path.exists(STBGEN) or os.path.getmtime(src) > os.path.getmtime(STBGEN):
            subprocess.check_call(["gcc", "-O2", "-w", "-fPIC", "-shared", "-I" + REF_SRC, src, "-o", STBGEN])
    return STBGEN if os.path.exists(STBGEN) else None


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_tools())
