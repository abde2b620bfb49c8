"""In-tree build of ``libmeshrcnn_b200.so`` (sm_100a only) with nvcc.  No torch headers are involved: the
library is a plain C-ABI shared object (``include/meshrcnn_b200.h``); cudart is linked statically so the
nvcc-12.9 objects do not depend on the cu128 runtime bundled with torch.

    python -m meshrcnn_b200.build            # (re)build if the sources differ from those the .so was built from
"""
import glob
import hashlib
import os
import platform
import shutil
import subprocess
import sys
import sysconfig
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libmeshrcnn_b200.so")
OBJ = os.path.join(HERE, "build")
STAMP = os.path.join(OBJ, "sources.sha256")         # digest of the inputs the library in the tree was built from

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
              "-I", os.path.join(ROOT, "include")]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def source_digest() -> str:
    """SHA-256 over the names and contents of every input of the library and the call shim (and of this file, which holds
    the flags).  Contents, not timestamps: a tree that was copied, or is read-only, is still judged right."""
    h = hashlib.sha256()
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(ROOT, "include", "*.h"))
    for p in sorted(deps + [FASTCALL_SRC, os.path.abspath(__file__)]):
        h.update(os.path.relpath(p, ROOT).encode() + b"\0")
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def needs_build() -> bool:
    """True unless the library in the tree was built from the sources as they are now."""
    try:
        with open(STAMP) as f:
            return not os.path.exists(LIB) or f.read().strip() != source_digest()
    except OSError:
        return True


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        build_fastcall()
        return LIB
    nvcc = _nvcc()
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = max([os.path.getmtime(p) for p in glob.glob(os.path.join(CSRC, "*.cuh")) +
                 glob.glob(os.path.join(ROOT, "include", "*.h"))] + [0.0])

    def compile_one(src):
        obj = os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")
        if (not force and os.path.exists(obj) and os.path.getmtime(obj) > os.path.getmtime(src)
                and os.path.getmtime(obj) > hdr_t):
            return obj
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, sources()))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcuda"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    build_fastcall(force=True)
    with open(STAMP, "w") as f:
        f.write(source_digest() + "\n")
    return LIB


FASTCALL_SRC = os.path.join(CSRC, "host", "fastcall.c")
FASTCALL = os.path.join(HERE, "_fastcall" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))


def build_fastcall(force: bool = False):
    """The optional host-side call shim (csrc/host/fastcall.c, plain C + the CPython API, gcc).  Returns its path, or None
    if it cannot be built here (no compiler / no Python headers): meshrcnn_b200._lib then calls through ctypes only."""
    if platform.machine() not in ("x86_64", "AMD64") or not sys.platform.startswith("linux"):
        return None
    if not force and os.path.exists(FASTCALL) and os.path.getmtime(FASTCALL) > os.path.getmtime(FASTCALL_SRC):
        return FASTCALL
    cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
    inc = sysconfig.get_paths().get("include")
    if not cc or not inc or not os.path.exists(os.path.join(inc, "Python.h")):
        return None
    r = subprocess.run([cc, "-O2", "-fPIC", "-shared", "-I", inc, FASTCALL_SRC, "-o", FASTCALL], capture_output=True, text=True)
    return FASTCALL if r.returncode == 0 else None


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_fastcall(force="--force" in sys.argv))
