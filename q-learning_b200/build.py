"""Build the CUDA shared library (libqlcuda.so) in-tree for sm_100a with nvcc (cross-compiles without a GPU).

The library embeds the SHA-256 of the sources it was built from ("QLC_BUILD_INFO:src_hash=...;" — also qlc_build_info()).
A library whose hash differs from the sources next to it is STALE: it is rebuilt, and if that fails the failure is raised —
a broken edit is never tested against yesterday's binary."""
import hashlib
import os
import re
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("QLC_LIB") or os.path.join(_HERE, "libqlcuda.so")   # QLC_LIB: A/B-test another build of the library
SOURCES = [os.path.join(_HERE, "csrc", "qlc_api.cu"), os.path.join(_HERE, "csrc", "host_pool.cpp"), os.path.join(_HERE, "csrc", "comm.cpp")]
HEADERS = [
    os.path.join(_HERE, "csrc", "kernels.cuh"),
    os.path.join(_HERE, "csrc", "physics.cuh"),
    os.path.join(_HERE, "csrc", "qnet.cuh"),
    os.path.join(_HERE, "csrc", "qnet_conv.cuh"),
    os.path.join(_HERE, "csrc", "qnet_train.cuh"),
    os.path.join(_HERE, "csrc", "per.cuh"),
    os.path.join(_HERE, "csrc", "nstep.cuh"),
    os.path.join(_HERE, "csrc", "host_pool.h"),
    os.path.join(_HERE, "csrc", "comm.h"),
    os.path.join(os.path.dirname(_HERE), "include", "ql_cuda.h"),
]
# -fmad=false: the reference's Rust never contracts a*b+c; results must be bit-identical to that arithmetic.
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
    "-shared", "-Xcompiler", "-fPIC", "-cudart", "static", "-Xcompiler", "-pthread", "-ldl",
]
PROFILING = bool(int(os.environ.get("QLC_PROFILING_BUILD", "0")))      # ablation build: -DQLC_PROFILING enables QLC_DEBUG_SKIP


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built")


def source_hash():
    """SHA-256 over the names and contents of every source and header, plus the compiler flags."""
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        h.update(os.path.basename(f).encode() + b"\0")
        h.update(open(f, "rb").read())
        h.update(b"\0")
    h.update(" ".join(NVCC_FLAGS).encode())
    h.update(b"profiling" if PROFILING else b"")
    return h.hexdigest()


def library_info(path=None):
    """{'src_hash': ..., 'profiling': ...} read from the marker string inside the library file (no dlopen), {} if there is none."""
    path = path or SO_PATH
    try:
        data = open(path, "rb").read()
    except OSError:
        return {}
    m = re.search(rb"QLC_BUILD_INFO:src_hash=([0-9a-z]+);profiling=([01]);", data)
    return {"src_hash": m.group(1).decode(), "profiling": m.group(2).decode()} if m else {}


def needs_build():
    if os.environ.get("QLC_LIB"):
        return False
    return library_info().get("src_hash") != source_hash()


def build(force=False, verbose=False):
    """Compile libqlcuda.so if it is missing or was built from other sources. Returns the path; raises if the build fails."""
    if not force and not needs_build():
        return SO_PATH
    want = source_hash()
    cmd = [_nvcc()] + NVCC_FLAGS + ['-DQLC_SRC_HASH="%s"' % want] + (["-DQLC_PROFILING"] if PROFILING else []) \
        + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO_PATH + ".tmp"] + SOURCES
    env = dict(os.environ)
    env.pop("CC", None)   # the image exports CC=/opt/gcc/bin/gcc; let nvcc use the system g++
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed (the stale libqlcuda.so is NOT used):\n" + res.stdout)
    os.replace(SO_PATH + ".tmp", SO_PATH)
    got = library_info().get("src_hash")
    if got != want:
        raise RuntimeError("libqlcuda.so does not carry the hash of its sources (%s != %s)" % (got, want))
    if verbose:
        print(res.stdout)
    return SO_PATH


def build_c_host_tool():
    """tools/cabi/c_abi_latency: the drop-in calls timed from a compiled host (plain C against include/ql_cuda.h, linked to the library).
    Returns the path, or None if it cannot be built (no gcc)."""
    root = os.path.dirname(_HERE)
    src, exe = os.path.join(root, "tools", "cabi", "c_abi_latency.c"), os.path.join(root, "tools", "cabi", "c_abi_latency")
    if os.path.exists(exe) and os.path.getmtime(exe) >= max(os.path.getmtime(src), os.path.getmtime(os.path.join(root, "include", "ql_cuda.h"))):
        return exe
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc:
        return None
    env = dict(os.environ); env.pop("CC", None)
    res = subprocess.run([cc, "-O2", "-I", os.path.join(root, "include"), src, "-L", _HERE, "-lqlcuda", "-Wl,-rpath,$ORIGIN/../../q-learning_b200", "-o", exe],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("gcc failed on tools/cabi/c_abi_latency.c:\n" + res.stdout)
    return exe


if __name__ == "__main__":
    print(build(force=True, verbose=True))
    print(build_c_host_tool())
