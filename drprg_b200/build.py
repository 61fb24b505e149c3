"""Builds drprg_b200/libdrprg_cuda.so (hand-written sm_100a kernels + C ABI) in-tree with nvcc: one object per
source, stale objects only, compiled in parallel, then linked."""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
SO = os.path.join(HERE, "libdrprg_cuda.so")
SOURCES = ["sketch.cu", "cluster.cu", "mlpath.cu", "genotype.cu", "capi.cu", "ingest.cu", "gzip_inflate.cpp",
           "prg_graph.cpp", "genotype_host.cpp", "discover.cpp", "assemble.cu", "fastq_frame.cpp"]
EXTRA = ["pandora_cuda_main.cpp"]
HEADERS = ["kernels.cuh", "kernels_common.cuh", "prg_graph.hpp", "genotype_host.hpp", "ingest.hpp", "cuda_owned.hpp",
           "gzip_inflate.hpp", "fastq_frame.hpp", "../../include/drprg_cuda.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false"]
HOST_FLAGS = "-fPIC,-O2,-Wall,-Wno-unused-function,-pthread"


def nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _headers_mtime():
    return max(os.path.getmtime(os.path.join(CSRC, h)) for h in HEADERS if os.path.exists(os.path.join(CSRC, h)))


def _obj(src):
    return os.path.join(OBJ, os.path.splitext(src)[0] + ".o")


def _stale_objects():
    hm = max(_headers_mtime(), os.path.getmtime(os.path.abspath(__file__)))
    out = []
    for s in _sources():
        o = _obj(s)
        if not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(os.path.join(CSRC, s)), hm):
            out.append(s)
    return out


def stale():
    if not os.path.exists(SO) or not os.path.exists(os.path.join(HERE, "pandora_cuda")):
        return True
    t = os.path.getmtime(SO)
    if any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in _sources() + EXTRA):
        return True
    return _headers_mtime() > t


def build(force=False, verbose=False):
    if not force and not stale():
        return SO
    os.makedirs(OBJ, exist_ok=True)
    host_cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    todo = _sources() if force else _stale_objects()

    def compile_one(src):
        cmd = [nvcc()] + NVCC_FLAGS + ["-ccbin", host_cxx, "-Xcompiler", HOST_FLAGS, "-c", os.path.join(CSRC, src), "-o", _obj(src)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(todo)))) as ex:
        list(ex.map(compile_one, todo))
    link = [nvcc()] + NVCC_FLAGS + ["-ccbin", host_cxx, "-Xcompiler", HOST_FLAGS, "-shared", "-cudart", "shared", "-o", SO]
    link += [_obj(s) for s in _sources()] + ["-lz", "-lpthread"]
    subprocess.check_call(link)
    # pandora-argv-compatible front end (drprg -p/--pandora can point at it)
    exe = os.path.join(HERE, "pandora_cuda")
    subprocess.check_call([host_cxx, "-std=c++17", "-O2", "-o", exe, os.path.join(CSRC, "pandora_cuda_main.cpp"),
                           "-L" + HERE, "-ldrprg_cuda", "-Wl,-rpath,$ORIGIN"])
    return SO


if __name__ == "__main__":
    build(force="-f" in sys.argv or "--force" in sys.argv, verbose="-v" in sys.argv)
    print(SO)
