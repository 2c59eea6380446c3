"""Builds the in-tree shared libraries (nvcc cross-compiles sm_100a without a GPU):
  libobgpu_scan.so   -- the product: CUDA kernels + C-ABI (include/obgpu_scan.h, obgpu_skip_index.h, obgpu_compaction.h)
  libobgpu_writer.so -- plain C++ micro-block / aggregate-row writer (include/obgpu_writer.h); no CUDA, so the
                        reference arm of bench.py and the CPU tests never map the product library to WRITE blocks.
"""
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
INC = os.path.join(_HERE, "..", "include")
LIB = os.path.join(CSRC, "libobgpu_scan.so")
WRITER_LIB = os.path.join(CSRC, "libobgpu_writer.so")
SOURCES = ["obgpu_scan.cu"]
HEADERS = ["ob_format.h", "scan_device.cuh", "scan_small.cuh", "merge_kernels.cuh", "merge_exchange.cuh", "merge_streamed.cuh", "encode_kernels.cuh", "encode_codecs.cuh", "macro_blocks.cuh", "dict_ops.cuh", "cg_bitmap.cuh", "result_strings.cuh", "skip_index.cuh", "stream_codecs.cuh", "mat_codecs.cuh", "host_pipeline.h",
           os.path.join(INC, "obgpu_scan.h"), os.path.join(INC, "obgpu_compaction.h"), os.path.join(INC, "obgpu_skip_index.h"), os.path.join(INC, "obgpu_pipeline.h")]
WRITER_SOURCES = ["sstable_writer.cpp"]
WRITER_HEADERS = ["ob_format.h", "stream_codecs_host.h", os.path.join(INC, "obgpu_writer.h"), os.path.join(INC, "obgpu_scan.h"),
                  os.path.join(INC, "obgpu_skip_index.h")]


def nvcc_path():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _stale(lib, deps):
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    return any(os.path.exists(os.path.join(CSRC, f)) and os.path.getmtime(os.path.join(CSRC, f)) > t for f in deps)


def needs_build():
    return _stale(LIB, SOURCES + HEADERS) or _stale(WRITER_LIB, WRITER_SOURCES + WRITER_HEADERS)


def build_writer(force=False):
    if not force and not _stale(WRITER_LIB, WRITER_SOURCES + WRITER_HEADERS):
        return WRITER_LIB
    cmd = ["g++", "-std=c++17", "-O3", "-fPIC", "-shared", "-pthread", "-o", WRITER_LIB] + WRITER_SOURCES
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ (writer) failed:\n" + r.stdout + r.stderr)
    return WRITER_LIB


def build(force=False, verbose=False):
    build_writer(force)
    if not force and not _stale(LIB, SOURCES + HEADERS):
        return LIB
    cmd = [nvcc_path(), "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
           "-Xcompiler", "-fPIC", "-shared", "-o", LIB] + SOURCES + ["-ldl"]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
