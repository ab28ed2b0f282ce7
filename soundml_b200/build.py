"""Build libsoundml_b200.so in-tree with nvcc for sm_100a.

    python soundml_b200/build.py          # rebuild if sources are newer

nvcc cross-compiles without a GPU.  The shared library lands next to this file
(``soundml_b200/libsoundml_b200.so``): git-ignored, but it travels with the
tree to the GPU box.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsoundml_b200.so")

CUDA_SOURCES = ["api.cu", "kernels_generic.cu", "stft2048.cu", "stft2048p.cu", "stft2048tc.cu", "resample_kernels.cu",
                "ols_kernels.cu", "ols2048.cu", "resample_gemm.cu", "db_kernels.cu", "istft_kernels.cu", "istft2048.cu", "ingest_kernels.cu",
                "effects_kernels.cu", "hpss_kernels.cu", "spectral_kernels.cu"]
HOST_SOURCES = ["host_design.cpp", "kernel_tables.cpp"]
HEADERS = ["host_design.h", "kernel_tables.h", "kernels.h", "fft32.cuh", "fft32x2.cuh", "max_key.cuh", "sm100.cuh", "stft_stage.cuh",
           os.path.join("..", "..", "include", "soundml_b200.h")]

NVCC_FLAGS = [
    "-std=c++17", "-O3", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC,-Wall",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libsoundml_b200.so")
    return nvcc


def needs_build():
    if not os.path.exists(LIB):
        return True
    built = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in CUDA_SOURCES + HOST_SOURCES + HEADERS]
    return any(os.path.getmtime(d) > built for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """Compile every CUDA translation unit for sm_100a and link the library.
    ``defines`` / ``out`` build a variant (e.g. -DSMB_FFT32_PACKED=1) next to it."""
    if out is None and not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build" if out is None else "build_variant")
    os.makedirs(objdir, exist_ok=True)
    objs, jobs = [], []
    newest_header = max(os.path.getmtime(os.path.join(CSRC, h)) for h in HEADERS)
    for src in CUDA_SOURCES + HOST_SOURCES:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        # an object newer than its source and every header is kept (variants and
        # forced builds recompile everything)
        if (out is None and not force and os.path.exists(obj) and
                os.path.getmtime(obj) > max(os.path.getmtime(os.path.join(CSRC, src)), newest_header)):
            continue
        cmd = [nvcc] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + [
            "-c", os.path.join(CSRC, src), "-o", obj]
        if src.endswith(".cpp"):
            cmd.insert(1, "-x")
            cmd.insert(2, "cu")
        jobs.append(cmd)
    # translation units are independent: compile them side by side
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1) or 1) as pool:
        list(pool.map(lambda c: _run(c, verbose), jobs))
    _run([nvcc, "-shared", "-o", out or LIB] + objs + ["-cudart", "static"], verbose)
    return out or LIB


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    else:   # compiler warnings are never silent (a missing return once hung a kernel)
        warn = [l for l in (res.stdout + res.stderr).splitlines() if "warning" in l.lower()]
        if warn:
            sys.stderr.write("\n".join(warn) + "\n")
    if res.returncode != 0:
        raise RuntimeError(f"build failed: {' '.join(cmd)}")


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[6:] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs,
                out=outs[0] if outs else None))
