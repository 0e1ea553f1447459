"""Build the CUDA shared library in-tree:  python -m grates_b200.build [-f] [-v]

nvcc cross-compiles for sm_100a without a GPU.  The resulting grates_b200/lib/libgrates_b200.so
has a plain C ABI (include/grates_b200.h), links cudart statically and has no Python or torch
dependency.
"""
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIBDIR, "libgrates_b200.so")
SOURCES = ["gb_plan.cu", "gb_pack.cu", "gb_synthesis.cu", "gb_analysis.cu", "gb_covprop.cu", "gb_filter.cu", "gb_points.cu", "gb_matrices.cu", "gb_reduce.cu", "gb_densefilter.cu", "gb_linalg.cu", "gb_gradient.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-extended-lambda"]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; grates_b200 cannot be built without the CUDA toolkit")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(PKG, "..", "include", "grates_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(nvcc, src, obj, verbose):
    extra = os.environ.get("GB_NVCC_EXTRA", "").split()       # development builds only (e.g. -DGB_TRACE)
    cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
    res = subprocess.run(cmd, capture_output=True, text=True)
    return res.returncode, res.stdout + res.stderr


def build(force=False, verbose=False):
    """One object per source (compiled in parallel, only when the source, a header or the flags changed), then one link."""
    if not force and not needs_build():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    nvcc = find_nvcc()
    os.makedirs(LIBDIR, exist_ok=True)
    extra = os.environ.get("GB_NVCC_EXTRA", "").strip()
    objdir = os.path.join(PKG, "..", "build", "obj" + ("_" + "".join(c if c.isalnum() else "_" for c in extra) if extra else ""))
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers += [os.path.join(PKG, "..", "include", "grates_b200.h"), os.path.abspath(__file__)]
    t_hdr = max(os.path.getmtime(h) for h in headers)
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs = [os.path.join(objdir, os.path.basename(s)[:-3] + ".o") for s in srcs]
    todo = [(s, o) for s, o in zip(srcs, objs)
            if force or verbose or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), t_hdr)]
    with ThreadPoolExecutor(max_workers=min(8, max(1, len(todo)))) as pool:
        results = list(pool.map(lambda so: _compile(nvcc, so[0], so[1], verbose), todo))
    for (src, _), (rc, log) in zip(todo, results):
        if rc != 0:
            sys.stderr.write(log)
            raise RuntimeError("nvcc failed on %s" % os.path.basename(src))
        if verbose:
            sys.stderr.write(log)
    res = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs,
                         capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed linking libgrates_b200.so")
    return LIB


if __name__ == "__main__":
    print(build(force="-f" in sys.argv, verbose="-v" in sys.argv))   # -f: recompile everything, -v: ptxas statistics
