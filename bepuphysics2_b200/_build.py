"""Builds the native libraries in-tree (the .so files travel to the GPU box with the repo snapshot).

    libbepucuda.so   hand-written sm_100a CUDA kernels + the C ABI of include/bepucuda.h
    libbepuhost.so   C++ host-side mirror of the reference's Bodies/Solver/Timestepper slice (links libbepucuda)

nvcc cross-compiles for sm_100a without a GPU. The solver kernels are compiled twice: once with FMA contraction
(`bepu_fast`) and once with -fmad=false (`bepu_strict`, bit-exact against a non-contracting CPU evaluation).
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(CSRC, "build")
LIB_CUDA = os.path.join(HERE, "libbepucuda.so")
LIB_HOST = os.path.join(HERE, "libbepuhost.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
GXX = "/usr/bin/g++"
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-ccbin", GXX]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _digest(sources, flag_sets):
    """Content hash of everything libbepucuda.so is compiled from (sources, headers, compiler flags)."""
    h = hashlib.sha256()
    for flags in flag_sets:
        h.update(("\0".join(flags) + "\n").encode())
    for path in sorted(sources, key=os.path.basename):
        h.update(os.path.basename(path).encode() + b"\0")
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _stamp_matches(stamp, digest):
    """Line 1 of the stamp: digest of the sources the library was built from (line 2: sha256 of the library itself, see binary_matches_stamp)."""
    try:
        with open(stamp) as f:
            return f.read().split("\n")[0].strip() == digest
    except OSError:
        return False


def _sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for block in iter(lambda: f.read(1 << 20), b""):
            h.update(block)
    return h.hexdigest()


def _write_stamp(stamp, digest, lib):
    with open(stamp, "w") as f:
        f.write(digest + "\n" + _sha256(lib) + "\n")


def binary_matches_stamp(lib=None):
    """True / False when the stamp next to the library records the library's own hash and it does / does not match the file (a stale or foreign
    binary next to a fresh stamp); None when there is no such record (stamp missing or written by an older build script)."""
    lib = lib or LIB_CUDA
    try:
        with open(lib + ".stamp") as f:
            lines = f.read().split("\n")
    except OSError:
        return None
    if len(lines) < 2 or len(lines[1].strip()) != 64:
        return None
    return lines[1].strip() == _sha256(lib)


def _run(cmd):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("command failed: %s\n%s" % (" ".join(cmd), r.stdout))
    return r.stdout


def build(force=False, verbose=False, variant=None, defines=()):
    """variant/defines: development A/B builds (libbepucuda_<variant>.so with extra -D flags, selected at run time with BEPUCUDA_VARIANT)."""
    global BUILD, LIB_CUDA
    if variant:
        BUILD = os.path.join(CSRC, "build_" + variant)
        LIB_CUDA = os.path.join(HERE, "libbepucuda_%s.so" % variant)
    os.makedirs(BUILD, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".inc"))]
    headers.append(os.path.join(HERE, "..", "include", "bepucuda.h"))
    flavours = [("fast", ["-DBEPU_NS=bepu_fast", "-prec-div=false", "-prec-sqrt=false"]), ("strict", ["-DBEPU_NS=bepu_strict", "-fmad=false"])]
    # (object, source, extra flags)
    units = [("solver_%s_%d.o" % (name, unit), "bepu_solver_kernels.cu", flags + ["-DBEPU_UNIT=%d" % unit]) for unit in (1, 0, 2, 3) for name, flags in flavours]
    units += [("layout.o", "bepu_layout_kernels.cu", []), ("coloring.o", "bepu_coloring.cu", []), ("bounds.o", "bepu_bounds.cu", ["-fmad=false"]), ("shape_bounds.o", "bepu_shape_bounds.cu", ["-fmad=false"]), ("api.o", "bepucuda_api.cu", [])]
    all_sources = [os.path.join(CSRC, f) for f in ("bepu_solver_kernels.cu", "bepu_layout_kernels.cu", "bepu_coloring.cu", "bepu_bounds.cu", "bepu_shape_bounds.cu", "bepucuda_api.cu")] + headers
    # Nothing to compile when the library was built from exactly these sources (content stamp written after a build: survives a snapshot that
    # does not keep modification times) or is newer than every source. Object files need not travel with a snapshot.
    stamp = LIB_CUDA + ".stamp"
    digest = _digest(all_sources, [NVCC_FLAGS] + [f for _, f in flavours] + [list(defines)])
    fresh = os.path.exists(LIB_CUDA) and (_stamp_matches(stamp, digest) or (not os.path.exists(stamp) and not _newer(LIB_CUDA, all_sources)))
    if not force and not defines and fresh:
        units = []
        if not os.path.exists(stamp):
            _write_stamp(stamp, digest, LIB_CUDA)
    jobs = []
    for obj, src, extra in units:
        o = os.path.join(BUILD, obj)
        s = os.path.join(CSRC, src)
        frozen = os.path.exists(o) and any(obj.endswith("_%s.o" % u) for u in os.environ.get("BEPUCUDA_FREEZE_UNITS", "").split(",") if u)
        if frozen:
            continue  # development shortcut: keep a stale object of a unit that is not being worked on (never set for release builds)
        if force or _newer(o, [s] + headers):
            jobs.append([NVCC] + NVCC_FLAGS + extra + list(defines) + ["-c", s, "-o", o])
    if jobs:
        with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 4))) as ex:
            for out in ex.map(_run, jobs):
                if verbose and out.strip():
                    print(out)
    objs = [os.path.join(BUILD, u[0]) for u in units]
    if units and (force or _newer(LIB_CUDA, objs) or not _stamp_matches(stamp, digest)):
        _run([NVCC] + NVCC_FLAGS + ["-shared", "-o", LIB_CUDA] + objs)
    if units and not os.environ.get("BEPUCUDA_FREEZE_UNITS"):
        _write_stamp(stamp, digest, LIB_CUDA)
    if variant:
        return LIB_CUDA, LIB_HOST
    host_src = os.path.join(CSRC, "host", "bepu_host.cpp")
    if force or _newer(LIB_HOST, [host_src, LIB_CUDA] + headers):
        _run([GXX, "-O2", "-std=c++17", "-fPIC", "-shared", "-o", LIB_HOST, host_src, "-L" + HERE, "-lbepucuda", "-Wl,-rpath,$ORIGIN"])
    return LIB_CUDA, LIB_HOST


if __name__ == "__main__":
    _variant = next((a.split("=", 1)[1] for a in sys.argv if a.startswith("--variant=")), None)
    build(force="--force" in sys.argv, verbose=True, variant=_variant, defines=[a for a in sys.argv if a.startswith("-D")])
    print("built", LIB_CUDA, LIB_HOST)
