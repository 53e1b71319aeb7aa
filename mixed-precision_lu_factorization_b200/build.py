"""Build libmplu.so (CUDA kernels + C++ host driver + C ABI) in-tree with nvcc for sm_100a.

The shared library is the product: Python only loads it through ctypes.  No torch extension machinery is used so
the very same .so serves the C++ drivers in drivers/ and any reference-side binding (INTEGRATION.md).
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB = PKG / "libmplu.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-I", str(ROOT / "include"),
]

# experiments: extra nvcc flags from the environment (e.g. MPLU_EXTRA_NVCC_FLAGS="-DMPLU_LEAF_LOOKAHEAD=1"); they are part
# of the build stamp, so a plain build() afterwards rebuilds the default library
NVCC_FLAGS += os.environ.get("MPLU_EXTRA_NVCC_FLAGS", "").split()

SOURCES = ["gemm_tc.cu", "getrf_fused.cu", "getrf_flow.cu", "panel.cu", "equil.cu", "ir.cu", "lu.cu", "gmres.cu", "dist.cu", "generate.cu", "mpf_compat.cu", "fp64_fallback.cu", "dropin_kernels.cu"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stamp() -> str:
    h = hashlib.sha256()
    for p in sorted(list(CSRC.glob("*")) + list((ROOT / "include").glob("*.h"))):
        if p.is_file():
            h.update(p.name.encode())
            h.update(p.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    stamp_file = PKG / ".libmplu.stamp"
    stamp = _stamp()
    if not force and LIB.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB
    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        sp = CSRC / src
        if not sp.exists():
            continue
        obj = objdir / (src.rsplit(".", 1)[0] + ".o")
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", str(sp), "-o", str(obj)]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out.strip():
            print(out, file=sys.stderr)
    link = [_nvcc(), "-shared", "-o", str(LIB), *objs, "-gencode", "arch=compute_100a,code=sm_100a",
            "-cudart", "static", "-ldl"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    # the two drop-in kernels also as a static archive: a foreign translation unit that launches them itself (the way the
    # reference's MPF.cu does) links this instead of taking the host stubs out of the shared library (INTEGRATION.md 2)
    ar = PKG / "libmplu_dropin.a"
    if ar.exists():
        ar.unlink()
    subprocess.run(["ar", "rcs", str(ar), str(objdir / "dropin_kernels.o")], check=True)
    stamp_file.write_text(stamp)
    return LIB


def build_drivers(force: bool = False) -> None:
    """drivers/benchmark and drivers/matrix_generator (C++ hosts of the reference's two CLI programs)."""
    ddir = ROOT / "drivers"
    gen, bench = ddir / "matrix_generator", ddir / "benchmark"
    if force or not gen.exists() or gen.stat().st_mtime < (ddir / "matrix_generator.cpp").stat().st_mtime:
        subprocess.run(["g++", "-O2", "-std=c++17", str(ddir / "matrix_generator.cpp"), "-o", str(gen)], check=True)
    src = ddir / "benchmark.cpp"
    if force or not bench.exists() or bench.stat().st_mtime < max(src.stat().st_mtime, LIB.stat().st_mtime):
        defs = []
        try:  # host LAPACK for the lapack_time column: scipy's OpenBLAS if present (loaded with dlopen at run time)
            import glob
            import scipy
            libs = glob.glob(os.path.join(os.path.dirname(os.path.dirname(scipy.__file__)), "scipy.libs", "libscipy_openblas*.so"))
            if libs:
                defs = [f'-DMPLU_DEFAULT_LAPACK_LIB="{libs[0]}"']
        except Exception:
            pass
        subprocess.run(["g++", "-O2", "-std=c++17", *defs, "-I", str(ROOT / "include"), str(src), "-o", str(bench),
                        f"-L{PKG}", "-lmplu", "-ldl", f"-Wl,-rpath,{PKG}"], check=True)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
