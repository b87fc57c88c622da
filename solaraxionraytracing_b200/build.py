"""Builds libsart.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

Run as ``python -m solaraxionraytracing_b200.build``. nvcc cross-compiles without a GPU. The built library
stays next to the sources (git-ignored, but it travels to the GPU box with the gpurun snapshot).
"""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
LIB = HERE / "libsart.so"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
HOST_CXX = "/usr/bin/g++"

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall",
          "-ccbin", HOST_CXX, "-I", str(HERE.parent / "include")]

# (source, extra flags). The exact pipeline must not contract a*b+c into FMA: its hit/miss decisions are
# compared bit for bit with the CPU oracle.
UNITS = [
    ("kernels_exact.cu", ["-fmad=false", "-prec-div=true", "-prec-sqrt=true"]),
    ("kernels_fast.cu", []),
    ("kernels_f32.cu", []),
    ("kernels_f32_rays.cu", []),
    ("kernels_util.cu", []),
    ("kernels_emission.cu", []),
    ("api.cu", []),
    ("comm.cu", []),
    ("derive.cpp", []),
    ("derive_fast.cpp", []),
    ("host_setup.cpp", []),
]


def _stale(out: Path, deps: list[Path]) -> bool:
    if not out.exists():
        return True
    t = out.stat().st_mtime
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False, defines: list[str] | None = None, out: Path | None = None) -> Path:
    """`defines`/`out` build an experimental variant (e.g. -DSART_FAST_MINBLOCKS=3) next to the default library."""
    if defines or out:
        return _build_variant(defines or [], out or LIB.with_name("libsart_variant.so"), verbose)
    hdrs = sorted(CSRC.glob("*.h")) + sorted(CSRC.glob("*.cuh")) + [HERE.parent / "include" / "sart.h",
                                                                    Path(__file__)]
    objdir = HERE / "build"
    objdir.mkdir(exist_ok=True)
    objs, cmds = [], []
    for src, extra in UNITS:
        s = CSRC / src
        o = objdir / (src + ".o")
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [NVCC, *ARCH, *COMMON, *extra, "-c", str(s), "-o", str(o)]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), flush=True)
            cmds.append(cmd)
    if cmds:   # the translation units are independent: compile them side by side
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(cmds), os.cpu_count() or 1)) as ex:
            for r in ex.map(lambda c: subprocess.run(c, check=False, capture_output=not verbose, text=True), cmds):
                if r.returncode != 0:
                    sys.stderr.write((r.stdout or "") + (r.stderr or ""))
                    raise subprocess.CalledProcessError(r.returncode, r.args)
    if force or _stale(LIB, objs):
        cmd = [NVCC, *ARCH, "-shared", "-ccbin", HOST_CXX, "-cudart", "static", "-o", str(LIB), *map(str, objs), "-ldl"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.run(cmd, check=True)
    return LIB


def _build_variant(defines: list[str], out: Path, verbose: bool) -> Path:
    objdir = HERE / "build" / out.stem
    objdir.mkdir(parents=True, exist_ok=True)
    objs = []
    for src, extra in UNITS:
        o = objdir / (src + ".o")
        objs.append(o)
        cmd = [NVCC, *ARCH, *COMMON, *extra, *[f"-D{d}" for d in defines], "-c", str(CSRC / src), "-o", str(o)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        subprocess.run(cmd, check=True)
    subprocess.run([NVCC, *ARCH, "-shared", "-ccbin", HOST_CXX, "-cudart", "static", "-o", str(out), *map(str, objs), "-ldl"],
                   check=True)
    return out


if __name__ == "__main__":
    if any(a.startswith("-D") for a in sys.argv[1:]):
        defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
        outs = [a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--out=")]
        print(build(defines=defs, out=HERE / outs[0] if outs else None, verbose="-v" in sys.argv))
        sys.exit(0)
    build(force="--force" in sys.argv, verbose="-v" in sys.argv or "--verbose" in sys.argv)
    print(LIB)
