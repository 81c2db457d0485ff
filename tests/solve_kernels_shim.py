"""Builds and loads tests/cuda/solve_kernels_shim.cu: C entry points over the solve-phase launchers, linked against
linalg.cu and block_matvec.cu compiled with exactly the library's flags (math_audio_b200.build).

TEST INFRASTRUCTURE ONLY.  The shim links the CUDA runtime statically and has no libcuda dependency, so it loads on a
machine without a GPU (where every launch would fail).
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

from math_audio_b200 import build as _b

ROOT = Path(__file__).resolve().parent.parent
SHIM_SRC = ROOT / "tests" / "cuda" / "solve_kernels_shim.cu"
UNITS = ("linalg.cu", "block_matvec.cu")

_P, _U64, _I = C.c_void_p, C.c_uint64, C.c_int
SIGNATURES = {
    "shim_zgemv": (_I, [_P, _U64, _U64, _U64, _P, _P]),
    "shim_zgemv_t": (_I, [_P, _U64, _U64, _U64, _P, _P]),
    "shim_zgemm_block": (_I, [_P, _U64, _U64, _U64, _P, _P, _I]),
    "shim_mgs": (_I, [_P, _U64, _P, _I, _U64, _P, _P, _P, _I, _P, _I, _P]),
    "shim_mgs_scratch_elems": (_U64, []),
    "shim_mgs_batched": (_I, [_I, _P, _U64, _U64, _P, _I, _U64, _P, _U64, _P, _P]),
    "shim_residual": (_I, [_P, _P, _P, _U64, _P, _P]),
    "shim_interleave": (_I, [_P, _P, _U64, _I, _I, _I]),
    "shim_sync": (_I, []),
}


def build_shim(outdir: Path, csrc: Path = _b.CSRC) -> Path:
    """Compile the shim and the kernel units from `csrc` into `outdir`; returns the shared library."""
    outdir = Path(outdir)
    outdir.mkdir(parents=True, exist_ok=True)
    nvcc = _b._nvcc()
    jobs = []
    for src, extra in [(Path(csrc) / u, _b.UNITS[u]) for u in UNITS] + [(SHIM_SRC, [])]:
        obj = outdir / (src.name + ".o")
        cmd = [nvcc, *_b.ARCH, *_b.COMMON, *extra, "-I", str(csrc), "-c", str(src), "-o", str(obj)]
        jobs.append((obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for obj, p in jobs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for {obj.name}:\n{out}")
    so = outdir / "libsolve_kernels_shim.so"
    subprocess.run([nvcc, *_b.ARCH, "-shared", "-o", str(so), *(str(o) for o, _ in jobs), "-Xcompiler", "-fPIC"], check=True)
    return so


def load(so: Path) -> C.CDLL:
    lib = C.CDLL(str(so))
    for name, (res, args) in SIGNATURES.items():
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    return lib
