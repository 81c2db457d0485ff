"""ctypes front end of tests/cpp/admittance_oracle.cpp: ``assemble_opts``, the CPU oracle of ``bemb200_assemble_staged_opts``
(admittance, forced dg_dn_sign, consistent beta; DESIGN.md 4.8), and the exact series of the sphere tests.

TEST INFRASTRUCTURE ONLY.  The library is compiled on first use into the temporary directory (the repository tree may be
read-only where the tests run), keyed by the sources it is built from.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
_SRC = ROOT / "tests" / "cpp" / "admittance_oracle.cpp"
_DEPS = [_SRC, ROOT / "oracle" / "bem_oracle.cpp", ROOT / "oracle" / "quad_tables.h"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(p.read_bytes() for p in _DEPS)).hexdigest()[:16]
        so = Path(tempfile.gettempdir()) / f"bemb200_admittance_oracle_{os.getuid()}_{h}.so"
        if not so.exists():
            tmp = so.with_suffix(f".{os.getpid()}.tmp")
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", str(tmp), str(_SRC), "-lpthread"],
                           check=True)
            os.replace(tmp, so)
        _lib = C.CDLL(str(so))
        _lib.orc_assemble_opts.restype = C.c_long
    return _lib


def assemble_opts(mesh, k, beta, dg_dn_sign=0, consistent_beta=False, admittance=None, row_begin=0, row_end=None, harmonic=1.0,
                  tau=1.0, nthreads=0):
    """(A, rhs, quadrature points) of rows [row_begin, row_end); ``admittance`` in DOF order (None: none)."""
    from oracle import oracle as orc

    cm = orc._cmesh(mesh)
    n = int((np.asarray(mesh.is_eval) == 0).sum())
    row_end = n if row_end is None else row_end
    A = np.zeros((row_end - row_begin, n), dtype=np.complex128)
    rhs = np.zeros(row_end - row_begin, dtype=np.complex128)
    y = None if admittance is None else np.ascontiguousarray(admittance, dtype=np.complex128)
    if y is not None and y.shape != (n,):
        raise ValueError("admittance must have one entry per DOF")
    beta = complex(beta)
    nq = lib().orc_assemble_opts(C.byref(cm), C.c_double(k), C.c_double(harmonic), C.c_double(tau), C.c_double(beta.real),
                                 C.c_double(beta.imag), C.c_int(int(dg_dn_sign)), C.c_int(int(consistent_beta)),
                                 y.ctypes.data_as(C.c_void_p) if y is not None else None, C.c_uint64(row_begin), C.c_uint64(row_end),
                                 A.ctypes.data_as(C.c_void_p), rhs.ctypes.data_as(C.c_void_p), C.c_int(nthreads))
    if nq == -1:
        raise ValueError("orc_assemble_opts: invalid options")
    if nq == -2:
        raise ValueError("orc_assemble_opts: consistent_beta needs tau > 0")
    return A, rhs, int(nq)


def robin_mie(k, a, Y, points, nterms=60):
    """Total pressure of a plane wave exp(ikz) on a sphere of radius a with dp/dr = Y p on r = a (e^{+ikr} convention)."""
    from scipy.special import eval_legendre, spherical_jn, spherical_yn

    pts = np.asarray(points, dtype=np.float64)
    r = np.linalg.norm(pts, axis=1)
    ct = pts[:, 2] / r
    p = np.zeros(len(pts), dtype=np.complex128)
    for m in range(nterms):
        j, jp = spherical_jn(m, k * a), spherical_jn(m, k * a, True)
        h, hp = j + 1j * spherical_yn(m, k * a), jp + 1j * spherical_yn(m, k * a, True)
        am = -(k * jp - Y * j) / (k * hp - Y * h)
        jr = spherical_jn(m, k * r)
        p += (2 * m + 1) * (1j ** m) * (jr + am * (jr + 1j * spherical_yn(m, k * r))) * eval_legendre(m, ct)
    return p


def rel_l2(x, ref) -> float:
    return float(np.linalg.norm(x - ref) / np.linalg.norm(ref))
