#!/usr/bin/env python3
"""Golden fixtures for the LARGE configurations (BASELINE.json configs[1] and configs[3]), generated once
by the CPU oracle (oracle/bem_oracle.cpp) and committed, so that neither `bench.py` nor the `-m gpu`
tests need the oracle at these sizes at run time:

  config4_rows.npz   121 680-element geodesic sphere (nu = 78), ka = 16, adaptive beta: 32 sampled rows
                     (4 per rank of an 8-way row partition: first/last row of the slab and two interior
                     ones), each at the 256 columns nearest to the collocation point (all subdivided
                     pairs, the self term) plus every 32nd column, and the dot product of the WHOLE row
                     with a seeded vector (sampled-row matvec parity, SURVEY.md 8d row 4).
  config2_x_kaXX.npz 20 480-element icosphere(5), ka in {0.25, 2, 8}: the plane-wave right-hand side is
                     recomputed by the test; the fixture holds the LAPACK (LU) solution of the oracle's
                     matrix and the oracle GMRES(50, 1e-10) iteration / restart counts.

  config3_rows.npz   50 176-element Quad4 cabinet (64 x 88 x 128) with the piston velocity BC, f = 1 kHz, beta = i/k:
                     16 sampled rows (4 per rank of a 4-way row partition) at the 256 nearest + every 32nd column,
                     whole-row dot products with a seeded vector, and the right-hand-side entries of those rows.
  config3_coarse_x.npz  the 4x-coarsened copy (32 x 44 x 64 = 12 544 elements, same box, piston and frequency) solved in
                     full: LAPACK solution of the oracle's matrix with the oracle's right-hand side, oracle GMRES counts
                     (SURVEY.md 8d row 3).

  config5_rhs32.npz  20 480-element icosphere(5), ka = 2, adaptive beta, 32 plane-wave directions on the Fibonacci sphere
                     (BASELINE.json configs[4]): oracle GMRES(50, 1e-10) iteration / restart counts of all 32 right-hand
                     sides (32 independent gmres() calls, the reference's semantics) and the LAPACK solutions of columns
                     0, 13 and 31.

  rowdot_fsum.npz    the whole-row dot products of config4_rows.npz and config3_rows.npz again, summed with exact_dot: the
                     same bits on every CPU, where np.dot's summation order follows the BLAS kernel chosen for the processor.
                     The rows are re-assembled and checked against those two fixtures first.

    python tests/golden/make_golden_large.py [config4] [config2] [config3] [config5] [rowdot]

config2 takes ~8 minutes per frequency on 8 cores (assembly 92 s, LU 4-5 min, GMRES 25 s).
"""
import math
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from math_audio_b200.incident import IncidentField  # noqa: E402
from math_audio_b200.mesh import generate_geodesic_sphere_mesh, generate_icosphere_mesh  # noqa: E402
from math_audio_b200.types import PhysicsParams  # noqa: E402
from oracle import oracle as orc  # noqa: E402

OUT = Path(__file__).resolve().parent

CONFIG4_NRANKS = 8
CONFIG4_STRIDE = 32
CONFIG4_NEAREST = 256


def config4_sample_rows(n: int):
    chunk = (n + CONFIG4_NRANKS - 1) // CONFIG4_NRANKS
    rows = []
    for p in range(CONFIG4_NRANKS):
        b, e = p * chunk, min(n, (p + 1) * chunk)
        rows += [b, b + (e - b) // 3, b + 2 * (e - b) // 3 + 1, e - 1]
    return np.array(rows, dtype=np.int64)


def config4_probe_vector(n: int) -> np.ndarray:
    rng = np.random.default_rng(1234)
    return rng.standard_normal(n) + 1j * rng.standard_normal(n)


def make_config4():
    a, ka = 1.0, 16.0
    mesh = generate_geodesic_sphere_mesh(a, 78)
    n = mesh.num_dofs
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    rows = config4_sample_rows(n)
    xprobe = config4_probe_vector(n)
    cols = np.zeros((len(rows), CONFIG4_NEAREST + (n + CONFIG4_STRIDE - 1) // CONFIG4_STRIDE), dtype=np.int64)
    vals = np.zeros(cols.shape, dtype=np.complex128)
    rowdot = np.zeros(len(rows), dtype=np.complex128)
    rhs = np.zeros(len(rows), dtype=np.complex128)
    rownorm = np.zeros(len(rows))
    t0 = time.time()
    for i, r in enumerate(rows):
        A, rh, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=int(r), row_end=int(r) + 1)
        d = np.linalg.norm(mesh.center - mesh.center[r], axis=1)
        near = np.argsort(d, kind="stable")[:CONFIG4_NEAREST]
        c = np.concatenate([near, np.arange(0, n, CONFIG4_STRIDE)])
        cols[i] = c
        vals[i] = A[0, c]
        rowdot[i] = np.dot(A[0], xprobe)
        rhs[i] = rh[0]
        rownorm[i] = np.linalg.norm(A[0])
    np.savez_compressed(OUT / "config4_rows.npz", rows=rows, cols=cols, vals=vals, rowdot=rowdot, rownorm=rownorm, rhs=rhs, k=ph.wave_number,
                        beta=beta, nu=78, a=a, n=n)
    print(f"config4_rows: {len(rows)} rows x {cols.shape[1]} columns in {time.time() - t0:.1f} s")


def make_config2(kas=(0.25, 2.0, 8.0)):
    import scipy.linalg as sla

    a = 0.1
    mesh = generate_icosphere_mesh(a, 5)
    inc = IncidentField.plane_wave_z()
    for ka in kas:
        t0 = time.time()
        ph = PhysicsParams.from_wave_number(ka / a)
        beta, _ = ph.burton_miller_beta_adaptive(a)
        A, rhs0, _ = orc.assemble(mesh, ph.wave_number, beta)
        b = rhs0 + inc.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
        t1 = time.time()
        xg, info = orc.gmres(A, b, max_iterations=1000, restart=50, tolerance=1e-10)
        t2 = time.time()
        lu, piv = sla.lu_factor(A, overwrite_a=True, check_finite=False)
        x = sla.lu_solve((lu, piv), b, check_finite=False)
        t3 = time.time()
        dx = float(np.linalg.norm(xg - x) / np.linalg.norm(x))
        tag = f"{ka:g}".replace(".", "p")
        np.savez_compressed(OUT / f"config2_x_ka{tag}.npz", x=x, ka=ka, a=a, sub=5, k=ph.wave_number, beta=beta,
                            iterations=info["iterations"], restarts=info["restarts"], residual=info["residual"],
                            gmres_vs_lu=dx)
        print(f"config2 ka={ka}: assemble {t1 - t0:.0f} s, gmres {t2 - t1:.0f} s ({info}), LU {t3 - t2:.0f} s, |x_gmres - x_lu|/|x_lu| = {dx:.2e}")


def cabinet_mesh(scale: float):
    """SURVEY.md 8d row 3 (same construction as tests/drivers/run_config.py and bench.py)."""
    from math_audio_b200.mesh import generate_box_mesh_quad

    nx, ny, nz = int(64 * scale), int(88 * scale), int(128 * scale)
    mesh = generate_box_mesh_quad(0.32, 0.44, 0.64, nx, ny, nz)
    front = (np.abs(mesh.center[:, 1] + 0.22) < 1e-9) & (np.hypot(mesh.center[:, 0], mesh.center[:, 2]) < 0.08)
    v = np.zeros((mesh.n_elem, 4), dtype=np.complex128)
    v[front] = 1.0
    mesh.set_velocity_bc(v)
    mesh.bc_len[~front] = 1
    return mesh


CONFIG3_NRANKS = 4


def make_config3():
    import scipy.linalg as sla

    ph = PhysicsParams.new(1000.0, 343.0, 1.21, False)
    beta = ph.burton_miller_beta()
    # sampled rows of the full-size box
    t0 = time.time()
    mesh = cabinet_mesh(1.0)
    n = mesh.num_dofs
    chunk = (n + CONFIG3_NRANKS - 1) // CONFIG3_NRANKS
    rows = []
    for p in range(CONFIG3_NRANKS):
        b, e = p * chunk, min(n, (p + 1) * chunk)
        rows += [b, b + (e - b) // 3, b + 2 * (e - b) // 3 + 1, e - 1]
    piston = np.flatnonzero(np.abs(mesh.bc_val[:, 0]) > 0)
    rows[1] = int(piston[len(piston) // 2])          # a row whose own element carries the piston velocity
    rows = np.array(sorted(set(rows)), dtype=np.int64)
    xprobe = config4_probe_vector(n)
    cols = np.zeros((len(rows), CONFIG4_NEAREST + (n + CONFIG4_STRIDE - 1) // CONFIG4_STRIDE), dtype=np.int64)
    vals = np.zeros(cols.shape, dtype=np.complex128)
    rowdot = np.zeros(len(rows), dtype=np.complex128)
    rhs = np.zeros(len(rows), dtype=np.complex128)
    rownorm = np.zeros(len(rows))
    for i, r in enumerate(rows):
        A, rh, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=int(r), row_end=int(r) + 1)
        d = np.linalg.norm(mesh.center - mesh.center[r], axis=1)
        c = np.concatenate([np.argsort(d, kind="stable")[:CONFIG4_NEAREST], np.arange(0, n, CONFIG4_STRIDE)])
        cols[i], vals[i], rowdot[i], rhs[i], rownorm[i] = c, A[0, c], np.dot(A[0], xprobe), rh[0], np.linalg.norm(A[0])
    np.savez_compressed(OUT / "config3_rows.npz", rows=rows, cols=cols, vals=vals, rowdot=rowdot, rownorm=rownorm, rhs=rhs,
                        k=ph.wave_number, beta=beta, n=n)
    print(f"config3_rows: {len(rows)} rows x {cols.shape[1]} columns in {time.time() - t0:.1f} s")
    # the 4x-coarsened copy, solved in full
    t0 = time.time()
    mesh = cabinet_mesh(0.5)
    A, b, _ = orc.assemble(mesh, ph.wave_number, beta)
    t1 = time.time()
    xg, info = orc.gmres(A, b, max_iterations=1000, restart=50, tolerance=1e-10)
    t2 = time.time()
    lu, piv = sla.lu_factor(A, overwrite_a=True, check_finite=False)
    x = sla.lu_solve((lu, piv), b, check_finite=False)
    dx = float(np.linalg.norm(xg - x) / np.linalg.norm(x))
    np.savez_compressed(OUT / "config3_coarse_x.npz", x=x, b=b, k=ph.wave_number, beta=beta, n=mesh.num_dofs, iterations=info["iterations"],
                        restarts=info["restarts"], residual=info["residual"], gmres_vs_lu=dx)
    print(f"config3 coarse ({mesh.num_dofs}): assemble {t1 - t0:.0f} s, gmres {t2 - t1:.0f} s ({info}), LU {time.time() - t2:.0f} s, |x_gmres - x_lu|/|x_lu| = {dx:.2e}")


def make_config5():
    import scipy.linalg as sla

    from math_audio_b200.mesh import fibonacci_directions

    a, ka = 0.1, 2.0
    mesh = generate_icosphere_mesh(a, 5)
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    t0 = time.time()
    A, rhs0, _ = orc.assemble(mesh, ph.wave_number, beta)
    dirs = fibonacci_directions(32)
    B = np.stack([rhs0 + IncidentField.plane_wave(d).compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta) for d in dirs])
    its, rst, res = [], [], []
    for m in range(32):
        _x, info = orc.gmres(A, B[m], max_iterations=1000, restart=50, tolerance=1e-10)
        its.append(info["iterations"]); rst.append(info["restarts"]); res.append(info["residual"])
        print(f"config5 rhs {m}: {info} ({time.time() - t0:.0f} s)", flush=True)
    cols = np.array([0, 13, 31])
    lu, piv = sla.lu_factor(A, overwrite_a=True, check_finite=False)
    X = np.stack([sla.lu_solve((lu, piv), B[m], check_finite=False) for m in cols])
    np.savez_compressed(OUT / "config5_rhs32.npz", iterations=np.array(its), restarts=np.array(rst), residual=np.array(res), x_cols=cols, x=X,
                        ka=ka, a=a, sub=5, k=ph.wave_number, beta=beta)
    print(f"config5: {time.time() - t0:.0f} s, iterations {its}")


def exact_dot(a: np.ndarray, x: np.ndarray) -> complex:
    """sum_j a_j x_j with every product rounded once and each of the two real sums correctly rounded (math.fsum)."""
    return complex(math.fsum(np.concatenate([a.real * x.real, -(a.imag * x.imag)])),
                   math.fsum(np.concatenate([a.real * x.imag, a.imag * x.real])))


def make_rowdot_fsum():
    out = {}
    for name in ("config4", "config3"):
        g = np.load(OUT / f"{name}_rows.npz")
        if name == "config4":
            mesh = generate_geodesic_sphere_mesh(float(g["a"]), int(g["nu"]))
            ph = PhysicsParams.from_wave_number(float(g["k"]))
            beta, _ = ph.burton_miller_beta_adaptive(float(g["a"]))
        else:
            mesh = cabinet_mesh(1.0)
            ph = PhysicsParams.new(1000.0, 343.0, 1.21, False)
            beta = ph.burton_miller_beta()
        xprobe = config4_probe_vector(mesh.num_dofs)
        out[name] = np.zeros(len(g["rows"]), dtype=np.complex128)
        for i, r in enumerate(g["rows"]):
            A, rh, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=int(r), row_end=int(r) + 1)
            assert np.array_equal(A[0, g["cols"][i]], g["vals"][i]) and rh[0] == g["rhs"][i], (name, i)
            out[name][i] = exact_dot(A[0], xprobe)
            assert abs(out[name][i] - g["rowdot"][i]) <= 1e-12 * abs(g["rowdot"][i]), (name, i)
    np.savez_compressed(OUT / "rowdot_fsum.npz", **out)
    print(f"rowdot_fsum: {len(out['config4'])} + {len(out['config3'])} rows")


if __name__ == "__main__":
    what = sys.argv[1:] or ["config4", "config2", "config3", "config5", "rowdot"]
    if "config5" in what:
        make_config5()
    if "config3" in what:
        make_config3()
    if "config4" in what:
        make_config4()
    if "config2" in what:
        make_config2()
    if "rowdot" in what:
        make_rowdot_fsum()
