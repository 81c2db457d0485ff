"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI
(math_audio_b200.bem -> ctypes -> libbemb200.so), against the CPU oracle and the committed
golden fixtures.

Tolerances (BASELINE.json north_star): matrix entries relative 1e-10 in FP64; surface
pressure after GMRES relative 1e-8 (GMRES tol 1e-10 on both sides, SURVEY 8d).
"""
import math
from pathlib import Path

import numpy as np
import pytest

from math_audio_b200.mesh import (BC_PRESSURE, BC_TRANSFER, generate_box_mesh_quad, generate_icosphere_mesh,
                                  generate_sphere_mesh, mesh_from_data)
from math_audio_b200.types import PhysicsParams

pytestmark = pytest.mark.gpu

ENTRY_TOL = 1e-10
X_TOL = 1e-8
GOLD = Path(__file__).resolve().parent / "golden"


@pytest.fixture(scope="module")
def bem():
    from math_audio_b200 import bem as b

    b.default_context()  # raises loudly if the extension or the GPU is missing
    return b


def entry_err(A, Aref):
    """max |dA_ij|/|A_ij| where the reference entry is not (numerically) zero, plus the
    row-normwise error everywhere (SURVEY 8d 'Tolerances & metrics')."""
    scale = np.max(np.abs(Aref), axis=1, keepdims=True)
    rownorm = np.max(np.abs(A - Aref) / scale)
    big = np.abs(Aref) > 1e-9 * scale
    rel = np.max(np.abs(A - Aref)[big] / np.abs(Aref)[big])
    return rel, rownorm


def box_piston_mesh(nx=4, ny=6, nz=8):
    mesh = generate_box_mesh_quad(0.32, 0.44, 0.64, nx, ny, nz)
    front = (np.abs(mesh.center[:, 1] + 0.22) < 1e-9) & (np.hypot(mesh.center[:, 0], mesh.center[:, 2]) < 0.12)
    v = np.zeros((mesh.n_elem, 4), dtype=np.complex128)
    v[front] = 1.0
    mesh.set_velocity_bc(v)
    mesh.bc_len[~front] = 1
    return mesh, front


def test_far_kernel_math(bem):
    ctx = bem.default_context()
    for xmax in (50.0, 200.0, 5000.0):
        sc, rs = ctx.selftest_math(1 << 21, xmax)
        # abs error of sin/cos against the EXACT phase kappa*r (double-double reference): 5e-16 + 1.5e-16 |kappa r| -- the
        # reference's sin(k*r) starts from a product that is itself rounded by up to 1.1e-16 |k r|
        assert sc < 5e-16 + 1.5e-16 * xmax, (xmax, sc)
        assert rs < 5e-16, rs                                    # rel error of 1/sqrt


@pytest.mark.parametrize("name", ["ico1_ka0p5", "ico2_ka0p2", "ico2_ka6"])
def test_golden_sphere(bem, name):
    g = np.load(GOLD / f"{name}.npz")
    a, k, beta = float(g["a"]), float(g["k"]), complex(g["beta"])
    mesh = generate_icosphere_mesh(a, int(g["sub"]))
    ph = PhysicsParams.from_wave_number(k)
    assert ph.wave_number == pytest.approx(k, rel=1e-15)
    ph.wave_number = k
    system = bem.build_tbem_system_with_beta(mesh, ph, beta)
    rel, rown = entry_err(system.matrix.rows(), g["A"])
    assert rel < ENTRY_TOL and rown < ENTRY_TOL, (rel, rown)
    op = bem.DenseOperator(system)
    sol = bem.gmres(op, g["b"], bem.GmresConfig(max_iterations=1000, restart=50, tolerance=1e-10))
    assert sol.converged and sol.iterations == int(g["iterations"]) and sol.restarts == int(g["restarts"])
    assert np.linalg.norm(sol.x - g["x"]) / np.linalg.norm(g["x"]) < X_TOL


def test_golden_box_piston_rhs(bem):
    g = np.load(GOLD / "box_4x6x8_piston.npz")
    mesh, front = box_piston_mesh()
    ph = PhysicsParams.new(500.0, 343.0, 1.21, False)
    system = bem.build_tbem_system_with_beta(mesh, ph, complex(g["beta"]))
    rel, rown = entry_err(system.matrix.rows(), g["A"])
    assert rown < ENTRY_TOL and rel < 1e-9, (rel, rown)  # coplanar pairs: H ~ 1e-17 noise vs exact 0
    assert np.max(np.abs(system.rhs - g["rhs"])) / np.max(np.abs(g["rhs"])) < ENTRY_TOL
    st = system.matrix.assembly_stats()
    assert st["special_pairs"] == 0  # piston (non-zero velocity) columns stay in the far kernel; rhs_far_kernel adds their RHS term


@pytest.mark.parametrize("sub,ka", [(3, 0.2), (3, 1.0), (3, 3.0), (3, 8.0), (3, 16.0)])
def test_full_matrix_parity_icosphere(bem, orc, sub, ka):
    """All N^2 entries.  ka=8/16 on icosphere(3) reach k*h_e >= 1 and >= 2: the nsec2 = 3 / 4
    duplicate-sub-triangle quirk of the singular integration (singular.rs:268-278)."""
    a = 0.1
    ph = PhysicsParams.from_wave_number(ka / a)
    mesh = generate_icosphere_mesh(a, sub)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    system = bem.build_tbem_system_with_beta(mesh, ph, beta)
    Ao, rhso, _ = orc.assemble(mesh, ph.wave_number, beta)
    rel, rown = entry_err(system.matrix.rows(), Ao)
    assert rel < ENTRY_TOL and rown < ENTRY_TOL, (rel, rown)
    assert np.abs(system.rhs).max() == 0.0 and np.abs(rhso).max() == 0.0  # rigid: v = 0
    assert system.matrix.ctx and bem.StagedMesh(mesh).dg_dn_sign(ph.wave_number) == orc.dg_dn_sign(mesh, ph.wave_number)


def test_config1_uv_sphere_solve_and_mie(bem, orc):
    """BASELINE.json configs[0]: rigid UV sphere (32x32 -> 1984 Tri3), ka = 1, plane wave +z,
    beta = adaptive (4i/k); GMRES(50) tol 1e-10; L2 vs the 50-term Mie series must EQUAL the
    oracle's (the reference's own accuracy here is ~27 %, qa_suite.rs:175-179)."""
    from math_audio_b200.incident import IncidentField

    a = 0.1
    ph = PhysicsParams.from_wave_number(1.0 / a)
    mesh = generate_sphere_mesh(a, 32, 32)
    assert mesh.n_elem == 1984
    beta, scale = ph.burton_miller_beta_adaptive(a)
    assert scale == 4.0
    system = bem.build_tbem_system_with_beta(mesh, ph, beta)
    Ao, rhso, _ = orc.assemble(mesh, ph.wave_number, beta)
    rel, rown = entry_err(system.matrix.rows(), Ao)
    assert rel < ENTRY_TOL and rown < ENTRY_TOL, (rel, rown)
    b = system.rhs + IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
    bo = rhso + orc.incident_rhs(0, [0, 0, 1.0], 1.0, mesh.center, mesh.normal, ph.wave_number, beta)[0]
    assert np.max(np.abs(b - bo)) < 1e-13
    cfg = bem.GmresConfig(max_iterations=1000, restart=50, tolerance=1e-10)
    sol = bem.solve_gmres(bem.DenseOperator(system), b, cfg)
    xo, io = orc.gmres(Ao, bo, max_iterations=1000, restart=50, tolerance=1e-10)
    assert sol.converged and abs(sol.iterations - io["iterations"]) <= 1
    assert np.linalg.norm(sol.x - xo) / np.linalg.norm(xo) < X_TOL
    xl = np.linalg.solve(Ao, bo)
    assert np.linalg.norm(sol.x - xl) / np.linalg.norm(xl) < X_TOL
    r = np.linalg.norm(mesh.center, axis=1)
    mie = orc.mie_rigid_sphere(ph.wave_number, a, 50, r, np.arccos(mesh.center[:, 2] / r))
    e_gpu, e_orc = orc.l2_relative(mie, sol.x), orc.l2_relative(mie, xo)
    assert abs(e_gpu - e_orc) < 1e-8 and e_gpu < 0.30
    # far field: 72 points on r = 10a in the xz-plane through the oracle's field evaluation
    th = np.linspace(0, 2 * math.pi, 72, endpoint=False)
    pts = np.stack([10 * a * np.sin(th), np.zeros_like(th), 10 * a * np.cos(th)], axis=1)
    fg = orc.scattered_field(mesh, pts, sol.x, ph.wave_number)
    fo = orc.scattered_field(mesh, pts, xo, ph.wave_number)
    assert np.linalg.norm(fg - fo) / np.linalg.norm(fo) < X_TOL


def test_cylinder_quad_mesh_parity(bem, orc):
    """generate_cylinder_mesh (generators.rs:242-285): an open Quad4 shell off the coordinate planes
    (rectangular, hence flat, quads through the affine far kernel; normals flipped outward by the generator)."""
    from math_audio_b200.mesh import generate_cylinder_mesh

    mesh = generate_cylinder_mesh(0.12, 0.4, 24, 16)
    assert mesh.n_elem == 384 and (mesh.etype == 4).all()
    for ka in (0.3, 2.5):
        ph = PhysicsParams.from_wave_number(ka / 0.12)
        beta = ph.burton_miller_beta_scaled(4.0)
        system = bem.build_tbem_system_with_beta(mesh, ph, beta)
        Ao, rhso, _ = orc.assemble(mesh, ph.wave_number, beta)
        rel, rown = entry_err(system.matrix.rows(), Ao)
        assert rel < ENTRY_TOL and rown < ENTRY_TOL, (ka, rel, rown)
        st = system.matrix.assembly_stats()
        assert st["special_pairs"] == 0 and st["near_pairs"] > 0


def test_mixed_bc_and_element_types(bem, orc):
    """Pressure / transfer BCs, 1-entry non-zero velocity (the N0-weighted quirk of
    regular.rs:159-164), Tri3 + Quad4 in one mesh, a warped (non-planar) Quad4."""
    box = generate_box_mesh_quad(0.3, 0.4, 0.5, 3, 4, 5)
    nodes = box.nodes.copy()
    quads = box.conn[:, :4].copy()
    # split every quad of the z = -0.25 wall into two triangles, keep the others as quads
    conn = []
    for q in quads:
        if abs(nodes[q, 2].mean() + 0.25) < 1e-12:
            conn.append([q[0], q[1], q[2]])
            conn.append([q[0], q[2], q[3]])
        else:
            conn.append(list(q))
    # warp one wall out of plane so that some quads are not flat
    warped = np.abs(nodes[:, 0] - 0.15) < 1e-12
    nodes[warped, 0] += 0.01 * np.sin(17.0 * nodes[warped, 1]) * np.cos(11.0 * nodes[warped, 2])
    mesh = mesh_from_data(nodes, conn)
    n = mesh.n_elem
    rng = np.random.default_rng(5)
    pick = rng.permutation(n)
    mesh.bc_type[pick[:9]] = BC_PRESSURE
    mesh.bc_val[pick[:5], 0] = 0.7 - 0.2j          # pressure, 1 value
    mesh.bc_type[pick[9:12]] = BC_TRANSFER
    mesh.bc_val[pick[12:20], 0] = 1.0 + 0.5j        # velocity, single entry -> v * N0
    full = pick[20:26]
    mesh.bc_len[full] = mesh.etype[full]
    mesh.bc_val[full] = 0.0
    for e in full:
        mesh.bc_val[e, : mesh.etype[e]] = rng.standard_normal(mesh.etype[e]) + 1j * rng.standard_normal(mesh.etype[e])
    assert set(np.unique(mesh.etype)) == {3, 4}
    for freq in (200.0, 2500.0):
        ph = PhysicsParams.new(freq, 343.0, 1.21, False)
        beta = ph.burton_miller_beta_scaled(2.0)
        system = bem.build_tbem_system_with_beta(mesh, ph, beta)
        Ao, rhso, _ = orc.assemble(mesh, ph.wave_number, beta)
        A = system.matrix.rows()
        rel, rown = entry_err(A, Ao)
        assert rown < ENTRY_TOL, (freq, rel, rown)
        assert np.abs(A[:, mesh.dof[pick[9:12]]]).max() == 0.0  # transfer columns contribute 0
        assert np.max(np.abs(system.rhs - rhso)) / np.max(np.abs(rhso)) < ENTRY_TOL
        assert system.matrix.assembly_stats()["special_pairs"] > 0


@pytest.mark.parametrize("tau,harmonic,beta", [
    (-1.0, 1.0, 0j),                 # interior problem: PhysicsParams::new(.., is_internal = true), beta = 0 (types.rs:45, 64-70)
    (-1.0, 1.0, 0.25j),              # interior with an explicit coupling passed to build_tbem_system_with_beta
    (1.0, 1.0, 0.03 + 0.4j),         # beta with a real part: the general (non purely imaginary) far-kernel instantiation
    (1.0, -1.0, 0.4j),               # harmonic_factor = -1, exp(-ikr): carried by the ABI, never set by PhysicsParams::new
    (-1.0, -1.0, -0.02 + 0.3j),
])
def test_interior_complex_beta_and_time_convention(bem, orc, tau, harmonic, beta):
    """Every parameter of `bemb200_physics` away from the exterior / exp(+ikr) / purely imaginary beta case the
    reference's callers use, against the oracle on all entries (Tri3 sphere across the dG/dn sign switch, and the
    Quad4 box with a vibrating piston, i.e. the right-hand-side path with its unscaled-beta quirk: 0 for tau < 0)."""
    a = 0.1
    mesh = generate_icosphere_mesh(a, 2)
    for ka in (0.3, 2.0):
        ph = PhysicsParams.from_wave_number(ka / a)
        ph.tau, ph.harmonic_factor = tau, harmonic
        system = bem.build_tbem_system_with_beta(mesh, ph, beta)
        Ao, rhso, _ = orc.assemble(mesh, ph.wave_number, beta, harmonic=harmonic, tau=tau)
        rel, rown = entry_err(system.matrix.rows(), Ao)
        assert rel < ENTRY_TOL and rown < 1e-13, (ka, rel, rown)
        assert not system.rhs.any() and not rhso.any()
    box, front = box_piston_mesh()
    ph = PhysicsParams.new(1000.0, 343.0, 1.21, tau < 0)
    ph.harmonic_factor = harmonic
    system = bem.build_tbem_system_with_beta(box, ph, beta)
    Ao, rhso, _ = orc.assemble(box, ph.wave_number, beta, harmonic=harmonic, tau=tau)
    rel, rown = entry_err(system.matrix.rows(), Ao)
    assert rown < 1e-13, (rel, rown)
    assert np.max(np.abs(system.rhs - rhso)) <= 1e-12 * max(1.0, np.max(np.abs(rhso)))
    assert np.abs(rhso).max() > 0.0


def test_tiny_offcentre_and_scaled_meshes(bem, orc):
    """Edge shapes of the input: the reference's own 2-element fixture (tbem.rs:542-598, hand-set centres/normals/areas,
    1-entry non-zero velocity -> RHS), a single element, 20 elements (less than one 128-column tile), a sphere translated
    away from the origin (the dG/dn sign heuristic of tbem.rs:108-123 then sees k*|centre| >= 0.5) and the same problem
    at two length scales (ka fixed)."""
    nodes = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.5, 1.0, 0.0], [1.5, 1.0, 0.0]])
    m = mesh_from_data(nodes, np.array([[0, 1, 2], [1, 3, 2]], dtype=np.uint32))
    m.normal[:] = [0.0, 0.0, 1.0]
    m.center[0] = [0.5, 1.0 / 3.0, 0.0]
    m.center[1] = [1.0, 2.0 / 3.0, 0.0]
    m.area[:] = 0.5
    m.bc_val[0, 0] = 1.0
    ph = PhysicsParams.new(100.0, 343.0, 1.21, False)
    system = bem.build_tbem_system(m, ph)
    A = system.matrix.rows()
    Ao, rhso, _ = orc.assemble(m, ph.wave_number, ph.burton_miller_beta())
    assert system.num_dofs == 2 and A.shape == (2, 2) and system.rhs.shape == (2,)
    assert abs(A[0, 0]) > 1e-15 and abs(A[1, 1]) > 1e-15                   # tbem.rs:594-597
    assert np.max(np.abs(A - Ao) / np.abs(Ao)) < ENTRY_TOL
    assert np.max(np.abs(system.rhs - rhso) / np.abs(rhso)) < ENTRY_TOL and abs(rhso[0]) > 0 and abs(rhso[1]) > 0
    one = mesh_from_data(nodes[:3], np.array([[0, 1, 2]], dtype=np.uint32))
    s1 = bem.build_tbem_system(one, ph)
    A1, _, _ = orc.assemble(one, ph.wave_number, ph.burton_miller_beta())
    assert s1.matrix.rows().shape == (1, 1) and abs(s1.matrix.rows()[0, 0] - A1[0, 0]) / abs(A1[0, 0]) < ENTRY_TOL
    sol = bem.gmres(bem.DenseOperator(s1), np.array([1.0 + 2.0j]), bem.GmresConfig(10, 5, 1e-12))
    assert sol.converged and abs(sol.x[0] - (1.0 + 2.0j) / A1[0, 0]) < 1e-12 * abs(sol.x[0])
    a = 0.1
    ico0 = generate_icosphere_mesh(a, 0)
    assert ico0.n_elem == 20
    for ka in (0.3, 1.0, 4.0):
        p = PhysicsParams.from_wave_number(ka / a)
        beta = p.burton_miller_beta_adaptive(a)[0]
        Ao, _, _ = orc.assemble(ico0, p.wave_number, beta)
        assert entry_err(bem.build_tbem_system_with_beta(ico0, p, beta).matrix.rows(), Ao)[0] < ENTRY_TOL
    # off-centre: same sphere shifted by (0.3, -0.2, 0.5) m
    mesh = generate_icosphere_mesh(a, 2)
    shift = np.array([0.3, -0.2, 0.5])
    moved = mesh_from_data(mesh.nodes + shift, mesh.conn[:, :3].copy())
    moved.normal[:] = mesh.normal
    p = PhysicsParams.from_wave_number(0.2 / a)                            # ka = 0.2 but k |centre| = 1.2 -> sign flips
    beta = p.burton_miller_beta()
    assert orc.dg_dn_sign(mesh, p.wave_number) == 1.0 and orc.dg_dn_sign(moved, p.wave_number) == -1.0
    Ao, _, _ = orc.assemble(moved, p.wave_number, beta)
    assert entry_err(bem.build_tbem_system_with_beta(moved, p, beta).matrix.rows(), Ao)[0] < ENTRY_TOL
    # length scales: a = 25 m and a = 2 mm at ka = 1.5
    for radius in (25.0, 2e-3):
        big = generate_icosphere_mesh(radius, 2)
        p = PhysicsParams.from_wave_number(1.5 / radius)
        beta = p.burton_miller_beta_adaptive(radius)[0]
        Ao, _, _ = orc.assemble(big, p.wave_number, beta)
        rel, rown = entry_err(bem.build_tbem_system_with_beta(big, p, beta).matrix.rows(), Ao)
        assert rel < ENTRY_TOL and rown < 1e-13, (radius, rel, rown)


def test_gmres_extreme_configurations(bem, orc):
    """restart = 1 (every iteration restarts), a tolerance already met by x0 = 0 never happens for b != 0 but a loose one
    stops after one iteration, max_iterations = 0 returns the initial residual unconverged (gmres.rs:137, 264-276)."""
    rng = np.random.default_rng(11)
    n = 300
    A = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))) / np.sqrt(n) + 3 * np.eye(n)
    b = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    op = bem.DenseOperator(A)
    for cfg in ((200, 1, 1e-8), (5, 3, 1e-12), (50, 7, 0.5), (0, 10, 1e-8), (3, 400, 1e-10)):
        sol = bem.gmres(op, b, bem.GmresConfig(*cfg))
        xo, io = orc.gmres(A, b, max_iterations=cfg[0], restart=cfg[1], tolerance=cfg[2])
        assert (sol.iterations, sol.restarts, sol.converged) == (io["iterations"], io["restarts"], io["converged"]), cfg
        assert abs(sol.residual - io["residual"]) <= 1e-9 * max(io["residual"], 1e-300) + 1e-15, cfg
        assert np.linalg.norm(sol.x - xo) <= 1e-10 * max(np.linalg.norm(xo), 1e-300), cfg
    # a long cycle: restart 150 > the 64 basis vectors of the low-synchronisation kernels (103 iterations without restart)
    A2 = A - 1.4 * np.eye(n)
    sol = bem.gmres(bem.DenseOperator(A2), b, bem.GmresConfig(3, 150, 1e-10))
    xo, io = orc.gmres(A2, b, max_iterations=3, restart=150, tolerance=1e-10)
    assert io["iterations"] > 64 and (sol.iterations, sol.restarts, sol.converged) == (io["iterations"], io["restarts"], io["converged"])
    assert np.linalg.norm(sol.x - xo) <= 1e-9 * np.linalg.norm(xo)


def test_row_blocks_eval_elements_and_dof_permutation(bem, orc):
    mesh = generate_icosphere_mesh(0.1, 2)
    ph = PhysicsParams.from_wave_number(15.0)
    beta = ph.burton_miller_beta_scaled(4.0)
    full = bem.build_tbem_system_with_beta(mesh, ph, beta).matrix.rows()
    st = bem.StagedMesh(mesh)
    parts = [bem.build_tbem_system_with_beta(st, ph, beta, rows=(r0, r1)).matrix.rows() for r0, r1 in [(0, 1), (1, 130), (130, 320)]]
    assert (np.vstack(parts) == full).all()  # row sharding changes no bit
    empty = bem.build_tbem_system_with_beta(st, ph, beta, rows=(7, 7))
    assert empty.matrix.rows().shape == (0, 320) and empty.rhs.shape == (0,)
    perm = np.random.default_rng(3).permutation(mesh.n_elem).astype(np.uint32)
    mesh.dof[:] = perm
    Ap = bem.build_tbem_system_with_beta(mesh, ph, beta).matrix.rows()
    Ao, _, _ = orc.assemble(mesh, ph.wave_number, beta)
    assert entry_err(Ap, Ao)[0] < ENTRY_TOL
    mesh = generate_icosphere_mesh(0.1, 2)
    mesh.is_eval[::7] = 1
    mesh.dof[mesh.is_eval == 0] = np.arange(mesh.num_dofs, dtype=np.uint32)
    Ae = bem.build_tbem_system_with_beta(mesh, ph, beta).matrix.rows()
    Ao, _, _ = orc.assemble(mesh, ph.wave_number, beta)
    assert Ae.shape == (mesh.num_dofs, mesh.num_dofs) and entry_err(Ae, Ao)[0] < ENTRY_TOL


def test_row_sum_correction(bem, orc):
    mesh = generate_icosphere_mesh(0.1, 2)
    ph = PhysicsParams.from_wave_number(2.0)
    system, avg = bem.build_tbem_system_corrected(mesh, ph)
    Ao, _, _ = orc.assemble(mesh, ph.wave_number, ph.burton_miller_beta())
    avg_o = orc.row_sum_correction(Ao)
    assert abs(avg - avg_o) < 1e-12
    assert entry_err(system.matrix.rows(), Ao)[1] < ENTRY_TOL
    assert np.abs(system.matrix.rows().sum(axis=1)).max() < 1e-11


def test_invalid_inputs_fail_loudly(bem):
    from math_audio_b200._capi import Bemb200Error

    mesh = generate_icosphere_mesh(0.1, 1)
    ph = PhysicsParams.from_wave_number(5.0)
    mesh.dof[3] = mesh.dof[4]
    with pytest.raises(Bemb200Error) as ei:
        bem.build_tbem_system(mesh, ph)
    assert ei.value.code == -1 and "permutation" in str(ei.value)
    mesh = generate_icosphere_mesh(0.1, 1)
    mesh.conn[0, 0] = 10_000
    with pytest.raises(Bemb200Error):
        bem.build_tbem_system(mesh, ph)
    mesh = generate_icosphere_mesh(0.1, 1)
    with pytest.raises(Bemb200Error):
        bem.build_tbem_system_with_beta(mesh, ph, 1j, rows=(10, 200))
    op = bem.DenseOperator(np.eye(4, dtype=np.complex128))
    with pytest.raises(ValueError):
        op.apply(np.zeros(5, dtype=np.complex128))  # the reference panics on shape mismatch
    with pytest.raises(ValueError):
        bem.gmres(op, np.zeros(3, dtype=np.complex128), bem.GmresConfig())
    with pytest.raises(Bemb200Error):  # gmres needs a square operator
        bem.gmres(bem.DenseOperator(np.ones((3, 5), dtype=np.complex128)), np.ones(3, dtype=np.complex128), bem.GmresConfig())


# ---- operator + GMRES: the reference's own tests through the GPU operator ----------------------
def tridiag(n, d, lo, up):
    A = np.zeros((n, n), dtype=np.complex128)
    for i in range(n):
        A[i, i] = d
        if i > 0:
            A[i, i - 1] = lo
        if i < n - 1:
            A[i, i + 1] = up
    return A


def test_dense_operator_apply(bem):
    rng = np.random.default_rng(1234)
    for shape in [(1, 1), (3, 5), (257, 300), (1000, 513), (2048, 2048)]:
        A = rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
        op = bem.DenseOperator(A)
        assert (op.num_rows(), op.num_cols()) == shape and op.is_square() == (shape[0] == shape[1])
        x = rng.standard_normal(shape[1]) + 1j * rng.standard_normal(shape[1])
        xt = rng.standard_normal(shape[0]) + 1j * rng.standard_normal(shape[0])
        for got, ref in [(op.apply(x), A @ x), (op.apply_transpose(xt), A.T @ xt), (op.apply_hermitian(xt), A.conj().T @ xt)]:
            assert np.linalg.norm(got - ref) <= 1e-13 * np.linalg.norm(ref) + 1e-300
        # linearity and determinism
        assert (op.apply(x) == op.apply(x)).all()
        assert np.linalg.norm(op.apply(2.5 * x) - 2.5 * op.apply(x)) <= 1e-13 * np.linalg.norm(A @ x) + 1e-300


def test_gmres_reference_kats(bem, orc):
    A = np.array([[4.0, 1.0], [1.0, 3.0]], dtype=np.complex128)        # gmres.rs:631-655
    b = np.array([1.0, 2.0], dtype=np.complex128)
    sol = bem.gmres(bem.DenseOperator(A), b, bem.GmresConfig(100, 10, 1e-10))
    assert sol.converged and np.linalg.norm(A @ sol.x - b) < 1e-8
    n = 5                                                               # gmres.rs:657-680
    b = np.arange(1, n + 1, dtype=np.complex128)
    sol = bem.gmres(bem.DenseOperator(np.eye(n, dtype=np.complex128)), b, bem.GmresConfig(10, 10, 1e-12))
    assert sol.converged and sol.iterations <= 2 and np.linalg.norm(sol.x - b) < 1e-10
    sol = bem.gmres(bem.DenseOperator(np.eye(3, dtype=np.complex128)), np.zeros(3, dtype=np.complex128), bem.GmresConfig())
    assert (sol.iterations, sol.restarts, sol.residual, sol.converged) == (0, 0, 0.0, True) and (sol.x == 0).all()
    n = 20                                                              # test_fmm_validation.rs:537-585
    A = tridiag(n, 10.0, complex(-1.0, 0.1), complex(-1.0, -0.1))
    b = np.array([math.sin(i * 0.3) for i in range(n)], dtype=np.complex128)
    sol = bem.solve_gmres(bem.DenseOperator(A), b, bem.GmresConfig(50, 15, 1e-10))
    xo, io = orc.gmres(A, b, max_iterations=50, restart=15, tolerance=1e-10)
    assert sol.converged and (sol.iterations, sol.restarts) == (io["iterations"], io["restarts"])
    assert np.linalg.norm(A @ sol.x - b) / np.linalg.norm(b) < 1e-8 and np.linalg.norm(sol.x - xo) < 1e-12
    n = 50                                                              # test_fmm_validation.rs:640-700
    A = tridiag(n, 4.0, -1.0, -1.0)
    b = np.ones(n, dtype=np.complex128)
    small = bem.gmres(bem.DenseOperator(A), b, bem.GmresConfig(100, 5, 1e-10))
    large = bem.gmres(bem.DenseOperator(A), b, bem.GmresConfig(100, 50, 1e-10))
    xs, osm = orc.gmres(A, b, max_iterations=100, restart=5, tolerance=1e-10)
    assert small.converged and large.converged and large.restarts <= small.restarts
    assert (small.iterations, small.restarts) == (osm["iterations"], osm["restarts"])
    assert np.linalg.norm(small.x - xs) / np.linalg.norm(xs) < 1e-10
    # budget exhausted: converged = false and the TRUE residual is reported (gmres.rs:264-276)
    sol = bem.gmres(bem.DenseOperator(A), b, bem.GmresConfig(1, 3, 1e-14))
    assert (not sol.converged) and sol.restarts == 1 and sol.iterations == 3
    assert abs(sol.residual - np.linalg.norm(b - A @ sol.x) / np.linalg.norm(b)) < 1e-12
    # initial guess (gmres_with_guess): starting from the solution converges in 0 iterations
    xl = np.linalg.solve(A, b)
    sol = bem.gmres_with_guess(bem.DenseOperator(A), b, xl, bem.GmresConfig(10, 10, 1e-10))
    assert sol.converged and sol.iterations == 0


def test_incident_rhs_and_field_evaluation_on_device(bem, orc):
    """SURVEY 8f ranks 1-2: IncidentField::compute_rhs_with_beta and compute_scattered_field."""
    from math_audio_b200.incident import IncidentField
    from math_audio_b200.mesh import fibonacci_directions

    a = 0.1
    ph = PhysicsParams.from_wave_number(25.0)
    beta = ph.burton_miller_beta_scaled(4.0)
    for mesh in (generate_icosphere_mesh(a, 3), generate_box_mesh_quad(0.3, 0.4, 0.5, 6, 8, 10)):
        st = bem.StagedMesh(mesh)
        n = mesh.n_elem
        for inc, kind, vec in [(IncidentField.plane_wave_z(), 0, [0, 0, 1.0]), (IncidentField.plane_wave([0.6, 0.0, 0.8]), 0, [0.6, 0.0, 0.8]),
                               (IncidentField.point_source([0.7, -0.2, 0.4]), 1, [0.7, -0.2, 0.4])]:
            got = bem.incident_rhs_device(st, ph, beta, inc)
            ref, _ = orc.incident_rhs(kind, vec, 1.0, mesh.center, mesh.normal, ph.wave_number, beta)
            assert np.max(np.abs(got - ref)) / np.max(np.abs(ref)) < 1e-13
        multi = IncidentField(plane_waves=[(d, 0.5 + 0.1j) for d in fibonacci_directions(5)])
        ref = sum(orc.incident_rhs(0, d, 0.5 + 0.1j, mesh.center, mesh.normal, ph.wave_number, beta)[0] for d in fibonacci_directions(5))
        assert np.max(np.abs(bem.incident_rhs_device(st, ph, beta, multi) - ref)) / np.max(np.abs(ref)) < 1e-13
        rng = np.random.default_rng(8)
        p = rng.standard_normal(n) + 1j * rng.standard_normal(n)
        v = rng.standard_normal(n) + 1j * rng.standard_normal(n)
        v[::3] = 0.0
        pts = rng.standard_normal((97, 3))
        pts *= (3.0 * a / np.linalg.norm(pts, axis=1))[:, None] * (1.0 + rng.random(97))[:, None]
        for vel in (None, v):
            got = bem.compute_scattered_field(pts, st, p, vel, ph)
            ref = orc.scattered_field(mesh, pts, p, ph.wave_number, surface_velocity=vel)
            assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 1e-12
        # compute_rcs (pressure.rs:438-478): 32 directions in one launch, and the scalar form
        dirs = np.array(fibonacci_directions(32))
        ref = orc.compute_rcs(mesh, p, dirs, ph.wave_number)
        got = bem.compute_rcs(p, st, dirs, ph)
        assert got.shape == (32,) and np.max(np.abs(got - ref) / ref) < 1e-11
        assert abs(bem.compute_rcs(p, st, dirs[3], ph) - ref[3]) / ref[3] < 1e-11


def test_sweep_driver_equals_sequential(bem):
    """The pipelined frequency sweep (assembly of f+1 on a second stream underneath the solve of f,
    persistent 'background' far kernel) must give the results of the plain sequential calls."""
    from math_audio_b200.incident import IncidentField
    from math_audio_b200.sweep import SweepDriver

    a = 0.1
    mesh = generate_icosphere_mesh(a, 3)
    inc = IncidentField.plane_wave_z()
    cfg = bem.GmresConfig(max_iterations=1000, restart=50, tolerance=1e-10)
    cases = []
    for ka in (0.3, 1.0, 2.5, 6.0, 0.7):
        ph = PhysicsParams.from_wave_number(ka / a)
        cases.append((ph, ph.burton_miller_beta_adaptive(a)[0]))
    ref = []
    for ph, beta in cases:
        system = bem.build_tbem_system_with_beta(mesh, ph, beta)
        b = system.rhs + inc.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
        ref.append((system.matrix.rows(), bem.gmres(bem.DenseOperator(system), b, cfg)))
    for overlap in (True, False):
        driver = SweepDriver(mesh, overlap=overlap, background_blocks_per_sm=1)

        def solve(i, system, op):
            ph, beta = cases[i]
            b = system.rhs_full() + inc.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
            return system.matrix.rows(), bem.gmres(op, b, cfg)

        out = driver.run(cases, cfg, solve)
        for (A0, s0), (A1, s1) in zip(ref, out):
            assert (A0 == A1).all()  # same kernels, same bits (the background grid only changes the schedule)
            assert (s0.iterations, s0.restarts) == (s1.iterations, s1.restarts) and (s0.x == s1.x).all()


def test_boosted_background_assembly_same_bits(bem):
    """bemb200_matrix_boost_assembly: a second launch of the far kernel on another stream joins a
    background assembly (both pull work items from one device counter).  Whatever the split between
    the polite grid and the helper blocks, the matrix must come out bit-identical to the foreground
    assembly (every entry is written by exactly one work item)."""
    import threading
    import time

    a = 0.1
    mesh = generate_icosphere_mesh(a, 4)  # 5 120 elements: 40 column tiles, enough items for a persistent grid
    ph = PhysicsParams.from_wave_number(3.0 / a)
    beta = ph.burton_miller_beta_adaptive(a)[0]
    ph2 = PhysicsParams.from_wave_number(0.7 / a)
    ctx_a, ctx_b = bem.Context(0), bem.Context(0)
    staged = bem.StagedMesh(mesh, ctx_a)
    system = bem.build_tbem_system_with_beta(staged, ph, beta, ctx=ctx_a)
    A0, rhs0 = system.matrix.rows(), system.rhs.copy()
    near0 = system.matrix.assembly_stats()["near_pairs"]
    for trial in range(3):
        ctx_a.set_background(0)
        bem.build_tbem_system_with_beta(staged, ph2, ph2.burton_miller_beta(), ctx=ctx_a, reuse=system)  # overwrite
        ctx_a.set_background(1)
        err = []

        def work():
            try:
                bem.build_tbem_system_with_beta(staged, ph, beta, ctx=ctx_a, reuse=system, fetch_rhs=False)
            except Exception as e:
                err.append(e)

        t = threading.Thread(target=work)
        t.start()
        time.sleep(0.002 * trial)
        while t.is_alive():
            system.matrix.boost_assembly(ctx_b)  # no-op until the far pass is in flight, and after the first boost
            time.sleep(0.0005)
        t.join()
        assert not err, err
        assert system.matrix.assembly_stats()["near_pairs"] == near0
        assert (system.matrix.rows() == A0).all()
        assert (system.matrix.rhs() == rhs0).all()
    ctx_a.set_background(0)


def test_gmres_preconditioned(bem, orc):
    """gmres_preconditioned (gmres.rs:282-585) with the identity and the Jacobi preconditioner on an
    assembled BEM matrix and on the reference's tridiagonal KAT."""
    from math_audio_b200.incident import IncidentField

    a = 0.1
    mesh = generate_icosphere_mesh(a, 3)
    ph = PhysicsParams.from_wave_number(3.0 / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    system = bem.build_tbem_system_with_beta(mesh, ph, beta)
    A = system.matrix.rows()
    b = system.rhs + IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
    op = bem.DenseOperator(system)
    cfg = bem.GmresConfig(max_iterations=100, restart=20, tolerance=1e-10)
    jac = bem.DiagonalPreconditioner.from_operator(op)
    assert np.max(np.abs(jac.inv_diag - orc.inverse_diagonal(np.diag(A)))) < 1e-13 * np.abs(jac.inv_diag).max()
    for pre, idg in [(bem.IdentityPreconditioner(), None), (jac, jac.inv_diag)]:
        sol = bem.gmres_preconditioned(op, pre, b, cfg)
        xo, io = orc.gmres_preconditioned(A, b, inv_diag=idg, max_iterations=100, restart=20, tolerance=1e-10)
        assert sol.converged and (sol.iterations, sol.restarts) == (io["iterations"], io["restarts"])
        assert abs(sol.residual - io["residual"]) < 1e-3 * io["residual"] + 1e-14
        assert np.linalg.norm(sol.x - xo) / np.linalg.norm(xo) < X_TOL
        assert np.linalg.norm(b - A @ sol.x) / np.linalg.norm(b) < 1e-8
    # initial guess + budget exhaustion report the PRECONDITIONED true residual
    sol = bem.gmres_preconditioned_with_guess(op, jac, b, np.ones_like(b), bem.GmresConfig(1, 4, 1e-14))
    xo, io = orc.gmres_preconditioned(A, b, inv_diag=jac.inv_diag, x0=np.ones_like(b), max_iterations=1, restart=4, tolerance=1e-14)
    assert not sol.converged and sol.iterations == io["iterations"] == 4
    assert abs(sol.residual - io["residual"]) < 1e-9 * io["residual"]
    n = 30  # test_fmm_validation.rs:587-637 matrix with Jacobi instead of ILU
    T = tridiag(n, complex(5.0, 0.5), complex(-2.0, 0.2), complex(-2.0, -0.2))
    for i in range(n - 3):
        T[i, i + 3] = 0.5
    bb = np.array([math.sin(i * 0.2) + 0.5 + 0.1j for i in range(n)], dtype=np.complex128)
    opT = bem.DenseOperator(T)
    sol = bem.gmres_preconditioned(opT, bem.DiagonalPreconditioner.from_operator(opT), bb, bem.GmresConfig(100, 20, 1e-8))
    assert sol.converged and np.linalg.norm(T @ sol.x - bb) / np.linalg.norm(bb) < 1e-5


def test_block_jacobi_schwarz_preconditioner(bem, orc):
    """AdditiveSchwarzPreconditioner (math-solvers/src/preconditioners/schwarz.rs) built on the device from the assembled
    operator: block-Jacobi on the reference's contiguous partition, explicit overlapping subdomains with the reference's
    weights, left-preconditioned GMRES (gmres.rs:282-585) -- against oracle/schwarz_oracle.py and the oracle's GMRES."""
    from math_audio_b200.incident import IncidentField
    from oracle import schwarz_oracle as so

    a = 0.1
    mesh = generate_icosphere_mesh(a, 3)
    ph = PhysicsParams.from_wave_number(8.0 / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    system = bem.build_tbem_system_with_beta(mesh, ph, beta)
    A = system.matrix.rows()
    n = A.shape[0]
    b = system.rhs + IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
    op = bem.DenseOperator(system)
    rng = np.random.default_rng(5)
    r = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    cfg = bem.GmresConfig(max_iterations=100, restart=50, tolerance=1e-10)
    plain = bem.gmres(op, b, cfg)
    for S in (10, 7, 20):  # blocks of 128, uneven blocks (183 / 182), blocks of 64 = one level-2 parent triangle each
        pre = bem.AdditiveSchwarzPreconditioner.from_operator(op, S)
        ds = so.DenseSchwarz(A, S)
        st = pre.stats()
        ns, mn, mx, avg = ds.stats()
        assert (st["num_subdomains"], st["min_size"], st["max_size"]) == (ns, mn, mx) and abs(st["avg_size"] - avg) < 1e-12
        assert st["disjoint"] == 1 and st["inverse_bytes"] == 16 * sum(len(s) ** 2 for s in ds.subs)
        z, zo = pre.apply(r), ds.apply(r)
        assert np.linalg.norm(z - zo) / np.linalg.norm(zo) < 1e-12
        sol = bem.gmres_preconditioned(op, pre, b, cfg)
        xo, io = orc.gmres_preconditioned_cb(lambda v: A @ v, ds.apply, n, b, max_iterations=100, restart=50, tolerance=1e-10)
        assert sol.converged and (sol.iterations, sol.restarts) == (io["iterations"], io["restarts"])
        assert abs(sol.residual - io["residual"]) < 1e-3 * io["residual"] + 1e-14
        assert np.linalg.norm(sol.x - xo) / np.linalg.norm(xo) < X_TOL
        assert np.linalg.norm(b - A @ sol.x) / np.linalg.norm(b) < 1e-8
        if S == 20:  # compact near-field patches do precondition the Burton-Miller operator (measured 47 against 80); blocks
            assert sol.iterations < 0.7 * plain.iterations  # of 128 at this k h (two patches each) make it worse -- parity only
        pre.close()
    # the committed fixture of the LINE-BY-LINE restatement of schwarz.rs on the ico1 golden system (tests/golden/make_golden_schwarz.py)
    g1, f1 = np.load(GOLD / "ico1_ka0p5.npz"), np.load(GOLD / "schwarz_ico1.npz")
    op1 = bem.DenseOperator(g1["A"])
    for S in (4, 7):
        pre1 = bem.AdditiveSchwarzPreconditioner.from_operator(op1, S)
        assert np.max(np.abs(pre1.apply(f1["r"]) - f1[f"z_S{S}"])) < 1e-13 * np.max(np.abs(f1[f"z_S{S}"]))
        s1 = bem.gmres_preconditioned(op1, pre1, g1["b"], bem.GmresConfig(100, 20, 1e-10))
        assert [s1.iterations, s1.restarts, int(s1.converged)] == list(f1[f"info_S{S}"])
        assert np.linalg.norm(s1.x - f1[f"x_S{S}"]) / np.linalg.norm(s1.x) < X_TOL
        pre1.close()
    # overlapping subdomains: the contiguous blocks grown by one layer of mesh neighbours (elements within 1.6 edge lengths),
    # exactly what extend_partition does with a sparsity pattern (schwarz.rs:177-203); weights 1 / multiplicity
    d = np.linalg.norm(mesh.center[:, None, :] - mesh.center[None, :, :], axis=2)
    h = np.sort(d, axis=1)[:, 1].mean()
    adj = [list(np.nonzero((d[i] < 1.6 * h) & (np.arange(n) != i))[0]) for i in range(n)]
    pre = bem.AdditiveSchwarzPreconditioner.from_operator(op, 10, overlap=1, adjacency=adj)
    subs = [so.extend_partition(p, adj, 1, n) for p in so.contiguous_partition(n, 10)]
    ds = so.DenseSchwarz(A, subdomains=subs)
    assert pre.stats()["disjoint"] == 0 and pre.stats()["max_size"] == max(len(s) for s in subs) > 128
    z, zo = pre.apply(r), ds.apply(r)
    assert np.linalg.norm(z - zo) / np.linalg.norm(zo) < 1e-12
    sol = bem.gmres_preconditioned(op, pre, b, cfg)
    xo, io = orc.gmres_preconditioned_cb(lambda v: A @ v, ds.apply, n, b, max_iterations=100, restart=50, tolerance=1e-10)
    assert sol.converged and sol.iterations == io["iterations"] and np.linalg.norm(sol.x - xo) / np.linalg.norm(xo) < X_TOL
    pre.close()
    # initial guess + exhausted budget: the preconditioned true residual is reported (gmres.rs:574-584)
    pre = bem.AdditiveSchwarzPreconditioner.from_operator(op, 10)
    ds = so.DenseSchwarz(A, 10)
    sol = bem.gmres_preconditioned_with_guess(op, pre, b, np.ones_like(b), bem.GmresConfig(1, 4, 1e-14))
    xo, io = orc.gmres_preconditioned_cb(lambda v: A @ v, ds.apply, n, b, x0=np.ones_like(b), max_iterations=1, restart=4, tolerance=1e-14)
    assert not sol.converged and sol.iterations == io["iterations"] == 4 and abs(sol.residual - io["residual"]) < 1e-9 * io["residual"]
    pre.close()
    # the reference's own test matrix (schwarz.rs:468-492) as a DENSE operator: 4 subdomains, GMRES(20) to 1e-8 converges
    T = np.zeros((20, 20), dtype=np.complex128)
    for i in range(20):
        T[i, i] = 4.0
        if i > 0:
            T[i, i - 1] = -1.0
        if i < 19:
            T[i, i + 1] = -1.0
        if i >= 5:
            T[i, i - 5] = -0.5
        if i < 15:
            T[i, i + 5] = -0.5
    bb = np.array([math.sin(i) for i in range(20)], dtype=np.complex128)
    opT = bem.DenseOperator(T)
    preT = bem.AdditiveSchwarzPreconditioner.from_operator(opT, 4)
    dsT = so.DenseSchwarz(T, 4)
    assert np.max(np.abs(preT.apply(bb) - dsT.apply(bb))) < 1e-14 and np.all(np.abs(preT.apply(bb)) < 100.0)
    sol = bem.gmres_preconditioned(opT, preT, bb, bem.GmresConfig(100, 20, 1e-8))
    xo, io = orc.gmres_preconditioned_cb(lambda v: T @ v, dsT.apply, 20, bb, max_iterations=100, restart=20, tolerance=1e-8)
    assert sol.converged and sol.iterations == io["iterations"] and np.linalg.norm(T @ sol.x - bb) / np.linalg.norm(bb) < 1e-7
    # a zero pivot is skipped, not divided by (schwarz.rs:283-285, :374-377)
    Z = np.array([[0.0, 2.0, 0.0], [3.0, 4.0, 1.0], [1.0, 0.0, 5.0]], dtype=np.complex128)
    rz = np.array([1.0, 2.0, 3.0], dtype=np.complex128)
    preZ = bem.AdditiveSchwarzPreconditioner.from_operator(bem.DenseOperator(Z), 1)
    assert np.max(np.abs(preZ.apply(rz) - so.DenseSchwarz(Z, 1).apply(rz))) < 1e-14
    # invalid subdomains fail loudly
    for bad in ([np.array([0, 1, 1], dtype=np.uint64)], [np.array([0, 25], dtype=np.uint64)]):
        with pytest.raises(Exception):
            bem.AdditiveSchwarzPreconditioner.from_operator(opT, subdomains=bad)
    with pytest.raises(Exception):
        bem.gmres_preconditioned(op, preT, b, cfg)  # built for another operator


def test_block_matvec_and_batched_gmres(bem, orc):
    """BASELINE config 5 at test size: several incident directions, reference semantics = one
    independent gmres() per right-hand side; the device runs them in lockstep on the FP64
    tensor-core block matvec."""
    from math_audio_b200.incident import IncidentField
    from math_audio_b200.mesh import fibonacci_directions

    rng = np.random.default_rng(11)
    for shape, nrhs in [((300, 257), 5), ((1024, 1024), 32), ((77, 1000), 16)]:
        A = rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
        X = rng.standard_normal((nrhs, shape[1])) + 1j * rng.standard_normal((nrhs, shape[1]))
        Y, ms = bem.apply_block(bem.DenseOperator(A), X)
        ref = X @ A.T
        assert np.linalg.norm(Y - ref) < 1e-13 * np.linalg.norm(ref) and ms > 0
    a = 0.1
    mesh = generate_icosphere_mesh(a, 3)
    ph = PhysicsParams.from_wave_number(2.0 / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    system = bem.build_tbem_system_with_beta(mesh, ph, beta)
    A = system.matrix.rows()
    op = bem.DenseOperator(system)
    cfg = bem.GmresConfig(max_iterations=1000, restart=20, tolerance=1e-10)
    for nrhs in (11, 32):
        dirs = fibonacci_directions(nrhs)
        B = np.stack([system.rhs + IncidentField.plane_wave(d).compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta) for d in dirs])
        if nrhs == 11:
            B[3] = 0.0  # a zero right-hand side returns at once (gmres.rs:125-135)
        sols, st = bem.gmres_batched(op, B, cfg)
        assert st["block_matvecs"] > 0 and len(sols) == nrhs
        for i, sol in enumerate(sols):
            xo, io = orc.gmres(A, B[i], max_iterations=1000, restart=20, tolerance=1e-10)
            assert sol.converged == io["converged"]
            assert (sol.iterations, sol.restarts) == (io["iterations"], io["restarts"]), (i, sol.iterations, io)
            if np.abs(B[i]).max() == 0:
                assert sol.iterations == 0 and (sol.x == 0).all()
                continue
            assert np.linalg.norm(sol.x - xo) / np.linalg.norm(xo) < X_TOL
            assert np.linalg.norm(B[i] - A @ sol.x) / np.linalg.norm(B[i]) < 2e-10
    # the same batch through gmres_preconditioned with block-Jacobi (20 blocks of 64): per right-hand side what the single call gives
    pre = bem.AdditiveSchwarzPreconditioner.from_operator(op, 20)
    solp, _ = bem.gmres_batched(op, B, cfg, precond=pre)
    for i in (0, 7, 31):
        one = bem.gmres_preconditioned(op, pre, B[i], cfg)
        assert solp[i].converged and (solp[i].iterations, solp[i].restarts) == (one.iterations, one.restarts)
        assert np.linalg.norm(solp[i].x - one.x) / np.linalg.norm(one.x) < 1e-9
        assert np.linalg.norm(solp[i].x - sols[i].x) / np.linalg.norm(sols[i].x) < X_TOL and solp[i].iterations < sols[i].iterations
    pre.close()
    # budget exhaustion: converged = false, true residual (per right-hand side)
    sols, _ = bem.gmres_batched(op, B[:8], bem.GmresConfig(max_iterations=1, restart=5, tolerance=1e-14))
    for i, sol in enumerate(sols):
        assert (not sol.converged) and sol.iterations == 5 and sol.restarts == 1
        assert abs(sol.residual - np.linalg.norm(B[i] - A @ sol.x) / np.linalg.norm(B[i])) < 1e-10


def test_batched_gmres_beyond_32768_unknowns(bem):
    """33 620 unknowns (geodesic sphere, nu = 41): the batched Gram-Schmidt step keeps its slice of w in shared memory
    instead of registers.  No oracle at this size: the batched solve must reproduce independent single-right-hand-side
    device solves (which the oracle pins at small sizes) -- iteration / restart counts, solutions, true residuals."""
    from math_audio_b200.incident import IncidentField
    from math_audio_b200.mesh import fibonacci_directions, generate_geodesic_sphere_mesh

    a = 0.1
    mesh = generate_geodesic_sphere_mesh(a, 41)
    n = mesh.num_dofs
    assert n == 33620
    ph = PhysicsParams.from_wave_number(3.0 / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    system = bem.build_tbem_system_with_beta(mesh, ph, beta, fetch_rhs=False)
    op = bem.DenseOperator(system)
    cfg = bem.GmresConfig(max_iterations=1000, restart=30, tolerance=1e-10)
    B = np.stack([IncidentField.plane_wave(d).compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta) for d in fibonacci_directions(5)])
    sols, st = bem.gmres_batched(op, B, cfg)
    assert st["block_matvecs"] > 0
    X = np.stack([s.x for s in sols])
    R, _ = bem.apply_block(op, X)
    for i, sol in enumerate(sols):
        single = bem.gmres(op, B[i], cfg)
        assert sol.converged and single.converged
        assert (sol.iterations, sol.restarts) == (single.iterations, single.restarts) and sol.restarts >= 1
        assert np.linalg.norm(sol.x - single.x) / np.linalg.norm(single.x) < 1e-9
        assert np.linalg.norm(B[i] - R[i]) / np.linalg.norm(B[i]) < 2e-10
    system.matrix.close()


# ---- full benchmark size: size-independent properties ---------------------------------------------
@pytest.fixture(scope="module")
def big(bem):
    a = 0.1
    mesh = generate_icosphere_mesh(a, 5)  # 20 480 elements: BASELINE.json configs[1]
    st = bem.StagedMesh(mesh)
    return a, mesh, st


@pytest.mark.parametrize("ka", [0.25, 2.0, 8.0])
def test_config2_sampled_rows_and_solve(bem, orc, big, ka):
    from math_audio_b200.incident import IncidentField

    a, mesh, st = big
    n = mesh.n_elem
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    system = bem.build_tbem_system_with_beta(st, ph, beta)
    # >= 64 sampled rows incl. the first/last, icosahedron-vertex neighbourhoods and random rows
    rng = np.random.default_rng(99)
    rows = sorted(set([0, 1, 2, 3, 4, n - 1, n - 2] + list(rng.integers(0, n, 57))))
    assert len(rows) >= 60
    worst = 0.0
    for r in rows:
        Ar = system.matrix.rows(r, r + 1)
        Ao, _, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=r, row_end=r + 1)
        worst = max(worst, *entry_err(Ar, Ao))
    assert worst < ENTRY_TOL, worst
    st_a = system.matrix.assembly_stats()
    assert 20 * n < st_a["near_pairs"] < 40 * n  # ~28 near pairs per row (SURVEY section 6)
    op = bem.DenseOperator(system)
    b = system.rhs + IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
    sol = bem.gmres(op, b, bem.GmresConfig(max_iterations=1000, restart=50, tolerance=1e-10))
    assert sol.converged and sol.residual < 1e-10
    # independent residual through the operator boundary + linearity of the operator
    res = np.linalg.norm(b - op.apply(sol.x)) / np.linalg.norm(b)
    assert res < 2e-10
    x2 = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    y1, y2 = op.apply(sol.x), op.apply(x2)
    assert np.linalg.norm(op.apply(sol.x + 3.0 * x2) - (y1 + 3.0 * y2)) < 1e-12 * np.linalg.norm(y1 + 3.0 * y2)
    # sampled-row matvec parity against the oracle rows
    for r in rows[:8]:
        Ao, _, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=r, row_end=r + 1)
        assert abs(y2[r] - (Ao @ x2)[0]) < 1e-12 * np.linalg.norm(Ao) * np.linalg.norm(x2)
    # full x parity against the committed oracle solution (LAPACK LU of the oracle's matrix, SURVEY 8d row 2) and the
    # oracle's GMRES iteration / restart counts at this size (tests/golden/make_golden_large.py config2)
    tag = f"{ka:g}".replace(".", "p")
    gold = np.load(Path(__file__).resolve().parent / "golden" / f"config2_x_ka{tag}.npz")
    assert np.linalg.norm(sol.x - gold["x"]) / np.linalg.norm(gold["x"]) < X_TOL
    assert sol.iterations == int(gold["iterations"]) and sol.restarts == int(gold["restarts"])
    if ka < 0.5:
        # +K' branch: closed-surface row sums = -1/2 + K'[1] + beta E[1] ~ -1 (tbem.rs:487-493); the
        # beta E[1] quadrature residue is O(0.1) here, exactly as in the oracle
        ones = op.apply(np.ones(n, dtype=np.complex128))
        assert np.abs(ones.real + 1.0).max() < 0.05 and np.abs(ones + 1.0).max() < 0.2


def test_bench_dump_outputs_are_the_last_timed_step(orc, tmp_path):
    """bench.py --dump-outputs: float64 arrays within 64 MB holding what the last timed step computed -- the sampled rows of its
    matrix and its GMRES solution agree with the oracle's assembly and solve of that frequency."""
    import json
    import os
    import subprocess
    import sys

    from math_audio_b200.incident import IncidentField

    root = Path(__file__).resolve().parent.parent
    steps, warmup = 2, 3
    p = subprocess.run([sys.executable, str(root / "bench.py"), "--workload", "sphere1k", "--steps", str(steps), "--warmup", str(warmup),
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, env=dict(os.environ, BENCH_NO_CONFIG5="1"), timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    assert json.loads(p.stdout)["steps"] == steps
    files = sorted(tmp_path.glob("*.npy"))
    assert {f.stem for f in files} == {"x", "gmres", "matrix_rows", "matrix_row_index"}
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    d = {f.stem: np.load(f) for f in files}
    assert all(a.dtype == np.float64 for a in d.values())
    if str(root) not in sys.path:
        sys.path.insert(0, str(root))
    import bench

    wl = bench.workload("sphere1k")
    mesh = wl["mesh"]
    _, ph, beta = bench.physics_for(wl, warmup + steps - 1)
    Ao, _, _ = orc.assemble(mesh, ph.wave_number, beta)
    rows = d["matrix_row_index"].astype(np.int64)
    assert len(rows) == mesh.num_dofs and (np.diff(rows) > 0).all()  # this small matrix fits the sample whole
    A = d["matrix_rows"][..., 0] + 1j * d["matrix_rows"][..., 1]
    assert max(entry_err(A, Ao[rows])) < ENTRY_TOL
    b = IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
    xo, _ = orc.gmres(Ao, b, max_iterations=1000, restart=50, tolerance=1e-10)
    x = d["x"][:, 0] + 1j * d["x"][:, 1]
    assert np.linalg.norm(x - xo) / np.linalg.norm(xo) < X_TOL
    _, _, residual, converged = d["gmres"]
    assert converged == 1.0 and residual < 1e-10
