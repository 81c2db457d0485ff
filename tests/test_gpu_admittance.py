"""Admittance boundaries and the sign-consistent formulation on the device (DESIGN.md 4.8): every matrix entry against the
CPU oracle of ``bemb200_assemble_staged_opts``, the bits of the assembly without options, row slabs, the sweep, and the
end-to-end solve against the exact Robin series of the sphere."""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import admittance_oracle as ao  # noqa: E402

from math_audio_b200.mesh import BC_PRESSURE, generate_box_mesh_quad, generate_icosphere_mesh, mesh_from_data  # noqa: E402
from math_audio_b200.types import PhysicsParams  # noqa: E402

pytestmark = pytest.mark.gpu
ENTRY_TOL = 1e-10
ROW_TOL = 1e-13


@pytest.fixture(scope="module")
def bem():
    from math_audio_b200 import bem as b

    b.default_context()
    return b


def entry_err(A, Aref):
    scale = np.max(np.abs(Aref), axis=1, keepdims=True)
    rownorm = np.max(np.abs(A - Aref) / scale)
    big = np.abs(Aref) > 1e-9 * scale
    return np.max(np.abs(A - Aref)[big] / np.abs(Aref)[big]), rownorm


def mixed_admittance(mesh, k, seed, frac=0.5):
    """Passive Y on a random subset of the velocity-BC boundary elements (enumeration order), 0 elsewhere."""
    rng = np.random.default_rng(seed)
    vel = np.flatnonzero(np.asarray(mesh.bc_type)[np.asarray(mesh.is_eval) == 0] == 0)
    y = np.zeros(int((np.asarray(mesh.is_eval) == 0).sum()), dtype=np.complex128)
    pick = rng.permutation(vel)[: max(1, int(frac * vel.size))]
    y[pick] = k * (rng.uniform(0.05, 0.6, pick.size) - 1j * rng.uniform(0.05, 0.6, pick.size))
    return y


def check_against_oracle(bem, mesh, ph, beta, opts):
    system = bem.build_tbem_system_with_beta(mesh, ph, beta, options=opts)
    e2d = bem.enumeration_to_dof(mesh)
    y = None if opts.admittance is None else bem.surface_values_in_dof_order(e2d, np.asarray(opts.admittance, dtype=np.complex128))
    Ao, rhso, _ = ao.assemble_opts(mesh, ph.wave_number, beta, opts.dg_dn_sign, opts.consistent_beta, y)
    A = system.matrix.rows()
    rel, rown = entry_err(A, Ao)
    assert rel < ENTRY_TOL and rown < ROW_TOL, (rel, rown)
    if np.abs(rhso).max() > 0:
        assert np.max(np.abs(system.rhs - rhso)) / np.max(np.abs(rhso)) < ENTRY_TOL
    return system, A


@pytest.mark.parametrize("sub", [2, 3])
@pytest.mark.parametrize("ka,sign", [(0.3, 0), (0.3, -1), (2.0, 0), (2.0, 1)])
def test_sphere_entries_mixed_admittance(bem, sub, ka, sign):
    a = 0.1
    mesh = generate_icosphere_mesh(a, sub)
    # a prescribed velocity on a few elements, some of them absorbing too: the v-bar right-hand side with both betas
    mesh.bc_len[:8] = 3
    mesh.bc_val[:8, :3] = 0.4 + 0.1j
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    y = mixed_admittance(mesh, ph.wave_number, sub)
    for consistent in (False, True):
        system, A = check_against_oracle(bem, mesh, ph, beta, bem.AssemblyOptions(sign, consistent, y))
        st = system.matrix.assembly_stats()
        assert st["near_pairs"] > 0


def test_quad_box_patch_and_warped_quads(bem):
    box = generate_box_mesh_quad(0.32, 0.44, 0.64, 4, 6, 8)
    patch = (np.abs(box.center[:, 1] + 0.22) < 1e-9) & (np.hypot(box.center[:, 0], box.center[:, 2]) < 0.15)
    ph = PhysicsParams.new(900.0, 343.0, 1.21, False)
    beta = ph.burton_miller_beta_scaled(4.0)
    y = np.where(patch, (0.4 - 0.7j) * ph.wave_number, 0.0)
    check_against_oracle(bem, box, ph, beta, bem.AssemblyOptions(0, False, y))
    check_against_oracle(bem, box, ph, beta, bem.AssemblyOptions(1, True, y))
    # warped quads: the special (generic) path
    nodes = box.nodes.copy()
    wall = np.abs(nodes[:, 0] - 0.16) < 1e-12
    nodes[wall, 0] += 0.01 * np.sin(17.0 * nodes[wall, 1]) * np.cos(11.0 * nodes[wall, 2])
    warped = mesh_from_data(nodes, box.conn[:, :4])
    on_wall = np.abs(warped.center[:, 0] - 0.16) < 0.02
    y = np.where(on_wall, (0.3 - 0.3j) * ph.wave_number, 0.0)
    system, _ = check_against_oracle(bem, warped, ph, beta, bem.AssemblyOptions(-1, True, y))
    assert system.matrix.assembly_stats()["special_pairs"] > 0


def test_eval_elements_and_permuted_dofs(bem):
    a = 0.1
    mesh = generate_icosphere_mesh(a, 2)
    mesh.is_eval[::7] = 1
    nd = int((mesh.is_eval == 0).sum())
    mesh.dof[mesh.is_eval == 0] = np.random.default_rng(4).permutation(nd).astype(np.uint32)
    mesh.bc_type[np.flatnonzero(mesh.is_eval == 0)[:5]] = BC_PRESSURE
    ph = PhysicsParams.from_wave_number(1.5 / a)
    beta = ph.burton_miller_beta_scaled(4.0)
    y = mixed_admittance(mesh, ph.wave_number, 7)
    assert bem.enumeration_to_dof(mesh) is not None
    check_against_oracle(bem, mesh, ph, beta, bem.AssemblyOptions(1, True, y))


def rhs_equal(r, ref, vbar_near_pairs):
    """TbemSystem.rhs of two assemblies that must compute the same thing.  The near-field kernel adds the prescribed-velocity
    term of each near pair to its row with an atomic add, in the order the far kernel's atomic compaction listed the pairs, so
    with a non-zero velocity the last bits differ between two calls of the plain assembly too; without one it is bit-exact."""
    if not vbar_near_pairs:
        return np.array_equal(r, ref)
    return np.max(np.abs(r - ref)) <= 1e-14 * np.max(np.abs(ref))


@pytest.mark.parametrize("vbar", [False, True])
def test_bits_of_the_plain_assembly_and_row_slabs(bem, vbar):
    a = 0.1
    mesh = generate_icosphere_mesh(a, 3)
    if vbar:  # a prescribed velocity on ten elements: their near pairs reach rhs through atomic adds
        mesh.bc_len[:10] = 3
        mesh.bc_val[:10, :3] = 1.0 - 0.5j
    st = bem.StagedMesh(mesh)
    n = st.num_dofs
    for ka in (0.3, 2.0):
        ph = PhysicsParams.from_wave_number(ka / a)
        beta, _ = ph.burton_miller_beta_adaptive(a)
        plain = bem.build_tbem_system_with_beta(st, ph, beta)
        A0, r0 = plain.matrix.rows(), plain.rhs
        again = bem.build_tbem_system_with_beta(st, ph, beta)
        assert np.array_equal(again.matrix.rows(), A0) and rhs_equal(again.rhs, r0, vbar)
        # NULL-equivalent options (defaults, an all-zero admittance) give the whole matrix bit for bit, and the rhs of the plain call
        for opts in (bem.AssemblyOptions(), bem.AssemblyOptions(admittance=np.zeros(n, dtype=np.complex128))):
            s = bem.build_tbem_system_with_beta(st, ph, beta, options=opts)
            assert np.array_equal(s.matrix.rows(), A0) and rhs_equal(s.rhs, r0, vbar)
        # Y = 0 columns of an admittance assembly keep the bits of the plain one
        y = mixed_admittance(mesh, ph.wave_number, 11, frac=0.1)
        s = bem.build_tbem_system_with_beta(st, ph, beta, options=bem.AssemblyOptions(admittance=y))
        A = s.matrix.rows()
        zero = y == 0
        assert np.array_equal(A[:, zero], A0[:, zero]) and rhs_equal(s.rhs, r0, vbar)
        assert not np.array_equal(A[:, ~zero], A0[:, ~zero])
        # two row slabs (two ranks' shares) equal the one-rank matrix bit for bit
        for opts in (bem.AssemblyOptions(admittance=y), bem.AssemblyOptions(1, True, y)):
            full = bem.build_tbem_system_with_beta(st, ph, beta, options=opts)
            parts = [bem.build_tbem_system_with_beta(st, ph, beta, rows=rr, options=opts) for rr in ((0, n // 2 + 3), (n // 2 + 3, n))]
            assert np.array_equal(np.vstack([p.matrix.rows() for p in parts]), full.matrix.rows())
            assert rhs_equal(np.concatenate([p.rhs for p in parts]), full.rhs, vbar)


def test_library_refuses_bad_options(bem):
    from math_audio_b200 import _capi
    import ctypes as C

    mesh = generate_icosphere_mesh(0.1, 1)
    mesh.bc_type[3] = BC_PRESSURE
    st = bem.StagedMesh(mesh)
    ph = bem._cphys(PhysicsParams.from_wave_number(10.0))
    y = np.zeros(st.num_dofs, dtype=np.complex128)
    y[3] = 1.0 - 1.0j
    lib = _capi.lib()
    for copts in (_capi.CAssemblyOptions(2, 0, None), _capi.CAssemblyOptions(0, 3, None), _capi.CAssemblyOptions(0, 0, _capi.ptr(y))):
        h = C.c_void_p()
        rc = lib.bemb200_assemble_staged_opts(st.ctx._h, st._h, C.byref(ph), 0.0, 0.1, C.byref(copts), 0, st.num_dofs, C.byref(h))
        assert rc == -1 and not h


@pytest.mark.parametrize("overlap", [False, True])
def test_sweep_carries_a_y_per_frequency(bem, overlap):
    from math_audio_b200.incident import IncidentField
    from math_audio_b200.sweep import Sweep

    a = 0.1
    mesh = generate_icosphere_mesh(a, 3)
    cfg = bem.GmresConfig(max_iterations=300, restart=50, tolerance=1e-10)
    cases = []
    for i, ka in enumerate((0.4, 1.0, 1.7, 2.5)):
        ph = PhysicsParams.from_wave_number(ka / a)
        beta, _ = ph.burton_miller_beta_adaptive(a)
        opts = bem.AssemblyOptions.sign_consistent(mixed_admittance(mesh, ph.wave_number, 20 + i, frac=0.3 + 0.2 * i))
        cases.append((ph, beta, IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta), opts))
    sw = Sweep(mesh, overlap=overlap)
    for ph, beta, rhs, opts in cases:
        sw.set_assembly_options(opts)
        sw.submit(ph, beta, rhs, cfg)
    sw.set_assembly_options(None)
    got = [sw.next() for _ in cases]
    sw.close()
    for (ph, beta, rhs, opts), (sol, stats, b) in zip(cases, got):
        system = bem.build_tbem_system_with_beta(mesh, ph, beta, options=opts)
        ref = bem.gmres(bem.DenseOperator(system), system.rhs + rhs, cfg)
        assert np.array_equal(b, system.rhs + rhs)
        assert (sol.iterations, sol.restarts, sol.converged) == (ref.iterations, ref.restarts, ref.converged) and sol.converged
        if overlap:  # the solver's Gram-Schmidt kernel differs beside a background assembly
            assert np.linalg.norm(sol.x - ref.x) / np.linalg.norm(ref.x) < 1e-9
        else:
            assert np.array_equal(sol.x, ref.x) and sol.residual == ref.residual


def test_end_to_end_robin_sphere(bem):
    """BemSolver with a passive admittance, the sign-consistent formulation, icosphere(4) at ka = 2: the surface pressure and
    the field at r = 2a against the exact Robin series."""
    from math_audio_b200.bem_solver import BemProblem, BemSolver, SolverMethod

    a, ka = 1.0, 2.0
    c = 343.0
    freq = ka / a * c / (2.0 * np.pi)
    problem = BemProblem.rigid_sphere_scattering(a, freq, c, 1.21)
    problem.mesh = generate_icosphere_mesh(a, 4)
    k = problem.physics.wave_number
    Y = (0.3 - 0.3j) * k
    problem.with_admittance(Y)
    solver = BemSolver().with_solver_method(SolverMethod.Direct).with_sign_consistent_formulation(True)
    solver.beta_scale = 16.0
    sol = solver.solve(problem)
    surf = ao.rel_l2(sol.surface_pressure, ao.robin_mie(k, a, Y, problem.mesh.center))
    assert surf < 0.08, surf
    rigid = BemSolver().with_solver_method(SolverMethod.Direct).with_sign_consistent_formulation(True)
    rigid.beta_scale = 16.0
    p_rigid = rigid.solve(BemProblem(problem.mesh, problem.physics, problem.incident_field)).surface_pressure
    assert ao.rel_l2(p_rigid, ao.robin_mie(k, a, 0.0, problem.mesh.center)) < 0.015
    th = np.linspace(0.1, np.pi - 0.1, 24)
    pts = 2.0 * a * np.stack([np.sin(th), np.zeros_like(th), np.cos(th)], axis=1)
    field = np.array([fp.p_total for fp in sol.evaluate_pressure_field(pts)])
    ferr = ao.rel_l2(field, ao.robin_mie(k, a, Y, pts))
    assert ferr < 0.08, ferr
