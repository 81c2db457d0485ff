"""The far-field amplitude on the device (DESIGN.md 4.9): ``bemb200_far_field`` against the numpy restatement
(tests/far_field_oracle.py), its bit-identity rules, and radiation / scattering through ``BemSolver`` against the exact sphere
series with the bars of tests/test_far_field_cpu.py."""
import dataclasses
import math
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import far_field_oracle as fo  # noqa: E402

from math_audio_b200.mesh import generate_box_mesh_quad, generate_icosphere_mesh  # noqa: E402
from math_audio_b200.types import PhysicsParams  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bem():
    from math_audio_b200 import bem as _bem

    return _bem


@pytest.fixture(scope="module")
def torch():
    import torch as _torch

    assert _torch.cuda.is_available()
    return _torch


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.complex128)).to("cuda:0")


def _bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def _mesh(case):
    rng = np.random.default_rng(5)
    if case == "sphere":
        return generate_icosphere_mesh(0.5, 2)
    if case == "box":
        return generate_box_mesh_quad(0.32, 0.44, 0.64, 4, 4, 8)
    if case == "warped":
        mesh = generate_box_mesh_quad(0.32, 0.44, 0.64, 4, 4, 8)
        mesh.nodes = mesh.nodes + 0.01 * rng.standard_normal(mesh.nodes.shape)  # non-planar quads
        return mesh
    mesh = generate_icosphere_mesh(0.5, 2)  # evaluation-only elements and a permuted DOF map
    mesh.is_eval[::11] = 1
    bnd = np.flatnonzero(mesh.is_eval == 0)
    mesh.dof[bnd] = rng.permutation(mesh.num_dofs).astype(np.uint32)
    return mesh


def _physics(k, s):
    return dataclasses.replace(PhysicsParams.from_wave_number(k), harmonic_factor=s)


def _values(rng, nsol, n):
    return rng.standard_normal((nsol, n)) + 1j * rng.standard_normal((nsol, n))


@pytest.mark.parametrize("case", ["sphere", "box", "warped", "permuted"])
@pytest.mark.parametrize("s", [1.0, -1.0])
def test_device_far_field_matches_restatement(bem, case, s):
    mesh = _mesh(case)
    st = bem.StagedMesh(mesh)
    rng = np.random.default_rng(7)
    n = st.num_dofs
    P, V = _values(rng, 3, n), _values(rng, 3, n)
    dirs, _ = fo.sphere_quadrature(9, 18)
    k = 8.0
    ph = _physics(k, s)
    for vel in (None, V):
        got = bem.compute_far_field(dirs, st, P, vel, ph)
        for i in range(3):
            ref = fo.far_field(mesh, dirs, P[i], None if vel is None else vel[i], k, s)
            err = np.linalg.norm(got[i] - ref) / np.linalg.norm(ref)
            assert err <= 1e-12, (case, s, i, err)


def test_bit_identity_batch_single_device_host_repeat(bem, torch):
    mesh = _mesh("permuted")
    st = bem.StagedMesh(mesh)
    rng = np.random.default_rng(11)
    n = st.num_dofs
    ph = PhysicsParams.from_wave_number(6.0)
    for nsol, grid in ((13, (7, 6)), (4096, (2, 3))):  # 13: not a multiple of the chunk; 4096: the batch limit
        P, V = _values(rng, nsol, n), _values(rng, nsol, n)
        dirs, _ = fo.sphere_quadrature(*grid)
        batch = bem.compute_far_field(dirs, st, P, V, ph)
        assert batch.shape == (nsol, len(dirs))
        assert _bits(batch, bem.compute_far_field(dirs, st, P, V, ph))  # repeated call
        for i in sorted({0, 7, 8, nsol - 1}):
            assert _bits(batch[i], bem.compute_far_field(dirs, st, P[i], V[i], ph)), (nsol, i)
        # device input, DOF order
        Pd, Vd = np.empty_like(P), np.empty_like(V)
        Pd[:, st.enum_to_dof], Vd[:, st.enum_to_dof] = P, V
        pd, vd = _dev(torch, Pd), _dev(torch, Vd)
        assert _bits(bem.compute_far_field(dirs, st, pd.data_ptr(), vd.data_ptr(), ph, nsol=nsol), batch)
        if nsol == 13:  # spot check against the restatement
            ref = fo.far_field(mesh, dirs, P[12], V[12], 6.0)
            assert np.linalg.norm(batch[12] - ref) / np.linalg.norm(ref) <= 1e-12
    rigid = bem.compute_far_field(dirs, st, P[:2], None, ph)
    assert _bits(rigid[1], bem.compute_far_field(dirs, st, P[1], None, ph))


def test_bad_direction_is_refused_by_the_library(bem):
    from math_audio_b200 import _capi

    st = bem.StagedMesh(generate_icosphere_mesh(0.5, 1))
    ph = bem._cphys(PhysicsParams.from_wave_number(2.0))
    p = np.zeros(st.num_dofs, np.complex128)
    d = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 1.5]])
    out = np.empty(2, np.complex128)
    import ctypes as C

    rc = _capi.lib().bemb200_far_field(st._h, C.byref(ph), 1, _capi.ptr(p), None, 0, 2, _capi.ptr(d), _capi.ptr(out))
    assert rc == -1 and "direction 1" in _capi.lib().bemb200_last_error(st.ctx._h).decode()
    rc = _capi.lib().bemb200_far_field(st._h, C.byref(ph), 1, _capi.ptr(p), None, 1, 1, _capi.ptr(d), _capi.ptr(out))
    assert rc == -1  # a host array passed as device memory


def _solver(scale):
    from math_audio_b200.bem_solver import BemSolver

    return BemSolver(beta_scale=scale).with_sign_consistent_formulation(True)


def test_solver_pulsating_sphere_far_field_and_power():
    """radiation through BemSolver: dp/dn = 1 on icosphere(3), ka = 2 (beta 16 i / k, as the CPU bars)"""
    from math_audio_b200 import postprocess
    from math_audio_b200.bem_solver import BemProblem
    from math_audio_b200.incident import IncidentField

    k = 2.0
    ph = PhysicsParams.from_wave_number(k)
    problem = BemProblem(generate_icosphere_mesh(1.0, 3), ph, IncidentField()).with_surface_velocity(1.0)
    sol = _solver(16.0).solve(problem)
    assert np.array_equal(sol.surface_velocity, np.ones(sol.num_dofs()))
    dirs, w = fo.sphere_quadrature(24, 48)
    F = sol.far_field(dirs)
    exact = fo.radiator_far_field(k, 1.0, 0, dirs[:, 2])
    err = np.linalg.norm(F - exact) / np.linalg.norm(exact)
    assert err <= 0.03, err  # CPU: 2.0e-2
    ws, wff = sol.radiated_power(), postprocess.far_field_power(F, w, ph)
    assert ws > 0 and abs(ws - wff) / wff <= 0.03, (ws, wff)  # CPU: 2.1e-2
    # the field kernel takes the prescribed velocity too: at R = 1e4 it approaches F exp(ikR) / R
    R = 1e4
    fp = sol.evaluate_pressure_field(R * dirs[:5])
    got = np.array([f.p_scattered for f in fp]) * R * np.exp(-1j * k * R)
    assert np.linalg.norm(got - F[:5]) / np.linalg.norm(F[:5]) < 1e-3


def test_solver_rigid_sphere_optical_theorem():
    from math_audio_b200.bem_solver import BemProblem
    from math_audio_b200.incident import IncidentField

    k = 1.0
    ph = PhysicsParams.from_wave_number(k)
    sol = _solver(4.0).solve(BemProblem(generate_icosphere_mesh(1.0, 3), ph, IncidentField.plane_wave_z()))
    dirs, w = fo.sphere_quadrature(24, 48)
    F = sol.far_field(dirs)
    sigma_ext = 4 * math.pi / k * sol.far_field(np.array([[0.0, 0.0, 1.0]]))[0].imag
    sigma_sc = float(np.abs(F) ** 2 @ w)
    assert sol.radiated_power() == 0.0
    assert abs(sigma_ext - sigma_sc) / sigma_sc <= 0.007, (sigma_ext, sigma_sc)  # CPU: 4.9e-3
    exact = fo.series_far_field(k, 1.0, dirs[:, 2])
    assert np.linalg.norm(F - exact) / np.linalg.norm(exact) <= 0.01  # CPU: 6.8e-3
