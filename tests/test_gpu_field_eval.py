"""Accurate field evaluation on the device (DESIGN.md 4.10): ``bemb200_evaluate_field`` against the numpy restatement
(tests/field_eval_oracle.py), its bit-identity rules, the NaN contract for points on the surface, and the near-surface field
of a rigid sphere through ``BemSolver`` against the exact series with the bars of tests/test_field_eval_cpu.py."""
import dataclasses
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import far_field_oracle as fo  # noqa: E402
import field_eval_oracle as fe  # noqa: E402

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
    return np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


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


def _points(mesh):
    """regular points far out, and near points above and below interior spots of a few boundary elements at
    delta h, delta in {1, 0.1, 0.01, 0.001}"""
    h = fe.mesh_h(mesh)
    bnd = np.flatnonzero(np.asarray(mesh.is_eval) == 0)
    pts = [3.0 * d for d in fo.sphere_quadrature(3, 4)[0]]
    for e in bnd[[1, 17, 40]]:
        et = int(mesh.etype[e])
        x = mesh.nodes[mesh.conn[e, :et].astype(np.int64)]
        foot = 0.7 * x.mean(axis=0) + 0.3 * x[1]
        for d in (1.0, 0.1, 0.01, 0.001):
            for side in (1.0, -1.0):
                pts.append(foot + side * d * h * mesh.normal[e])
    return np.array(pts)


def _physics(k, s):
    return dataclasses.replace(PhysicsParams.from_wave_number(k), harmonic_factor=s)


def _values(rng, nsol, n):
    return rng.standard_normal((nsol, n)) + 1j * rng.standard_normal((nsol, n))


@pytest.mark.parametrize("case", ["sphere", "box", "warped", "permuted"])
@pytest.mark.parametrize("s", [1.0, -1.0])
def test_device_field_matches_restatement(bem, case, s):
    mesh = _mesh(case)
    st = bem.StagedMesh(mesh)
    rng = np.random.default_rng(7)
    n = st.num_dofs
    P, V = _values(rng, 2, n), _values(rng, 2, n)
    pts = _points(mesh)
    k = 8.0
    ph = _physics(k, s)
    for vel in (None, V):
        got = bem.evaluate_field(pts, st, P, vel, ph)
        for i in range(2):
            ref = fe.evaluate_field(mesh, pts, P[i], None if vel is None else vel[i], k, s)
            err = np.linalg.norm(got[i] - ref) / np.linalg.norm(ref)
            assert err <= 1e-12, (case, s, i, err)


def test_bit_identity_batch_single_device_host_repeat(bem, torch):
    mesh = _mesh("permuted")
    st = bem.StagedMesh(mesh)
    rng = np.random.default_rng(11)
    n = st.num_dofs
    ph = PhysicsParams.from_wave_number(6.0)
    all_pts = _points(mesh)
    for nsol, pts in ((13, all_pts), (4096, all_pts[::5])):  # 13: not a multiple of the chunk; 4096: the batch limit
        P, V = _values(rng, nsol, n), _values(rng, nsol, n)
        batch = bem.evaluate_field(pts, st, P, V, ph)
        assert batch.shape == (nsol, len(pts))
        assert _bits(batch, bem.evaluate_field(pts, st, P, V, ph))  # repeated call
        for i in sorted({0, 7, 8, nsol - 1}):
            assert _bits(batch[i], bem.evaluate_field(pts, st, P[i], V[i], ph)), (nsol, i)
        Pd, Vd = np.empty_like(P), np.empty_like(V)  # device input, DOF order
        Pd[:, st.enum_to_dof], Vd[:, st.enum_to_dof] = P, V
        pd, vd = _dev(torch, Pd), _dev(torch, Vd)
        assert _bits(bem.evaluate_field(pts, st, pd.data_ptr(), vd.data_ptr(), ph, nsol=nsol), batch)
    rigid = bem.evaluate_field(pts, st, P[:2], None, ph)
    assert _bits(rigid[1], bem.evaluate_field(pts, st, P[1], None, ph))


def test_tri3_all_regular_points_equal_compute_scattered_field(bem):
    mesh = generate_icosphere_mesh(0.5, 3)
    st = bem.StagedMesh(mesh)
    rng = np.random.default_rng(4)
    p, v = _values(rng, 1, st.num_dofs)[0], _values(rng, 1, st.num_dofs)[0]
    pts = 5.0 * fo.sphere_quadrature(8, 16)[0]
    ph = PhysicsParams.from_wave_number(7.0)
    for vel in (None, v):
        got, ref = bem.evaluate_field(pts, st, p, vel, ph), bem.compute_scattered_field(pts, st, p, vel, ph)
        assert np.max(np.abs(got - ref)) <= 1e-13 * np.max(np.abs(ref))


def test_point_on_the_surface_is_nan_and_leaves_the_others_alone(bem):
    """a point on a mesh node is NaN for every solution; the other points have the bits of the same call with that point
    moved off the surface"""
    mesh = _mesh("box")
    st = bem.StagedMesh(mesh)
    rng = np.random.default_rng(2)
    P, V = _values(rng, 3, st.num_dofs), _values(rng, 3, st.num_dofs)
    ph = PhysicsParams.from_wave_number(5.0)
    pts = _points(mesh)
    on = pts.copy()
    on[4] = mesh.nodes[10]
    got, ref = bem.evaluate_field(on, st, P, V, ph), bem.evaluate_field(pts, st, P, V, ph)
    assert np.all(np.isnan(got[:, 4]))
    keep = np.arange(len(pts)) != 4
    assert np.all(np.isfinite(got[:, keep])) and _bits(got[:, keep], ref[:, keep])


def test_bad_points_are_refused_by_the_library(bem):
    import ctypes as C

    from math_audio_b200 import _capi

    st = bem.StagedMesh(generate_icosphere_mesh(0.5, 1))
    ph = bem._cphys(PhysicsParams.from_wave_number(2.0))
    p = np.zeros(st.num_dofs, np.complex128)
    x = np.array([[0.0, 0.0, 1.0], [0.0, np.nan, 1.5]])
    out = np.empty(2, np.complex128)
    rc = _capi.lib().bemb200_evaluate_field(st._h, C.byref(ph), 1, _capi.ptr(p), None, 0, 2, _capi.ptr(x), _capi.ptr(out))
    assert rc == -1 and "evaluation point 1" in _capi.lib().bemb200_last_error(st.ctx._h).decode()
    rc = _capi.lib().bemb200_evaluate_field(st._h, C.byref(ph), 1, _capi.ptr(p), None, 1, 1, _capi.ptr(x), _capi.ptr(out))
    assert rc == -1  # a host array passed as device memory


def test_solver_rigid_sphere_near_surface_field():
    """BemSolver (sign-consistent, beta 4 i / k) on icosphere(3), ka = 1: the total pressure at c_e + delta h n_e against
    the exact series with the CPU bar, and the default (reference) path unchanged"""
    from math_audio_b200.bem_solver import BemProblem, BemSolver
    from math_audio_b200.incident import IncidentField

    k = 1.0
    mesh = generate_icosphere_mesh(1.0, 3)
    sol = BemSolver(beta_scale=4.0).with_sign_consistent_formulation(True).solve(
        BemProblem(mesh, PhysicsParams.from_wave_number(k), IncidentField.plane_wave_z()))
    h = fe.mesh_h(mesh)
    es = np.flatnonzero(np.abs(mesh.center[:, 2]) < 2.0)[:: max(1, mesh.n_elem // 12)]
    pts = np.array([mesh.center[e] + d * h * mesh.normal[e] for e in es for d in (1.0, 0.1, 0.01)])
    got = np.array([f.p_total for f in sol.evaluate_pressure_field(pts, accurate=True)])
    exact = fe.sphere_total_field(k, 1.0, pts)
    assert np.linalg.norm(got - exact) / np.linalg.norm(exact) <= 0.003  # CPU: 2.2e-3
    assert abs(sol.evaluate_pressure(pts[0], accurate=True) - got[0]) <= 1e-14 * abs(got[0])
    plain = np.array([f.p_total for f in sol.evaluate_pressure_field(pts)])
    assert np.linalg.norm(plain - exact) / np.linalg.norm(exact) > 0.1  # the reference's rule this close to the surface
