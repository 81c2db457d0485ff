"""The far-field amplitude, radiated power and directivity (DESIGN.md 4.9) on the CPU, no GPU: the numpy restatement
(tests/far_field_oracle.py) against the field representation it is the limit of, against itself with finer rules, and against
the exact sphere series on sign-consistent oracle solutions (tests/admittance_oracle.py); the energy identities; the host
helpers of ``postprocess``; and the argument checks of the Python and C entries.

Every physics bar is a number measured here on icosphere(2) -> icosphere(3) (radius 1; the Quad4 box: 4x4x8 -> 8x8x16), and
each error must also shrink by a ratio < 0.75 with the refinement.  DESIGN.md 4.9 records the table."""
from __future__ import annotations

import ctypes as C
import functools
import math
import subprocess
import sys
import types
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import admittance_oracle as ao  # noqa: E402
import far_field_oracle as fo  # noqa: E402

from math_audio_b200 import _capi, bem, postprocess  # noqa: E402
from math_audio_b200.mesh import generate_box_mesh_quad, generate_icosphere_mesh, mesh_from_data  # noqa: E402
from math_audio_b200.types import PhysicsParams  # noqa: E402

ROOT = Path(__file__).resolve().parent.parent
EINVAL = -1
DIRS, WTS = fo.sphere_quadrature(24, 48)


def adaptive_beta(ka, k):
    scale = 1.0 if ka < 0.5 else (4.0 if ka < 1.2 else (8.0 if ka < 1.8 else 16.0))
    return 1j * scale / k


def set_velocity(mesh, v):
    """constant dp/dn = v_j on element j: one value per node (BemSolver.prepare_elements does the same)"""
    mesh.bc_len[:] = mesh.etype
    mesh.bc_val[:] = 0.0
    for i in range(4):
        mesh.bc_val[:, i] = np.where(i < mesh.etype, v, 0.0)


def sign_consistent_solution(mesh, k, beta, Y=None, v=None, incident=True):
    """(p, v) of the sign-consistent formulation (forced sign +1, consistent beta) on the CPU oracle"""
    if v is not None:
        set_velocity(mesh, v)
    A, rhs, _ = ao.assemble_opts(mesh, k, beta, dg_dn_sign=1, consistent_beta=True,
                                 admittance=None if Y is None else np.full(mesh.n_elem, Y))
    if incident:
        from oracle import oracle as orc

        inc, _ = orc.incident_rhs(0, [0, 0, 1], 1.0, mesh.center, mesh.normal, k, beta)
        rhs = rhs + inc
    p = np.linalg.solve(A, rhs)
    vel = np.zeros_like(p) if v is None else np.asarray(v, dtype=np.complex128)
    if Y is not None:
        vel = vel + Y * p
    return p, vel


@functools.lru_cache(maxsize=None)
def sphere_case(kind, sub, ka, yk=0.0):
    """(mesh, physics, p, v, F over DIRS, exact F over DIRS) on icosphere(sub), radius 1, k = ka"""
    mesh = generate_icosphere_mesh(1.0, sub)
    k = ka
    ph = PhysicsParams.from_wave_number(k)
    beta = adaptive_beta(ka, k)
    if kind == "scatter":
        Y = yk * k if yk else None
        p, v = sign_consistent_solution(mesh, k, beta, Y=Y)
        exact = fo.series_far_field(k, 1.0, DIRS[:, 2], Y=0.0 if Y is None else Y)
    else:
        order = {"pulsating": 0, "oscillating": 1}[kind]
        ct = mesh.center[:, 2] / np.linalg.norm(mesh.center, axis=1)
        p, v = sign_consistent_solution(mesh, k, beta, v=np.ones(mesh.n_elem) if order == 0 else ct, incident=False)
        exact = fo.radiator_far_field(k, 1.0, order, DIRS[:, 2])
    return mesh, ph, p, v, fo.far_field(mesh, DIRS, p, v, k), exact


def converges(err2, err3, bar):
    assert err3 <= bar and err3 < 0.75 * err2, (err2, err3, bar)


# ---- the definition ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("s", [1.0, -1.0])
def test_far_field_is_the_limit_of_the_scattered_field(s):
    """R exp(-i s k R) p_scat(R d) of the field representation -> F(d), with a difference falling as 1/R (Tri3)."""
    mesh = generate_icosphere_mesh(1.0, 1)
    rng = np.random.default_rng(3)
    n = mesh.n_elem
    p = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    v = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    k = 2.0
    d = DIRS[::97]
    F = fo.far_field(mesh, d, p, v, k, s)
    diff = []
    for R in (1e4, 1e6):
        FR = fo.scattered_field(mesh, R * d, p, v, k, s) * R * np.exp(-1j * s * k * R)
        diff.append(np.linalg.norm(FR - F) / np.linalg.norm(F))
    assert diff[0] < 1e-3 and 0.005 < diff[1] / diff[0] < 0.02, diff


def test_planar_quad_equals_its_two_triangles():
    nodes = np.array([[0.0, 0.0, 0.0], [0.12, 0.01, 0.0], [0.15, 0.11, 0.0], [0.02, 0.09, 0.0]])
    quad = mesh_from_data(nodes, [[0, 1, 2, 3]])
    tris = mesh_from_data(nodes, [[0, 1, 2], [0, 2, 3]])
    k = 10.0
    for p, v in ((1.0 + 0.5j, 0.0), (0.0, 2.0 - 1.0j), (0.3 - 0.2j, -0.7j)):
        Fq = fo.far_field(quad, DIRS, np.array([p]), np.array([v]), k)
        Ft = fo.far_field(tris, DIRS, np.array([p, p]), np.array([v, v]), k)
        assert np.linalg.norm(Fq - Ft) / np.linalg.norm(Ft) < 3e-6  # measured 3.6e-7 .. 9.5e-7 (k h ~ 1.5)


def test_warped_quad_against_a_fine_gauss_rule():
    """the 3 x 3 rule on a warped (non-planar) quad against 10 x 10: the error of the 3 x 3 rule is small and shrinks
    fast with the element size (O(h^6) of the rule)"""
    errs = []
    for h in (0.2, 0.1):
        nodes = h * np.array([[0.0, 0.0, 0.0], [1.0, 0.1, 0.15], [1.1, 1.0, -0.1], [0.0, 0.9, 0.2]])
        quad = mesh_from_data(nodes, [[0, 1, 2, 3]])
        p, v = np.array([1.0 - 0.3j]), np.array([0.4 + 0.8j])
        F3 = fo.far_field(quad, DIRS, p, v, 12.0, gauss=3)
        F10 = fo.far_field(quad, DIRS, p, v, 12.0, gauss=10)
        errs.append(np.linalg.norm(F3 - F10) / np.linalg.norm(F10))
    assert errs[0] < 5e-5 and errs[1] < 0.1 * errs[0], errs  # measured 2.1e-5 -> 6.4e-7


def test_compute_rcs_is_4pi_times_the_squared_4pi_far_field():
    """compute_rcs (centroid rule, no velocity term) = 4 pi |4 pi F|^2 of a rigid body to centroid-rule accuracy"""
    from oracle import oracle as orc

    for sub, bar in ((2, 8e-3), (3, 2e-3)):
        mesh, _, p, _, F, _ = sphere_case("scatter", sub, 2.0)
        rcs = orc.compute_rcs(mesh, p, DIRS, 2.0)
        err = np.max(np.abs(rcs - 4 * math.pi * np.abs(4 * math.pi * F) ** 2)) / np.max(rcs)
        assert err < bar, (sub, err)  # measured 5.5e-3 (icosphere 2) and 1.3e-3 (icosphere 3)


# ---- against the exact sphere far fields ------------------------------------------------------------------------------
@pytest.mark.parametrize("ka,bar", [(1.0, 0.01), (2.0, 0.015)])
def test_rigid_sphere_far_field(ka, bar):
    e = [ao.rel_l2(sphere_case("scatter", s, ka)[4], sphere_case("scatter", s, ka)[5]) for s in (2, 3)]
    converges(*e, bar)  # measured ka = 1: 2.3e-2 -> 6.8e-3; ka = 2: 3.9e-2 -> 1.0e-2


@pytest.mark.parametrize("kind,bar", [("pulsating", 0.03), ("oscillating", 0.02)])
def test_radiating_sphere_far_field(kind, bar):
    e = [ao.rel_l2(sphere_case(kind, s, 2.0)[4], sphere_case(kind, s, 2.0)[5]) for s in (2, 3)]
    converges(*e, bar)  # measured at ka = 2: pulsating 3.7e-2 -> 2.0e-2, oscillating 3.4e-2 -> 1.5e-2


@pytest.mark.parametrize("ka,bar", [(1.0, 0.025), (2.0, 0.065)])
def test_robin_sphere_far_field(ka, bar):
    e = [ao.rel_l2(sphere_case("scatter", s, ka, -0.5j)[4], sphere_case("scatter", s, ka, -0.5j)[5]) for s in (2, 3)]
    converges(*e, bar)  # measured ka = 1: 4.0e-2 -> 1.8e-2; ka = 2: 8.7e-2 -> 5.0e-2


# ---- energy identities ------------------------------------------------------------------------------------------------
def _power_mismatch(mesh, ph, p, v, F):
    ws = postprocess.surface_power(mesh, p, v, ph)
    wff = postprocess.far_field_power(F, WTS, ph)
    assert ws > 0 and wff > 0
    return abs(ws - wff) / wff


def test_pulsating_sphere_surface_power_is_far_field_power():
    e = [_power_mismatch(*sphere_case("pulsating", s, 2.0)[:5]) for s in (2, 3)]
    converges(*e, 0.03)  # measured 4.0e-2 -> 2.1e-2


@functools.lru_cache(maxsize=None)
def box_case(refine):
    """a small config 3: the 0.32 x 0.44 x 0.64 m Quad4 cabinet with a 0.16 x 0.22 m piston (v = 1) on top, 300 Hz"""
    mesh = generate_box_mesh_quad(0.32, 0.44, 0.64, 4 * refine, 4 * refine, 8 * refine)
    ph = PhysicsParams.new(300.0, 343.0, 1.21, False)
    k = ph.wave_number
    c = mesh.center
    piston = (np.abs(c[:, 2] - 0.32) < 1e-9) & (np.abs(c[:, 0]) < 0.08) & (np.abs(c[:, 1]) < 0.11)
    p, v = sign_consistent_solution(mesh, k, 4j / k, v=piston.astype(np.float64), incident=False)
    return mesh, ph, p, v, fo.far_field(mesh, DIRS, p, v, k)


def test_box_piston_surface_power_is_far_field_power():
    assert int(box_case(1)[3].real.sum()) == 4 and int(box_case(2)[3].real.sum()) == 16
    e = [_power_mismatch(*box_case(r)) for r in (1, 2)]
    converges(*e, 0.045)  # measured 8.5e-2 -> 3.2e-2


def _optical(sub, ka, yk=0.0):
    mesh, ph, p, v, F, _ = sphere_case("scatter", sub, ka, yk)
    fwd = fo.far_field(mesh, [[0.0, 0.0, 1.0]], p, v, ka)[0]
    sigma_ext = ph.harmonic_factor * 4 * math.pi / ka * fwd.imag
    sigma_sc = float(np.abs(F) ** 2 @ WTS)
    sigma_abs = -postprocess.surface_power(mesh, p, v, ph) * 2 * ph.density * ph.speed_of_sound
    return sigma_ext, sigma_sc, sigma_abs


def test_rigid_sphere_optical_theorem():
    e = []
    for sub in (2, 3):
        ext, sc, ab = _optical(sub, 1.0)
        assert ab == 0.0
        e.append(abs(ext - sc) / sc)
    converges(*e, 0.007)  # measured 1.5e-2 -> 4.9e-3
    ext, sc, _ = _optical(3, 2.0)
    assert abs(ext - sc) / sc < 1e-3  # at ka = 2 both meshes sit at a 4-5e-4 floor, exempt from the ratio


@pytest.mark.parametrize("ka,bar", [(1.0, 0.025), (2.0, 0.045)])
def test_robin_sphere_extinction_is_scattering_plus_absorption(ka, bar):
    e = []
    for sub in (2, 3):
        ext, sc, ab = _optical(sub, ka, -0.5j)
        assert ab > 0.5 * ext  # an absorber: sigma_abs is most of sigma_ext here
        e.append(abs(ext - sc - ab) / ext)
    converges(*e, bar)  # measured ka = 1: 3.5e-2 -> 1.9e-2; ka = 2: 5.2e-2 -> 3.3e-2


# ---- host helpers -----------------------------------------------------------------------------------------------------
def test_sphere_quadrature_integrates_low_order_harmonics():
    d, w = postprocess.sphere_quadrature(6, 12)
    d0, w0 = fo.sphere_quadrature(6, 12)
    assert np.allclose(d, d0, atol=1e-15, rtol=0) and np.allclose(w, w0, atol=1e-15, rtol=0)
    x, y, z = d.T
    four_pi = 4 * math.pi
    for f, exact in ((1.0, four_pi), (x, 0.0), (z, 0.0), (x * y, 0.0), (x * x, four_pi / 3), (z * z, four_pi / 3),
                     (x * x * y * y, four_pi / 15), (z ** 4, four_pi / 5), (x * y * z, 0.0), (x ** 2 * z ** 3, 0.0),
                     (x ** 6, four_pi / 7)):
        assert abs(float(np.sum(w * f)) - exact) < 1e-13, (f, exact)


def test_power_and_directivity_helpers():
    ph = PhysicsParams.from_wave_number(2.0)
    d, w = postprocess.sphere_quadrature(12, 24)
    omni = np.full(len(d), 0.5 + 0.5j)
    assert postprocess.far_field_power(omni, w, ph) == pytest.approx(4 * math.pi * 0.5 / (2 * ph.density * ph.speed_of_sound))
    assert np.allclose(postprocess.far_field_power(np.stack([omni, 2 * omni]), w, ph),
                       [1, 4] * np.asarray(postprocess.far_field_power(omni, w, ph)))
    assert abs(postprocess.directivity_index(omni, w, 0)) < 1e-12
    dipole = d[:, 2]  # |F|^2 = cos^2: DI = 10 log10(3) on axis
    on_axis = int(np.argmax(d[:, 2]))
    assert postprocess.directivity_index(dipole, w, on_axis) == pytest.approx(10 * math.log10(3 * d[on_axis, 2] ** 2), abs=1e-12)
    mesh, _, p, v, _, _ = sphere_case("pulsating", 2, 2.0)
    assert postprocess.surface_power(mesh, p, v, ph) == pytest.approx(fo.surface_power(mesh, p, v, ph), rel=1e-14)
    with pytest.raises(ValueError):
        postprocess.surface_power(mesh, p[:-1], v, ph)
    with pytest.raises(ValueError):
        postprocess.far_field_power(omni[:-1], w, ph)
    with pytest.raises(ValueError):
        postprocess.sphere_quadrature(0, 4)


def test_solver_radiation_problem_prepares_constant_velocity():
    from math_audio_b200.bem_solver import BemProblem, BemSolver
    from math_audio_b200.incident import IncidentField

    mesh = generate_box_mesh_quad(1.0, 1.0, 1.0, 1, 1, 1)
    ph = PhysicsParams.from_wave_number(1.0)
    problem = BemProblem(mesh, ph, IncidentField())
    plain = BemSolver().prepare_elements(problem)
    assert (plain.bc_len == 1).all() and (plain.bc_val == 0).all()  # without v_bar: exactly the rigid preparation
    v = np.arange(mesh.n_elem) * (1 - 1j)
    prepared = BemSolver().prepare_elements(problem.with_surface_velocity(v))
    assert (prepared.bc_len == 4).all() and np.array_equal(prepared.bc_val, np.repeat(v[:, None], 4, axis=1))
    from math_audio_b200.bem_solver import BemError

    with pytest.raises(BemError):
        BemSolver().prepare_elements(problem.with_surface_velocity(np.ones(3)))


# ---- argument checks --------------------------------------------------------------------------------------------------
def _staged(n=10, enum_to_dof=None):
    return types.SimpleNamespace(num_dofs=n, enum_to_dof=enum_to_dof, _h=None, ctx=types.SimpleNamespace(_h=None))


def test_python_wrapper_refuses_bad_arguments():
    st = _staged(10)
    ph = PhysicsParams.from_wave_number(2.0)
    dirs = np.eye(3)
    p = np.zeros(10, np.complex128)
    for bad in (np.ones(3), np.ones((0, 3)), np.ones((2, 2)), [[1.0, 1e-4, 0.0]], [[np.nan, 0.0, 1.0]], [[0.0, 0.0, 1.0 + 2e-9]]):
        with pytest.raises(ValueError):
            bem.compute_far_field(bad, st, p, None, ph)
    for bad in (np.zeros(9), np.zeros((2, 9)), np.zeros((0, 10)), np.zeros((4097, 10))):
        with pytest.raises(ValueError):
            bem.compute_far_field(dirs, st, bad, None, ph)
    with pytest.raises(ValueError):
        bem.compute_far_field(dirs, st, p, np.zeros((1, 10)), ph)  # 1-D pressure, 2-D velocity
    with pytest.raises(ValueError):
        bem.compute_far_field(dirs, st, p, np.zeros(9), ph)
    with pytest.raises(ValueError):
        bem.compute_far_field(dirs, st, np.zeros((2, 10)), None, ph, nsol=3)
    for ptr, nsol in ((1 << 20, None), (1 << 20, 0), (1 << 20, 5000), (True, 1), (-5, 1)):
        with pytest.raises(ValueError):
            bem.compute_far_field(dirs, st, ptr, None, ph, nsol=nsol)
    with pytest.raises(ValueError):  # mixed host / device inputs
        bem.compute_far_field(dirs, st, 1 << 20, np.zeros((2, 10)), ph, nsol=2)


def test_c_entry_refuses_bad_arguments_without_a_device():
    lib = _capi.lib()
    ph = _capi.CPhysics(1.0, 1.0, 1.0, 1.0)
    d = (C.c_double * 6)(0.0, 0.0, 1.0, 1.0, 0.0, 0.0)
    vals = (C.c_double * 64)()
    out = (C.c_double * 64)()

    def call(sm=None, phys=C.byref(ph), nsol=1, p=vals, v=None, on_device=0, n_dirs=2, dirs=d, o=out):
        rc = lib.bemb200_far_field(sm, phys, nsol, p, v, on_device, n_dirs, dirs, o)
        return rc, lib.bemb200_last_error(None).decode()

    assert call() == (EINVAL, "NULL staged mesh")  # every other argument is valid
    for kw, msg in ((dict(phys=None), "NULL"), (dict(p=None), "NULL"), (dict(dirs=None), "NULL"), (dict(o=None), "NULL"),
                    (dict(nsol=0), "solutions"), (dict(nsol=4097), "solutions"), (dict(on_device=2), "on_device"),
                    (dict(n_dirs=0), "directions")):
        rc, err = call(**kw)
        assert rc == EINVAL and msg in err, (kw, err)
    for bad in ((0.0, 0.0, 1.0 + 2e-9), (0.0, 0.0, 0.0), (float("nan"), 0.0, 1.0), (float("inf"), 0.0, 0.0), (0.6, 0.8, 1e-4)):
        rc, err = call(dirs=(C.c_double * 6)(0.0, 0.0, 1.0, *bad))
        assert rc == EINVAL and "direction 1 " in err, (bad, err)
    rc, _ = call(dirs=(C.c_double * 6)(0.0, 0.0, 1.0, 0.6, 0.8, 1e-10))  # within 1e-9 of unit length: only the mesh is missing
    assert rc == EINVAL and _ == "NULL staged mesh"


def test_cpp_far_field_wrapper_compiles_and_links(tmp_path):
    """bemb200::compute_far_field (include/bemb200.hpp) against the library's exported symbols, warnings as errors."""
    exe = tmp_path / "instantiate_far_field"
    libdir = _capi.LIB_PATH.parent
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "instantiate_far_field.cpp"),
           "-o", str(exe), f"-L{libdir}", "-lbemb200", f"-Wl,-rpath,{libdir}"]
    subprocess.run(cmd, check=True)
    assert subprocess.run([str(exe)]).returncode == 0  # nothing is executed: main returns before touching the GPU
