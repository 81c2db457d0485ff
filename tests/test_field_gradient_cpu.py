"""Field gradient, particle velocity and intensity (DESIGN.md 4.11) on the CPU, no GPU: the numpy restatement
(tests/field_gradient_oracle.py) against central differences of the pressure restatement, against the vanishing gradient of
the static double layer on closed surfaces, against single elements with a much stricter acceptance, against
Kirchhoff-Helmholtz reproductions of a point source and the exact rigid-sphere series, and against the radiated power of
pulsating and oscillating spheres; the incident gradient, the host helpers, and the argument checks of the Python and C
entries.

Every physics bar is a number measured here on two meshes (icosphere(2) -> icosphere(3); the Quad4 box of config 3 at
184 -> 784 elements); where an error converges with the mesh it must also shrink by a ratio < 0.75.  DESIGN.md 4.11 records
the table."""
from __future__ import annotations

import ctypes as C
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
import field_eval_oracle as fe  # noqa: E402
import field_gradient_oracle as fg  # noqa: E402

from math_audio_b200 import _capi, bem, postprocess  # noqa: E402
from math_audio_b200.incident import IncidentField  # noqa: E402
from math_audio_b200.mesh import generate_box_mesh_quad, generate_icosphere_mesh  # noqa: E402
from math_audio_b200.types import PhysicsParams  # noqa: E402

ROOT = Path(__file__).resolve().parent.parent
EINVAL = -1
DELTAS = (1.0, 0.1, 0.01, 0.001)


def converges(err_coarse, err_fine, bar):
    assert err_fine <= bar and err_fine < 0.75 * err_coarse, (err_coarse, err_fine, bar)


def _mesh(case):
    if case == "sphere":
        return generate_icosphere_mesh(1.0, 2)
    mesh = generate_box_mesh_quad(0.32, 0.44, 0.64, 4, 4, 8)
    if case == "warped":  # shared nodes: the jittered surface stays closed
        mesh.nodes = mesh.nodes + 0.01 * np.random.default_rng(1).standard_normal(mesh.nodes.shape)
    return mesh


def _central_differences(f, pts, eps):
    """(M, 3) central differences of f ((K, 3) points -> (K,)) at the points, one call for all"""
    vals = f(np.concatenate([pts + eps * e for e in np.eye(3)] + [pts - eps * e for e in np.eye(3)])).reshape(6, -1)
    return ((vals[:3] - vals[3:]) / (2 * eps)).T


# ---- the definition: the gradient of the pressure restatement ---------------------------------------------------------
@pytest.mark.parametrize("case", ["sphere", "box", "warped"])
@pytest.mark.parametrize("kh", [0.1, 1.0, 3.0])
def test_gradient_equals_central_differences_of_the_field(case, kh):
    """regular points and points at delta in {1, 0.1} h on both sides of three elements, s = +-1, steps of 1e-5 h"""
    mesh = _mesh(case)
    h = fe.mesh_h(mesh)
    R = float(np.linalg.norm(mesh.nodes, axis=1).max())
    pts = [3 * R * np.array([0.3, 0.5, 0.81]), 3 * R * np.array([-0.6, 0.2, -0.77])]
    for e in (1, 17, 40):
        et = int(mesh.etype[e])
        x = mesh.nodes[mesh.conn[e, :et].astype(np.int64)]
        foot = 0.7 * x.mean(axis=0) + 0.3 * x[1]
        pts += [foot + side * d * h * mesh.normal[e] for d in (1.0, 0.1) for side in (1.0, -1.0)]
    pts = np.array(pts)
    rng = np.random.default_rng(3)
    n = mesh.num_dofs
    p, v = rng.standard_normal(n) + 1j * rng.standard_normal(n), rng.standard_normal(n) + 1j * rng.standard_normal(n)
    k = kh / h
    for s in (1.0, -1.0):
        g = fg.evaluate_field_gradient(mesh, pts, p, v, k, s)
        fd = _central_differences(lambda x: fe.evaluate_field(mesh, x, p, v, k, s), pts, 1e-5 * h)
        err = np.linalg.norm(g - fd, axis=1) / np.linalg.norm(g, axis=1)
        assert err.max() <= 1e-6, (s, err.max())  # measured <= 8.6e-10


def test_point_on_the_surface_is_nan():
    mesh = _mesh("box")
    one = np.ones(mesh.num_dofs)
    g = fg.evaluate_field_gradient(mesh, np.array([mesh.nodes[7], [0.0, 0.0, 2.0]]), one, one, 1.0)
    assert np.all(np.isnan(g[0])) and np.all(np.isfinite(g[1]))


# ---- the static double layer: grad D[1] = 0 off a closed surface -------------------------------------------------------
@pytest.mark.parametrize("case", ["sphere", "box", "warped"])
def test_static_double_layer_gradient_vanishes(case):
    """the probes of the solid-angle test (above a centroid, an edge midpoint and a vertex at DELTAS h, both sides), measured
    against sum_q |w_q n_q| / (4 pi r_q^3)"""
    mesh = _mesh(case)
    e = 5 if case == "sphere" else int(np.argmin(np.linalg.norm(mesh.center - [-0.04, -0.055, 0.32], axis=1)))
    et = int(mesh.etype[e])
    x = mesh.nodes[mesh.conn[e, :et].astype(np.int64)]
    h = fe.mesh_h(mesh)
    worst = 0.0
    for base in (x.mean(axis=0), 0.5 * (x[0] + x[1]), x[0]):
        for d in DELTAS:
            for side in (1.0, -1.0):
                g, scale = fg.static_double_layer_gradient(mesh, base + side * d * h * mesh.normal[e])
                worst = max(worst, float(np.linalg.norm(g)) / scale)
    assert worst <= 1e-6, worst  # measured <= 5.0e-7 (the Quad4 box)


# ---- single elements against a much stricter acceptance ------------------------------------------------------------------
H = 0.1
ELEMENTS = {
    "tri": (3, H * np.array([[0.0, 0.0, 0.0], [1.0, 0.1, 0.0], [0.2, 0.9, 0.0]])),
    "planar_quad": (4, H * np.array([[0.0, 0.0, 0.0], [1.0, 0.05, 0.0], [1.1, 1.0, 0.0], [-0.1, 0.9, 0.0]])),
    "warped_quad": (4, H * np.array([[0.0, 0.0, 0.0], [1.0, 0.1, 0.15], [1.1, 1.0, -0.1], [0.0, 0.9, 0.2]])),
}


@pytest.mark.parametrize("name", list(ELEMENTS))
@pytest.mark.parametrize("kh", [0.1, 1.0, 3.0])
def test_single_element_gradient_integrals(name, kh):
    """int grad_x G and int grad_x dG/dn_y against acceptance ratio 12 (which agrees with ratio 16 to 1.4e-11)"""
    et, x = ELEMENTS[name]
    n = np.cross(x[1] - x[0], x[2] - x[0])
    n = n / np.linalg.norm(n)
    foot = 0.7 * x[:et].mean(axis=0) + 0.3 * x[0]
    k = kh / H
    for d in (1.0, 0.1, 0.01):
        pt = foot + d * H * n
        a, b = fg.element_gradient_integrals(x, et, pt, k)
        ra, rb = fg.element_gradient_integrals(x, et, pt, k, accept=12.0)
        ea, eb = np.linalg.norm(a - ra) / np.linalg.norm(ra), np.linalg.norm(b - rb) / np.linalg.norm(rb)
        assert ea <= 1e-6, (d, ea)  # measured <= 6.6e-8
        # measured <= 4.3e-7 on the quads and at delta >= 0.1, 1.8e-6 on the triangle at delta = 0.01 (2.9e-8 of the
        # measure sum_q |w_q n_q| / (4 pi r_q^3) of the static test)
        assert eb <= (2e-6 if (et == 3 and d == 0.01) else 1e-6), (d, eb)


# ---- Kirchhoff-Helmholtz: a point source inside, its gradient outside ----------------------------------------------------
X0 = np.array([0.02, -0.03, 0.05])


def _point_source_errors(mesh, k):
    """relative gradient error at c_e + delta h n_e (e in 3, 40, 97) for delta in {2, 1} h together, then for delta = 0.1 and
    0.01 h each"""
    c, n = mesh.center, mesh.normal
    rv = c - X0
    r = np.linalg.norm(rv, axis=1)
    p = np.exp(1j * k * r) / (4 * math.pi * r)
    v = p * (1j * k - 1 / r) * (np.sum(rv * n, axis=1) / r)
    h = fe.mesh_h(mesh)
    pts = np.array([c[e] + d * h * n[e] for e in (3, 40, 97) for d in (2.0, 1.0, 0.1, 0.01)])
    dv = pts - X0
    rx = np.linalg.norm(dv, axis=1)
    exact = ((1j * k - 1 / rx) * np.exp(1j * k * rx) / (4 * math.pi * rx) / rx)[:, None] * dv
    err = (fg.evaluate_field_gradient(mesh, pts, p, v, k) - exact).reshape(3, 4, 3)
    ex = exact.reshape(3, 4, 3)
    far = float(np.linalg.norm(err[:, :2]) / np.linalg.norm(ex[:, :2]))
    return far, [float(np.linalg.norm(err[:, i]) / np.linalg.norm(ex[:, i])) for i in (2, 3)]


def test_kirchhoff_helmholtz_gradient_quad4_box():
    coarse, fine = [_point_source_errors(generate_box_mesh_quad(0.32, 0.44, 0.64, nx, ny, nz), 10.0)
                    for nx, ny, nz in ((4, 5, 8), (8, 11, 16))]
    converges(coarse[0], fine[0], 0.011)  # measured 2.6e-2 -> 9.6e-3
    # delta = 0.1 h / 0.01 h: measured 0.21 / 0.27 -> 0.14 / 0.19, the piecewise-constant surface values' own error
    assert max(fine[1]) <= 0.22, fine


def test_kirchhoff_helmholtz_gradient_sphere():
    coarse, fine = [_point_source_errors(generate_icosphere_mesh(0.3, sub), 10.0) for sub in (2, 3)]
    converges(coarse[0], fine[0], 0.003)  # measured 1.05e-2 -> 2.6e-3
    assert max(fine[1]) <= 0.11, fine  # delta = 0.1 h / 0.01 h: measured 0.074 / 0.10 -> 0.068 / 0.095


# ---- close to a rigid sphere: the exact series -----------------------------------------------------------------------------
def _rigid_sphere_errors(sub):
    """(error at delta in {2, 1} h, error at delta in {0.1, 0.01} h) of the total gradient at c_e + delta h n_e against
    central differences of the exact series: sign-consistent oracle solution, icosphere(sub), radius 1, ka = 1"""
    from oracle import oracle as orc

    k = 1.0
    mesh = generate_icosphere_mesh(1.0, sub)
    beta = 4j / k
    A, rhs, _ = ao.assemble_opts(mesh, k, beta, dg_dn_sign=1, consistent_beta=True)
    inc, _ = orc.incident_rhs(0, [0, 0, 1], 1.0, mesh.center, mesh.normal, k, beta)
    p = np.linalg.solve(A, rhs + inc)
    h = fe.mesh_h(mesh)
    es = np.flatnonzero(np.abs(mesh.center[:, 2]) < 2.0)[:: max(1, mesh.n_elem // 12)]
    out = []
    for deltas in ((2.0, 1.0), (0.1, 0.01)):
        pts = np.array([mesh.center[e] + d * h * mesh.normal[e] for e in es for d in deltas])
        g = fg.evaluate_field_gradient(mesh, pts, p, None, k)
        g = g + IncidentField.plane_wave_z().evaluate_gradient(pts, PhysicsParams.from_wave_number(k))
        exact = _central_differences(lambda x: fe.sphere_total_field(k, 1.0, x), pts, 1e-6)
        out.append(float(np.linalg.norm(g - exact) / np.linalg.norm(exact)))
    return out


def test_rigid_sphere_near_surface_gradient():
    coarse, fine = _rigid_sphere_errors(2), _rigid_sphere_errors(3)
    converges(coarse[0], fine[0], 0.0095)  # measured 1.4e-2 -> 8.8e-3
    # at 0.1 h and 0.01 h the gradient of piecewise-constant surface values is off by a fraction that does not shrink with h
    # at a fixed delta / h (measured 0.37 .. 0.52 at each delta on both meshes)
    assert fine[1] <= 0.55, fine


# ---- energy balance: the flux of I equals the radiated power ---------------------------------------------------------------
def _radiator_flux_errors(kind, sub):
    """(|flux - W_s| / W_s at R = 1.5 and 3, max |flux - W_ff| / W_ff) of a pulsating or oscillating unit sphere, ka = 1,
    sign-consistent oracle solution on icosphere(sub); the flux over a 12 x 24 sphere rule"""
    k = 1.0
    mesh = generate_icosphere_mesh(1.0, sub)
    ph = PhysicsParams.from_wave_number(k)
    ct = mesh.center[:, 2] / np.linalg.norm(mesh.center, axis=1)
    v = np.ones(mesh.n_elem) if kind == "pulsating" else ct
    mesh.bc_len[:] = mesh.etype
    mesh.bc_val[:] = 0.0
    for i in range(4):
        mesh.bc_val[:, i] = np.where(i < mesh.etype, v, 0.0)
    A, rhs, _ = ao.assemble_opts(mesh, k, 4j / k, dg_dn_sign=1, consistent_beta=True)
    p, v = np.linalg.solve(A, rhs), np.asarray(v, dtype=np.complex128)
    ws = postprocess.surface_power(mesh, p, v, ph)
    D, W = fo.sphere_quadrature(24, 48)
    wff = postprocess.far_field_power(fo.far_field(mesh, D, p, v, k), W, ph)
    dirs, wts = postprocess.sphere_quadrature(12, 24)
    to_ws, to_wff = [], []
    for R in (1.5, 3.0):
        pts = R * dirs
        intensity = postprocess.sound_intensity(fe.evaluate_field(mesh, pts, p, v, k), fg.evaluate_field_gradient(mesh, pts, p, v, k), ph)
        flux = R * R * float(np.sum(wts * np.sum(intensity * dirs, axis=1)))
        to_ws.append(abs(flux - ws) / abs(ws))
        to_wff.append(abs(flux - wff) / abs(wff))
    return max(to_ws), max(to_wff)


@pytest.mark.parametrize("kind,bar", [("pulsating", 0.03), ("oscillating", 0.04)])
def test_intensity_flux_is_the_radiated_power(kind, bar):
    coarse, fine = _radiator_flux_errors(kind, 2), _radiator_flux_errors(kind, 3)
    # against W_s: measured pulsating 5.4e-2 -> 2.9e-2, oscillating 5.7e-2 -> 3.7e-2 (W_s and W_ff differ by as much)
    converges(coarse[0], fine[0], bar)
    # against W_ff of the same surface values: energy conservation outside the body, up to the sphere rule at R = 1.5
    assert max(coarse[1], fine[1]) <= 1e-5, (coarse, fine)  # measured <= 3.6e-6


# ---- incident field and host helpers -----------------------------------------------------------------------------------------
def test_incident_gradient_equals_central_differences():
    ph = PhysicsParams.from_wave_number(7.0)
    pts = np.random.default_rng(0).uniform(-1.0, 1.0, (20, 3)) + [0.0, 0.0, 2.0]
    for inc in (IncidentField.plane_wave([0.3, -0.5, 0.8], 2.0), IncidentField.point_source([0.1, 0.2, -0.3], 3.0),
                IncidentField(plane_waves=IncidentField.plane_wave_z().plane_waves,
                              point_sources=IncidentField.point_source([0.0, 0.5, 0.0]).point_sources)):
        g = inc.evaluate_gradient(pts, ph)
        fd = _central_differences(lambda x: inc.evaluate_pressure(x, ph), pts, 1e-6)
        assert np.max(np.linalg.norm(g - fd, axis=1) / np.linalg.norm(g, axis=1)) <= 1e-8


@pytest.mark.parametrize("s", [1.0, -1.0])
def test_plane_wave_velocity_and_intensity(s):
    """a plane wave exp(i s k d.x): u = p d / (rho c), I = |p|^2 d / (2 rho c), and I.n is surface_power's integrand"""
    import dataclasses

    ph = dataclasses.replace(PhysicsParams.from_wave_number(3.0), harmonic_factor=s)
    d = np.array([0.36, 0.48, 0.8])
    x = np.random.default_rng(1).standard_normal((5, 3))
    p = 2.0 * np.exp(1j * s * ph.wave_number * (x @ d))
    grad = (1j * s * ph.wave_number * p)[:, None] * d
    rc = ph.density * ph.speed_of_sound
    assert np.allclose(postprocess.particle_velocity(grad, ph), p[:, None] * d / rc, rtol=1e-13, atol=0)
    intensity = postprocess.sound_intensity(p, grad, ph)
    assert np.allclose(intensity, 2.0 * d[None, :] / rc, rtol=1e-13, atol=0)
    n = np.array([0.0, 0.6, 0.8])
    dpdn = grad @ n
    assert np.allclose(intensity @ n, -s / (2 * ph.omega * ph.density) * np.imag(p * np.conj(dpdn)), rtol=1e-13, atol=0)


# ---- argument checks --------------------------------------------------------------------------------------------------------
def _staged(n=10):
    return types.SimpleNamespace(num_dofs=n, enum_to_dof=None, _h=None, ctx=types.SimpleNamespace(_h=None))


def test_python_wrapper_refuses_bad_arguments():
    st = _staged(10)
    ph = PhysicsParams.from_wave_number(2.0)
    pts = np.ones((2, 3))
    p = np.zeros(10, np.complex128)
    for bad in (np.ones(3), np.ones((0, 3)), np.ones((2, 2)), [[np.nan, 0.0, 1.0]], [[0.0, np.inf, 1.0]]):
        with pytest.raises(ValueError):
            bem.evaluate_field_gradient(bad, st, p, None, ph)
    for bad in (np.zeros(9), np.zeros((2, 9)), np.zeros((0, 10)), np.zeros((4097, 10))):
        with pytest.raises(ValueError):
            bem.evaluate_field_gradient(pts, st, bad, None, ph)
    with pytest.raises(ValueError):
        bem.evaluate_field_gradient(pts, st, p, np.zeros((1, 10)), ph)  # 1-D pressure, 2-D velocity
    with pytest.raises(ValueError):
        bem.evaluate_field_gradient(pts, st, np.zeros((2, 10)), None, ph, nsol=3)
    for ptr, nsol in ((1 << 20, None), (1 << 20, 0), (1 << 20, 5000), (True, 1), (-5, 1)):
        with pytest.raises(ValueError):
            bem.evaluate_field_gradient(pts, st, ptr, None, ph, nsol=nsol)
    with pytest.raises(ValueError):  # mixed host / device inputs
        bem.evaluate_field_gradient(pts, st, 1 << 20, np.zeros((2, 10)), ph, nsol=2)
    with pytest.raises(ValueError):
        postprocess.evaluate_field_gradient(np.ones((1, 2)), st, p, None, ph)


def test_c_entry_refuses_bad_arguments_without_a_device():
    lib = _capi.lib()
    ph = _capi.CPhysics(1.0, 1.0, 1.0, 1.0)
    x = (C.c_double * 6)(0.0, 0.0, 1.0, 1.0, 0.0, 0.0)
    vals = (C.c_double * 64)()
    out_p = (C.c_double * 64)()
    out_g = (C.c_double * 64)()

    def call(sm=None, phys=C.byref(ph), nsol=1, p=vals, v=None, on_device=0, n_eval=2, pts=x, op=out_p, og=out_g):
        rc = lib.bemb200_evaluate_field_gradient(sm, phys, nsol, p, v, on_device, n_eval, pts, op, og)
        return rc, lib.bemb200_last_error(None).decode()

    assert call() == (EINVAL, "NULL staged mesh")  # every other argument is valid
    assert call(op=None) == (EINVAL, "NULL staged mesh")  # out_p is optional
    for kw, msg in ((dict(phys=None), "NULL"), (dict(p=None), "NULL"), (dict(pts=None), "NULL"), (dict(og=None), "NULL"),
                    (dict(nsol=0), "solutions"), (dict(nsol=4097), "solutions"), (dict(on_device=2), "on_device"),
                    (dict(on_device=-1), "on_device"), (dict(n_eval=0), "evaluation points"),
                    (dict(n_eval=1 << 31), "evaluation points")):
        rc, err = call(**kw)
        assert rc == EINVAL and msg in err, (kw, err)
    for bad in ((float("nan"), 0.0, 1.0), (0.0, float("inf"), 0.0), (0.0, 0.0, -float("inf"))):
        rc, err = call(pts=(C.c_double * 6)(0.0, 0.0, 1.0, *bad))
        assert rc == EINVAL and "evaluation point 1 " in err, (bad, err)


def test_cpp_evaluate_field_gradient_wrapper_compiles_and_links(tmp_path):
    """bemb200::evaluate_field_gradient (include/bemb200.hpp) against the library's exported symbols, warnings as errors."""
    exe = tmp_path / "instantiate_evaluate_field_gradient"
    libdir = _capi.LIB_PATH.parent
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", str(ROOT / "include"),
           str(ROOT / "tests" / "cpp" / "instantiate_evaluate_field_gradient.cpp"), "-o", str(exe), f"-L{libdir}", "-lbemb200",
           f"-Wl,-rpath,{libdir}"]
    subprocess.run(cmd, check=True)
    assert subprocess.run([str(exe)]).returncode == 0  # nothing is executed: main returns before touching the GPU
