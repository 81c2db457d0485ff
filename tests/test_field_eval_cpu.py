"""Accurate field evaluation (DESIGN.md 4.10) on the CPU, no GPU: the numpy restatement (tests/field_eval_oracle.py) against
Gauss's solid-angle identity, against independent single-element integrals, against Kirchhoff-Helmholtz reproductions of a
point source and the exact rigid-sphere series close to the surface, and against the far field it tends to; plus the argument
checks of the Python and C entries.

Every physics bar is a number measured here on two meshes (icosphere(2) -> icosphere(3); the Quad4 box of config 3 at
184 -> 784 elements), and each error must also shrink by a ratio < 0.75 with the refinement.  DESIGN.md 4.10 records the
table."""
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
import field_eval_oracle as fe  # noqa: E402

from math_audio_b200 import _capi, bem, postprocess  # noqa: E402
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
    if case == "warped":  # the nodes are shared, so the jittered surface stays closed: a closed warped bilinear surface
        mesh.nodes = mesh.nodes + 0.01 * np.random.default_rng(1).standard_normal(mesh.nodes.shape)
    return mesh


def _probe_points(mesh, e):
    """points above the centroid, an edge midpoint and a vertex of element e along its normal at DELTAS h, outside then
    inside: (points, expected static double layer of density 1)"""
    et = int(mesh.etype[e])
    x = mesh.nodes[mesh.conn[e, :et].astype(np.int64)]
    n = mesh.normal[e]
    h = fe.mesh_h(mesh)
    pts, want = [], []
    for base in (x.mean(axis=0), 0.5 * (x[0] + x[1]), x[0]):
        for d in DELTAS:
            for side, w in ((1.0, 0.0), (-1.0, -1.0)):
                pts.append(base + side * d * h * n)
                want.append(w)
    return np.array(pts), np.array(want)


# ---- Gauss's solid-angle identity -------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["sphere", "box", "warped"])
def test_solid_angle_identity_close_to_the_surface(case):
    """the static double layer of density 1 over a closed surface is -1 inside and 0 outside at every point off it"""
    mesh = _mesh(case)
    # a facet whose nodes are off the box's edges (a point above a node on an edge, along one face's normal, lies on the
    # other face: NaN by contract)
    e = 5 if case == "sphere" else int(np.argmin(np.linalg.norm(mesh.center - [-0.04, -0.055, 0.32], axis=1)))
    pts, want = _probe_points(mesh, e)
    one = np.ones(mesh.num_dofs)
    got = fe.evaluate_field(mesh, pts, one, None, 1e-9)
    err = np.abs(got - want)
    assert err.max() <= 1e-6, err.max()  # measured <= 1.1e-7 (icosphere(2), above a vertex at delta = 1)
    # the reference's rule at the same points misses by more than 1e-2 at every distance delta <= 0.1 (at single points its
    # errors can cancel: 8.4e-3 above an icosphere edge at delta = 0.01)
    today = np.abs(fo.scattered_field(mesh, pts, one, None, 1e-9) - want).reshape(3, len(DELTAS), 2)
    worst = today.max(axis=(0, 2))
    assert np.all(worst[np.array(DELTAS) <= 0.1] > 1e-2), worst


def test_point_on_the_surface_is_nan():
    mesh = _mesh("box")
    one = np.ones(mesh.num_dofs)
    pts = np.array([mesh.nodes[7], [0.0, 0.0, 2.0]])
    got = fe.evaluate_field(mesh, pts, one, None, 1.0)
    assert np.isnan(got[0]) and np.isfinite(got[1])


# ---- single elements ----------------------------------------------------------------------------------------------------
def _flat_reference(x, et, pt, w):
    """(int G, int dG/dn_y) over a flat convex polygon by polar coordinates about the foot point of pt: the radial integrals
    in closed form, the angular one by scipy quad with breaks at the vertex angles"""
    from scipy.integrate import quad

    poly = x[:et]
    n = np.cross(poly[1] - poly[0], poly[2] - poly[0])
    n = n / np.linalg.norm(n)
    z0 = float((pt - poly[0]) @ n)
    foot, az = pt - z0 * n, abs(z0)
    t1 = (poly[1] - poly[0]) / np.linalg.norm(poly[1] - poly[0])
    t2 = np.cross(n, t1)
    P = np.array([[(v - foot) @ t1, (v - foot) @ t2] for v in poly])

    def radius(th):
        u, best = np.array([math.cos(th), math.sin(th)]), np.inf
        for i in range(len(P)):
            a, e = P[i], P[(i + 1) % len(P)] - P[i]
            s, t = np.linalg.solve(np.array([[u[0], -e[0]], [u[1], -e[1]]]), a)
            if s > 0 and -1e-12 <= t <= 1 + 1e-12:
                best = min(best, s)
        return best

    def radial(th):
        r1 = math.hypot(radius(th), az)
        a = (np.exp(1j * w * r1) - np.exp(1j * w * az)) / (4 * math.pi * 1j * w)
        b = -z0 / (4 * math.pi) * (np.exp(1j * w * r1) / r1 - np.exp(1j * w * az) / az)
        return a, b

    breaks = list(np.sort(np.mod(np.arctan2(P[:, 1], P[:, 0]), 2 * math.pi))) + [2 * math.pi]
    out = [0j, 0j]
    lo = 0.0
    for hi in breaks:
        for i in range(2):
            for part in (np.real, np.imag):
                val = quad(lambda th: float(part(radial(th)[i])), lo, hi, epsabs=0, epsrel=1e-12, limit=200)[0]
                out[i] += val if part is np.real else 1j * val
        lo = hi
    return tuple(out)


H = 0.1
ELEMENTS = {
    "tri": (3, H * np.array([[0.0, 0.0, 0.0], [1.0, 0.1, 0.0], [0.2, 0.9, 0.0]])),
    "planar_quad": (4, H * np.array([[0.0, 0.0, 0.0], [1.0, 0.05, 0.0], [1.1, 1.0, 0.0], [-0.1, 0.9, 0.0]])),
    "warped_quad": (4, H * np.array([[0.0, 0.0, 0.0], [1.0, 0.1, 0.15], [1.1, 1.0, -0.1], [0.0, 0.9, 0.2]])),
}


@pytest.mark.parametrize("name", list(ELEMENTS))
@pytest.mark.parametrize("kh", [0.1, 1.0, 3.0])
def test_single_element_integrals(name, kh):
    """flat elements against polar integration about the foot point; the warped quad against itself with acceptance
    ratio 6 instead of 3"""
    et, x = ELEMENTS[name]
    n = np.cross(x[1] - x[0], x[2] - x[0])
    n = n / np.linalg.norm(n)
    foot = 0.7 * x[:et].mean(axis=0) + 0.3 * x[0]
    k = kh / H
    for d in (1.0, 0.1, 0.01):
        pt = foot + d * H * n
        a, b = fe.element_integrals(x, et, pt, k)
        ra, rb = fe.element_integrals(x, et, pt, k, accept=6.0) if name == "warped_quad" else _flat_reference(x, et, pt, k)
        assert abs(a - ra) <= 1e-6 * abs(ra) and abs(b - rb) <= 1e-6 * abs(rb), (d, a, ra, b, rb)  # measured <= 6.6e-8


# ---- Kirchhoff-Helmholtz: a point source inside, reproduced outside from its own surface values -------------------------
X0 = np.array([0.02, -0.03, 0.05])


def _point_source_error(mesh, k):
    c, n = mesh.center, mesh.normal
    rv = c - X0
    r = np.linalg.norm(rv, axis=1)
    p = np.exp(1j * k * r) / (4 * math.pi * r)
    v = p * (1j * k - 1 / r) * (np.sum(rv * n, axis=1) / r)
    h = fe.mesh_h(mesh)
    pts = np.array([c[e] + d * h * n[e] for e in (3, 40, 97) for d in (2.0, 1.0, 0.1, 0.01)])
    rx = np.linalg.norm(pts - X0, axis=1)
    exact = np.exp(1j * k * rx) / (4 * math.pi * rx)
    got = fe.evaluate_field(mesh, pts, p, v, k)
    return float(np.linalg.norm(got - exact) / np.linalg.norm(exact))


def test_kirchhoff_helmholtz_quad4_box():
    e = [_point_source_error(generate_box_mesh_quad(0.32, 0.44, 0.64, nx, ny, nz), 10.0) for nx, ny, nz in ((4, 5, 8), (8, 11, 16))]
    converges(*e, 0.006)  # measured 1.7e-2 -> 4.8e-3 (the reference's rule: 35 %)


def test_kirchhoff_helmholtz_sphere():
    e = [_point_source_error(generate_icosphere_mesh(0.3, sub), 10.0) for sub in (2, 3)]
    converges(*e, 0.0025)  # measured 7.9e-3 -> 2.0e-3


# ---- close to a rigid sphere: exact series outside, extinction inside ---------------------------------------------------
@functools.lru_cache(maxsize=None)
def rigid_sphere(sub, ka):
    """(mesh, p) of the sign-consistent formulation (forced sign +1, consistent beta, adaptive beta) on icosphere(sub),
    radius 1, plane wave exp(ikz)"""
    from oracle import oracle as orc

    mesh = generate_icosphere_mesh(1.0, sub)
    k = ka
    scale = 4.0 if ka < 1.2 else (8.0 if ka < 1.8 else 16.0)
    beta = 1j * scale / k
    A, rhs, _ = ao.assemble_opts(mesh, k, beta, dg_dn_sign=1, consistent_beta=True)
    inc, _ = orc.incident_rhs(0, [0, 0, 1], 1.0, mesh.center, mesh.normal, k, beta)
    return mesh, np.linalg.solve(A, rhs + inc)


def _near_sphere_errors(sub, ka):
    """(outside error against the series, inside |p_total|) at c_e +- delta h n_e, delta in {1, 0.1, 0.01}, above a few
    facets: normwise relative to the series outside, to the unit incident wave inside"""
    mesh, p = rigid_sphere(sub, ka)
    h = fe.mesh_h(mesh)
    es = np.flatnonzero(np.abs(mesh.center[:, 2]) < 2.0)[:: max(1, mesh.n_elem // 12)]
    out_pts = np.array([mesh.center[e] + d * h * mesh.normal[e] for e in es for d in (1.0, 0.1, 0.01)])
    in_pts = np.array([mesh.center[e] - d * h * mesh.normal[e] for e in es for d in (1.0, 0.1, 0.01)])
    got = fe.evaluate_field(mesh, np.vstack([out_pts, in_pts]), p, None, ka)
    tot = got + np.exp(1j * ka * np.vstack([out_pts, in_pts])[:, 2])
    m = len(out_pts)
    exact = fe.sphere_total_field(ka, 1.0, out_pts)
    return float(np.linalg.norm(tot[:m] - exact) / np.linalg.norm(exact)), float(np.linalg.norm(tot[m:]) / math.sqrt(m))


@pytest.mark.parametrize("ka,bar_out", [(1.0, 0.003), (2.0, 0.005)])
def test_rigid_sphere_near_surface(ka, bar_out):
    coarse, fine = _near_sphere_errors(2, ka), _near_sphere_errors(3, ka)
    converges(coarse[0], fine[0], bar_out)  # measured ka = 1: 7.3e-3 -> 2.2e-3; ka = 2: 1.4e-2 -> 4.2e-3
    if ka == 1.0:
        converges(coarse[1], fine[1], 0.0035)  # measured 5.0e-3 -> 3.0e-3
    else:
        # at ka = 2 the interior value sits at 5e-3 on both meshes, as large at delta = 1 as at delta = 0.01: a floor of
        # the discrete solution, not of the evaluation near the surface, so no ratio is asked
        assert fine[1] <= 0.006, fine  # measured 5.2e-3 -> 5.4e-3


# ---- the far field and the reference's rule ----------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["sphere", "warped"])
@pytest.mark.parametrize("s", [1.0, -1.0])
def test_far_field_is_the_limit(case, s):
    """R exp(-i s k R) p(R d) -> far_field(d) on Tri3 and on (warped) Quad4, with a difference falling as 1/R"""
    mesh = generate_icosphere_mesh(1.0, 1) if case == "sphere" else _mesh("warped")
    rng = np.random.default_rng(3)
    n = mesh.num_dofs
    p = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    v = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    k = 2.0 if case == "sphere" else 9.0
    d, _ = fo.sphere_quadrature(5, 7)
    F = fo.far_field(mesh, d, p, v, k, s)
    diff = []
    for R in (1e4, 1e6):
        FR = fe.evaluate_field(mesh, R * d, p, v, k, s) * R * np.exp(-1j * s * k * R)
        diff.append(np.linalg.norm(FR - F) / np.linalg.norm(F))
    assert diff[0] < 1e-3 and 0.005 < diff[1] / diff[0] < 0.02, diff


def test_tri3_all_regular_points_equal_the_reference_rule():
    mesh = generate_icosphere_mesh(0.5, 2)
    rng = np.random.default_rng(4)
    n = mesh.num_dofs
    p = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    v = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    pts = 5.0 * fo.sphere_quadrature(4, 6)[0]
    for vel in (None, v):
        got, ref = fe.evaluate_field(mesh, pts, p, vel, 7.0), fo.scattered_field(mesh, pts, p, vel, 7.0)
        assert np.max(np.abs(got - ref)) <= 1e-13 * np.max(np.abs(ref))


# ---- argument checks --------------------------------------------------------------------------------------------------
def _staged(n=10, enum_to_dof=None):
    return types.SimpleNamespace(num_dofs=n, enum_to_dof=enum_to_dof, _h=None, ctx=types.SimpleNamespace(_h=None))


def test_python_wrapper_refuses_bad_arguments():
    st = _staged(10)
    ph = PhysicsParams.from_wave_number(2.0)
    pts = np.ones((2, 3))
    p = np.zeros(10, np.complex128)
    for bad in (np.ones(3), np.ones((0, 3)), np.ones((2, 2)), [[np.nan, 0.0, 1.0]], [[0.0, np.inf, 1.0]]):
        with pytest.raises(ValueError):
            bem.evaluate_field(bad, st, p, None, ph)
    for bad in (np.zeros(9), np.zeros((2, 9)), np.zeros((0, 10)), np.zeros((4097, 10))):
        with pytest.raises(ValueError):
            bem.evaluate_field(pts, st, bad, None, ph)
    with pytest.raises(ValueError):
        bem.evaluate_field(pts, st, p, np.zeros((1, 10)), ph)  # 1-D pressure, 2-D velocity
    with pytest.raises(ValueError):
        bem.evaluate_field(pts, st, p, np.zeros(9), ph)
    with pytest.raises(ValueError):
        bem.evaluate_field(pts, st, np.zeros((2, 10)), None, ph, nsol=3)
    for ptr, nsol in ((1 << 20, None), (1 << 20, 0), (1 << 20, 5000), (True, 1), (-5, 1)):
        with pytest.raises(ValueError):
            bem.evaluate_field(pts, st, ptr, None, ph, nsol=nsol)
    with pytest.raises(ValueError):  # mixed host / device inputs
        bem.evaluate_field(pts, st, 1 << 20, np.zeros((2, 10)), ph, nsol=2)
    with pytest.raises(ValueError):
        postprocess.evaluate_field(np.ones((1, 2)), st, p, None, ph)


def test_c_entry_refuses_bad_arguments_without_a_device():
    lib = _capi.lib()
    ph = _capi.CPhysics(1.0, 1.0, 1.0, 1.0)
    x = (C.c_double * 6)(0.0, 0.0, 1.0, 1.0, 0.0, 0.0)
    vals = (C.c_double * 64)()
    out = (C.c_double * 64)()

    def call(sm=None, phys=C.byref(ph), nsol=1, p=vals, v=None, on_device=0, n_eval=2, pts=x, o=out):
        rc = lib.bemb200_evaluate_field(sm, phys, nsol, p, v, on_device, n_eval, pts, o)
        return rc, lib.bemb200_last_error(None).decode()

    assert call() == (EINVAL, "NULL staged mesh")  # every other argument is valid
    for kw, msg in ((dict(phys=None), "NULL"), (dict(p=None), "NULL"), (dict(pts=None), "NULL"), (dict(o=None), "NULL"),
                    (dict(nsol=0), "solutions"), (dict(nsol=4097), "solutions"), (dict(on_device=2), "on_device"),
                    (dict(on_device=-1), "on_device"), (dict(n_eval=0), "evaluation points"),
                    (dict(n_eval=1 << 31), "evaluation points")):
        rc, err = call(**kw)
        assert rc == EINVAL and msg in err, (kw, err)
    for bad in ((float("nan"), 0.0, 1.0), (0.0, float("inf"), 0.0), (0.0, 0.0, -float("inf"))):
        rc, err = call(pts=(C.c_double * 6)(0.0, 0.0, 1.0, *bad))
        assert rc == EINVAL and "evaluation point 1 " in err, (bad, err)


def test_cpp_evaluate_field_wrapper_compiles_and_links(tmp_path):
    """bemb200::evaluate_field (include/bemb200.hpp) against the library's exported symbols, warnings as errors."""
    exe = tmp_path / "instantiate_evaluate_field"
    libdir = _capi.LIB_PATH.parent
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", str(ROOT / "include"),
           str(ROOT / "tests" / "cpp" / "instantiate_evaluate_field.cpp"), "-o", str(exe), f"-L{libdir}", "-lbemb200",
           f"-Wl,-rpath,{libdir}"]
    subprocess.run(cmd, check=True)
    assert subprocess.run([str(exe)]).returncode == 0  # nothing is executed: main returns before touching the GPU
