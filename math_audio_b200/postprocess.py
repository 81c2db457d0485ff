"""Host-side mirror of ``math-bem/src/core/postprocess/pressure.rs``: evaluation-point generators
(:311-424), ``FieldPoint`` (:24-56), ``compute_scattered_field`` (:81-137), ``compute_total_field``
(:273-309) and ``compute_rcs`` (:438-478).  The O(M N) sums run on the device
(``csrc/postprocess.cu`` behind ``bemb200_scattered_field`` / ``bemb200_compute_rcs``).

Beyond the reference: the complex far-field amplitude with the surface-velocity term (``compute_far_field``, device) and the
host-side quantities built on it -- ``sphere_quadrature``, ``far_field_power``, ``surface_power`` and ``directivity_index``
(DESIGN.md 4.9)."""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import bem
from .incident import IncidentField
from .types import PhysicsParams


@dataclass
class FieldPoint:
    """pressure.rs:24-56."""
    position: np.ndarray
    p_incident: complex
    p_scattered: complex

    @property
    def p_total(self) -> complex:
        return self.p_incident + self.p_scattered

    def magnitude(self) -> float:
        return abs(self.p_total)

    def spl_db(self) -> float:
        return 20.0 * math.log10(abs(self.p_total) / 20e-6)


def generate_sphere_eval_points(radius: float, n_theta: int, n_phi: int) -> np.ndarray:
    """pressure.rs:311-330: theta at cell centres, phi from 0."""
    pts = np.empty((n_theta * n_phi, 3))
    r = 0
    for i in range(n_theta):
        theta = math.pi * (i + 0.5) / n_theta
        st, ct = math.sin(theta), math.cos(theta)
        for j in range(n_phi):
            phi = 2.0 * math.pi * j / n_phi
            pts[r] = (radius * st * math.cos(phi), radius * st * math.sin(phi), radius * ct)
            r += 1
    return pts


def generate_line_eval_points(start, end, n_points: int) -> np.ndarray:
    """pressure.rs:332-343."""
    pts = np.empty((n_points, 3))
    den = max(n_points - 1, 1)
    for i in range(n_points):
        t = i / den
        pts[i] = [start[d] + t * (end[d] - start[d]) for d in range(3)]
    return pts


def generate_plane_eval_points(center, normal, extent: float, n_points: int) -> np.ndarray:
    """pressure.rs:345-424: n_points x n_points grid spanning [-extent, extent]^2 in the plane through ``center``."""
    n = np.asarray(normal, dtype=np.float64)
    n = n / math.sqrt(float(n @ n))
    arbitrary = np.array([1.0, 0.0, 0.0]) if abs(n[0]) < 0.9 else np.array([0.0, 1.0, 0.0])
    u = np.array([n[1] * arbitrary[2] - n[2] * arbitrary[1], n[2] * arbitrary[0] - n[0] * arbitrary[2], n[0] * arbitrary[1] - n[1] * arbitrary[0]])
    u = u / math.sqrt(float(u @ u))
    v = np.array([n[1] * u[2] - n[2] * u[1], n[2] * u[0] - n[0] * u[2], n[0] * u[1] - n[1] * u[0]])
    den = max(n_points - 1, 1)
    pts = np.empty((n_points * n_points, 3))
    r = 0
    for i in range(n_points):
        s = -extent + 2.0 * extent * i / den
        for j in range(n_points):
            t = -extent + 2.0 * extent * j / den
            pts[r] = [center[d] + s * u[d] + t * v[d] for d in range(3)]
            r += 1
    return pts


def compute_scattered_field(eval_points, staged: bem.StagedMesh, surface_pressure, surface_velocity, physics: PhysicsParams) -> np.ndarray:
    """pressure.rs:81-137 (device)."""
    return bem.compute_scattered_field(eval_points, staged, surface_pressure, surface_velocity, physics)


def evaluate_field(eval_points, staged: bem.StagedMesh, surface_pressure, surface_velocity, physics: PhysicsParams,
                   nsol: Optional[int] = None) -> np.ndarray:
    """Accurate scattered pressure, whole elements and adaptive near-surface quadrature (device; ``bem.evaluate_field``)."""
    return bem.evaluate_field(eval_points, staged, surface_pressure, surface_velocity, physics, nsol)


def compute_total_field(eval_points, staged: bem.StagedMesh, surface_pressure, surface_velocity: Optional[np.ndarray],
                        incident_field: IncidentField, physics: PhysicsParams, accurate: bool = False) -> List[FieldPoint]:
    """pressure.rs:273-309: incident (host, O(M)) + scattered (device, O(M N)).  ``accurate``: the scattered part from
    ``evaluate_field`` (whole elements, adaptive near the surface) instead of the reference's rule."""
    pts = np.ascontiguousarray(eval_points, dtype=np.float64).reshape(-1, 3)
    p_inc = incident_field.evaluate_pressure(pts, physics)
    if accurate:
        p_sc = bem.evaluate_field(pts, staged, surface_pressure, surface_velocity, physics)
    else:
        p_sc = bem.compute_scattered_field(pts, staged, surface_pressure, surface_velocity, physics)
    return [FieldPoint(pts[i].copy(), complex(p_inc[i]), complex(p_sc[i])) for i in range(pts.shape[0])]


def compute_rcs(surface_pressure, staged: bem.StagedMesh, direction, physics: PhysicsParams):
    """pressure.rs:438-478 (device)."""
    return bem.compute_rcs(surface_pressure, staged, direction, physics)


def compute_far_field(directions, staged: bem.StagedMesh, surface_pressure, surface_velocity, physics: PhysicsParams,
                      nsol: Optional[int] = None) -> np.ndarray:
    """Complex far-field amplitude F, p_scat(R d) = F(d) exp(i s k R) / R + O(1/R^2) (device; ``bem.compute_far_field``)."""
    return bem.compute_far_field(directions, staged, surface_pressure, surface_velocity, physics, nsol)


def sphere_quadrature(n_theta: int, n_phi: int):
    """(directions (n_theta * n_phi, 3), solid-angle weights) of a product rule on the unit sphere: Gauss-Legendre in
    cos(theta), uniform in phi (phi_j = 2 pi j / n_phi).  The weights sum to 4 pi; spherical harmonics of degree
    < min(2 n_theta, n_phi) are integrated exactly."""
    if int(n_theta) < 1 or int(n_phi) < 1:
        raise ValueError("n_theta and n_phi must be >= 1")
    x, w = np.polynomial.legendre.leggauss(int(n_theta))
    phi = 2.0 * math.pi * np.arange(int(n_phi)) / int(n_phi)
    st = np.sqrt(1.0 - x * x)
    dirs = np.stack([np.outer(st, np.cos(phi)), np.outer(st, np.sin(phi)), np.outer(x, np.ones_like(phi))], axis=-1).reshape(-1, 3)
    return dirs, np.repeat(w * (2.0 * math.pi / int(n_phi)), int(n_phi))


def far_field_power(F, weights, physics: PhysicsParams):
    """Radiated (or scattered) power W = 1/(2 rho c) sum_q w_q |F(d_q)|^2 of far-field amplitudes F ((M,) or (nsol, M)) over
    a sphere quadrature; a float, or one per solution."""
    F = np.asarray(F)
    w = np.asarray(weights, dtype=np.float64)
    if F.shape[-1] != w.shape[0] or w.ndim != 1:
        raise ValueError("F must have one entry per quadrature weight (last axis)")
    out = (np.abs(F) ** 2) @ w / (2.0 * physics.density * physics.speed_of_sound)
    return float(out) if np.ndim(out) == 0 else out


def surface_power(mesh, p, v, physics: PhysicsParams) -> float:
    """Power through the surface W = -(s / (2 omega rho)) sum_j A_j Im(p_j conj(v_j)) (s = harmonic_factor, v = dp/dn on
    the outward normal, A_j = Element.area), for surface vectors in enumeration order (entry j <-> the j-th non-evaluation
    element).  Positive when the surface radiates, negative when it absorbs."""
    rows = np.asarray(mesh.is_eval) == 0
    area = np.asarray(mesh.area, dtype=np.float64)[rows]
    p = np.asarray(p, dtype=np.complex128)
    v = np.asarray(v, dtype=np.complex128)
    if p.shape != area.shape or v.shape != area.shape:
        raise ValueError("p and v must have one entry per boundary element")
    return float(-physics.harmonic_factor / (2.0 * physics.omega * physics.density) * float(np.sum(area * np.imag(p * np.conj(v)))))


def directivity_index(F, weights, on_axis: int) -> float:
    """DI = 10 log10(4 pi |F(d_on_axis)|^2 / sum_q w_q |F(d_q)|^2) in dB, ``on_axis`` the index of the on-axis direction
    among the quadrature directions of ``F`` (M,)."""
    F = np.asarray(F)
    w = np.asarray(weights, dtype=np.float64)
    if F.ndim != 1 or w.shape != F.shape:
        raise ValueError("F and weights must be (M,) arrays of the same length")
    total = float(np.abs(F) ** 2 @ w)
    return 10.0 * math.log10(4.0 * math.pi * abs(F[int(on_axis)]) ** 2 / total)
