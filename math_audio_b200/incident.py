"""Incident fields and the Burton-Miller right-hand side (host side, O(N)).

Mirror of math-bem/src/core/incident.rs: ``IncidentField::{plane_wave_z, plane_wave,
point_source}``, ``evaluate_pressure`` (:93-166), ``evaluate_normal_derivative`` (:177-280),
``compute_rhs`` / ``compute_rhs_with_beta`` (:293-342):  rhs = -(gamma p_inc + beta tau dp_inc/dn).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Tuple

import numpy as np

from .types import PhysicsParams


@dataclass
class IncidentField:
    plane_waves: List[Tuple[np.ndarray, complex]] = field(default_factory=list)    # (unit direction, amplitude)
    point_sources: List[Tuple[np.ndarray, complex]] = field(default_factory=list)  # (position, strength)

    @staticmethod
    def plane_wave_z() -> "IncidentField":  # incident.rs:46-51
        return IncidentField(plane_waves=[(np.array([0.0, 0.0, 1.0]), 1.0 + 0j)])

    @staticmethod
    def plane_wave_neg_z() -> "IncidentField":  # incident.rs:54-59
        return IncidentField.plane_wave([0.0, 0.0, -1.0], 1.0)

    @staticmethod
    def plane_wave(direction, amplitude: float = 1.0) -> "IncidentField":  # incident.rs:62-76
        d = np.asarray(direction, dtype=np.float64)
        ln = math.sqrt(d[0] ** 2 + d[1] ** 2 + d[2] ** 2)
        d = d / ln if ln > 1e-10 else np.array([0.0, 0.0, -1.0])
        return IncidentField(plane_waves=[(d, complex(amplitude, 0.0))])

    @staticmethod
    def point_source(position, strength: float = 1.0) -> "IncidentField":  # incident.rs:79-84
        return IncidentField(point_sources=[(np.asarray(position, dtype=np.float64), complex(strength, 0.0))])

    def evaluate_pressure(self, points: np.ndarray, physics: PhysicsParams) -> np.ndarray:
        k = physics.wave_number
        p = np.zeros(points.shape[0], dtype=np.complex128)
        for d, amp in self.plane_waves:
            kdotx = k * (d[0] * points[:, 0] + d[1] * points[:, 1] + d[2] * points[:, 2])
            p += amp * (np.cos(kdotx) + 1j * np.sin(kdotx))
        for pos, s in self.point_sources:
            dx, dy, dz = points[:, 0] - pos[0], points[:, 1] - pos[1], points[:, 2] - pos[2]
            r = np.sqrt(dx * dx + dy * dy + dz * dz)
            ok = r > 1e-10
            kr = k * r[ok]
            g = (np.cos(kr) + 1j * np.sin(kr)) / (4.0 * math.pi * r[ok])
            p[ok] += s * g
        return p

    def evaluate_gradient(self, points: np.ndarray, physics: PhysicsParams) -> np.ndarray:
        """(M, 3) gradient of ``evaluate_pressure`` as written (wave number k): i k d p for a plane wave, s (i k - 1/r) G
        (x - x_s) / r for a point source (0 where ``evaluate_pressure`` skips the source, r <= 1e-10)."""
        k = physics.wave_number
        points = np.asarray(points, dtype=np.float64).reshape(-1, 3)
        g = np.zeros(points.shape, dtype=np.complex128)
        for d, amp in self.plane_waves:
            kdotx = k * (d[0] * points[:, 0] + d[1] * points[:, 1] + d[2] * points[:, 2])
            p = amp * (np.cos(kdotx) + 1j * np.sin(kdotx))
            g += (1j * k * p)[:, None] * np.asarray(d, dtype=np.float64)[None, :]
        for pos, s in self.point_sources:
            dv = points - np.asarray(pos, dtype=np.float64)[None, :]
            r = np.sqrt(dv[:, 0] * dv[:, 0] + dv[:, 1] * dv[:, 1] + dv[:, 2] * dv[:, 2])
            ok = r > 1e-10
            kr = k * r[ok]
            gr = (np.cos(kr) + 1j * np.sin(kr)) / (4.0 * math.pi * r[ok])
            g[ok] += (s * (1j * k - 1.0 / r[ok]) * gr / r[ok])[:, None] * dv[ok]
        return g

    def evaluate_normal_derivative(self, points: np.ndarray, normals: np.ndarray, physics: PhysicsParams) -> np.ndarray:
        k = physics.wave_number
        out = np.zeros(points.shape[0], dtype=np.complex128)
        for d, amp in self.plane_waves:
            kdotx = k * (d[0] * points[:, 0] + d[1] * points[:, 1] + d[2] * points[:, 2])
            kdotn = k * (d[0] * normals[:, 0] + d[1] * normals[:, 1] + d[2] * normals[:, 2])
            p = amp * (np.cos(kdotx) + 1j * np.sin(kdotx))
            out += (1j * kdotn) * p
        for pos, s in self.point_sources:
            dx, dy, dz = points[:, 0] - pos[0], points[:, 1] - pos[1], points[:, 2] - pos[2]
            r = np.sqrt(dx * dx + dy * dy + dz * dz)
            ok = r > 1e-10
            kr = k * r[ok]
            g = (np.cos(kr) + 1j * np.sin(kr)) / (4.0 * math.pi * r[ok])
            dgdr = (1j * k - 1.0 / r[ok]) * g
            drdn = (dx[ok] * normals[ok, 0] + dy[ok] * normals[ok, 1] + dz[ok] * normals[ok, 2]) / r[ok]
            out[ok] += s * dgdr * drdn
        return out

    def compute_rhs_with_beta(self, centers: np.ndarray, normals: np.ndarray, physics: PhysicsParams, beta: complex) -> np.ndarray:
        p_inc = self.evaluate_pressure(centers, physics)
        dpdn = self.evaluate_normal_derivative(centers, normals, physics)
        return -(physics.gamma() * p_inc + beta * physics.tau * dpdn)

    def compute_rhs(self, centers, normals, physics: PhysicsParams, use_burton_miller: bool) -> np.ndarray:
        if use_burton_miller:
            return self.compute_rhs_with_beta(centers, normals, physics, physics.burton_miller_beta())
        return -physics.gamma() * self.evaluate_pressure(centers, physics)
