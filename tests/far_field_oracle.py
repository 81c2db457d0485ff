"""numpy restatement of the far-field amplitude of ``bemb200_far_field`` (DESIGN.md 4.9), of ``compute_scattered_field``'s
representation it is the limit of, and of the power and sphere-quadrature helpers, plus the exact far fields of the sphere
tests.  TEST INFRASTRUCTURE ONLY: element by element in enumeration order, the rules written out again.

Surface vectors are in enumeration order (entry j <-> the j-th non-evaluation element); s = harmonic_factor.
"""
from __future__ import annotations

import math

import numpy as np

TR7 = np.array([  # the 7-point triangle rule of csrc/postprocess.cu (xi, eta, weight on the unit triangle x 2)
    [0.333333333333333, 0.333333333333333, 0.225],
    [0.797426985353087, 0.101286507323456, 0.125939180544827],
    [0.101286507323456, 0.797426985353087, 0.125939180544827],
    [0.101286507323456, 0.101286507323456, 0.125939180544827],
    [0.470142064105115, 0.059715871789770, 0.132394152788506],
    [0.059715871789770, 0.470142064105115, 0.132394152788506],
    [0.470142064105115, 0.470142064105115, 0.132394152788506],
])


def element_points(x, etype, gauss=3):
    """(y (Q, 3), w J (Q,), w N (Q, 3)) of one element with node coordinates x (4, 3): Tri3 with TR7, Quad4 with a
    gauss x gauss Gauss-Legendre rule on the bilinear map (N = dy/dxi x dy/deta, J = |N|)."""
    if etype == 3:
        e1, e2 = x[1] - x[0], x[2] - x[0]
        nv = np.cross(e1, e2)
        y = (1.0 - TR7[:, :1] - TR7[:, 1:2]) * x[0] + TR7[:, :1] * x[1] + TR7[:, 1:2] * x[2]
        w = TR7[:, 2] * 0.5
        return y, w * np.linalg.norm(nv), w[:, None] * nv
    g, gw = np.polynomial.legendre.leggauss(gauss)
    xi, eta = np.repeat(g, gauss), np.tile(g, gauss)
    w = np.repeat(gw, gauss) * np.tile(gw, gauss)
    sh = 0.25 * np.stack([(1 - xi) * (1 - eta), (1 + xi) * (1 - eta), (1 + xi) * (1 + eta), (1 - xi) * (1 + eta)], axis=1)
    y = sh @ x
    dxi = 0.25 * ((1 - eta)[:, None] * (x[1] - x[0]) + (1 + eta)[:, None] * (x[2] - x[3]))
    deta = 0.25 * ((1 - xi)[:, None] * (x[3] - x[0]) + (1 + xi)[:, None] * (x[2] - x[1]))
    nv = np.cross(dxi, deta)
    return y, w * np.linalg.norm(nv, axis=1), w[:, None] * nv


def _elements(mesh):
    for e in np.flatnonzero(np.asarray(mesh.is_eval) == 0):
        et = int(mesh.etype[e])
        yield et, mesh.nodes[mesh.conn[e, :et].astype(np.int64)]


def far_field(mesh, dirs, p, v, k, s=1.0, gauss=3):
    """F(d) = 1/(4 pi) sum_j [-i s k (d.n) p_j - v_j] int_{E_j} exp(-i s k d.y) dS_y (v None: 0) -> (M,)"""
    d = np.asarray(dirs, dtype=np.float64).reshape(-1, 3)
    w = s * k
    F = np.zeros(len(d), dtype=np.complex128)
    for j, (et, x) in enumerate(_elements(mesh)):
        y, wj, wn = element_points(x, et, gauss)
        e = np.exp(-1j * w * (d @ y.T))  # (M, Q)
        a, b = e @ wj, ((d @ wn.T) * e).sum(axis=1)
        F += p[j] * (-1j * w) * b - (0.0 if v is None else v[j]) * a
    return F / (4.0 * math.pi)


def scattered_field(mesh, pts, p, v, k, s=1.0):
    """compute_scattered_field (csrc/postprocess.cu, pressure.rs:81-137): sum_j p_j int dG/dn_y - v_j int G on each element's
    first triangle with TR7 and its normal e1 x e2 / |e1 x e2|."""
    x = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
    w = s * k
    out = np.zeros(len(x), dtype=np.complex128)
    for j, (_, xe) in enumerate(_elements(mesh)):
        y, wj, wn = element_points(xe[:3], 3)
        en = wn[0] / np.linalg.norm(wn[0])
        rv = y[None, :, :] - x[:, None, :]
        r = np.linalg.norm(rv, axis=2)
        g = np.exp(1j * w * r) / (4.0 * math.pi * r)
        dgdn = g * (-1.0 / r + 1j * w) * (rv @ en) / r
        out += p[j] * (dgdn @ wj) - (0.0 if v is None else v[j]) * (g @ wj)
    return out


def sphere_quadrature(n_theta, n_phi):
    """Gauss-Legendre in cos(theta) x uniform phi: (directions, weights summing to 4 pi)"""
    x, w = np.polynomial.legendre.leggauss(n_theta)
    dirs, wts = [], []
    for xi, wi in zip(x, w):
        st = math.sqrt(1.0 - xi * xi)
        for j in range(n_phi):
            ph = 2.0 * math.pi * j / n_phi
            dirs.append([st * math.cos(ph), st * math.sin(ph), xi])
            wts.append(wi * 2.0 * math.pi / n_phi)
    return np.array(dirs), np.array(wts)


def surface_power(mesh, p, v, physics):
    """W_s = -(s / (2 omega rho)) sum_j A_j Im(p_j conj(v_j))"""
    area = mesh.area[np.asarray(mesh.is_eval) == 0]
    return -physics.harmonic_factor / (2.0 * physics.omega * physics.density) * float(np.sum(area * np.imag(p * np.conj(v))))


def _h(n, x, derivative=False):
    from scipy.special import spherical_jn, spherical_yn

    return spherical_jn(n, x, derivative) + 1j * spherical_yn(n, x, derivative)


def series_far_field(k, a, cos_theta, Y=0.0, R_over_a=1e5, nterms=40):
    """R exp(-i k R) p_scat(R) at R = R_over_a * a of a plane wave exp(ikz) on a sphere of radius a with dp/dr = Y p (Y = 0:
    rigid): the exact Robin series evaluated at a large distance."""
    from scipy.special import eval_legendre, spherical_jn

    R = R_over_a * a
    out = np.zeros(np.shape(cos_theta), dtype=np.complex128)
    for m in range(nterms):
        j, jp = spherical_jn(m, k * a), spherical_jn(m, k * a, True)
        am = -(k * jp - Y * j) / (k * _h(m, k * a, True) - Y * _h(m, k * a))
        out += (2 * m + 1) * (1j ** m) * am * _h(m, k * R) * eval_legendre(m, cos_theta)
    return out * R * np.exp(-1j * k * R)


def radiator_far_field(k, a, order, cos_theta, R_over_a=1e5):
    """R exp(-i k R) p(R) of the sphere with dp/dr = P_order(cos theta) on r = a (order 0: pulsating, 1: oscillating):
    p = h_order(kr) P_order / (k h_order'(ka))."""
    from scipy.special import eval_legendre

    R = R_over_a * a
    return _h(order, k * R) * eval_legendre(order, cos_theta) / (k * _h(order, k * a, True)) * R * np.exp(-1j * k * R)
