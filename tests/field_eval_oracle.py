"""numpy restatement of the accurate field evaluation of ``bemb200_evaluate_field`` (DESIGN.md 4.10), plus the exact sphere
fields of its tests.  TEST INFRASTRUCTURE ONLY: element by element in enumeration order, the pair split, the subdivision
rule and the quadrature written out again.

  p_sc(x) = sum_j p_j int_{E_j} dG/dn_y dS - v_j int_{E_j} G dS,  G = exp(i w r) / (4 pi r),  w = s k

over the whole element (Tri3: flat triangle, normal e1 x e2 / |e1 x e2|; Quad4: bilinear map, its Jacobian and normal).
A pair is regular when |x - c_e|^2 >= (ETA rho_e)^2 (c_e: node mean, rho_e: largest centroid-to-node distance) and takes
the rule of ``far_field_oracle.element_points``; otherwise the element is split 4 ways in its parameter domain until
|x - y(sub-centre)| >= ACCEPT sqrt(sub-area), and accepted pieces take TR13 (Tri3) or 4 x 4 Gauss-Legendre (Quad4).  A
piece not accepted at depth L_MAX makes the point's value NaN.
"""
from __future__ import annotations

import math

import numpy as np

import far_field_oracle as fo

ETA = 4.0
ACCEPT = 3.0
L_MAX = 30

TR13 = np.array([  # BEMQ_TR13 of csrc/quad_tables.h (xi, eta, weight on the unit triangle x 2)
    [0.333333333333333, 0.333333333333333, -0.149570044467682],
    [0.260345966079040, 0.260345966079040, 0.175615257433208],
    [0.260345966079040, 0.479308067841920, 0.175615257433208],
    [0.479308067841920, 0.260345966079040, 0.175615257433208],
    [0.065130102902216, 0.065130102902216, 0.053347235608838],
    [0.065130102902216, 0.869739794195568, 0.053347235608838],
    [0.869739794195568, 0.065130102902216, 0.053347235608838],
    [0.638444188569810, 0.048690315425316, 0.077113760890257],
    [0.048690315425316, 0.638444188569810, 0.077113760890257],
    [0.638444188569810, 0.312865496004874, 0.077113760890257],
    [0.312865496004874, 0.638444188569810, 0.077113760890257],
    [0.048690315425316, 0.312865496004874, 0.077113760890257],
    [0.312865496004874, 0.048690315425316, 0.077113760890257],
])
GL4_X = np.array([-0.8611363115940526, -0.3399810435848563, 0.3399810435848563, 0.8611363115940526])
GL4_W = np.array([0.3478548451374538, 0.6521451548625461, 0.6521451548625461, 0.3478548451374538])


def centroid_rho2(x, et):
    """(node mean, largest squared centroid-to-node distance)"""
    c = x[:et].sum(axis=0) / et
    d = x[:et] - c
    return c, float(np.max(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]))


def is_regular(pt, c, rho2, eta=ETA):
    d = pt - c
    return d[0] * d[0] + d[1] * d[1] + d[2] * d[2] >= eta * eta * rho2


def _quad_map(x, xi, eta):
    """y, N = dy/dxi x dy/deta of the bilinear map at arrays xi, eta"""
    sh = 0.25 * np.stack([(1 - xi) * (1 - eta), (1 + xi) * (1 - eta), (1 + xi) * (1 + eta), (1 - xi) * (1 + eta)], axis=-1)
    y = sh @ x[:4]
    dxi = 0.25 * ((1 - eta)[..., None] * (x[1] - x[0]) + (1 + eta)[..., None] * (x[2] - x[3]))
    deta = 0.25 * ((1 - xi)[..., None] * (x[3] - x[0]) + (1 + xi)[..., None] * (x[2] - x[1]))
    return y, np.cross(dxi, deta)


def _tri_sub(P, child):
    m01, m12, m20 = (P[0] + P[1]) / 2, (P[1] + P[2]) / 2, (P[2] + P[0]) / 2
    return np.array(((P[0], m01, m20), (m01, P[1], m12), (m20, m12, P[2]), (m01, m12, m20))[child])


def _pieces(x, et, pt, accept):
    """accepted pieces of the near pair (point pt, element x) in depth-first order, children in order: Tri3 (parametric
    vertices (3, 2), depth), Quad4 ((xi0, eta0, side), depth); None when a piece reaches L_MAX unaccepted"""
    out = []
    if et == 3:
        nv = np.cross(x[1] - x[0], x[2] - x[0])
        area = 0.5 * np.linalg.norm(nv)
        stack = [(np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0]]), 0)]
    else:
        stack = [((-1.0, -1.0, 2.0), 0)]
    while stack:
        P, lvl = stack.pop()
        if et == 3:
            cp = P.sum(axis=0) / 3.0
            yc = (1.0 - cp[0] - cp[1]) * x[0] + cp[0] * x[1] + cp[1] * x[2]
            sub_area = area * 0.25 ** lvl
        else:
            h = P[2]
            yc, N = _quad_map(x, np.array(P[0] + 0.5 * h), np.array(P[1] + 0.5 * h))
            sub_area = float(np.linalg.norm(N)) * h * h
        d = yc - pt
        if d @ d >= accept * accept * sub_area:
            out.append((P, lvl))
            continue
        if lvl == L_MAX:
            return None
        if et == 3:
            kids = [_tri_sub(P, c) for c in range(4)]
        else:
            xi0, eta0, h = P
            g = 0.5 * h
            kids = [(xi0, eta0, g), (xi0 + g, eta0, g), (xi0, eta0 + g, g), (xi0 + g, eta0 + g, g)]
        stack.extend((kid, lvl + 1) for kid in reversed(kids))
    return out


def piece_points(x, et, P, lvl):
    """(y (Q, 3), w J (Q,), w N (Q, 3)) of an accepted piece: TR13 on the sub-triangle, 4 x 4 Gauss on the sub-square"""
    if et == 3:
        nv = np.cross(x[1] - x[0], x[2] - x[0])
        J = np.linalg.norm(nv) * 0.25 ** lvl
        u = P[0] + TR13[:, :1] * (P[1] - P[0]) + TR13[:, 1:2] * (P[2] - P[0])
        y = (1.0 - u[:, :1] - u[:, 1:2]) * x[0] + u[:, :1] * x[1] + u[:, 1:2] * x[2]
        w = TR13[:, 2] * 0.5 * J
        return y, w, w[:, None] * (nv / np.linalg.norm(nv))
    xi0, eta0, h = P
    g = 0.5 * h
    xi = np.repeat(xi0 + g + g * GL4_X, 4)
    eta = np.tile(eta0 + g + g * GL4_X, 4)
    w = np.repeat(GL4_W, 4) * np.tile(GL4_W, 4) * g * g
    y, N = _quad_map(x, xi, eta)
    return y, w * np.linalg.norm(N, axis=1), w[:, None] * N


def _ab(pt, y, wj, wn, w):
    """(int G, int dG/dn_y) of one point over quadrature points"""
    rv = y - pt
    r = np.linalg.norm(rv, axis=1)
    g = np.exp(1j * w * r) / (4.0 * math.pi * r)
    return complex(g @ wj), complex(np.sum(g * (-1.0 / r + 1j * w) * np.sum(rv * wn, axis=1) / r))


def near_pair(x, et, pt, w, accept=ACCEPT):
    """(int G, int dG/dn_y) of a near pair by adaptive subdivision; (nan, nan) on a point the rule cannot resolve"""
    pieces = _pieces(x, et, pt, accept)
    if pieces is None:
        return complex(np.nan, np.nan), complex(np.nan, np.nan)
    a = b = 0.0
    for P, lvl in pieces:
        da, db = _ab(pt, *piece_points(x, et, P, lvl), w)
        a, b = a + da, b + db
    return a, b


def evaluate_field(mesh, pts, p, v, k, s=1.0, eta=ETA, accept=ACCEPT):
    """p_sc at the (M, 3) points (v None: 0) -> (M,) complex"""
    x_all = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
    w = s * k
    out = np.zeros(len(x_all), dtype=np.complex128)
    for j, (et, xe) in enumerate(fo._elements(mesh)):
        vj = 0.0 if v is None else v[j]
        c, rho2 = centroid_rho2(xe, et)
        reg = np.array([is_regular(pt, c, rho2, eta) for pt in x_all])
        if reg.any():
            y, wj, wn = fo.element_points(xe, et)
            rv = y[None, :, :] - x_all[reg][:, None, :]
            r = np.linalg.norm(rv, axis=2)
            g = np.exp(1j * w * r) / (4.0 * math.pi * r)
            dgdn = g * (-1.0 / r + 1j * w) * np.einsum("mqd,qd->mq", rv, wn) / r
            out[reg] += p[j] * dgdn.sum(axis=1) - vj * (g @ wj)
        for m in np.flatnonzero(~reg):
            a, b = near_pair(xe, et, x_all[m], w, accept)
            out[m] += p[j] * b - vj * a
    return out


def element_integrals(x, et, pt, k, accept=ACCEPT):
    """(int G, int dG/dn_y) of one element (node coordinates x (et, 3)) at pt, as the evaluation treats the pair"""
    c, rho2 = centroid_rho2(x, et)
    if is_regular(pt, c, rho2):
        y, wj, wn = fo.element_points(x, et)
        return _ab(pt, y, wj, wn, k)
    return near_pair(x, et, pt, k, accept)


def mesh_h(mesh):
    return math.sqrt(float(np.mean(mesh.area[np.asarray(mesh.is_eval) == 0])))


def sphere_total_field(k, a, pts, Y=0.0, nterms=60):
    """exact p_inc + p_sc of the plane wave exp(ikz) on a sphere of radius a with dp/dr = Y p (Y = 0: rigid), outside"""
    from scipy.special import eval_legendre, spherical_jn

    pts = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
    r = np.linalg.norm(pts, axis=1)
    ct = pts[:, 2] / r
    out = np.exp(1j * k * pts[:, 2])
    for m in range(nterms):
        j, jp = spherical_jn(m, k * a), spherical_jn(m, k * a, True)
        am = -(k * jp - Y * j) / (k * fo._h(m, k * a, True) - Y * fo._h(m, k * a))
        out = out + (2 * m + 1) * (1j ** m) * am * fo._h(m, k * r) * eval_legendre(m, ct)
    return out
