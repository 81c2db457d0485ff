"""numpy restatement of the field gradient of ``bemb200_evaluate_field_gradient`` (DESIGN.md 4.11), on the pairs, pieces and
rules of ``field_eval_oracle``.  TEST INFRASTRUCTURE ONLY: element by element in enumeration order, the formulas written out
as the documentation states them.

  grad p_sc(x) = sum_j p_j int_{E_j} grad_x dG/dn_y dS - v_j int_{E_j} grad_x G dS,
  rv = y - x, G' = (i w - 1/r) G, G'' = ((i w - 1/r)^2 + 1/r^2) G, w = s k,
  grad_x G = -G' rv / r,   grad_x dG/dn_y = -(G'/r) n - (G'' - G'/r) (rv.n) rv / r^2.
"""
from __future__ import annotations

import math

import numpy as np

import far_field_oracle as fo
import field_eval_oracle as fe


def element_points_at(x, et, pt, eta=fe.ETA, accept=fe.ACCEPT):
    """(y, w J, w N) of every quadrature point the evaluation uses for the pair (pt, element x): the element's rule when the
    pair is regular, else the accepted pieces' rules concatenated; None when a piece reaches L_MAX unaccepted"""
    c, rho2 = fe.centroid_rho2(x, et)
    if fe.is_regular(pt, c, rho2, eta):
        return fo.element_points(x, et)
    pieces = fe._pieces(x, et, pt, accept)
    if pieces is None:
        return None
    parts = [fe.piece_points(x, et, P, lvl) for P, lvl in pieces]
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))


def gradient_integrals(pt, y, wj, wn, w):
    """(int grad_x G (3,), int grad_x dG/dn_y (3,)) over quadrature points (y, w J, w N)"""
    rv = y - pt
    r = np.linalg.norm(rv, axis=1)
    g = np.exp(1j * w * r) / (4.0 * math.pi * r)
    g1 = (1j * w - 1.0 / r) * g
    g2 = ((1j * w - 1.0 / r) ** 2 + 1.0 / r ** 2) * g
    rn = np.sum(rv * wn, axis=1)
    grad_g = -(g1 / r)[:, None] * rv
    grad_d = -(g1 / r)[:, None] * wn - ((g2 - g1 / r) * rn / r ** 2)[:, None] * rv
    return (wj[:, None] * grad_g).sum(axis=0), grad_d.sum(axis=0)


def element_gradient_integrals(x, et, pt, k, accept=fe.ACCEPT):
    """(int grad_x G, int grad_x dG/dn_y) of one element at pt, as the evaluation treats the pair (NaN when unresolved)"""
    q = element_points_at(x, et, pt, accept=accept)
    if q is None:
        nan = np.full(3, complex(np.nan, np.nan))
        return nan, nan
    return gradient_integrals(pt, *q, k)


def evaluate_field_gradient(mesh, pts, p, v, k, s=1.0, eta=fe.ETA, accept=fe.ACCEPT):
    """grad p_sc at the (M, 3) points (v None: 0) -> (M, 3) complex; NaN rows at points the rule cannot resolve"""
    x_all = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
    w = s * k
    out = np.zeros((len(x_all), 3), dtype=np.complex128)
    for j, (et, xe) in enumerate(fo._elements(mesh)):
        vj = 0.0 if v is None else v[j]
        c, rho2 = fe.centroid_rho2(xe, et)
        reg = np.array([fe.is_regular(pt, c, rho2, eta) for pt in x_all])
        if reg.any():  # the regular pairs of the element at once: the formulas of gradient_integrals, per point
            y, wj, wn = fo.element_points(xe, et)
            rv = y[None, :, :] - x_all[reg][:, None, :]
            r = np.linalg.norm(rv, axis=2)
            g = np.exp(1j * w * r) / (4.0 * math.pi * r)
            g1 = (1j * w - 1.0 / r) * g
            g2 = ((1j * w - 1.0 / r) ** 2 + 1.0 / r ** 2) * g
            rn = np.einsum("mqd,qd->mq", rv, wn)
            grad_g = (-(g1 / r) * wj[None, :])[:, :, None] * rv
            grad_d = -(g1 / r)[:, :, None] * wn[None, :, :] - ((g2 - g1 / r) * rn / r ** 2)[:, :, None] * rv
            out[reg] += p[j] * grad_d.sum(axis=1) - vj * grad_g.sum(axis=1)
        for m in np.flatnonzero(~reg):
            pieces = fe._pieces(xe, et, x_all[m], accept)
            if pieces is None:
                out[m] = np.nan
                continue
            parts = [fe.piece_points(xe, et, P, lvl) for P, lvl in pieces]
            ga, gb = gradient_integrals(x_all[m], *(np.concatenate([q[i] for q in parts]) for i in range(3)), w)
            out[m] += p[j] * gb - vj * ga
    return out


def static_double_layer_gradient(mesh, pt):
    """(grad D[1](pt), sum_q |w_q n_q| / (4 pi r_q^3)) of the static (k -> 0) double layer of density 1 on the evaluation's
    quadrature points: the identity grad D[1] = 0 off a closed surface, and the scale it is measured against"""
    g = np.zeros(3)
    scale = 0.0
    for et, xe in fo._elements(mesh):
        y, wj, wn = element_points_at(xe, et, pt)
        rv = y - pt
        r = np.linalg.norm(rv, axis=1)
        rn = np.sum(rv * wn, axis=1)
        # k -> 0: G = 1/(4 pi r), G' = -G/r, G'' = 2G/r^2, G'' - G'/r = 3G/r^2
        g += (wn / r[:, None] ** 3 - 3.0 * (rn / r ** 5)[:, None] * rv).sum(axis=0) / (4.0 * math.pi)
        scale += float(np.sum(np.linalg.norm(wn, axis=1) / r ** 3)) / (4.0 * math.pi)
    return g, scale
