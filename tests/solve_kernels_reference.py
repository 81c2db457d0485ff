"""Extended-precision reference of the solve-phase kernels (linalg.cu, block_matvec.cu), and a Python mirror of the
stream-K work split of the block product.

TEST INFRASTRUCTURE ONLY.  Arithmetic is numpy ``longdouble``: on x86-64 the 80-bit x87 format, 64-bit mantissa, eleven
bits beyond FP64, so the reference's own rounding (~1e-19 relative) is far below the FP64 kernels' (~1e-16).

One Arnoldi step of the solver is a pure function of the stored basis v_0..v_j, the new vector w and the optional
elementwise preconditioner pinv.  Modified Gram-Schmidt of pinv * w against v_0..v_j defines its exact result; the
low-synchronisation kernels solve (I + L) h = V^H w with L_kl = v_k^H v_l (k > l), which in exact arithmetic gives the
same h for any V, orthonormal or not, so this one reference covers every kernel.
"""
from __future__ import annotations

import numpy as np

LD = np.longdouble


def _split(z) -> tuple[np.ndarray, np.ndarray]:
    z = np.asarray(z)
    return np.ascontiguousarray(z.real, dtype=LD), np.ascontiguousarray(z.imag, dtype=LD)


def mgs(V, w, pinv=None):
    """Modified Gram-Schmidt of w (times pinv elementwise, when given) against the basis vectors V[0], ..., V[m-1]
    (V: m x n, one FP64 complex vector per row, as the solver stores its basis).

    Returns (h, nrm, q): h[l] = v_l^H (w - sum_{k<l} h_k v_k) as clongdouble, nrm = ||w_perp|| as longdouble and
    q = w_perp / nrm as clongdouble (None when nrm == 0)."""
    V = np.asarray(V)
    wr, wi = _split(w)
    if pinv is not None:
        pr, pi = _split(pinv)
        wr, wi = wr * pr - wi * pi, wr * pi + wi * pr
    m = V.shape[0]
    h = np.zeros(m, dtype=np.clongdouble)
    for l in range(m):
        vr, vi = _split(V[l])
        hr = np.dot(vr, wr) + np.dot(vi, wi)  # conj(v) . w
        hi = np.dot(vr, wi) - np.dot(vi, wr)
        wr = wr - (hr * vr - hi * vi)
        wi = wi - (hr * vi + hi * vr)
        h[l] = hr + 1j * hi
    nrm = np.sqrt(np.dot(wr, wr) + np.dot(wi, wi))
    q = (wr / nrm + 1j * (wi / nrm)).astype(np.clongdouble) if nrm > 0 else None
    return h, nrm, q


def gram_lower(V) -> np.ndarray:
    """L_kl = v_k^H v_l for k > l, zero elsewhere (clongdouble), V one vector per row as in mgs: the loss of
    orthogonality the low-sync kernels carry."""
    Vl = np.asarray(V).astype(np.clongdouble)
    G = Vl.conj() @ Vl.T
    return np.tril(G, -1)


def matmul(A, X) -> np.ndarray:
    """A @ X in clongdouble (for Gaussian inputs; exact-integer checks use exact_int_matmul)."""
    return np.asarray(A).astype(np.clongdouble) @ np.asarray(X).astype(np.clongdouble)


def exact_int_matmul(A, X, check_integers: bool = True) -> np.ndarray:
    """A @ X for complex inputs whose parts are small integers, exactly, as complex128.

    Every product and partial sum of such inputs is an integer; while they stay below 2**53 FP64 represents them exactly
    and any summation order (BLAS included) gives the exact result, the same as an int64 product.  The bound is checked;
    so is integrality, unless the caller generated the inputs as integers (check_integers=False saves a pass)."""
    A = np.asarray(A)
    X = np.asarray(X)
    for Z in (A, X) if check_integers else ():
        if Z.size and not (np.all(Z.real == np.round(Z.real)) and np.all(Z.imag == np.round(Z.imag))):
            raise ValueError("exact_int_matmul needs integer-valued parts")
    amax = max(float(np.max(np.abs(A.real), initial=0)), float(np.max(np.abs(A.imag), initial=0)))
    xmax = max(float(np.max(np.abs(X.real), initial=0)), float(np.max(np.abs(X.imag), initial=0)))
    if 2.0 * A.shape[-1] * amax * xmax >= 2.0**53:
        raise ValueError("partial sums could exceed 2**53: the FP64 product would not be exact")
    Ar, Ai, Xr, Xi = (np.ascontiguousarray(z) for z in (A.real, A.imag, X.real, X.imag))
    return (Ar @ Xr - Ai @ Xi) + 1j * (Ar @ Xi + Ai @ Xr)


# ---- stream-K work split of the block product (block_matvec.cu) -----------------------------------------------------
SK_BM = 256  # rows per tile
SK_BK = 8  # k per work unit
FIXUP_MAX = 8  # block_fixup_kernel's table of contributors per tile (s_src[8])


def sk_range(c: int, G: int, U: int) -> tuple[int, int]:
    """Work units [u0, u1) of CTA c (mirror of sk_range)."""
    return c * U // G, (c + 1) * U // G


def streamk_grid(nrows: int, ncols: int, sms: int = 148) -> tuple[int, int, int]:
    """(G, ntiles, nk) as launch_streamk_t chooses them on a device with `sms` SMs."""
    nk = (ncols + SK_BK - 1) // SK_BK
    ntiles = (nrows + SK_BM - 1) // SK_BM
    G = sms
    if ntiles * nk < G:
        G = ntiles * nk
    if 6 * ntiles < G:
        G = 6 * ntiles
    return G, ntiles, nk


def fixup_sources(tile: int, nk: int, G: int, U: int) -> list[tuple[int, int]]:
    """(cta, slot) of every partial tile block_fixup_kernel adds for `tile`, in its order, WITHOUT its cap of 8 (so a
    ninth contributor shows); [] when one CTA covered the tile and wrote it directly.  Mirror of the kernel's walk."""
    t0, t1 = tile * nk, tile * nk + nk
    cg0 = t0 * G // U
    c = cg0 if cg0 < G - 1 else G - 1
    while c > 0 and sk_range(c, G, U)[0] > t0:
        c -= 1
    while sk_range(c, G, U)[1] <= t0:
        c += 1
    out = []
    while c < G:
        u0, u1 = sk_range(c, G, U)
        if u0 >= t1:
            break
        a, b = max(u0, t0), min(u1, t1)
        if a < b:
            if a == t0 and b == t1:
                return []
            out.append((c, 0 if a > t0 else 1))
        c += 1
    return out


def contributor_counts(ntiles: int, nks: np.ndarray, sms: int = 148) -> np.ndarray:
    """Contributors per tile, shape (len(nks), ntiles), for every k-chunk count in `nks` (closed form of fixup_sources:
    with G <= U every CTA owns at least one unit, and unit u belongs to CTA floor(((u + 1) G - 1) / U))."""
    nks = np.asarray(nks, dtype=np.int64)[:, None]
    U = ntiles * nks
    G = np.minimum(np.minimum(sms, U), 6 * ntiles)
    t = np.arange(ntiles, dtype=np.int64)[None, :]
    first = t * nks
    last = first + nks - 1
    cta = lambda u: ((u + 1) * G - 1) // U  # noqa: E731
    return cta(last) - cta(first) + 1


def scan_contributors(max_tiles: int = 200, max_nk: int = 4000, sms: int = 148):
    """Exhaustive scan of ntiles <= max_tiles, nk <= max_nk.  Returns (max contributors, [(ntiles, nk) reaching it],
    [(ntiles, nk) where some CTA's range begins and ends inside one tile])."""
    nks = np.arange(1, max_nk + 1, dtype=np.int64)
    best, at_max, interior = 0, [], []
    for ntiles in range(1, max_tiles + 1):
        cnt = contributor_counts(ntiles, nks, sms).max(axis=1)
        m = int(cnt.max())
        if m > best:
            best, at_max = m, []
        if m == best:
            at_max += [(ntiles, int(nk)) for nk in nks[cnt == best]]
        interior += [(ntiles, int(nk)) for nk in nks[cnt >= 3]]  # a middle contributor lies wholly inside the tile
    return best, at_max, interior


def shape_of(ntiles: int, nk: int) -> tuple[int, int]:
    """An (nrows, ncols) with this tile / k-chunk count whose last tile and last chunk are both partial (when possible)."""
    nrows = ntiles * SK_BM - (37 if ntiles > 0 else 0)
    ncols = nk * SK_BK - (3 if nk > 0 else 0)
    return nrows, ncols


# Block-product shapes of the GPU test (G = 148), as (ntiles, nk), picked from scan_contributors' lists (the CPU test
# checks them against a fresh scan): tiles with the most contributors (7; 148 CTAs over 25..29 tiles), and tiles where a
# CTA's whole range lies inside one tile so that it writes only its slot-0 partial, plus a one-unit and a one-chunk case.
STREAMK_MAX_CASES = [(25, 7), (27, 501), (26, 1333)]
STREAMK_INTERIOR_CASES = [(1, 3), (3, 3), (7, 45), (40, 11)]
STREAMK_EDGE_CASES = [(1, 1), (150, 1)]
