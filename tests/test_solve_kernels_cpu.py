"""Solve-phase kernel tests that need no GPU: the test shim over the launchers cross-compiles for sm_100a and exports its
entry points, the extended-precision reference is checked against numpy and against hand-built cases, and the stream-K
split of the block product is checked never to give a tile more partials than block_fixup_kernel can add."""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import solve_kernels_reference as R  # noqa: E402
import solve_kernels_shim as shim  # noqa: E402

LD = np.longdouble


@pytest.fixture(scope="module")
def shim_so(tmp_path_factory):
    return shim.build_shim(tmp_path_factory.mktemp("solve_shim"))


def test_shim_compiles_and_exports_every_entry_point(shim_so):
    lib = shim.load(shim_so)  # no libcuda needed: the CUDA runtime is linked in statically
    for name in shim.SIGNATURES:
        assert getattr(lib, name) is not None
    assert lib.shim_mgs_scratch_elems() == 148 * 2 * 64 + 148


def _crandn(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


@pytest.mark.parametrize("n,m", [(5, 1), (7, 3), (40, 12), (300, 64)])
def test_reference_mgs_matches_qr(n, m):
    rng = np.random.default_rng(n * 100 + m)
    Q, _ = np.linalg.qr(_crandn(rng, n, m + 1))
    V, w = Q[:, :m], _crandn(rng, n)
    h, nrm, q = R.mgs(V.T, w)
    # with an orthonormal V, h = V^H w and w_perp = w - V h
    assert np.max(np.abs(h.astype(np.complex128) - V.conj().T @ w)) < 1e-13 * np.linalg.norm(w)
    wp = w - V @ (V.conj().T @ w)
    assert abs(float(nrm) - np.linalg.norm(wp)) < 1e-13 * np.linalg.norm(w)
    assert np.linalg.norm(q.astype(np.complex128) - wp / np.linalg.norm(wp)) < 1e-13
    # and against QR of [V w]: the last column of Q is q up to a unit phase, |R_mm| = ||w_perp||
    Q2, R2 = np.linalg.qr(np.column_stack([V, w]))
    assert abs(abs(R2[m, m]) - float(nrm)) < 1e-12 * np.linalg.norm(w)
    assert abs(abs(np.vdot(Q2[:, m], q.astype(np.complex128))) - 1.0) < 1e-12


def test_reference_mgs_known_coefficients():
    # V = first three unit vectors times exact unit phases, w = V c + 2 e_3: h = c, ||w_perp|| = 2, q = e_3, all exactly
    n = 6
    ph = np.array([1, 1j, -1j])
    V = np.zeros((n, 3), dtype=np.complex128)
    V[[0, 1, 2], [0, 1, 2]] = ph
    c = np.array([1 - 2j, 0.5 + 0.25j, -3 + 0j])
    w = V @ c
    w[3] = 2.0
    h, nrm, q = R.mgs(V.T, w)
    assert np.array_equal(h, c.astype(np.clongdouble))
    assert nrm == 2
    assert np.array_equal(q.astype(np.complex128), np.eye(n)[3])
    # pinv scales w first
    pinv = np.full(n, 0.5 - 0.5j)
    h2, nrm2, _ = R.mgs(V.T, w, pinv)
    assert np.array_equal(h2, (c * (0.5 - 0.5j)).astype(np.clongdouble))
    assert abs(nrm2 - np.sqrt(LD(2))) < 1e-18


def _mgs_fp64(V, w):
    w = w.copy()
    h = np.zeros(V.shape[1], dtype=np.complex128)
    for l in range(V.shape[1]):
        h[l] = np.vdot(V[:, l], w)
        w -= h[l] * V[:, l]
    return h


def test_reference_lowsync_identity_on_nonorthonormal_basis():
    # (I + L) h = V^H w with L_kl = v_k^H v_l (k > l) holds for ANY V; take one visibly non-orthonormal (|L| ~ 0.1)
    rng = np.random.default_rng(7)
    n, m = 50, 9
    V = np.linalg.qr(_crandn(rng, n, m))[0] + 0.03 * _crandn(rng, n, m)
    w = _crandn(rng, n)
    h, _, _ = R.mgs(V.T, w)
    L = R.gram_lower(V.T)
    lhs = (np.eye(m, dtype=np.clongdouble) + L) @ h
    rhs = V.astype(np.clongdouble).conj().T @ w.astype(np.clongdouble)
    assert np.max(np.abs(L)) > 0.05
    assert np.max(np.abs(lhs - rhs)) < 1e-17 * np.max(np.abs(rhs))
    # an FP64 MGS of the same inputs is off by ~1e-16: the longdouble reference resolves the kernels' rounding
    assert np.max(np.abs(lhs - rhs)) < 1e-2 * np.max(np.abs(h.astype(np.complex128) - _mgs_fp64(V, w)))


def test_reference_exact_int_matmul():
    rng = np.random.default_rng(3)
    A = rng.integers(-4, 5, (33, 70)) + 1j * rng.integers(-4, 5, (33, 70))
    X = rng.integers(-4, 5, (70, 8)) + 1j * rng.integers(-4, 5, (70, 8))
    Ai = A.real.astype(np.int64), A.imag.astype(np.int64)
    Xi = X.real.astype(np.int64), X.imag.astype(np.int64)
    want = (Ai[0] @ Xi[0] - Ai[1] @ Xi[1]) + 1j * (Ai[0] @ Xi[1] + Ai[1] @ Xi[0])
    assert np.array_equal(R.exact_int_matmul(A, X), want)
    with pytest.raises(ValueError):
        R.exact_int_matmul(A + 0.5, X)


def test_streamk_tile_contributors_fit_the_fixup_table():
    """block_fixup_kernel keeps at most 8 partial tiles per tile (s_src[8]); a ninth would be dropped without a trace.
    launch_streamk_t prevents it with G <= 6 ntiles.  Exhaustive over G0 = 148 SMs, ntiles <= 200, nk <= 4000."""
    best, at_max, interior = R.scan_contributors(200, 4000, 148)
    print(f"stream-K: at most {best} contributors per tile; reached at {len(at_max)} (ntiles, nk), e.g. "
          f"{sorted(at_max, key=lambda p: p[0] * p[1])[:6]}; a CTA range inside one tile at {len(interior)}, e.g. "
          f"{sorted(interior, key=lambda p: p[0] * p[1])[:6]}")
    print("GPU test shapes (nrows, ncols):", [R.shape_of(*c) for c in R.STREAMK_MAX_CASES + R.STREAMK_INTERIOR_CASES])
    assert best <= R.FIXUP_MAX
    at_max, interior = set(at_max), set(interior)
    assert all(c in at_max for c in R.STREAMK_MAX_CASES)
    assert all(c in interior for c in R.STREAMK_INTERIOR_CASES)
    for nt, nk in R.STREAMK_MAX_CASES + R.STREAMK_INTERIOR_CASES + R.STREAMK_EDGE_CASES:
        assert R.streamk_grid(*R.shape_of(nt, nk))[1:] == (nt, nk)


def test_streamk_closed_form_matches_fixup_walk():
    # the scan's closed form against a line-by-line mirror of block_fixup_kernel's walk, including its slot choice
    rng = np.random.default_rng(11)
    cases = [(int(rng.integers(1, 201)), int(rng.integers(1, 4001))) for _ in range(300)]
    for nt, nk in cases + R.STREAMK_MAX_CASES + R.STREAMK_INTERIOR_CASES + R.STREAMK_EDGE_CASES:
        G, _, _ = R.streamk_grid(nt * R.SK_BM, nk * R.SK_BK)
        U = nt * nk
        cnt = R.contributor_counts(nt, np.array([nk]))[0]
        for t in range(nt):
            src = R.fixup_sources(t, nk, G, U)
            assert (len(src) or 1) == cnt[t]
            if src:  # the first contributor started before the tile (slot 1 = a range's last segment), the others inside
                assert [s for _, s in src] == [1] + [0] * (len(src) - 1)
                assert [c for c, _ in src] == list(range(src[0][0], src[0][0] + len(src)))
