"""Every size-dispatched branch of the solve-phase kernels against an extended-precision reference, at the edges of its
size range, called through a test shim over the launchers (tests/cuda/solve_kernels_shim.cu) with no matrix assembled.

One Arnoldi step (launch_mgs) is checked along whole bases built the way gmres.cu builds them, so the Gram rows kept in
Lmat carry real state; the batched step, ZGEMV / ZGEMV^T, the stream-K block product and the residual kernel are checked
on their own.  Every kernel's name (and, where it tells placements apart, its grid and shared memory) is read back from
the profiler: the launchers demote silently to another kernel when one cannot be placed, and a test that passed on the
wrong kernel would prove nothing.

mgs_lowsync_kernel<4> and <8> are not tested: launch_mgs reaches them only for 4096 <= n <= 32768 after the cooperative
grid kernel has been demoted on the device, which a healthy B200 never does.

Bounds.  h, ||w_perp||: 4e-14 ||w|| (the longest chain of sequential additions is ~170: 148 CTA partials in order, a warp
tree and a slice; ~1.9e-14 ||w|| worst case), v_{j+1}: 4e-14 in 2-norm.  A dropped or twice-counted element moves h by
~||w|| / n, at least 3.8e-6 ||w|| at the largest n here.  The GEMV pair and the block product are fed small integers, so
every partial sum is exact and their results must match bit for bit.
"""
from __future__ import annotations

import json
import math
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import solve_kernels_reference as R  # noqa: E402
import solve_kernels_shim as shim  # noqa: E402

pytestmark = pytest.mark.gpu

BOUND = 4e-14
CPLX = 16  # bytes per complex128
INVALID_VALUE = 1  # cudaErrorInvalidValue
GR_CTAS, LS_MAXV = 148, 64


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    return shim.load(shim.build_shim(tmp_path_factory.mktemp("solve_shim")))


@pytest.fixture(scope="module")
def torch():
    import torch as t

    assert t.cuda.is_available(), "the solve-kernel tests need a CUDA device"
    t.cuda.init()
    return t


def _ptr(t, off=0):
    return None if t is None else t.data_ptr() + off * CPLX


def _ok(lib, rc):
    assert rc == 0, f"launcher returned cudaError {rc}"
    assert lib.shim_sync() == 0


def _nan(torch, *shape):
    return torch.full(shape, complex(float("nan"), float("nan")), dtype=torch.complex128, device="cuda")


def _crandn(torch, g, *shape):
    return torch.complex(torch.randn(*shape, generator=g, device="cuda", dtype=torch.float64),
                         torch.randn(*shape, generator=g, device="cuda", dtype=torch.float64))


def _bits(t):
    import torch as _t

    return _t.view_as_real(t).cpu().numpy().view(np.int64)


def _all_nan(t):
    import torch as _t

    return bool(_t.isnan(_t.view_as_real(t)).all())


def _profiled(torch, tmp_path, fn):
    """Runs fn under torch.profiler; returns (fn's result, [kernel trace events])."""
    from torch.profiler import ProfilerActivity, profile

    # A window that held nothing but the shim's launches came back from the profiler without kernel events on a B200
    # (torch 2.11); torch kernels on both sides of fn keep the window's device activity anchored, and show that the
    # profiler was recording when the expected kernel is missing.
    marker = torch.zeros(1, device="cuda")
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        marker.add_(1)
        torch.cuda.synchronize()
        out = fn()
        torch.cuda.synchronize()
        marker.add_(1)
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    kern = [e for e in json.loads(path.read_text())["traceEvents"] if e.get("cat") == "kernel"]
    if not kern:
        pytest.fail("the profiler recorded no kernel events: cannot tell which kernel ran")
    return out, kern


def _find(kern, name):
    return [e for e in kern if name in e.get("name", "")]


def _check_kernel(kern, name, grid=None, smem_min=None, smem_max=None):
    hits = _find(kern, name)
    assert hits, f"{name} did not run; kernels seen: {sorted({e['name'].split('(')[0] for e in kern})}"
    if grid is not None and all("grid" in e.get("args", {}) for e in hits):
        match = [e for e in hits if list(e["args"]["grid"]) == list(grid)]
        assert match, f"{name}: grids {sorted({tuple(e['args']['grid']) for e in hits})}, expected {grid}"
        hits = match
    e = hits[0]
    args = e.get("args", {})
    smem = args.get("shared memory")
    if smem is not None:
        if smem_min is not None:
            assert smem >= smem_min, f"{name}: {smem} B of shared memory, expected >= {smem_min}"
        if smem_max is not None:
            assert smem <= smem_max, f"{name}: {smem} B of shared memory, expected <= {smem_max}"
    return f"{e['name'].split('(')[0].split('::')[-1]} grid={args.get('grid')} smem={smem}"


# ---- which kernel launch_mgs picks (mirror of linalg.cu's dispatch on a device that demotes nothing) ----------------
def _cl_ept(n, threads=256):
    cl = 16 if n >= 2048 else (4 if n >= 512 else 1)
    S = -(-n // cl)
    ept = -(-S // threads)
    return cl, 1 if ept <= 1 else 2 if ept <= 2 else 4 if ept <= 4 else 8


def expected_mgs(n, j):
    """(kernel name, grid, min dynamic shared memory, max shared memory) of launch_mgs at (n, j)."""
    if j + 1 <= LS_MAXV and 4096 <= n <= GR_CTAS * 1024:
        S = -(-n // GR_CTAS)
        e, t = (1, 128) if S <= 128 else (2, 128) if S <= 256 else (2, 256) if S <= 512 else (4, 256)
        return f"mgs_grid_kernel<{e}, {t}>", (GR_CTAS, 1, 1), None, None
    if n <= 16 * 256 * 8:
        cl, e = _cl_ept(n)
        kind = "mgs_lowsync_kernel" if j + 1 <= LS_MAXV else "mgs_cluster_reg_kernel"
        return f"{kind}<{e}>", (cl, 1, 1), None, None
    cl = 8
    S = -(-n // cl)
    if S * CPLX > 200 * 1024:
        cl, S = 16, -(-n // 16)
    if S * CPLX <= 200 * 1024:
        return "mgs_cluster_kernel(", (cl, 1, 1), S * CPLX, None
    return "mgs_cluster_kernel(", (cl, 1, 1), None, 64 * 1024  # w in global memory


def _run_basis(torch, lib, n, restart, steps, seed, pinv, direct_scale, keep, breakdown_at=()):
    """Builds a basis with launch_mgs as gmres.cu does (one Lmat + scratch for the whole cycle); returns device V, H and
    the host copies of w taken before each step in `keep`, plus the breakdown launches' results."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    ldv, ldl = n + 13, restart + 1
    V = _nan(torch, steps + 2, ldv)  # padding rows and unwritten columns stay NaN
    H = _nan(torch, steps, steps + 2)
    Lm = _nan(torch, ldl * ldl + lib.shim_mgs_scratch_elems())
    v0 = _crandn(torch, g, n)
    V[0, :n] = v0 / torch.linalg.vector_norm(v0)
    ws, brk = {}, {}
    scratch = _ptr(Lm, ldl * ldl)
    for j in range(steps):
        w = _crandn(torch, g, n) / math.sqrt(2 * n)
        if j in breakdown_at:  # w in span(v_0..v_j) after pinv: ||w_perp|| ~ 1e-16, v_{j+1} must stay untouched
            c = _crandn(torch, g, j + 1)
            c /= torch.linalg.vector_norm(c)
            wb = (c[None, :] @ V[: j + 1, :n]).reshape(n)
            if pinv is not None:
                wb = wb / pinv
            hb = _nan(torch, j + 3)
            wb_h = wb.cpu().numpy()
            torch.cuda.synchronize()
            _ok(lib, lib.shim_mgs(_ptr(V), ldv, _ptr(wb), j, n, _ptr(hb), _ptr(V, (j + 1) * ldv), _ptr(pinv), direct_scale,
                                  _ptr(Lm), ldl, scratch))
            brk[j] = (wb_h, c.cpu().numpy(), hb.cpu().numpy(), _all_nan(V[j + 1]))
        if j in keep:
            ws[j] = w.cpu().numpy()
        torch.cuda.synchronize()
        _ok(lib, lib.shim_mgs(_ptr(V), ldv, _ptr(w), j, n, _ptr(H, j * (steps + 2)), _ptr(V, (j + 1) * ldv), _ptr(pinv),
                              direct_scale, _ptr(Lm), ldl, scratch))
    return V, H, ws, brk


COMPARE = (0, 1, 7, 8, 9, 31, 32, 33, 62, 63, 64, 65, 99)
COMPARE_SHORT = (0, 9, 33, 63, 64, 99)
LOWSYNC_N = (1, 2, 256, 257, 511, 512, 1024, 1025, 2047, 2048, 4095)
GRID_N = (4096, 4097, 18944, 18945, 37888, 37889, 75776, 75777, 151552)
GENERIC_N = (151553, 204800, 204801)
LONG_N = (4096, 4097, 8192, 8193, 16384, 16385, 32768, 32769, 102400, 102401)  # restart 100: j = 64 leaves LS_MAXV
MGS_CASES = ([(n, 64, "plain") for n in LOWSYNC_N + GRID_N + GENERIC_N] + [(n, 100, "plain") for n in LONG_N]
             + [(n, 64, v) for n in (257, 2048, 4097, 37889, 75777, 204801) for v in ("pinv", "pinv-direct")]
             + [(n, 100, v) for n in (8193, 16385, 102401) for v in ("pinv", "pinv-direct")])


@pytest.mark.parametrize("n,restart,variant", MGS_CASES)
def test_mgs_step_matches_reference(torch, lib, tmp_path, n, restart, variant):
    steps = min(restart, n)  # n <= restart: the basis is complete at j = n - 1, which must report a breakdown
    seed = n * 7 + restart
    pinv = pinv_h = None
    if variant != "plain":
        g = torch.Generator(device="cuda").manual_seed(seed + 1)
        mag = 0.5 * 4.0 ** torch.rand(n, generator=g, device="cuda", dtype=torch.float64)  # |pinv| in [0.5, 2]
        pinv = torch.polar(mag, 2 * math.pi * torch.rand(n, generator=g, device="cuda", dtype=torch.float64))
        pinv_h = pinv.cpu().numpy()
    ds = 1 if variant == "pinv-direct" else 0
    compare = [j for j in (COMPARE if variant == "plain" else COMPARE_SHORT) if j < steps] + [steps - 1]
    breakdown_at = tuple(j for j in (9, 65) if j + 1 < steps) if variant == "plain" else ()

    (V, H, ws, brk), kern = _profiled(torch, tmp_path, lambda: _run_basis(torch, lib, n, restart, steps, seed, pinv, ds,
                                                                          set(compare), breakdown_at))
    seen = []
    for j in sorted({0, steps - 1} | ({63, 64} & set(range(steps)))):
        name, grid, smin, smax = expected_mgs(n, j)
        seen.append(_check_kernel(kern, name, grid, smin, smax))

    # fixed summation order: the same inputs give the same bits (row-sharded ranks rely on it)
    V2, H2, _, _ = _run_basis(torch, lib, n, restart, steps, seed, pinv, ds, set(), breakdown_at)
    assert np.array_equal(_bits(V), _bits(V2)) and np.array_equal(_bits(H), _bits(H2))

    Vh, Hh = V.cpu().numpy(), H.cpu().numpy()
    assert np.isnan(Vh[:, n:]).all(), "a kernel wrote into the padding of the basis"
    assert np.isnan(Vh[steps + 1]).all(), "a kernel wrote past v_{j+1}"
    err = 0.0
    for j in sorted(set(compare)):
        w = ws[j]
        weff = w * pinv_h if pinv_h is not None else w
        wn = float(np.linalg.norm(weff))
        h_ref, nrm_ref, q_ref = R.mgs(Vh[: j + 1, :n], w, pinv_h)
        dh = float(np.max(np.abs(Hh[j, : j + 1] - h_ref))) / wn
        dn = abs(complex(Hh[j, j + 1]) - complex(nrm_ref)) / wn
        assert dh <= BOUND and dn <= BOUND, f"j={j}: |h - h_ref| = {dh:.2e} ||w||, |norm - ref| = {dn:.2e} ||w||"
        assert np.isnan(Hh[j, j + 2:]).all(), f"j={j}: the kernel wrote past hcol[j + 1]"
        err = max(err, dh, dn)
        if j == n - 1:  # the basis spans the space: breakdown, v_{j+1} untouched
            assert Hh[j, j + 1].real < 1e-14 and np.isnan(Vh[j + 1]).all()
            continue
        dv = float(np.linalg.norm(Vh[j + 1, :n] - q_ref))
        assert dv <= BOUND, f"j={j}: ||v_(j+1) - ref|| = {dv:.2e}"
        err = max(err, dv)
    for j, (wb, c, hb, untouched) in brk.items():
        h_ref, _, _ = R.mgs(Vh[: j + 1, :n], wb, pinv_h)
        wn = float(np.linalg.norm(wb * pinv_h if pinv_h is not None else wb))
        assert float(np.max(np.abs(hb[: j + 1] - h_ref))) <= BOUND * wn
        assert float(np.max(np.abs(hb[: j + 1] - c))) <= BOUND * wn
        assert hb[j + 1].real < 1e-14 and hb[j + 1].imag == 0 and untouched, f"j={j}: breakdown not reported / v_(j+1) written"
    print(f"\nROW mgs n={n} restart={restart} {variant}: {'; '.join(seen)}; max err {err:.2e} (bound {BOUND:.0e})")


# ---- batched step (launch_mgs_batched) ----------------------------------------------------------------------------
BATCHED_N = (2048, 4096, 4097, 8193, 16385, 32768, 32769, 196608)


def expected_batched(n, width):
    if n > 16 * 256 * 8:
        return "mgs_batched_smem_kernel", (16, width, 1)
    cl, e = _cl_ept(n)
    return f"mgs_batched_kernel<{e}>", (cl, width, 1)


@pytest.mark.parametrize("width", (8, 16, 24, 32))
@pytest.mark.parametrize("n", BATCHED_N)
def test_mgs_batched_step_matches_reference(torch, lib, tmp_path, n, width):
    steps, compare = 10, (0, 1, 9)
    ldv = n + 13
    vstride, hstride = (steps + 2) * ldv, steps * (steps + 1)
    g = torch.Generator(device="cuda").manual_seed(n + width)
    Vall = _nan(torch, width, steps + 2, ldv)
    Hb = _nan(torch, width, steps, steps + 1)
    off = [0, width // 2, width - 1]  # right-hand sides switched off: first, a middle one, last
    active = torch.ones(width, dtype=torch.uint8, device="cuda")
    active[off] = 0
    v0 = _crandn(torch, g, width, n)
    Vall[:, 0, :n] = v0 / torch.linalg.vector_norm(v0, dim=1, keepdim=True)
    ys = {}

    def run():
        for j in range(steps):
            Y = _crandn(torch, g, n, width) / math.sqrt(2 * n)  # interleaved [k][S]
            if j in compare:
                ys[j] = Y.cpu().numpy()
            X = _nan(torch, n, width)
            torch.cuda.synchronize()
            _ok(lib, lib.shim_mgs_batched(width, _ptr(Vall), ldv, vstride, _ptr(Y), j, n, _ptr(Hb, j * (steps + 1)), hstride,
                                          _ptr(X), _ptr(active)))
            Xh, Vn = X.cpu().numpy(), Vall[:, j + 1, :n].cpu().numpy()
            on = [s for s in range(width) if s not in off]
            assert np.isnan(Xh[:, off]).all(), "Xblk column of an inactive right-hand side written"
            assert np.array_equal(Xh[:, on].T, Vn[on]), "Xblk and the basis disagree"

    _, kern = _profiled(torch, tmp_path, run)
    name, grid = expected_batched(n, width)
    seen = _check_kernel(kern, name, grid)
    Vh, Hh = Vall.cpu().numpy(), Hb.cpu().numpy()
    assert np.isnan(Vh[off, 1:]).all() and np.isnan(Hh[off]).all(), "an inactive right-hand side was touched"
    assert np.isnan(Vh[:, :, n:]).all() and np.isnan(Vh[:, steps + 1]).all()
    err = 0.0
    for s in range(width):
        if s in off:
            continue
        for j in compare:
            w = ys[j][:, s]
            wn = float(np.linalg.norm(w))
            h_ref, nrm_ref, q_ref = R.mgs(Vh[s, : j + 1, :n], w)
            dh = float(np.max(np.abs(Hh[s, j, : j + 1] - h_ref))) / wn
            dn = abs(complex(Hh[s, j, j + 1]) - complex(nrm_ref)) / wn
            dv = float(np.linalg.norm(Vh[s, j + 1, :n] - q_ref))
            assert dh <= BOUND and dn <= BOUND and dv <= BOUND, f"rhs {s} j={j}: h {dh:.2e}, norm {dn:.2e}, v {dv:.2e}"
            err = max(err, dh, dn, dv)
    print(f"\nROW batched n={n} S={width}: {seen}; max err {err:.2e} (bound {BOUND:.0e})")


def test_mgs_batched_refuses_n_beyond_shared_memory(torch, lib, tmp_path):
    n, width = 196609, 8  # a 16-CTA slice of 12 289 > 12 288 complex numbers
    ldv = n + 13
    Vall = _nan(torch, width, 3, ldv)
    Vall[:, 0, :n] = 1.0 / math.sqrt(n)
    Hb, X = _nan(torch, width, 2), _nan(torch, n, width)
    Y = torch.ones(n, width, dtype=torch.complex128, device="cuda")
    torch.cuda.synchronize()
    rc, kern = None, []
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc = lib.shim_mgs_batched(width, _ptr(Vall), ldv, 3 * ldv, _ptr(Y), 0, n, _ptr(Hb), 2, _ptr(X), None)
        assert lib.shim_sync() == 0
    kern = [e.name for e in prof.events() if "mgs_batched" in e.name]
    assert rc == INVALID_VALUE and not kern
    assert _all_nan(Hb) and _all_nan(X) and _all_nan(Vall[:, 1:])


# ---- ZGEMV / ZGEMV^T / block product with exact integer inputs ---------------------------------------------------------
def _randint_c(torch, g, *shape):
    re = torch.randint(-4, 5, shape, generator=g, device="cuda", dtype=torch.float64)
    im = torch.randint(-4, 5, shape, generator=g, device="cuda", dtype=torch.float64)
    return torch.complex(re, im)


def _exact_rows(A, ncols, X, block=2048):
    """A[:, :ncols] @ X exactly (host), A on the device, in row blocks."""
    out = []
    for r0 in range(0, A.shape[0], block):
        out.append(R.exact_int_matmul(A[r0:r0 + block, :ncols].cpu().numpy(), X, check_integers=False))
    return np.concatenate(out)


GEMV_ROWS = (0, 1, 2, 3, 18943, 18944, 18945, 18946, 40001)
GEMV_COLS = (20480, 2049, 1025, 1024, 1023, 256, 255, 1)  # descending: each pass NaN-fills the columns it must not read


def test_zgemv_exact(torch, lib, tmp_path):
    g = torch.Generator(device="cuda").manual_seed(5)
    lda = GEMV_COLS[0] + 3
    A = _randint_c(torch, g, max(GEMV_ROWS), lda)
    x = _randint_c(torch, g, lda)
    nan = complex(float("nan"), float("nan"))

    def check(ncols):
        A[:, ncols:] = nan
        x[ncols:] = nan
        ref = _exact_rows(A, ncols, x[:ncols].cpu().numpy()[:, None])[:, 0]
        for nrows in GEMV_ROWS:
            y = _nan(torch, nrows + 3)
            torch.cuda.synchronize()
            _ok(lib, lib.shim_zgemv(_ptr(A), lda, nrows, ncols, _ptr(x), _ptr(y)))
            yh = y.cpu().numpy()
            assert np.array_equal(yh[:nrows], ref[:nrows]), f"ZGEMV {nrows} x {ncols}: not the exact product"
            assert np.isnan(yh[nrows:]).all(), f"ZGEMV {nrows} x {ncols}: wrote past y[nrows - 1]"

    for ncols in GEMV_COLS[:-1]:
        check(ncols)
    _, kern = _profiled(torch, tmp_path, lambda: check(GEMV_COLS[-1]))
    print(f"\nROW zgemv: {_check_kernel(kern, 'zgemv_kernel<2, 4, false>')}; bit-exact")


def test_zgemv_t_exact(torch, lib, tmp_path):
    g = torch.Generator(device="cuda").manual_seed(6)
    nrows_max, ncols_set = 40001, (1025, 257, 1)
    lda = ncols_set[0] + 5
    A = _randint_c(torch, g, nrows_max, lda)
    x = _randint_c(torch, g, nrows_max)
    nan = complex(float("nan"), float("nan"))

    def check(ncols):
        A[:, ncols:] = nan
        for nrows in (0, 1, 31, 32, 33, 1000, 40001):
            ref = R.exact_int_matmul(A[:nrows, :ncols].cpu().numpy().T, x[:nrows].cpu().numpy()[:, None])[:, 0]
            y = _nan(torch, ncols + 3)
            xs = x.clone()
            xs[nrows:] = nan  # x beyond nrows must not be read
            torch.cuda.synchronize()
            _ok(lib, lib.shim_zgemv_t(_ptr(A), lda, nrows, ncols, _ptr(xs), _ptr(y)))
            yh = y.cpu().numpy()
            assert np.array_equal(yh[:ncols], ref), f"ZGEMV^T {nrows} x {ncols}: not the exact product"
            assert np.isnan(yh[ncols:]).all()

    for ncols in ncols_set[:-1]:
        check(ncols)
    _, kern = _profiled(torch, tmp_path, lambda: check(ncols_set[-1]))
    print(f"\nROW zgemv_t: {_check_kernel(kern, 'zgemv_t_partial_kernel', (1, 32, 1))}, "
          f"{_check_kernel(kern, 'zgemv_t_reduce_kernel')}; bit-exact")


STREAMK_SHAPES = [R.shape_of(*c) for c in R.STREAMK_MAX_CASES + R.STREAMK_INTERIOR_CASES + R.STREAMK_EDGE_CASES]


def _block_case(torch, lib, nrows, ncols, nrhs, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    lda = ncols + 5
    A = _randint_c(torch, g, max(nrows, 1), lda)
    A[:, ncols:] = complex(float("nan"), float("nan"))
    X = _randint_c(torch, g, max(ncols, 1), nrhs)
    Y = _nan(torch, nrows + 1, nrhs)
    torch.cuda.synchronize()
    rc = lib.shim_zgemm_block(_ptr(A), lda, nrows, ncols, _ptr(X), _ptr(Y), nrhs)
    assert lib.shim_sync() == 0
    return rc, A, X, Y


@pytest.mark.parametrize("nrhs", (8, 16, 24, 32))
def test_zgemm_block_exact(torch, lib, tmp_path, nrhs):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    seen = None
    for i, (nrows, ncols) in enumerate(STREAMK_SHAPES + ([(20480, 20480)] if nrhs == 32 else [])):
        if i == 0:
            (rc, A, X, Y), kern = _profiled(torch, tmp_path, lambda: _block_case(torch, lib, nrows, ncols, nrhs, i))
            G = R.streamk_grid(nrows, ncols, sms)[0]
            seen = (_check_kernel(kern, f"zgemm_streamk_kernel<{nrhs // 8}>", (G, 1, 1)) + ", "
                    + _check_kernel(kern, f"block_fixup_kernel<{nrhs}>"))
        else:
            rc, A, X, Y = _block_case(torch, lib, nrows, ncols, nrhs, i)
        assert rc == 0
        ref = _exact_rows(A, ncols, X.cpu().numpy())
        Yh = Y.cpu().numpy()
        bad = np.argwhere(Yh[:nrows] != ref)
        assert bad.size == 0, f"{nrows} x {ncols}, S={nrhs}: {len(bad)} entries differ, first at row {bad[0][0]}"
        assert np.isnan(Yh[nrows]).all()
        del A, X, Y
    print(f"\nROW block S={nrhs} (G={sms}): {seen}; {len(STREAMK_SHAPES)} stream-K shapes bit-exact")


def test_zgemm_block_edges(torch, lib):
    for nrhs in (1, 9, 33):  # only 8, 16, 24 and 32 right-hand sides have a kernel
        rc, _, _, Y = _block_case(torch, lib, 300, 40, nrhs, 1)
        assert rc == INVALID_VALUE and _all_nan(Y)
    rc, _, _, Y = _block_case(torch, lib, 300, 0, 16, 2)  # empty sum: zeros
    assert rc == 0 and int(torch.count_nonzero(torch.view_as_real(Y[:300]))) == 0 and _all_nan(Y[300])
    rc, _, _, Y = _block_case(torch, lib, 0, 40, 16, 3)  # no rows: nothing written
    assert rc == 0 and _all_nan(Y)


@pytest.mark.parametrize("nrows,ncols,nrhs", [(6363, 53, 8), (1755, 357, 32), (731, 21, 16), (2000, 1003, 24)])
def test_zgemm_block_gaussian(torch, lib, nrows, ncols, nrhs):
    g = torch.Generator(device="cuda").manual_seed(nrows + ncols)
    A, X = _crandn(torch, g, nrows, ncols), _crandn(torch, g, ncols, nrhs)
    Y = _nan(torch, nrows, nrhs)
    torch.cuda.synchronize()
    _ok(lib, lib.shim_zgemm_block(_ptr(A), ncols, nrows, ncols, _ptr(X), _ptr(Y), nrhs))
    Ah, Xh = A.cpu().numpy(), X.cpu().numpy()
    ref = R.matmul(Ah, Xh)
    scale = np.abs(Ah) @ np.abs(Xh)
    assert np.all(np.abs(Y.cpu().numpy() - ref) <= 1e-14 * scale)


@pytest.mark.parametrize("n", (1, 4095, 4096, 4097, 151553))
@pytest.mark.parametrize("with_pinv", (False, True))
@pytest.mark.parametrize("with_ax", (False, True))
def test_residual_matches_reference(torch, lib, n, with_pinv, with_ax):
    g = torch.Generator(device="cuda").manual_seed(n)
    b, ax = _crandn(torch, g, n), _crandn(torch, g, n) if with_ax else None
    pinv = _crandn(torch, g, n) if with_pinv else None
    r = _nan(torch, n + 1)
    out = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    _ok(lib, lib.shim_residual(_ptr(b), _ptr(ax), _ptr(r), n, out.data_ptr(), _ptr(pinv)))
    br, bi = R._split(b.cpu().numpy())
    if with_ax:
        ar, ai = R._split(ax.cpu().numpy())
        br, bi = br - ar, bi - ai
    mag = np.abs(b.cpu().numpy()) + (np.abs(ax.cpu().numpy()) if with_ax else 0)
    if with_pinv:
        pr, pi = R._split(pinv.cpu().numpy())
        br, bi = br * pr - bi * pi, br * pi + bi * pr
        mag = mag * np.abs(pinv.cpu().numpy())
    rh = r.cpu().numpy()
    assert np.all(np.abs(rh[:n] - (br + 1j * bi)) <= 1e-15 * mag) and np.isnan(rh[n])
    nn = np.sum(br * br + bi * bi)
    assert abs(float(out.item()) - nn) <= 1e-14 * nn


def test_interleave_round_trip(torch, lib):
    g = torch.Generator(device="cuda").manual_seed(9)
    n, nsrc, nrhs = 4097, 5, 8
    src = _crandn(torch, g, nsrc, n)
    blk = _nan(torch, n, nrhs)
    _ok(lib, lib.shim_interleave(_ptr(src), _ptr(blk), n, nsrc, nrhs, 1))
    want = torch.zeros(n, nrhs, dtype=torch.complex128, device="cuda")
    want[:, :nsrc] = src.T
    assert torch.equal(blk, want)
    back = _nan(torch, nrhs, n)
    _ok(lib, lib.shim_interleave(_ptr(blk), _ptr(back), n, nsrc, nrhs, 0))
    assert torch.equal(back[:nsrc], src) and _all_nan(back[nsrc:])
