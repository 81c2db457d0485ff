"""Single-rank solves forced onto the persistent fused GMRES kernel (run with BEMB200_GMRES_FUSED=1: the switch is read
once, when the library loads), on arbitrary matrices, against the oracle and an extended-precision GMRES cycle.  Writes
one JSON record per case; tests/test_gpu_fused_gmres.py runs this in a child process and asserts on the records.

    BEMB200_GMRES_FUSED=1 python tests/drivers/fused_forced.py OUT.json
"""
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import fused_split_reference as F  # noqa: E402
import solve_kernels_reference as R  # noqa: E402
from math_audio_b200 import bem  # noqa: E402
from oracle import oracle as orc  # noqa: E402

LD, CLD = np.longdouble, np.clongdouble


def crandn(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def well_conditioned(n, seed, radius=0.5):
    """I + radius G / sqrt(2 n), G complex Gaussian: eigenvalues in a disk of `radius` around 1, GMRES converges at about
    that rate per iteration."""
    rng = np.random.default_rng(seed)
    return np.eye(n, dtype=np.complex128) + radius * crandn(rng, n, n) / np.sqrt(2 * n)


def profile_kernels(torch, fn, trace_path):
    """fn() under torch.profiler; returns (result, [(kernel name, shared memory)]), the trace written to and read back from
    `trace_path`.  Torch kernels on both sides anchor the window: one that held only the library's launches has come back
    without kernel events."""
    from torch.profiler import ProfilerActivity, profile

    marker = torch.zeros(1, device="cuda")
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        marker.add_(1)
        torch.cuda.synchronize()
        out = fn()
        torch.cuda.synchronize()
        marker.add_(1)
        torch.cuda.synchronize()
    path = Path(trace_path)
    prof.export_chrome_trace(str(path))
    ev = [e for e in json.loads(path.read_text())["traceEvents"] if e.get("cat") == "kernel"]
    path.unlink()
    return out, [(e["name"], e.get("args", {}).get("shared memory")) for e in ev]


def one_cycle_reference(A, b, x0, m):
    """One restart cycle of GMRES(m) in clongdouble: MGS Arnoldi (solve_kernels_reference.mgs), Givens least squares,
    x = x0 + V y; returns (x, ||b - A x|| / ||b||)."""
    Al = A.astype(CLD)
    bl, xl = b.astype(CLD), x0.astype(CLD)
    r = bl - Al @ xl
    beta = np.sqrt(np.sum(r.real * r.real + r.imag * r.imag))
    V = [r / beta]
    H = np.zeros((m + 1, m), dtype=CLD)
    k = m
    for j in range(m):
        h, nrm, q = R.mgs(np.array(V), Al @ V[j])
        H[: j + 1, j] = h
        H[j + 1, j] = nrm
        if q is None or nrm < 1e-14:
            k = j + 1
            break
        V.append(q)
    # least squares min || beta e1 - H y || by Givens rotations
    Hk = H[: k + 1, :k].copy()
    g = np.zeros(k + 1, dtype=CLD)
    g[0] = beta
    for j in range(k):
        a, c = Hk[j, j], Hk[j + 1, j]
        rr = np.sqrt(abs(a) ** 2 + abs(c) ** 2)
        cs, sn = a / rr, c / rr
        for col in range(j, k):
            t0, t1 = Hk[j, col], Hk[j + 1, col]
            Hk[j, col] = np.conj(cs) * t0 + np.conj(sn) * t1
            Hk[j + 1, col] = -sn * t0 + cs * t1
        g[j], g[j + 1] = np.conj(cs) * g[j] + np.conj(sn) * g[j + 1], -sn * g[j] + cs * g[j + 1]
    y = np.zeros(k, dtype=CLD)
    for i in range(k - 1, -1, -1):
        y[i] = (g[i] - Hk[i, i + 1:k] @ y[i + 1:k]) / Hk[i, i]
    x = xl + np.array(V[:k]).T @ y
    res = bl - Al @ x
    bn = np.sqrt(np.sum(bl.real * bl.real + bl.imag * bl.imag))
    return x, np.sqrt(np.sum(res.real * res.real + res.imag * res.imag)) / bn


def main(out_path):
    import torch

    torch.cuda.init()
    records = []
    trace = out_path.with_suffix(".trace.json")
    ctx = bem.Context(0)
    polite_ctx = bem.Context(0)
    polite_ctx.set_shared_gpu(True)

    def run(name, A, b, *, x0=None, restart=30, max_it=50, tol=1e-10, inv_diag=None, polite=False, one_cycle=False):
        n = A.shape[0]
        op = bem.DenseOperator(A, polite_ctx if polite else ctx)
        cfg = bem.GmresConfig(max_iterations=max_it, restart=restart, tolerance=tol)
        if inv_diag is None:
            sol, kern = profile_kernels(torch, lambda: bem.gmres_with_guess(op, b, x0, cfg), trace)
            xo, io = orc.gmres(A, b, x0=x0, max_iterations=max_it, restart=restart, tolerance=tol)
        else:
            pc = bem.DiagonalPreconditioner(inv_diag)
            sol, kern = profile_kernels(torch, lambda: bem.gmres_preconditioned_with_guess(op, pc, b, x0, cfg), trace)
            xo, io = orc.gmres_preconditioned(A, b, inv_diag=inv_diag, x0=x0, max_iterations=max_it, restart=restart, tolerance=tol)
        launches = op.matrix.solver_stats()["kernel_launches"]
        bn = float(np.linalg.norm(b))
        # the preconditioned variant reports ||M^-1 (b - A x)|| / ||M^-1 b||
        w = np.ones(n) if inv_diag is None else inv_diag
        true_res = float(np.linalg.norm(w * (b - A @ sol.x)) / np.linalg.norm(w * b)) if bn > 0 else 0.0
        xn = float(np.linalg.norm(xo))
        dx = float(np.linalg.norm(sol.x - xo) / xn) if xn > 0 else float(np.linalg.norm(sol.x))
        pl = F.plan_rank(n, 1, 0, 148, restart)
        rec = dict(name=name, n=n, restart=restart, max_it=max_it, polite=polite, precond=inv_diag is not None,
                   dev=[sol.iterations, sol.restarts, sol.converged], orc=[io["iterations"], io["restarts"], io["converged"]],
                   residual=sol.residual, orc_residual=io["residual"], true_residual=true_res, dx=dx, launches=launches,
                   kernels=sorted(set(kern)), mode=pl.mode, mirror_smem=pl.smem)
        if one_cycle:
            xr, rr = one_cycle_reference(A, b, x0 if x0 is not None else np.zeros(n, dtype=np.complex128), restart)
            rec["cycle_dx"] = float(np.linalg.norm((sol.x.astype(CLD) - xr)) / np.linalg.norm(xr))
            rec["cycle_residual"] = float(rr)
            rec["cycle_dres"] = float(abs(LD(sol.residual) - rr) / rr)
        op.matrix.close()
        records.append(rec)
        print(json.dumps(rec), flush=True)

    rng = np.random.default_rng(1)
    for n in sorted(F.FORCED_SIZES):
        A = well_conditioned(n, seed=n)
        b = crandn(rng, n)
        run(f"rand_n{n}", A, b)
        run(f"rand_n{n}_guess", A, b, x0=crandn(rng, n))
    n = 300
    A = well_conditioned(n, seed=5)
    b = crandn(rng, n)
    run("identity", np.eye(n, dtype=np.complex128), b)
    run("tiny_scale", A * 1e-16, b)
    # b inside a 3-dimensional invariant subspace (a block-diagonal matrix under a random permutation): the Krylov space
    # ends after 3 vectors and the fourth is rounding of three-term sums, far below the absolute 1e-14 breakdown threshold
    perm = rng.permutation(n)
    Blk = np.zeros((n, n), dtype=np.complex128)
    Blk[:3, :3] = np.eye(3) * 2 + 0.3 * crandn(rng, 3, 3)
    Blk[3:, 3:] = np.eye(n - 3) + 0.3 * crandn(rng, n - 3, n - 3) / np.sqrt(2 * n)
    Ainv = np.empty_like(Blk)
    Ainv[np.ix_(perm, perm)] = Blk
    binv = np.zeros(n, dtype=np.complex128)
    binv[perm[:3]] = crandn(rng, 3)
    run("invariant3", Ainv, binv, tol=1e-20)
    run("zero_b", A, np.zeros(n, dtype=np.complex128))
    run("guess_is_solution", A, b, x0=np.linalg.solve(A, b))
    run("max_it0", A, b, x0=crandn(rng, n), max_it=0)
    run("budget", A, b, max_it=1, restart=5)
    run("restart1", A, b, restart=1, max_it=40)
    run("restart63", A, b, restart=63, max_it=3)
    run("restart64", A, b, restart=64, max_it=3)
    # diagonal preconditioner on a badly scaled matrix
    d = np.exp(rng.uniform(0, 3, n)) * np.exp(1j * rng.uniform(0, 6.28, n))
    Ad = d[:, None] * A
    run("precond", Ad, b, inv_diag=1 / d)
    run("precond_guess", Ad, b, x0=crandn(rng, n), inv_diag=1 / d)
    run("precond_budget", Ad, b, x0=crandn(rng, n), inv_diag=1 / d, max_it=2, restart=5)
    n2 = 2100
    A2 = well_conditioned(n2, seed=21)
    b2 = crandn(rng, n2)
    run("polite_n300", A, b, polite=True)
    run("polite_n2100", A2, b2, polite=True)
    run("polite_precond", Ad, b, inv_diag=1 / d, polite=True)
    # one restart cycle against extended precision: nothing converges (tolerance 0), the true residual is reported
    for nn, Am, bm in ((300, well_conditioned(300, seed=9, radius=0.9), crandn(rng, 300)), (n2, well_conditioned(n2, seed=23, radius=0.9), b2)):
        for m in (1, 7, 63):
            run(f"cycle_n{nn}_m{m}", Am, bm, restart=m, max_it=1, tol=0.0, one_cycle=True)
    ctx.close()
    polite_ctx.close()
    out_path.write_text(json.dumps(records, indent=1))


if __name__ == "__main__":
    main(Path(sys.argv[1]))
