"""The persistent fused GMRES kernel (csrc/gmres_fused.cu) on one GPU, at every row-ownership branch and stopping rule.

a. Single-process groups (bem.MultiGpu([0] * k)): k ranks share device 0, 148 // k CTAs each, the fused kernel by default.
   The cases of fused_split_reference.GROUP_CASES put the split into each of its branches; test_fused_gmres_cpu.py pins
   which.  Iteration / restart / converged counts must equal the oracle's on the device's own matrix (for 38 720
   unknowns: a single-rank per-iteration solve), x must agree to 1e-9 and the true residual must match the reported one.
b. Single-rank solves forced onto the kernel (tests/drivers/fused_forced.py with BEMB200_GMRES_FUSED=1 in a child
   process): identity, 1e-16-scaled and invariant-subspace breakdowns, zero b, exact and random guesses, no cycle,
   budget exhaustion, restart 1 / 63 / 64, the diagonal preconditioner, the polite build, and one restart cycle against
   an extended-precision GMRES.
c. Every case reads back from the profiler which kernel ran and its shared memory, and compares that with the mirror.

Modes the profiler confirmed on an NVIDIA B200 (1000 W power limit), from the shared memory of every rank's launch:
  k1_equal: equal (S = 4)          k1_units: units, one segment a row      k1_frag: units with head fragments
  k2_frag, k3_frag: units, then calibrated units (per-rank sizes differ, e.g. 72 240 / 72 528 B)
  k8_tiny: equal, ranks 5 .. 7 without rows, solved
  k8_big: equal with S = 269 (two matvec passes), then the calibrated row table (136 080 / 136 112 B across ranks)
  forced single rank: equal for n <= 300, units with fragments for n = 2100, the polite build for set_shared_gpu(True),
  no fused launch for restart 64.
One restart cycle against extended precision (n = 300 and 2100, restart 1, 7, 63; worst of the six): x within 9.7e-16,
the reported true residual within 1.7e-13 relative (bound: ONE_CYCLE_BOUND).  The whole file ran in 30 s there; the
38 720-unknown case (mesh, two assemblies, three solves) took 1.9 s.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
sys.path.insert(0, str(Path(__file__).resolve().parent / "drivers"))
import fused_split_reference as F  # noqa: E402
from fused_forced import profile_kernels  # noqa: E402

from math_audio_b200.mesh import generate_geodesic_sphere_mesh, generate_icosphere_mesh  # noqa: E402
from math_audio_b200.types import PhysicsParams  # noqa: E402

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
X_BOUND = 1e-9
ONE_CYCLE_BOUND = 1e-11
STATIC_SMEM_MAX = 2048  # the kernel's static shared memory (a few flags and per-warp partials) on top of the dynamic part
CASES = {c[0]: c for c in F.GROUP_CASES}


@pytest.fixture(scope="module")
def bem():
    from math_audio_b200 import bem as _bem

    return _bem


@pytest.fixture(scope="module")
def torch():
    import torch as t

    assert t.cuda.is_available(), "the fused GMRES tests need a CUDA device"
    t.cuda.init()
    return t


_static_smem = []


def _profiled(torch, tmp_path, fn):
    """fn() under torch.profiler -> (result, [(kernel name, shared memory)])."""
    out, kern = profile_kernels(torch, fn, tmp_path / "trace.json")
    if not kern:
        pytest.fail("the profiler recorded no kernel events: cannot tell which kernel ran")
    return out, kern


def _confirmed_mode(launches, plans, calibrated):
    """The split the profiler's shared-memory figures show: the mirror's exact sizes before the calibration; afterwards a
    unit table needs at most 256 row slots and the row table more (rblk = 256 in both), so the dynamic part tells them
    apart (the static part is known from the uncalibrated launches checked before)."""
    if not calibrated:
        return plans[0].mode
    assert _static_smem, "no uncalibrated launch has fixed the static shared memory yet"
    dyn = min(launches) - _static_smem[0]
    return "row_off" if dyn > F.fused_smem_bytes(256, 256, F.GROUP_RESTART) else "units"


def _check_static(total, dynamic):
    """The profiler reports static + dynamic shared memory; the static part is the same for every launch."""
    st = total - dynamic
    assert 0 <= st < STATIC_SMEM_MAX, f"{total} B of shared memory for {dynamic} B dynamic"
    if _static_smem:
        assert st == _static_smem[0], f"static shared memory {st} B, earlier launches {_static_smem[0]} B"
    else:
        _static_smem.append(st)


def _fused_launches(kern, polite=False):
    """Shared memory of every launch of the fused kernel (of its polite build when `polite`); kern holds full demangled
    names such as bemb::(anonymous namespace)::gmres_fused_kernel(bemb::FusedParams)."""
    return [s for k, s in kern if "gmres_fused_kernel" in k and ("gmres_fused_kernel_polite" in k) == polite]


def _mesh(name, n):
    a = 0.1
    if n == 38720:
        mesh = generate_geodesic_sphere_mesh(a, 44)
    else:
        sub = 0 if n <= 20 else 3 if n <= 1280 else 4
        mesh = generate_icosphere_mesh(a, sub)
    mesh.is_eval[n:] = 1
    assert mesh.num_dofs == n
    return mesh


def _system(bem, grp, n, ka=2.0):
    from math_audio_b200.incident import IncidentField

    a = 0.1
    mesh = _mesh("", n)
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    system = grp.build_tbem_system_with_beta(mesh, ph, beta)
    b = system.rhs + IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center[:n], mesh.normal[:n], ph, beta)
    return mesh, ph, beta, system, b


def _check_solve(sol, io, xo, A, b, what):
    assert (sol.iterations, sol.restarts, sol.converged) == (io["iterations"], io["restarts"], io["converged"]), \
        f"{what}: device {(sol.iterations, sol.restarts, sol.converged)}, oracle {io}"
    xn = np.linalg.norm(xo)
    dx = np.linalg.norm(sol.x - xo) / xn if xn > 0 else np.linalg.norm(sol.x)
    assert dx < X_BOUND, f"{what}: |x - x_oracle| / |x_oracle| = {dx:.2e}"
    bn = np.linalg.norm(b)
    if bn == 0:
        assert sol.residual == 0 and not np.any(sol.x), what
        return
    true = np.linalg.norm(b - A @ sol.x) / bn
    assert abs(true - sol.residual) <= 1e-3 * sol.residual + 1e-13, f"{what}: reported residual {sol.residual:.3e}, true {true:.3e}"


def _group_variants(bem, orc, system, A, b, n, tmp_path, torch, k, label):
    """x0, a one-cycle budget with restart 5, restart 1 and 63, zero b: counts and x against the oracle on A."""
    rng = np.random.default_rng(n + k)
    x0 = (rng.standard_normal(n) + 1j * rng.standard_normal(n)) * 0.01
    variants = [
        ("guess", b, x0, 30, F.GROUP_RESTART),
        ("budget", b, None, 1, 5),
        ("restart1", b, None, 20, 1),
        ("restart63", b, x0, 3, 63),
        ("zero_b", np.zeros(n, dtype=np.complex128), None, 30, F.GROUP_RESTART),
    ]
    for vname, bb, xx, max_it, restart in variants:
        cfg = bem.GmresConfig(max_iterations=max_it, restart=restart, tolerance=1e-10)
        sol, kern = _profiled(torch, tmp_path, lambda: system.gmres(bb, cfg, x0=xx))
        xo, io = orc.gmres(A, bb, x0=xx, max_iterations=max_it, restart=restart, tolerance=1e-10)
        _check_solve(sol, io, xo, A, bb, f"{label} {vname}")
        launches = _fused_launches(kern)
        assert len(launches) == k, f"{label} {vname}: {len(launches)} fused launches for {k} ranks"
        plans = F.plan(n, k, F.group_ctas(k), restart)
        if all(pl.nloc < 16 * F.group_ctas(k) for pl in plans):  # never calibrated: the split is the mirror's exactly
            for s, pl in zip(sorted(launches), sorted(plans, key=lambda p: p.smem)):
                _check_static(s, pl.smem)


@pytest.mark.parametrize("name", ["k1_equal", "k1_units", "k1_frag", "k2_frag", "k3_frag"])
def test_group_solve_matches_oracle(bem, orc, torch, tmp_path, name):
    _, k, n, mode = CASES[name]
    G = F.group_ctas(k)
    grp = bem.MultiGpu([0] * k)
    system = None
    try:
        mesh, ph, beta, system, b = _system(bem, grp, n)
        A = system.rows()
        cfg = bem.GmresConfig(max_iterations=30, restart=F.GROUP_RESTART, tolerance=1e-10)
        xo, io = orc.gmres(A, b, max_iterations=30, restart=F.GROUP_RESTART, tolerance=1e-10)
        plans = F.plan(n, k, G, F.GROUP_RESTART)
        assert all(pl.mode == mode for pl in plans)
        sizeable = all(pl.nloc >= 16 * G for pl in plans)
        # uncalibrated split, first refinement, frozen table: the same system three times in one group.  The ranks calibrate
        # separately, so from the second solve on they launch with different shared-memory sizes.
        for solve in range(3 if sizeable else 1):
            sol, kern = _profiled(torch, tmp_path, lambda: system.gmres(b, cfg))
            _check_solve(sol, io, xo, A, b, f"{name} solve {solve}")
            launches = _fused_launches(kern)
            assert len(launches) == k, f"{name}: kernels {sorted(set(kern))}"
            if solve == 0:
                for s, pl in zip(sorted(launches), sorted(plans, key=lambda p: p.smem)):
                    _check_static(s, pl.smem)
            else:
                # calibrated unit table: S between the equal share and 256 slots
                lo = min(pl.smem for pl in plans)
                hi = F.fused_smem_bytes(256, 256, F.GROUP_RESTART) + STATIC_SMEM_MAX
                assert all(lo <= s <= hi for s in launches), (name, launches, lo, hi)
            seen = _confirmed_mode(launches, plans, solve > 0)
            assert seen == mode
            print(f"MODE {name} solve {solve}: {seen}{' (calibrated)' if solve else ''}, it {sol.iterations} restarts "
                  f"{sol.restarts} res {sol.residual:.2e}, shared memory {sorted(launches)}")
        _group_variants(bem, orc, system, A, b, n, tmp_path, torch, k, name)
    finally:
        if system is not None:
            system.close()
        grp.close()


def test_group_ranks_without_rows(bem, orc, torch, tmp_path):
    """Eight ranks, five unknowns: ranks 5 .. 7 own no rows.  The solve must be right or refused with an error."""
    from math_audio_b200 import _capi

    _, k, n, mode = CASES["k8_tiny"]
    grp = bem.MultiGpu([0] * k)
    system = None
    try:
        mesh, ph, beta, system, b = _system(bem, grp, n)
        A = system.rows()
        cfg = bem.GmresConfig(max_iterations=10, restart=F.GROUP_RESTART, tolerance=1e-10)
        try:
            sol, kern = _profiled(torch, tmp_path, lambda: system.gmres(b, cfg))
        except _capi.Bemb200Error as e:
            assert "timed out" not in str(e), f"ranks without rows stalled the group: {e}"
            print(f"k8_tiny refused: {e}")
            return
        xo, io = orc.gmres(A, b, max_iterations=10, restart=F.GROUP_RESTART, tolerance=1e-10)
        _check_solve(sol, io, xo, A, b, "k8_tiny")
        launches = _fused_launches(kern)
        assert len(launches) == k
        for s in launches:
            _check_static(s, F.plan_rank(n, k, 0, F.group_ctas(k), F.GROUP_RESTART).smem)
        print(f"MODE k8_tiny solve 0: {mode}, it {sol.iterations} res {sol.residual:.2e}, shared memory {sorted(set(launches))}")
    finally:
        if system is not None:
            system.close()
        grp.close()


def test_group_multipass_and_row_table(bem, torch, tmp_path):
    """Eight ranks, 38 720 unknowns (about 24 GB): 269 rows a CTA, two matvec passes of 256 and 13 rows on the first
    solve; the calibrated row table (more than 256 rows on the CTAs measured fastest, a different size on every rank) on
    the second.  Compared with a single-rank per-iteration solve of the same system."""
    _, k, n, mode = CASES["k8_big"]
    G = F.group_ctas(k)
    cfg = bem.GmresConfig(max_iterations=30, restart=F.GROUP_RESTART, tolerance=1e-10)
    grp = bem.MultiGpu([0] * k)
    system = None
    sols = []
    try:
        mesh, ph, beta, system, b = _system(bem, grp, n, ka=1.0)
        plans = F.plan(n, k, G, F.GROUP_RESTART)
        for solve in range(2):
            sol, kern = _profiled(torch, tmp_path, lambda: system.gmres(b, cfg))
            launches = _fused_launches(kern)
            assert len(launches) == k, f"k8_big: kernels {sorted(set(kern))}"
            if solve == 0:
                for s in launches:
                    _check_static(s, plans[0].smem)
            else:
                assert all(s <= F.SMEM_LIMIT + STATIC_SMEM_MAX for s in launches), launches
            seen = _confirmed_mode(launches, plans, solve > 0)
            assert seen == ("equal" if solve == 0 else "row_off"), (solve, launches)
            print(f"MODE k8_big solve {solve}: {seen}{' (calibrated)' if solve else ' (S = 269, two passes)'}, it "
                  f"{sol.iterations} restarts {sol.restarts} res {sol.residual:.2e}, shared memory {sorted(launches)}")
            sols.append(sol)
    finally:
        if system is not None:
            system.close()
        grp.close()
    ref_sys = bem.build_tbem_system_with_beta(_mesh("", n), ph, beta)
    try:
        op = bem.DenseOperator(ref_sys)
        ref = bem.gmres(op, b, cfg)
        bn = np.linalg.norm(b)
        for sol in sols:
            assert (sol.iterations, sol.restarts, sol.converged) == (ref.iterations, ref.restarts, ref.converged)
            assert np.linalg.norm(sol.x - ref.x) / np.linalg.norm(ref.x) < X_BOUND
            true = np.linalg.norm(b - op.apply(sol.x)) / bn
            assert abs(true - sol.residual) <= 1e-3 * sol.residual + 1e-13, (true, sol.residual)
    finally:
        ref_sys.matrix.close()


@pytest.fixture(scope="module")
def forced(tmp_path_factory):
    out = tmp_path_factory.mktemp("fused_forced") / "records.json"
    env = dict(os.environ, BEMB200_GMRES_FUSED="1")
    r = subprocess.run([sys.executable, str(ROOT / "tests" / "drivers" / "fused_forced.py"), str(out)], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return {rec["name"]: rec for rec in json.loads(out.read_text())}


def _forced_names():
    names = []
    for n in sorted(F.FORCED_SIZES):
        names += [f"rand_n{n}", f"rand_n{n}_guess"]
    names += ["identity", "tiny_scale", "invariant3", "zero_b", "guess_is_solution", "max_it0", "budget", "restart1",
              "restart63", "restart64", "precond", "precond_guess", "precond_budget", "polite_n300", "polite_n2100",
              "polite_precond"]
    names += [f"cycle_n{nn}_m{m}" for nn in (300, 2100) for m in (1, 7, 63)]
    return names


@pytest.mark.parametrize("name", _forced_names())
def test_forced_single_rank(forced, name):
    rec = forced[name]
    print(json.dumps(rec))
    assert rec["dev"] == rec["orc"], f"{name}: device (it, restarts, conv) {rec['dev']}, oracle {rec['orc']}"
    assert rec["dx"] < X_BOUND, f"{name}: dx {rec['dx']:.2e}"
    if rec["true_residual"] > 0 or rec["residual"] > 0:
        assert abs(rec["true_residual"] - rec["residual"]) <= 1e-3 * rec["residual"] + 1e-13, rec
    kern = [tuple(k) for k in rec["kernels"]]
    polite = rec["polite"]
    launches = _fused_launches(kern, polite)
    other = _fused_launches(kern, not polite)
    assert not other, f"{name}: the {'normal' if polite else 'polite'} build ran"
    if rec["restart"] > F.FUSED_MAX_RESTART:
        assert rec["mode"] == "not fused" and not launches, f"{name}: {kern}"
        assert rec["launches"] > 1
        return
    assert rec["mode"] in ("equal", "units")
    assert len(launches) == 1, f"{name}: kernels {kern}"
    assert rec["launches"] == 1, f"{name}: {rec['launches']} launches"
    _check_static(launches[0], rec["mirror_smem"])
    if name.startswith("cycle_"):
        m = rec["restart"]
        assert rec["dev"] == [m, 1, False]
        assert rec["cycle_dx"] < ONE_CYCLE_BOUND, f"{name}: x vs extended precision {rec['cycle_dx']:.2e}"
        assert rec["cycle_dres"] < ONE_CYCLE_BOUND, f"{name}: residual vs extended precision {rec['cycle_dres']:.2e}"
    if name in ("identity", "tiny_scale", "invariant3"):
        assert rec["dev"][0] <= {"identity": 1, "tiny_scale": 1, "invariant3": 4}[name] and rec["dev"][2], rec
    if name == "max_it0":
        assert rec["dev"] == [0, 0, False] and rec["residual"] > 0.1
