"""Multi-direction scattering on the device (DESIGN.md section 4.7): the batch entry points against the single-vector calls they
batch (bit for bit) and against the oracle.

incident_rhs_batch -> gmres_batched_device -> compute_rcs_batch / compute_scattered_field_batch, and the sweep's
submit_incident / next_batch."""
import numpy as np
import pytest

from math_audio_b200.mesh import fibonacci_directions, generate_icosphere_mesh
from math_audio_b200.types import PhysicsParams

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bem():
    from math_audio_b200 import bem as _bem

    return _bem


@pytest.fixture(scope="module")
def torch():
    import torch as _torch

    assert _torch.cuda.is_available()
    return _torch


def _dev(torch, a):
    """complex128 host array -> device tensor (kept alive by the caller)"""
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.complex128)).to("cuda:0")


def _host(t):
    return t.cpu().numpy()


def _bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def _incidents(rng, nrhs):
    """plane waves, point sources, multi-source groups and complex amplitudes"""
    from math_audio_b200.incident import IncidentField

    out = []
    for i, d in enumerate(fibonacci_directions(nrhs)):
        f = IncidentField.plane_wave(d)
        if i % 3 == 1:
            f = IncidentField(point_sources=[(rng.standard_normal(3) * 0.5, complex(*rng.standard_normal(2)))])
        elif i % 3 == 2:
            f.plane_waves.append((-d, complex(*rng.standard_normal(2))))
            f.point_sources.append((np.array([0.3, -0.2, 0.25]), 0.5 - 0.25j))
        out.append(f)
    return out


def _sphere(level, ka=2.0):
    a = 0.1
    mesh = generate_icosphere_mesh(a, level)
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    return mesh, ph, beta


@pytest.mark.parametrize("level", [3, 4])
def test_incident_batch_matches_single_calls_and_oracle(bem, orc, torch, level):
    mesh, ph, beta = _sphere(level)
    st = bem.StagedMesh(mesh)
    rng = np.random.default_rng(level)
    inc = _incidents(rng, 13)
    B = bem.incident_rhs_batch(st, ph, beta, inc)
    assert B.shape == (13, st.num_dofs)
    for s, f in enumerate(inc):
        assert _bits(B[s], bem.incident_rhs_device(st, ph, beta, f)), s
        ref = np.zeros(st.num_dofs, dtype=np.complex128)
        for kind, group in ((0, f.plane_waves), (1, f.point_sources)):
            for v, a in group:
                ref += a * orc.incident_rhs(kind, v, 1.0, mesh.center, mesh.normal, ph.wave_number, beta)[0]
        assert np.abs(B[s] - ref).max() <= 1e-13 * np.abs(ref).max()
    # device output, with TbemSystem.rhs added on the device: b = rhs + incident, one IEEE add
    system = bem.build_tbem_system_with_beta(st, ph, beta)
    bd = torch.empty((13, st.num_dofs), dtype=torch.complex128, device="cuda:0")
    got = bem.incident_rhs_batch(st, ph, beta, inc, system=system, b_dev=bd.data_ptr())
    assert _bits(got, system.rhs_full()[None, :] + B) and _bits(_host(bd), got)
    assert bem.incident_rhs_batch(st, ph, beta, inc[:2], b_dev=bd.data_ptr(), fetch=False) is None
    assert _bits(_host(bd)[:2], B[:2])


def test_gmres_batched_device_matches_host_batched(bem, torch):
    mesh, ph, beta = _sphere(3)
    st = bem.StagedMesh(mesh)
    system = bem.build_tbem_system_with_beta(st, ph, beta)
    op = bem.DenseOperator(system)
    from math_audio_b200.incident import IncidentField

    cfg = bem.GmresConfig(max_iterations=1000, restart=20, tolerance=1e-10)
    pre = bem.AdditiveSchwarzPreconditioner.from_operator(op, 20)
    for nrhs in (11, 32):
        B = bem.incident_rhs_batch(st, ph, beta, [IncidentField.plane_wave(d) for d in fibonacci_directions(nrhs)], system=system)
        if nrhs == 11:
            B[3] = 0.0
        bd = _dev(torch, B)
        for precond, c in ((None, cfg), (pre, cfg), (None, bem.GmresConfig(max_iterations=1, restart=5, tolerance=1e-14))):
            ref, _ = bem.gmres_batched(op, B, c, precond=precond)
            xd = torch.full((nrhs, st.num_dofs), complex(np.nan, np.nan), dtype=torch.complex128, device="cuda:0")
            sols, stats = bem.gmres_batched_device(op, bd.data_ptr(), nrhs, c, xd.data_ptr(), precond=precond)
            assert stats["block_matvecs"] > 0 and all(s.x is None for s in sols)
            X = _host(xd)
            for i in range(nrhs):
                assert _bits(X[i], ref[i].x), (nrhs, precond is not None, i)
                assert (sols[i].iterations, sols[i].restarts, sols[i].converged) == (ref[i].iterations, ref[i].restarts, ref[i].converged)
                assert _bits(np.float64(sols[i].residual), np.float64(ref[i].residual))
            if c.max_iterations == 1:
                assert not any(s.converged for i, s in enumerate(sols) if np.abs(B[i]).max() > 0)
    pre.close()


def _permuted_mesh():
    a = 0.1
    mesh = generate_icosphere_mesh(a, 2)
    rng = np.random.default_rng(21)
    mesh.is_eval[::11] = 1
    bnd = np.flatnonzero(mesh.is_eval == 0)
    mesh.dof[bnd] = rng.permutation(mesh.num_dofs).astype(np.uint32)
    return mesh, PhysicsParams.from_wave_number(25.0)


@pytest.mark.parametrize("case", ["ico3", "permuted"])
def test_rcs_and_field_batches_match_single_calls(bem, torch, case):
    if case == "ico3":
        mesh, ph, _ = _sphere(3)
    else:
        mesh, ph = _permuted_mesh()
    st = bem.StagedMesh(mesh)
    n = st.num_dofs
    rng = np.random.default_rng(5)
    dirs = rng.standard_normal((37, 3))
    dirs /= np.linalg.norm(dirs, axis=1)[:, None]
    pts = rng.standard_normal((29, 3))
    pts *= (0.35 / np.linalg.norm(pts, axis=1))[:, None]
    for nsol in (1, 7, 8, 33):
        P = rng.standard_normal((nsol, n)) + 1j * rng.standard_normal((nsol, n))
        V = rng.standard_normal((nsol, n)) + 1j * rng.standard_normal((nsol, n))
        V[nsol // 2] = 0.0  # has_v is decided per solution
        rcs = bem.compute_rcs_batch(P, st, dirs, ph)
        assert rcs.shape == (nsol, len(dirs))
        for vel in (None, V):
            fld = bem.compute_scattered_field_batch(pts, st, P, vel, ph)
            for s in range(nsol):
                assert _bits(fld[s], bem.compute_scattered_field(pts, st, P[s], None if vel is None else vel[s], ph)), (nsol, s)
        for s in range(nsol):
            assert _bits(rcs[s], bem.compute_rcs(P[s], st, dirs, ph)), (nsol, s)
        # device inputs are in DOF order, as the solver leaves them
        Pd = np.stack([bem.surface_values_in_dof_order(st.enum_to_dof, p) for p in P])
        Vd = np.stack([bem.surface_values_in_dof_order(st.enum_to_dof, v) for v in V])
        pd, vd = _dev(torch, Pd), _dev(torch, Vd)
        assert _bits(bem.compute_rcs_batch(pd.data_ptr(), st, dirs, ph, nsol=nsol), rcs)
        assert _bits(bem.compute_scattered_field_batch(pts, st, pd.data_ptr(), vd.data_ptr(), ph, nsol=nsol),
                     bem.compute_scattered_field_batch(pts, st, P, V, ph))


def test_end_to_end_directions_to_rcs_matches_oracle(bem, orc, torch):
    from math_audio_b200.incident import IncidentField

    mesh, ph, beta = _sphere(3)
    st = bem.StagedMesh(mesh)
    n = st.num_dofs
    system = bem.build_tbem_system_with_beta(st, ph, beta)
    op = bem.DenseOperator(system)
    A = system.matrix.rows()
    cfg = bem.GmresConfig(max_iterations=50, restart=50, tolerance=1e-10)
    incs = [IncidentField.plane_wave(d) for d in fibonacci_directions(32)]
    bd = torch.empty((32, n), dtype=torch.complex128, device="cuda:0")
    xd = torch.empty((32, n), dtype=torch.complex128, device="cuda:0")
    bem.incident_rhs_batch(st, ph, beta, incs, system=system, b_dev=bd.data_ptr(), fetch=False)
    sols, _ = bem.gmres_batched_device(op, bd.data_ptr(), 32, cfg, xd.data_ptr())
    obs = fibonacci_directions(200)
    rcs = bem.compute_rcs_batch(xd.data_ptr(), st, obs, ph, nsol=32)
    B, X = _host(bd), _host(xd)
    for i in range(32):
        xo, io = orc.gmres(A, B[i], max_iterations=50, restart=50, tolerance=1e-10)
        assert sols[i].converged and (sols[i].iterations, sols[i].restarts) == (io["iterations"], io["restarts"]), i
        assert np.linalg.norm(X[i] - xo) / np.linalg.norm(xo) < 1e-8
        ref = orc.compute_rcs(mesh, xo, obs, ph.wave_number)
        assert np.max(np.abs(rcs[i] - ref) / ref) < 1e-8


@pytest.mark.parametrize("overlap", [True, False])
def test_sweep_incident_jobs_match_existing_calls(bem, overlap):
    from math_audio_b200.sweep import Sweep

    mesh, _, _ = _sphere(3)
    a = 0.1
    cases = []
    for ka in (1.5, 2.0, 2.5):
        ph = PhysicsParams.from_wave_number(ka / a)
        cases.append((ph, ph.burton_miller_beta_adaptive(a)[0]))
    cfg = bem.GmresConfig(max_iterations=100, restart=30, tolerance=1e-10)
    rng = np.random.default_rng(3)
    inc = _incidents(rng, 5)
    st = bem.StagedMesh(mesh)
    # nrhs = 1: the same schedule through submit(rhs_extra = incident_rhs_device(...)) and submit_incident
    for nsub in (0, 16):
        swa, swb = Sweep(mesh, overlap=overlap), Sweep(mesh, overlap=overlap)
        swa.set_block_jacobi(nsub)
        swb.set_block_jacobi(nsub)
        for ph, beta in cases[:2]:
            swa.submit(ph, beta, bem.incident_rhs_device(st, ph, beta, inc[0]), cfg)
            swb.submit_incident(ph, beta, inc[:1], cfg)
        for i in range(len(cases)):
            ref, _, _ = swa.next()
            got, stats = swb.next_batch()
            assert len(got) == 1 and _bits(got[0].x, ref.x), (nsub, i)
            assert (got[0].iterations, got[0].restarts, got[0].converged) == (ref.iterations, ref.restarts, ref.converged)
            assert stats["near_pairs"] > 0
            if i + 2 < len(cases):
                ph, beta = cases[i + 2]
                swa.submit(ph, beta, bem.incident_rhs_device(st, ph, beta, inc[0]), cfg)
                swb.submit_incident(ph, beta, inc[:1], cfg)
        swa.close()
        swb.close()
    # nrhs = 5: gmres_batched on the same frequency's matrix and B, plain and block-Jacobi
    for nsub in (0, 16):
        sw = Sweep(mesh, overlap=overlap)
        sw.set_block_jacobi(nsub)
        for ph, beta in cases:
            sw.submit_incident(ph, beta, inc, cfg)
        for ph, beta in cases:
            got, _ = sw.next_batch()
            system = bem.build_tbem_system_with_beta(st, ph, beta)
            op = bem.DenseOperator(system)
            B = bem.incident_rhs_batch(st, ph, beta, inc, system=system)
            pre = bem.AdditiveSchwarzPreconditioner.from_operator(op, nsub) if nsub else None
            ref, _ = bem.gmres_batched(op, B, cfg, precond=pre)
            assert len(got) == 5
            for s in range(5):
                assert _bits(got[s].x, ref[s].x), (nsub, s)
                assert (got[s].iterations, got[s].restarts, got[s].converged) == (ref[s].iterations, ref[s].restarts, ref[s].converged)
            if pre is not None:
                pre.close()
        sw.close()


def test_sweep_queue_rules(bem):
    from math_audio_b200 import _capi
    from math_audio_b200.sweep import Sweep

    mesh, ph, beta = _sphere(3)
    cfg = bem.GmresConfig(max_iterations=100, restart=30, tolerance=1e-8)
    inc = _incidents(np.random.default_rng(1), 3)
    sw = Sweep(mesh)
    sw.submit_incident(ph, beta, inc, cfg)
    sw.submit(ph, beta, None, cfg)
    with pytest.raises(_capi.Bemb200Error) as ei:  # three right-hand sides, room for two: stays queued
        sw.next_batch(capacity=2)
    assert ei.value.code == -1
    with pytest.raises(_capi.Bemb200Error) as ei:  # next() takes one right-hand side: stays queued
        sw.next()
    assert ei.value.code == -1
    got, _ = sw.next_batch()
    assert len(got) == 3 and all(s.converged for s in got)
    sol, _ = sw.next_batch()  # a job of submit() through next_batch: one solution
    assert len(sol) == 1 and sol[0].converged
    # overlapping subdomains with nrhs > 1: EUNSUPPORTED in next_batch, the job is consumed
    n = sw.n
    subs = [np.arange(0, n // 2 + 8, dtype=np.uint64), np.arange(n // 2 - 8, n, dtype=np.uint64)]
    sw.set_block_jacobi(subdomains=subs)
    sw.submit_incident(ph, beta, inc, cfg)
    sw.submit_incident(ph, beta, inc[:1], cfg)
    with pytest.raises(_capi.Bemb200Error) as ei:
        sw.next_batch()
    assert ei.value.code == -6
    got, _ = sw.next_batch()  # the next job, a single right-hand side, solves with the overlapping Schwarz preconditioner
    assert len(got) == 1 and got[0].converged
    sw.close()
