"""Admittance boundaries and the sign-consistent formulation (DESIGN.md 4.8) on the CPU oracle, no GPU: the options oracle
against the reference-faithful one, against the reference's own velocity system, and against the exact sphere series; and
the argument checks of the Python layer."""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import admittance_oracle as ao  # noqa: E402

from math_audio_b200 import bem  # noqa: E402
from math_audio_b200.mesh import BC_PRESSURE, generate_icosphere_mesh  # noqa: E402

PASSIVE = (0.0, -0.5j, 0.3 - 0.3j)  # Y / k


def adaptive_beta(ka, k):  # burton_miller_beta_adaptive of the sphere tests (scale 1 / 4 / 8 / 16)
    scale = 1.0 if ka < 0.5 else (4.0 if ka < 1.2 else (8.0 if ka < 1.8 else 16.0))
    return 1j * scale / k


def test_default_options_are_orc_assemble(orc):
    mesh = generate_icosphere_mesh(0.1, 1)
    mesh.bc_len[:4] = 3
    mesh.bc_val[:4, :3] = 0.5 - 0.2j
    for k in (2.0, 15.0):  # both sides of the dg_dn_sign switch
        A0, r0, nq0 = orc.assemble(mesh, k, 4j / k)
        for y in (None, np.zeros(mesh.n_elem, dtype=np.complex128)):
            A, r, nq = ao.assemble_opts(mesh, k, 4j / k, admittance=y)
            assert np.array_equal(A, A0) and np.array_equal(r, r0) and nq == nq0


def test_admittance_is_the_velocity_system_with_v_equal_y_p(orc):
    """Reference sign, beta = the unscaled i/k (both betas coincide): the admittance solution p solves the existing velocity
    system with the full-length (bc_len = 3, constant) prescribed velocity v_j = Y_j p_j."""
    mesh = generate_icosphere_mesh(1.0, 2)
    k = 1.0
    beta = 1j / k
    assert orc.dg_dn_sign(mesh, k) == -1.0
    rng = np.random.default_rng(1)
    y = k * (rng.uniform(0.1, 0.6, mesh.n_elem) - 1j * rng.uniform(0.1, 0.6, mesh.n_elem))
    inc, _ = orc.incident_rhs(0, [0, 0, 1], 1.0, mesh.center, mesh.normal, k, beta)
    A, rhs, _ = ao.assemble_opts(mesh, k, beta, admittance=y)
    p = np.linalg.solve(A, rhs + inc)
    mesh.bc_len[:] = 3
    mesh.bc_val[:] = 0.0
    mesh.bc_val[:, :3] = (y * p)[:, None]
    Av, rv, _ = orc.assemble(mesh, k, beta)
    res = np.linalg.norm(Av @ p - (rv + inc)) / np.linalg.norm(rv + inc)
    assert res <= 1e-12, res


def _robin_error(sub, ka, yk):
    mesh = generate_icosphere_mesh(1.0, sub)
    k = ka
    beta = adaptive_beta(ka, k)
    from oracle import oracle as orc

    inc, _ = orc.incident_rhs(0, [0, 0, 1], 1.0, mesh.center, mesh.normal, k, beta)
    Y = yk * k
    A, rhs, _ = ao.assemble_opts(mesh, k, beta, dg_dn_sign=1, consistent_beta=True, admittance=np.full(mesh.n_elem, Y))
    return ao.rel_l2(np.linalg.solve(A, rhs + inc), ao.robin_mie(k, 1.0, Y, mesh.center))


@pytest.mark.parametrize("ka", [0.3, 2.0])
@pytest.mark.parametrize("yk", PASSIVE)
def test_robin_sphere_converges(orc, ka, yk):
    """Forced sign +1 and the consistent beta against the exact Robin series (plane wave along +z, radius 1, passive Y,
    Im Y <= 0 for exp(+ikr)).  Rigid at ka = 0.3 sits at a 0.44-0.47 % floor on both meshes and is exempt from the ratio."""
    e2, e3 = _robin_error(2, ka, yk), _robin_error(3, ka, yk)
    assert e3 <= (0.015 if yk == 0.0 else 0.08), (e2, e3)
    if not (yk == 0.0 and ka < 0.5):
        assert e3 < 0.75 * e2, (e2, e3)


def _pulsating_error(sub, ka, beta=None):
    from scipy.special import spherical_jn, spherical_yn

    mesh = generate_icosphere_mesh(1.0, sub)
    mesh.bc_len[:] = 3
    mesh.bc_val[:] = 0.0
    mesh.bc_val[:, :3] = 1.0
    k = ka
    beta = adaptive_beta(ka, k) if beta is None else beta
    A, rhs, _ = ao.assemble_opts(mesh, k, beta, dg_dn_sign=1, consistent_beta=True)
    r = np.linalg.norm(mesh.center, axis=1)
    h0 = lambda x: spherical_jn(0, x) + 1j * spherical_yn(0, x)  # noqa: E731
    h0p = lambda x: spherical_jn(0, x, True) + 1j * spherical_yn(0, x, True)  # noqa: E731
    return ao.rel_l2(np.linalg.solve(A, rhs), h0(k * r) / (k * h0p(k)))


@pytest.mark.parametrize("ka", [0.3, 2.0])
def test_pulsating_sphere_converges(ka):
    """Radiation of a pulsating sphere (dp/dn = 1): p = h0(kr) / (k h0'(ka)).  The error is a phase error of the
    beta-weighted hypersingular equation, O(h) and amplified by |beta| = 1/k at low ka (13.6 % on icosphere(2) at ka = 0.3,
    2.0 % with beta -> 0); it shrinks with the mesh: icosphere(2) -> (3) ratios 0.56 (ka = 0.3) and 0.43 (ka = 2)."""
    e2, e3 = _pulsating_error(2, ka), _pulsating_error(3, ka)
    assert e3 < 0.10 and e3 < 0.75 * e2, (e2, e3)
    if ka < 0.5:
        assert _pulsating_error(2, ka, beta=0.01j / ka) < 0.03  # the CBIE alone: the beta-weighted part carries the error


def test_option_validation():
    mesh = generate_icosphere_mesh(0.1, 1)
    mesh.bc_type[5] = BC_PRESSURE
    bct = np.asarray(mesh.bc_type, dtype=np.int32)
    y = np.zeros(mesh.n_elem, dtype=np.complex128)
    copts, ydof = bem.AssemblyOptions(1, True, y).to_c(bct)
    assert copts.dg_dn_sign == 1 and copts.consistent_beta == 1 and copts.admittance and ydof.shape == (mesh.n_elem,)
    with pytest.raises(ValueError, match="dg_dn_sign"):
        bem.AssemblyOptions(dg_dn_sign=2).to_c(bct)
    with pytest.raises(ValueError, match="entries"):
        bem.AssemblyOptions(admittance=np.ones(mesh.n_elem - 1)).to_c(bct)
    y[5] = 1.0 - 1.0j
    with pytest.raises(ValueError, match="velocity-BC"):
        bem.AssemblyOptions(admittance=y).to_c(bct)
    # the DOF order of a permuted map: entry j of the enumeration-order vector lands at DOF perm[j]
    perm = np.random.default_rng(0).permutation(mesh.n_elem)
    ye = np.arange(mesh.n_elem) * (1 - 1j)
    _, ydof = bem.AssemblyOptions(admittance=ye).to_c(np.zeros(mesh.n_elem, dtype=np.int32), perm)
    assert np.array_equal(ydof[perm], ye)
    with pytest.raises(ValueError, match="invalid"):  # the oracle refuses what the library refuses
        ao.assemble_opts(mesh, 10.0, 0.1j, admittance=y)
    with pytest.raises(ValueError, match="invalid"):
        ao.assemble_opts(mesh, 10.0, 0.1j, dg_dn_sign=3)
    v = bem.surface_velocity(mesh, 2.0 - 1.0j, np.ones(mesh.n_elem), v_bar=np.full(mesh.n_elem, 0.5))
    assert np.allclose(v, 2.5 - 1.0j)
    with pytest.raises(ValueError):
        bem.surface_velocity(mesh, 1.0, np.ones(3))
