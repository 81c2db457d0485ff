"""Argument checks of the multi-direction entry points (DESIGN.md section 4.7) that need no GPU: the Python wrappers refuse bad
shapes, types and source groups with ValueError before calling the library, and the C entries refuse NULL arguments with
BEMB200_EINVAL before touching a device."""
import ctypes as C
import types

import numpy as np
import pytest

from math_audio_b200 import _capi, bem
from math_audio_b200.incident import IncidentField
from math_audio_b200.types import PhysicsParams

EINVAL = -1
PH = PhysicsParams.from_wave_number(20.0)


def _staged(n=10, enum_to_dof=None):
    """stand-in for a StagedMesh: the wrappers read num_dofs / enum_to_dof before any library call"""
    return types.SimpleNamespace(num_dofs=n, enum_to_dof=enum_to_dof, _h=None, ctx=types.SimpleNamespace(_h=None))


def test_source_groups_follow_incident_rhs_device_order():
    f = IncidentField(plane_waves=[(np.array([0.0, 0.0, 1.0]), 1.0 + 2.0j)], point_sources=[(np.array([1.0, 2.0, 3.0]), 0.5)])
    g = IncidentField.plane_wave([1.0, 0.0, 0.0])
    src_ptr, kinds, vecs, amps = bem.source_groups([f, g])
    assert src_ptr.tolist() == [0, 2, 3] and kinds.tolist() == [0, 1, 0]
    assert vecs.tolist() == [[0, 0, 1], [1, 2, 3], [1, 0, 0]] and amps.tolist() == [1 + 2j, 0.5, 1]


@pytest.mark.parametrize("incidents", [[], "abc", [1, 2], None, [IncidentField(point_sources=[(np.zeros(2), 1.0)])]])
def test_bad_incidents_are_refused(incidents):
    with pytest.raises(ValueError):
        bem.incident_rhs_batch(_staged(), PH, 0j, incidents)


@pytest.mark.parametrize("src_ptr", [[1, 2], [0, 2, 1], [0], [[0, 1]], [0.0, 1.0], [0, 70000]])
def test_bad_src_ptr_is_refused(src_ptr):
    ns = 1
    with pytest.raises(ValueError):
        bem.check_source_groups(np.asarray(src_ptr), np.zeros(ns, np.int32), np.zeros((ns, 3)), np.ones(ns, np.complex128))


def test_bad_source_arrays_are_refused():
    ok = (np.array([0, 1, 2]), np.array([0, 1]), np.zeros((2, 3)), np.ones(2))
    bem.check_source_groups(*ok)
    with pytest.raises(ValueError):
        bem.check_source_groups(ok[0], np.array([0, 2]), ok[2], ok[3])  # unknown kind
    with pytest.raises(ValueError):
        bem.check_source_groups(ok[0], ok[1], np.zeros((2, 2)), ok[3])
    with pytest.raises(ValueError):
        bem.check_source_groups(ok[0], ok[1], ok[2], np.ones(3))
    with pytest.raises(ValueError):
        bem.check_source_groups(np.arange(34), np.zeros(33, np.int32), np.zeros((33, 3)), np.ones(33), max_groups=32)
    with pytest.raises(ValueError):  # fetch=False without a device buffer
        bem.incident_rhs_batch(_staged(), PH, 0j, [IncidentField.plane_wave_z()], fetch=False)
    with pytest.raises(ValueError):
        bem.incident_rhs_batch(_staged(), PH, 0j, [IncidentField.plane_wave_z()], system=object())


def test_batch_postprocess_wrappers_refuse_bad_arguments():
    st = _staged(10)
    dirs = np.eye(3)
    pts = np.ones((4, 3))
    for bad in (np.zeros(10), np.zeros((2, 9)), np.zeros((0, 10)), np.zeros((4097, 10))):
        with pytest.raises(ValueError):
            bem.compute_rcs_batch(bad, st, dirs, PH)
        with pytest.raises(ValueError):
            bem.compute_scattered_field_batch(pts, st, bad, None, PH)
    P = np.zeros((2, 10), np.complex128)
    with pytest.raises(ValueError):
        bem.compute_rcs_batch(P, st, np.ones(3), PH)  # directions must be (M, 3)
    with pytest.raises(ValueError):
        bem.compute_rcs_batch(P, st, dirs, PH, nsol=3)  # nsol does not match
    with pytest.raises(ValueError):
        bem.compute_scattered_field_batch(np.ones((4, 2)), st, P, None, PH)
    with pytest.raises(ValueError):
        bem.compute_scattered_field_batch(pts, st, P, np.zeros((3, 10)), PH)
    for ptr, nsol in ((1 << 20, None), (1 << 20, 0), (1 << 20, 5000), (True, 1), (-5, 1), (0, 1)):
        with pytest.raises(ValueError):
            bem.compute_rcs_batch(ptr, st, dirs, PH, nsol=nsol)
    with pytest.raises(ValueError):  # mixed host / device inputs
        bem.compute_scattered_field_batch(pts, st, 1 << 20, P, PH, nsol=2)


def test_gmres_batched_device_wrapper_refuses_bad_arguments():
    op = types.SimpleNamespace(matrix=types.SimpleNamespace(_h=None, ctx=types.SimpleNamespace(_h=None)))
    cfg = bem.GmresConfig()
    for b, nrhs, x in ((0, 1, 1 << 20), (1 << 20, 0, 1 << 20), (1 << 20, 33, 1 << 20), (1 << 20, 2, None), (1 << 20, 2.0, 1 << 20),
                       (np.zeros(3), 1, 1 << 20)):
        with pytest.raises(ValueError):
            bem.gmres_batched_device(op, b, nrhs, cfg, x)
    with pytest.raises(ValueError):
        bem.gmres_batched_device(op, 1 << 20, 2, cfg, 1 << 21, precond=bem.IdentityPreconditioner())


def test_c_entries_refuse_null_arguments_without_a_device():
    lib = _capi.lib()
    ph = _capi.CPhysics(1.0, 1.0, 1.0, 1.0)
    grp = (C.c_uint32 * 2)(0, 1)
    kinds = (C.c_int32 * 1)(0)
    v = (C.c_double * 3)(0.0, 0.0, 1.0)
    amp = (C.c_double * 2)(1.0, 0.0)
    out = (C.c_double * 64)()
    info = (_capi.CGmresInfo * 4)()
    cnt = C.c_uint32()
    assert lib.bemb200_incident_rhs_batch(None, C.byref(ph), 0.0, 0.0, 1, grp, kinds, v, amp, None, out, None) == EINVAL
    assert lib.bemb200_incident_rhs_batch(None, C.byref(ph), 0.0, 0.0, 1, None, kinds, v, amp, None, out, None) == EINVAL
    assert lib.bemb200_gmres_batched_device(None, None, out, 1, 10, 5, 1e-6, out, info, None, None) == EINVAL
    assert lib.bemb200_compute_rcs_batch(None, C.byref(ph), 1, out, 0, 1, v, out) == EINVAL
    assert lib.bemb200_scattered_field_batch(None, C.byref(ph), 1, out, None, 0, 1, v, out) == EINVAL
    assert lib.bemb200_sweep_submit_incident(None, C.byref(ph), 0.0, 0.0, 1, grp, kinds, v, amp, 10, 5, 1e-6) == EINVAL
    assert lib.bemb200_sweep_next_batch(None, 4, out, info, C.byref(cnt), None) == EINVAL
