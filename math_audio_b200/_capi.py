"""ctypes binding of libbemb200.so -- exactly the declarations of include/bemb200.h.

This is the same boundary a Rust `extern "C"` block binds (INTEGRATION.md).  The product
has no CPU fallback: if the library is missing or no B200 is visible, calls raise.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "libbemb200.so"

OK = 0
ERRORS = {-1: "EINVAL", -2: "ENODEVICE", -3: "ECUDA", -4: "ENOMEM", -5: "ENCCL", -6: "EUNSUPPORTED", -7: "ESINGULAR", -8: "ECALLBACK"}


class Bemb200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libbemb200 {ERRORS.get(code, code)}: {msg}")
        self.code = code


class CMesh(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_uint64), ("n_elem", C.c_uint64),
        ("nodes", C.c_void_p), ("conn", C.c_void_p), ("etype", C.c_void_p),
        ("center", C.c_void_p), ("normal", C.c_void_p), ("area", C.c_void_p),
        ("bc_type", C.c_void_p), ("bc_len", C.c_void_p), ("bc_val", C.c_void_p),
        ("dof", C.c_void_p), ("is_eval", C.c_void_p),
    ]


class CPhysics(C.Structure):
    _fields_ = [("wave_number", C.c_double), ("harmonic_factor", C.c_double), ("tau", C.c_double), ("gamma", C.c_double)]


class CGmresInfo(C.Structure):
    _fields_ = [("iterations", C.c_uint64), ("restarts", C.c_uint64), ("residual", C.c_double), ("converged", C.c_int32)]


class CAssemblyStats(C.Structure):
    _fields_ = [("near_pairs", C.c_uint64), ("special_pairs", C.c_uint64), ("far_kernel_launches", C.c_uint64),
                ("total_launches", C.c_uint64), ("far_ms", C.c_double), ("total_ms", C.c_double)]


class CAssemblyOptions(C.Structure):
    _fields_ = [("dg_dn_sign", C.c_int32), ("consistent_beta", C.c_int32), ("admittance", C.c_void_p)]


class CPrecondStats(C.Structure):
    _fields_ = [("num_subdomains", C.c_uint32), ("local_subdomains", C.c_uint32), ("min_size", C.c_uint32), ("max_size", C.c_uint32),
                ("avg_size", C.c_double), ("inverse_bytes", C.c_uint64), ("factor_ms", C.c_double), ("disjoint", C.c_int32)]


class CRoomSource(C.Structure):
    _fields_ = [("position", C.c_double * 3), ("amplitude", C.c_double), ("directivity", C.c_void_p),
                ("n_horizontal", C.c_uint32), ("n_vertical", C.c_uint32)]


# every symbol include/bemb200.h declares: (restype, argtypes)
_VP = C.c_void_p
_PP = C.POINTER(C.c_void_p)
# bemb200_precond_fn: int apply(void* user, const double* r, double* z, uint64_t n)  (Preconditioner::apply, traits.rs:366-371)
PRECOND_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_uint64)

SYMBOLS = {
    "bemb200_device_count": (C.c_int, []),
    "bemb200_ctx_create": (C.c_int, [C.c_int, _PP]),
    "bemb200_nccl_unique_id": (C.c_int, [_VP]),
    "bemb200_ctx_create_dist": (C.c_int, [C.c_int, C.c_int, C.c_int, _VP, _PP]),
    "bemb200_ctx_create_ex": (C.c_int, [C.c_int, C.c_int, C.c_int, _VP, _VP, _PP]),
    "bemb200_ctx_destroy": (None, [_VP]),
    "bemb200_matrix_set_context": (C.c_int, [_VP, _VP]),
    "bemb200_ctx_set_background": (C.c_int, [_VP, C.c_int]),
    "bemb200_ctx_set_shared_gpu": (C.c_int, [_VP, C.c_int]),
    "bemb200_matrix_boost_assembly": (C.c_int, [_VP, _VP]),
    "bemb200_ctx_peer_exchange_active": (C.c_int, [_VP, C.POINTER(C.c_int)]),
    "bemb200_last_error": (C.c_char_p, [_VP]),
    "bemb200_partition": (None, [C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "bemb200_mesh_stage": (C.c_int, [_VP, C.POINTER(CMesh), _PP]),
    "bemb200_staged_mesh_free": (None, [_VP]),
    "bemb200_staged_num_dofs": (C.c_uint64, [_VP]),
    "bemb200_assemble_staged": (C.c_int, [_VP, _VP, C.POINTER(CPhysics), C.c_double, C.c_double, C.c_uint64, C.c_uint64, _PP]),
    "bemb200_assemble_staged_opts": (C.c_int, [_VP, _VP, C.POINTER(CPhysics), C.c_double, C.c_double, C.POINTER(CAssemblyOptions),
                                               C.c_uint64, C.c_uint64, _PP]),
    "bemb200_assemble": (C.c_int, [_VP, C.POINTER(CMesh), C.POINTER(CPhysics), C.c_double, C.c_double, C.c_uint64, C.c_uint64, _PP]),
    "bemb200_assembly_stats_get": (C.c_int, [_VP, C.POINTER(CAssemblyStats)]),
    "bemb200_dg_dn_sign": (C.c_double, [_VP, C.c_double]),
    "bemb200_matrix_from_host": (C.c_int, [_VP, _VP, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, _PP]),
    "bemb200_matrix_free": (None, [_VP]),
    "bemb200_num_rows": (C.c_uint64, [_VP]),
    "bemb200_num_cols": (C.c_uint64, [_VP]),
    "bemb200_local_row_begin": (C.c_uint64, [_VP]),
    "bemb200_local_row_end": (C.c_uint64, [_VP]),
    "bemb200_matrix_download": (C.c_int, [_VP, C.c_uint64, C.c_uint64, _VP]),
    "bemb200_rhs_download": (C.c_int, [_VP, _VP]),
    "bemb200_rhs_download_full": (C.c_int, [_VP, _VP]),
    "bemb200_row_sum_correction": (C.c_int, [_VP, C.POINTER(C.c_double)]),
    "bemb200_apply": (C.c_int, [_VP, _VP, _VP]),
    "bemb200_apply_transpose": (C.c_int, [_VP, _VP, _VP]),
    "bemb200_apply_device": (C.c_int, [_VP, _VP, _VP]),
    "bemb200_gmres": (C.c_int, [_VP, _VP, _VP, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo)]),
    "bemb200_gmres_preconditioned": (C.c_int, [_VP, _VP, _VP, _VP, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo)]),
    "bemb200_matrix_diagonal": (C.c_int, [_VP, _VP]),
    "bemb200_schwarz_create": (C.c_int, [_VP, C.c_uint32, _VP, _VP, _PP]),
    "bemb200_precond_free": (None, [_VP]),
    "bemb200_precond_stats_get": (C.c_int, [_VP, C.POINTER(CPrecondStats)]),
    "bemb200_precond_apply": (C.c_int, [_VP, _VP, _VP]),
    "bemb200_gmres_schwarz": (C.c_int, [_VP, _VP, _VP, _VP, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo)]),
    "bemb200_gmres_callback": (C.c_int, [_VP, PRECOND_FN, _VP, _VP, _VP, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo),
                                         C.POINTER(C.c_uint64)]),
    "bemb200_gmres_device": (C.c_int, [_VP, _VP, _VP, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo)]),
    "bemb200_gmres_batched": (C.c_int, [_VP, _VP, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo),
                                        C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "bemb200_gmres_batched_schwarz": (C.c_int, [_VP, _VP, _VP, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo),
                                                C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "bemb200_gmres_batched_device": (C.c_int, [_VP, _VP, _VP, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo),
                                               C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "bemb200_apply_block": (C.c_int, [_VP, _VP, C.c_uint32, _VP, C.POINTER(C.c_double)]),
    "bemb200_solver_stats": (C.c_int, [_VP, C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "bemb200_incident_rhs": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_double, C.c_double, C.c_uint32, _VP, _VP, _VP, _VP, _VP]),
    "bemb200_scattered_field": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_uint64, _VP, _VP, _VP, _VP]),
    "bemb200_compute_rcs": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_uint32, _VP, _VP, _VP]),
    "bemb200_incident_rhs_batch": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_double, C.c_double, C.c_uint32, _VP, _VP, _VP, _VP, _VP, _VP,
                                             _VP]),
    "bemb200_compute_rcs_batch": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_uint32, _VP, C.c_int, C.c_uint32, _VP, _VP]),
    "bemb200_scattered_field_batch": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_uint32, _VP, _VP, C.c_int, C.c_uint64, _VP, _VP]),
    "bemb200_far_field": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_uint32, _VP, _VP, C.c_int, C.c_uint32, _VP, _VP]),
    "bemb200_evaluate_field": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_uint32, _VP, _VP, C.c_int, C.c_uint64, _VP, _VP]),
    "bemb200_evaluate_field_gradient": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_uint32, _VP, _VP, C.c_int, C.c_uint64, _VP, _VP, _VP]),
    "bemb200_bicgstab": (C.c_int, [_VP, _VP, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo)]),
    "bemb200_cgs": (C.c_int, [_VP, _VP, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo)]),
    "bemb200_lu_solve": (C.c_int, [_VP, _VP, _VP, C.c_int, C.POINTER(C.c_double)]),
    "bemb200_room_mesh_stage": (C.c_int, [_VP, _VP, C.c_uint64, _VP, C.c_uint64, _PP]),
    "bemb200_room_mesh_free": (None, [_VP]),
    "bemb200_room_mesh_num_elements": (C.c_uint64, [_VP]),
    "bemb200_room_mesh_geometry": (C.c_int, [_VP, _VP, _VP, _VP]),
    "bemb200_room_assemble": (C.c_int, [_VP, _VP, C.c_double, C.c_uint64, C.c_uint64, _PP, C.POINTER(C.c_double)]),
    "bemb200_room_incident_rhs": (C.c_int, [_VP, C.c_double, C.c_uint32, C.POINTER(CRoomSource), _VP, _VP]),
    "bemb200_room_field_pressure": (C.c_int, [_VP, C.c_double, C.c_uint32, C.POINTER(CRoomSource), C.c_uint64, _VP, _VP, _VP]),
    "bemb200_measure_fp64_peak": (C.c_int, [_VP, C.POINTER(C.c_double)]),
    "bemb200_selftest_math": (C.c_int, [_VP, C.c_uint64, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "bemb200_measure_allgather": (C.c_int, [_VP, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "bemb200_matrix_device_ptr": (_VP, [_VP]),
    "bemb200_sweep_create": (C.c_int, [C.c_int, C.c_int, C.c_int, _VP, C.POINTER(CMesh), C.c_int, C.c_int, _PP]),
    "bemb200_sweep_num_dofs": (C.c_uint64, [_VP]),
    "bemb200_sweep_submit": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_double, C.c_double, _VP, C.c_uint32, C.c_uint32, C.c_double]),
    "bemb200_sweep_next": (C.c_int, [_VP, _VP, C.POINTER(CGmresInfo), C.POINTER(CAssemblyStats), _VP]),
    "bemb200_sweep_submit_incident": (C.c_int, [_VP, C.POINTER(CPhysics), C.c_double, C.c_double, C.c_uint32, _VP, _VP, _VP, _VP,
                                                C.c_uint32, C.c_uint32, C.c_double]),
    "bemb200_sweep_next_batch": (C.c_int, [_VP, C.c_uint32, _VP, C.POINTER(CGmresInfo), C.POINTER(C.c_uint32), C.POINTER(CAssemblyStats)]),
    "bemb200_sweep_boosts": (C.c_uint64, [_VP]),
    "bemb200_sweep_set_block_jacobi": (C.c_int, [_VP, C.c_uint32, _VP, _VP]),
    "bemb200_sweep_set_assembly_options": (C.c_int, [_VP, C.POINTER(CAssemblyOptions)]),
    "bemb200_sweep_destroy": (None, [_VP]),
    "bemb200_multi_create": (C.c_int, [C.POINTER(C.c_int), C.c_int, _PP]),
    "bemb200_multi_destroy": (None, [_VP]),
    "bemb200_multi_num_ranks": (C.c_int, [_VP]),
    "bemb200_multi_last_error": (C.c_char_p, [_VP]),
    "bemb200_multi_assemble": (C.c_int, [_VP, C.POINTER(CMesh), C.POINTER(CPhysics), C.c_double, C.c_double, _PP]),
    "bemb200_multi_matrix_free": (None, [_VP]),
    "bemb200_multi_num_rows": (C.c_uint64, [_VP]),
    "bemb200_multi_rhs_download": (C.c_int, [_VP, _VP]),
    "bemb200_multi_matrix_download": (C.c_int, [_VP, C.c_uint64, C.c_uint64, _VP]),
    "bemb200_multi_gmres": (C.c_int, [_VP, _VP, _VP, C.c_uint32, C.c_uint32, C.c_double, _VP, C.POINTER(CGmresInfo)]),
}

_lib = None


def lib():
    """Load libbemb200.so (built in-tree by math_audio_b200.build). Raises if it is missing."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise FileNotFoundError(
                f"{LIB_PATH} not found: build it with `python -m math_audio_b200.build` (nvcc, sm_100a). "
                "There is no CPU fallback.")
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, ctx=None):
    if rc != OK:
        msg = lib().bemb200_last_error(ctx)
        if (not msg) and ctx is not None:
            msg = lib().bemb200_last_error(None)
        raise Bemb200Error(rc, (msg or b"").decode(errors="replace"))


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def cmesh(mesh) -> CMesh:
    arrs = dict(
        nodes=np.ascontiguousarray(mesh.nodes, dtype=np.float64),
        conn=np.ascontiguousarray(mesh.conn, dtype=np.uint32),
        etype=np.ascontiguousarray(mesh.etype, dtype=np.uint8),
        center=np.ascontiguousarray(mesh.center, dtype=np.float64),
        normal=np.ascontiguousarray(mesh.normal, dtype=np.float64),
        area=np.ascontiguousarray(mesh.area, dtype=np.float64),
        bc_type=np.ascontiguousarray(mesh.bc_type, dtype=np.int32),
        bc_len=np.ascontiguousarray(mesh.bc_len, dtype=np.uint8),
        bc_val=np.ascontiguousarray(mesh.bc_val, dtype=np.complex128),
        dof=np.ascontiguousarray(mesh.dof, dtype=np.uint32),
        is_eval=np.ascontiguousarray(mesh.is_eval, dtype=np.uint8),
    )
    m = CMesh(mesh.n_nodes, mesh.n_elem, *[ptr(arrs[k]) for k in
              ("nodes", "conn", "etype", "center", "normal", "area", "bc_type", "bc_len", "bc_val", "dof", "is_eval")])
    m._keep = arrs
    return m


def mesh_nbytes(mesh) -> int:
    return int(sum(getattr(mesh, k).nbytes for k in
                   ("nodes", "conn", "etype", "center", "normal", "area", "bc_type", "bc_len", "bc_val", "dof", "is_eval")))
