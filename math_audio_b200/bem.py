"""Host-side mirror of the reference's operator interface for the assemble + GMRES path,
over the C ABI of libbemb200 (no torch types, no CPU fallback).

Reference interface (same names, argument meaning, error behaviour):

* ``build_tbem_system{,_with_beta,_scaled,_bounded}`` -> ``TbemSystem``   math-bem/src/core/assembly/tbem.rs:13-101
* ``apply_row_sum_correction`` / ``build_tbem_system_corrected``          tbem.rs:500-534
* ``DenseOperator`` (``LinearOperator``: num_rows/num_cols/apply/apply_transpose/apply_hermitian)
                                                                          math-bem/src/core/solver/fmm_interface.rs:25-52,
                                                                          math-solvers/src/traits.rs:316-364
* ``GmresConfig`` / ``GmresSolution`` / ``gmres`` / ``gmres_with_guess`` / ``solve_gmres``
                                                                          math-solvers/src/iterative/gmres.rs:16-36,74-105,
                                                                          fmm_interface.rs:378-384

Differences forced by the device: ``TbemSystem.matrix`` stays on the GPU behind an opaque
handle (a 120k x 120k complex128 matrix is 237 GB, it can never be an ``Array2``); rows can be
fetched with ``matrix_rows``.  Shape mismatches raise (the reference panics).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _capi
from .mesh import Mesh
from .types import PhysicsParams


class Context:
    """One GPU (optionally one rank of a row-sharded job: one process per GPU)."""

    def __init__(self, device: int = 0, rank: int = 0, nranks: int = 1, nccl_id: Optional[bytes] = None,
                 cuda_stream: int = 0):
        """``cuda_stream``: raw cudaStream_t (e.g. ``torch.cuda.current_stream().cuda_stream``) to submit
        all work to, so that the caller's CUDA events bracket it; 0 = library-owned stream."""
        self._lib = _capi.lib()
        self._h = C.c_void_p()
        idp = None
        if nranks > 1 and nccl_id is not None:  # nccl_id None: context without communicator (assembly only)
            assert len(nccl_id) == 128
            self._idbuf = (C.c_uint8 * 128).from_buffer_copy(nccl_id)
            idp = C.cast(self._idbuf, C.c_void_p)
        _capi.check(self._lib.bemb200_ctx_create_ex(device, rank, nranks, idp, C.c_void_p(cuda_stream or None), C.byref(self._h)))
        self.device, self.rank, self.nranks = device, rank, nranks

    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = (C.c_uint8 * 128)()
        _capi.check(_capi.lib().bemb200_nccl_unique_id(C.cast(buf, C.c_void_p)))
        return bytes(buf)

    def partition(self, n: int):
        b, e = C.c_uint64(), C.c_uint64()
        self._lib.bemb200_partition(n, self.nranks, self.rank, C.byref(b), C.byref(e))
        return int(b.value), int(e.value)

    def measure_fp64_peak(self) -> float:
        t = C.c_double()
        _capi.check(self._lib.bemb200_measure_fp64_peak(self._h, C.byref(t)), self._h)
        return float(t.value)

    def selftest_math(self, n: int = 1 << 22, xmax: float = 200.0):
        a, b = C.c_double(), C.c_double()
        _capi.check(self._lib.bemb200_selftest_math(self._h, n, xmax, C.byref(a), C.byref(b)), self._h)
        return float(a.value), float(b.value)

    def set_background(self, blocks_per_sm: int) -> None:
        _capi.check(self._lib.bemb200_ctx_set_background(self._h, blocks_per_sm), self._h)

    def peer_exchange_active(self) -> bool:
        """True once row-sharded solves exchange A v through peer memory (fused ZGEMV epilogue) instead of NCCL."""
        a = C.c_int(0)
        _capi.check(self._lib.bemb200_ctx_peer_exchange_active(self._h, C.byref(a)), self._h)
        return bool(a.value)

    def set_shared_gpu(self, shared: bool) -> None:
        """Tell this context's solver that other streams share the GPU (no whole-GPU cooperative kernels)."""
        _capi.check(self._lib.bemb200_ctx_set_shared_gpu(self._h, 1 if shared else 0), self._h)

    def measure_allgather(self, bytes_per_rank: int, iters: int = 200, sync_each: bool = False) -> float:
        t = C.c_double()
        _capi.check(self._lib.bemb200_measure_allgather(self._h, bytes_per_rank, iters, 1 if sync_each else 0, C.byref(t)), self._h)
        return float(t.value)

    def close(self):
        if self._h:
            self._lib.bemb200_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Optional[Context] = None


class MultiGpu:
    """One process, several devices (`bemb200_multi_*`, csrc/sweep.cu): the shape of every reference caller
    (BemSolver::solve, qa_suite are single processes).  Rows are block partitioned over `devices`; the solve is the
    persistent fused GMRES kernel on every device with peer-memory exchange.  The same device may be listed twice (its SMs
    are split): that is how the sharded solver is exercised on a single GPU."""

    def __init__(self, devices):
        self._lib = _capi.lib()
        self._h = C.c_void_p()
        arr = (C.c_int * len(devices))(*[int(d) for d in devices])
        _capi.check(self._lib.bemb200_multi_create(arr, len(devices), C.byref(self._h)), None)
        self.nranks = len(devices)

    def build_tbem_system_with_beta(self, mesh: Mesh, physics: PhysicsParams, beta: complex) -> "MultiSystem":
        cm = _capi.cmesh(mesh)
        ph = _cphys(physics)
        beta = complex(beta)
        h = C.c_void_p()
        _capi.check(self._lib.bemb200_multi_assemble(self._h, C.byref(cm), C.byref(ph), beta.real, beta.imag, C.byref(h)), None)
        return MultiSystem(self, h)

    def close(self):
        if self._h:
            self._lib.bemb200_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiSystem:
    """TbemSystem whose matrix is row-sharded over the devices of a MultiGpu group."""

    def __init__(self, group: MultiGpu, handle):
        self.group, self._h, self._lib = group, handle, _capi.lib()
        self.num_dofs = int(self._lib.bemb200_multi_num_rows(self._h))

    @property
    def rhs(self) -> np.ndarray:
        out = np.empty(self.num_dofs, dtype=np.complex128)
        _capi.check(self._lib.bemb200_multi_rhs_download(self._h, _capi.ptr(out)), None)
        return out

    def rows(self, row_begin: int = 0, row_end: Optional[int] = None) -> np.ndarray:
        row_end = self.num_dofs if row_end is None else row_end
        out = np.empty((row_end - row_begin, self.num_dofs), dtype=np.complex128)
        _capi.check(self._lib.bemb200_multi_matrix_download(self._h, row_begin, row_end, _capi.ptr(out)), None)
        return out

    def gmres(self, b: np.ndarray, config: "GmresConfig", x0: Optional[np.ndarray] = None) -> "GmresSolution":
        b = np.ascontiguousarray(b, dtype=np.complex128)
        if b.shape != (self.num_dofs,):
            raise ValueError("gmres: b has the wrong length")
        x0a = np.ascontiguousarray(x0, dtype=np.complex128) if x0 is not None else None
        x = np.empty(self.num_dofs, dtype=np.complex128)
        info = _capi.CGmresInfo()
        _capi.check(self._lib.bemb200_multi_gmres(self._h, _capi.ptr(b), _capi.ptr(x0a) if x0a is not None else None,
                                                  config.max_iterations, config.restart, config.tolerance, _capi.ptr(x), C.byref(info)), None)
        return GmresSolution(x=x, iterations=int(info.iterations), restarts=int(info.restarts), residual=float(info.residual),
                             converged=bool(info.converged))

    def close(self):
        if self._h:
            self._lib.bemb200_multi_matrix_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


def enumeration_to_dof(mesh: Mesh) -> Optional[np.ndarray]:
    """DOF address of the j-th non-evaluation element, or None when that is j itself (every generator's sequential map).
    The reference pairs entry j of a surface vector with the j-th non-evaluation element (postprocess/pressure.rs:96-113,
    452-458); the device kernels pair an element with the entry at its DOF address (the C ABI's contract, include/bemb200.h)."""
    dof = np.asarray(mesh.dof, dtype=np.int64)[np.asarray(mesh.is_eval) == 0]
    if np.array_equal(dof, np.arange(dof.size)):
        return None
    if not np.array_equal(np.sort(dof), np.arange(dof.size)):
        return None  # not a permutation of 0..num_dofs-1: bemb200_mesh_stage has the say on such a mesh
    return dof


def surface_values_in_dof_order(enum_to_dof: Optional[np.ndarray], values: np.ndarray) -> np.ndarray:
    """Re-address a surface vector given as the reference takes it (entry j belongs to the j-th non-evaluation element) to the
    DOF order of the C ABI.  The pairing of values and elements -- including what it does to a solution vector of a mesh with
    a permuted DOF map -- is then the reference's."""
    if enum_to_dof is None:
        return values
    out = np.empty_like(values)
    out[enum_to_dof] = values
    return out


class StagedMesh:
    """Frequency-independent device copy of a mesh (reused across a sweep)."""

    def __init__(self, mesh: Mesh, ctx: Optional[Context] = None):
        self.ctx = ctx or default_context()
        self._lib = _capi.lib()
        self._h = C.c_void_p()
        cm = _capi.cmesh(mesh)
        _capi.check(self._lib.bemb200_mesh_stage(self.ctx._h, C.byref(cm), C.byref(self._h)), self.ctx._h)
        self.num_dofs = int(self._lib.bemb200_staged_num_dofs(self._h))
        self.nbytes_host = _capi.mesh_nbytes(mesh)
        self.enum_to_dof = enumeration_to_dof(mesh)
        self.bc_type = surface_values_in_dof_order(self.enum_to_dof, np.asarray(mesh.bc_type, dtype=np.int32)[np.asarray(mesh.is_eval) == 0])

    def dg_dn_sign(self, wave_number: float) -> float:
        return float(self._lib.bemb200_dg_dn_sign(self._h, wave_number))

    def close(self):
        if self._h:
            self._lib.bemb200_staged_mesh_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _cphys(physics: PhysicsParams) -> _capi.CPhysics:
    return _capi.CPhysics(physics.wave_number, physics.harmonic_factor, physics.tau, physics.gamma())


class DeviceMatrix:
    """Opaque handle of the local row slab of a dense complex128 operator on the GPU."""

    def __init__(self, ctx: Context, handle: C.c_void_p):
        self.ctx = ctx
        self._lib = _capi.lib()
        self._h = handle

    @property
    def shape(self):
        return int(self._lib.bemb200_num_rows(self._h)), int(self._lib.bemb200_num_cols(self._h))

    @property
    def local_rows(self):
        return int(self._lib.bemb200_local_row_begin(self._h)), int(self._lib.bemb200_local_row_end(self._h))

    def rows(self, row_begin: Optional[int] = None, row_end: Optional[int] = None) -> np.ndarray:
        lb, le = self.local_rows
        row_begin = lb if row_begin is None else row_begin
        row_end = le if row_end is None else row_end
        out = np.empty((row_end - row_begin, self.shape[1]), dtype=np.complex128)
        _capi.check(self._lib.bemb200_matrix_download(self._h, row_begin, row_end, _capi.ptr(out)), self.ctx._h)
        return out

    def rhs(self) -> np.ndarray:
        lb, le = self.local_rows
        out = np.empty(le - lb, dtype=np.complex128)
        _capi.check(self._lib.bemb200_rhs_download(self._h, _capi.ptr(out)), self.ctx._h)
        return out

    def assembly_stats(self) -> dict:
        st = _capi.CAssemblyStats()
        _capi.check(self._lib.bemb200_assembly_stats_get(self._h, C.byref(st)), self.ctx._h)
        return {k: getattr(st, k) for k, _ in st._fields_}

    def solver_stats(self) -> dict:
        a, b, c = C.c_uint64(), C.c_double(), C.c_uint64()
        _capi.check(self._lib.bemb200_solver_stats(self._h, C.byref(a), C.byref(b), C.byref(c)), self.ctx._h)
        return dict(kernel_launches=int(a.value), matvec_ms=float(b.value), matvecs=int(c.value))

    def device_ptr(self) -> int:
        return int(self._lib.bemb200_matrix_device_ptr(self._h) or 0)

    def boost_assembly(self, ctx: "Context") -> None:
        """Join a background assembly into this matrix (running in another thread/context) with extra far-kernel blocks
        on ``ctx``'s stream; no-op when none is in flight."""
        _capi.check(self._lib.bemb200_matrix_boost_assembly(self._h, ctx._h), ctx._h)

    def set_context(self, ctx: "Context") -> None:
        """Hand the matrix to another context of the same device (frequency-sweep pipelining)."""
        _capi.check(self._lib.bemb200_matrix_set_context(self._h, ctx._h), ctx._h)
        self.ctx = ctx

    def close(self):
        if self._h:
            self._lib.bemb200_matrix_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class TbemSystem:
    """tbem.rs:13-20.  ``matrix`` is device resident; ``rhs`` holds the local rows' entries."""

    matrix: DeviceMatrix
    rhs: Optional[np.ndarray]
    num_dofs: int

    def rhs_full(self, n: Optional[int] = None) -> np.ndarray:
        """TbemSystem.rhs for ALL rows (on a row-sharded system the slices are all-gathered)."""
        out = np.empty(self.num_dofs, dtype=np.complex128)
        _capi.check(_capi.lib().bemb200_rhs_download_full(self.matrix._h, _capi.ptr(out)), self.matrix.ctx._h)
        return out


@dataclass
class AssemblyOptions:
    """Options of one assembly (DESIGN.md 4.8, ``bemb200_assembly_options``); the defaults are the reference's assembly.

    * ``dg_dn_sign``: 0 = the reference's heuristic (tbem.rs:108-123, -1 once k * mean radius >= 0.5), or a forced +1 / -1.
    * ``consistent_beta``: the prescribed-velocity right-hand-side integrals use the assembly's beta instead of the unscaled
      i/k.  With ``dg_dn_sign=+1`` this is the sign-consistent Burton-Miller formulation, which converges to the exact
      solution at every ka (the reference's formulation does not above ka = 0.5).
    * ``admittance``: None, or one complex Y per boundary element in enumeration order (entry j <-> the j-th
      non-evaluation element, as surface vectors are passed everywhere else).  An absorbing velocity-BC element satisfies
      v = vbar + Y p with v = dp/dn (outward normal), Y in 1/m and constant over the element.  Passive surfaces have
      Im Y <= 0 for harmonic_factor = +1.  Only velocity-BC elements may carry a non-zero Y.
    """

    dg_dn_sign: int = 0
    consistent_beta: bool = False
    admittance: Optional[np.ndarray] = None

    @staticmethod
    def sign_consistent(admittance=None) -> "AssemblyOptions":
        return AssemblyOptions(dg_dn_sign=1, consistent_beta=True, admittance=admittance)

    def to_c(self, bc_type: np.ndarray, enum_to_dof: Optional[np.ndarray] = None):
        """(CAssemblyOptions, admittance array it points to, in DOF order) for a mesh whose boundary elements have the
        DOF-order BC types ``bc_type``.  Raises ValueError for options the library would refuse."""
        if self.dg_dn_sign not in (-1, 0, 1):
            raise ValueError(f"dg_dn_sign must be 0 (heuristic), +1 or -1, not {self.dg_dn_sign!r}")
        if self.consistent_beta not in (False, True, 0, 1):
            raise ValueError(f"consistent_beta must be a bool, not {self.consistent_beta!r}")
        y = None
        if self.admittance is not None:
            y = np.asarray(self.admittance, dtype=np.complex128)
            if y.ndim == 0:
                y = np.full(len(bc_type), complex(y))
            if y.shape != (len(bc_type),):
                raise ValueError(f"admittance has {y.size} entries, the mesh has {len(bc_type)} boundary elements")
            y = np.ascontiguousarray(surface_values_in_dof_order(enum_to_dof, y))
            bad = np.flatnonzero((y != 0) & (np.asarray(bc_type) != 0))
            if bad.size:
                raise ValueError(f"admittance is allowed on velocity-BC elements only (DOF {int(bad[0])} has bc_type {int(bc_type[bad[0]])})")
        c = _capi.CAssemblyOptions(int(self.dg_dn_sign), 1 if self.consistent_beta else 0, _capi.ptr(y) if y is not None else None)
        return c, y


def surface_velocity(mesh: Mesh, admittance, p: np.ndarray, v_bar: Optional[np.ndarray] = None) -> np.ndarray:
    """v = vbar + Y p on the boundary elements (enumeration order), the surface velocity ``compute_scattered_field`` needs
    for a solution ``p`` of a system assembled with ``AssemblyOptions(admittance=admittance)``; vbar defaults to 0."""
    n = int((np.asarray(mesh.is_eval) == 0).sum())
    p = np.asarray(p, dtype=np.complex128)
    y = np.broadcast_to(np.asarray(admittance, dtype=np.complex128), (n,))
    if p.shape != (n,):
        raise ValueError("p has the wrong length")
    v = y * p
    if v_bar is not None:
        v = np.asarray(v_bar, dtype=np.complex128) + v
    return v


def build_tbem_system_with_beta(elements: Mesh | StagedMesh, physics: PhysicsParams, beta: complex,
                                ctx: Optional[Context] = None, rows=None, reuse: Optional[TbemSystem] = None,
                                fetch_rhs: bool = True, options: Optional[AssemblyOptions] = None) -> TbemSystem:
    """tbem.rs:96-222.  ``elements`` carries nodes + elements (SoA).  ``rows=(r0, r1)`` assembles
    one row block (default: this rank's canonical block, i.e. everything on one GPU).
    ``fetch_rhs=False`` leaves TbemSystem.rhs on the device (``rhs`` is None).
    ``options`` (``AssemblyOptions``): admittance boundaries and the sign-consistent formulation; None is the reference's
    assembly."""
    lib = _capi.lib()
    staged = elements if isinstance(elements, StagedMesh) else StagedMesh(elements, ctx)
    ctx = staged.ctx
    n = staged.num_dofs
    r0, r1 = rows if rows is not None else ctx.partition(n)
    h = reuse.matrix._h if reuse is not None else C.c_void_p()
    ph = _cphys(physics)
    beta = complex(beta)
    if options is None:
        _capi.check(lib.bemb200_assemble_staged(ctx._h, staged._h, C.byref(ph), beta.real, beta.imag, r0, r1, C.byref(h)), ctx._h)
    else:
        copts, _y = options.to_c(staged.bc_type, staged.enum_to_dof)
        _capi.check(lib.bemb200_assemble_staged_opts(ctx._h, staged._h, C.byref(ph), beta.real, beta.imag, C.byref(copts), r0, r1,
                                                     C.byref(h)), ctx._h)
    mat = reuse.matrix if reuse is not None else DeviceMatrix(ctx, h)
    return TbemSystem(matrix=mat, rhs=mat.rhs() if fetch_rhs else None, num_dofs=n)


def build_tbem_system(elements, physics: PhysicsParams, **kw) -> TbemSystem:  # tbem.rs:45-51
    return build_tbem_system_with_beta(elements, physics, physics.burton_miller_beta(), **kw)


def build_tbem_system_scaled(elements, physics: PhysicsParams, scale: float, **kw) -> TbemSystem:  # tbem.rs:85-93
    return build_tbem_system_with_beta(elements, physics, physics.burton_miller_beta_scaled(scale), **kw)


def build_tbem_system_bounded(elements, physics: PhysicsParams, avg_element_size: float, **kw) -> TbemSystem:  # tbem.rs:64-72
    return build_tbem_system_with_beta(elements, physics, physics.burton_miller_beta_optimal(avg_element_size), **kw)


def apply_row_sum_correction(system: TbemSystem) -> float:  # tbem.rs:500-520
    avg = C.c_double()
    _capi.check(_capi.lib().bemb200_row_sum_correction(system.matrix._h, C.byref(avg)), system.matrix.ctx._h)
    return float(avg.value)


def build_tbem_system_corrected(elements, physics: PhysicsParams, **kw):  # tbem.rs:526-534
    system = build_tbem_system(elements, physics, **kw)
    return system, apply_row_sum_correction(system)


class DenseOperator:
    """fmm_interface.rs:25-52: ``DenseOperator::new(matrix)`` + the ``LinearOperator`` trait."""

    def __init__(self, matrix, ctx: Optional[Context] = None):
        if isinstance(matrix, TbemSystem):
            matrix = matrix.matrix
        if isinstance(matrix, DeviceMatrix):
            self.matrix = matrix
        else:
            a = np.ascontiguousarray(matrix, dtype=np.complex128)
            if a.ndim != 2:
                raise ValueError("DenseOperator needs a 2-D matrix")
            ctx = ctx or default_context()
            r0, r1 = ctx.partition(a.shape[0])
            h = C.c_void_p()
            loc = np.ascontiguousarray(a[r0:r1])
            _capi.check(_capi.lib().bemb200_matrix_from_host(ctx._h, _capi.ptr(loc), a.shape[0], a.shape[1], r0, r1, C.byref(h)), ctx._h)
            self.matrix = DeviceMatrix(ctx, h)
        self._lib = _capi.lib()

    def num_rows(self) -> int:
        return self.matrix.shape[0]

    def num_cols(self) -> int:
        return self.matrix.shape[1]

    def is_square(self) -> bool:
        return self.num_rows() == self.num_cols()

    def apply(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.complex128)
        if x.shape != (self.num_cols(),):
            raise ValueError(f"apply: x has shape {x.shape}, operator has {self.num_cols()} columns")
        y = np.empty(self.num_rows(), dtype=np.complex128)
        _capi.check(self._lib.bemb200_apply(self.matrix._h, _capi.ptr(x), _capi.ptr(y)), self.matrix.ctx._h)
        return y

    def apply_transpose(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.complex128)
        if x.shape != (self.num_rows(),):
            raise ValueError(f"apply_transpose: x has shape {x.shape}, operator has {self.num_rows()} rows")
        y = np.empty(self.num_cols(), dtype=np.complex128)
        _capi.check(self._lib.bemb200_apply_transpose(self.matrix._h, _capi.ptr(x), _capi.ptr(y)), self.matrix.ctx._h)
        return y

    def apply_hermitian(self, x: np.ndarray) -> np.ndarray:  # traits.rs:331-358 default: conj(A^T conj(x))
        return np.conj(self.apply_transpose(np.conj(x)))


@dataclass
class GmresConfig:
    """gmres.rs:16-36 (defaults of ``GmresConfig<f64>``)."""

    max_iterations: int = 100  # restart CYCLES
    restart: int = 30
    tolerance: float = 1e-6
    print_interval: int = 0

    @staticmethod
    def for_small_problems() -> "GmresConfig":  # gmres.rs:52-59
        return GmresConfig(max_iterations=50, restart=50, tolerance=1e-8)

    @staticmethod
    def with_restart(restart: int) -> "GmresConfig":  # gmres.rs:62-70
        return GmresConfig(restart=restart)


@dataclass
class GmresSolution:
    """gmres.rs:74-85."""

    x: np.ndarray
    iterations: int
    restarts: int
    residual: float
    converged: bool


def gmres_with_guess(operator: DenseOperator, b: np.ndarray, x0: Optional[np.ndarray], config: GmresConfig) -> GmresSolution:
    """gmres.rs:105-277 on the device."""
    b = np.ascontiguousarray(b, dtype=np.complex128)
    n = operator.num_rows()
    if b.shape != (n,):
        raise ValueError(f"gmres: b has shape {b.shape}, operator has {n} rows")
    x0a = None
    if x0 is not None:
        x0a = np.ascontiguousarray(x0, dtype=np.complex128)
        if x0a.shape != (n,):
            raise ValueError("gmres: x0 has the wrong length")
    x = np.empty(n, dtype=np.complex128)
    info = _capi.CGmresInfo()
    _capi.check(_capi.lib().bemb200_gmres(operator.matrix._h, _capi.ptr(b), _capi.ptr(x0a) if x0a is not None else None,
                                          config.max_iterations, config.restart, config.tolerance, _capi.ptr(x), C.byref(info)),
                operator.matrix.ctx._h)
    return GmresSolution(x=x, iterations=int(info.iterations), restarts=int(info.restarts), residual=float(info.residual),
                         converged=bool(info.converged))


def gmres_device(operator: DenseOperator, b_dev: int, x_dev: int, config: GmresConfig, x0_dev: int = 0) -> GmresSolution:
    """Same solve with DEVICE pointers (complex128 vectors of num_rows entries); ``x`` of the
    returned solution is None, the result is in ``x_dev``."""
    info = _capi.CGmresInfo()
    _capi.check(_capi.lib().bemb200_gmres_device(operator.matrix._h, C.c_void_p(b_dev), C.c_void_p(x0_dev or None),
                                                 config.max_iterations, config.restart, config.tolerance, C.c_void_p(x_dev),
                                                 C.byref(info)), operator.matrix.ctx._h)
    return GmresSolution(x=None, iterations=int(info.iterations), restarts=int(info.restarts), residual=float(info.residual),
                         converged=bool(info.converged))


def apply_device(operator: DenseOperator, x_dev: int, y_dev: int) -> None:
    _capi.check(_capi.lib().bemb200_apply_device(operator.matrix._h, C.c_void_p(x_dev), C.c_void_p(y_dev)), operator.matrix.ctx._h)


def incident_rhs_device(staged: StagedMesh, physics: PhysicsParams, beta: complex, incident, rhs_dev: int = 0,
                        fetch: bool = True) -> Optional[np.ndarray]:
    """IncidentField::compute_rhs_with_beta (incident.rs:317-342) on the device, at the staged
    mesh's collocation points (DOF order).  ``incident`` is a math_audio_b200.incident.IncidentField;
    ``rhs_dev``: optional device pointer receiving the vector (sweeps that never leave the GPU)."""
    kinds, vecs, amps = [], [], []
    for d, a in incident.plane_waves:
        kinds.append(0); vecs.append(np.asarray(d, dtype=np.float64)); amps.append(complex(a))
    for p, a in incident.point_sources:
        kinds.append(1); vecs.append(np.asarray(p, dtype=np.float64)); amps.append(complex(a))
    kinds_a = np.ascontiguousarray(kinds, dtype=np.int32)
    vecs_a = np.ascontiguousarray(np.stack(vecs), dtype=np.float64)
    amps_a = np.ascontiguousarray(amps, dtype=np.complex128)
    out = np.empty(staged.num_dofs, dtype=np.complex128) if fetch else None
    ph = _cphys(physics)
    beta = complex(beta)
    _capi.check(_capi.lib().bemb200_incident_rhs(staged._h, C.byref(ph), beta.real, beta.imag, len(kinds), _capi.ptr(kinds_a),
                                                 _capi.ptr(vecs_a), _capi.ptr(amps_a), _capi.ptr(out) if fetch else None,
                                                 C.c_void_p(rhs_dev or None)), staged.ctx._h)
    return out


def source_groups(incidents, max_groups: int = 4096) -> tuple:
    """``(src_ptr, kinds, vecs, amps)`` of a sequence of IncidentField objects, one group per field: its plane waves, then its
    point sources (the source order of ``incident_rhs_device``).  Raises ValueError for anything else."""
    if isinstance(incidents, (str, bytes)) or not hasattr(incidents, "__len__") or len(incidents) == 0:
        raise ValueError("incidents must be a non-empty sequence of IncidentField objects")
    src_ptr, kinds, vecs, amps = [0], [], [], []
    for f in incidents:
        if not (hasattr(f, "plane_waves") and hasattr(f, "point_sources")):
            raise ValueError(f"incidents must hold IncidentField objects, got {type(f).__name__}")
        for kind, group in ((0, f.plane_waves), (1, f.point_sources)):
            for v, a in group:
                v = np.asarray(v, dtype=np.float64)
                if v.shape != (3,):
                    raise ValueError("a source direction / position must have 3 components")
                kinds.append(kind); vecs.append(v); amps.append(complex(a))
        src_ptr.append(len(kinds))
    return check_source_groups(np.asarray(src_ptr, dtype=np.uint32), np.asarray(kinds, dtype=np.int32),
                               np.asarray(vecs, dtype=np.float64).reshape(-1, 3), np.asarray(amps, dtype=np.complex128),
                               max_groups)


def check_source_groups(src_ptr, kinds, vecs, amps, max_groups: int = 4096) -> tuple:
    """Validate the source groups of ``bemb200_incident_rhs_batch`` / ``bemb200_sweep_submit_incident`` before they reach the
    library: src_ptr[0] = 0, non-decreasing, at most ``max_groups`` groups and 65536 sources, kinds 0 / 1, vecs (ns, 3),
    amps (ns,).  Returns the contiguous arrays."""
    src_ptr = np.ascontiguousarray(src_ptr)
    if src_ptr.ndim != 1 or src_ptr.size < 2 or not np.issubdtype(src_ptr.dtype, np.integer):
        raise ValueError("src_ptr must be a 1-D integer array of nrhs + 1 entries")
    nrhs = src_ptr.size - 1
    if nrhs > max_groups:
        raise ValueError(f"at most {max_groups} right-hand sides per call")
    if src_ptr[0] != 0 or np.any(np.diff(src_ptr.astype(np.int64)) < 0):
        raise ValueError("src_ptr must start at 0 and be non-decreasing")
    ns = int(src_ptr[-1])
    if ns > 65536:
        raise ValueError("at most 65536 sources in all")
    kinds = np.ascontiguousarray(kinds, dtype=np.int32)
    vecs = np.ascontiguousarray(vecs, dtype=np.float64)
    amps = np.ascontiguousarray(amps, dtype=np.complex128)
    if kinds.shape != (ns,) or vecs.shape != (ns, 3) or amps.shape != (ns,):
        raise ValueError("kinds / vecs / amps must have src_ptr[-1] entries (vecs: 3 per source)")
    if np.any((kinds != 0) & (kinds != 1)):
        raise ValueError("source kind must be 0 (plane wave) or 1 (point source)")
    if ns == 0:  # the library takes no NULL arrays: one unused entry each
        kinds, vecs, amps = np.zeros(1, np.int32), np.zeros((1, 3)), np.zeros(1, np.complex128)
    return np.ascontiguousarray(src_ptr, dtype=np.uint32), kinds, vecs, amps


def _device_ptr(p, what: str) -> int:
    if isinstance(p, (bool, np.bool_)) or not isinstance(p, (int, np.integer)) or int(p) <= 0:
        raise ValueError(f"{what} must be a device pointer (a positive int)")
    return int(p)


def incident_rhs_batch(staged: StagedMesh, physics: PhysicsParams, beta: complex, incidents, system: Optional[TbemSystem] = None,
                       b_dev: int = 0, fetch: bool = True) -> Optional[np.ndarray]:
    """``incident_rhs_device`` for every IncidentField of ``incidents`` in one launch: row s of the (nrhs, n) result (DOF order)
    has the bits of ``incident_rhs_device(staged, physics, beta, incidents[s])``.  ``system``: add TbemSystem.rhs (b = rhs +
    incident, as the sweep forms it).  ``b_dev``: device pointer receiving the block; ``fetch=False`` returns None."""
    src_ptr, kinds, vecs, amps = source_groups(incidents)
    nrhs = src_ptr.size - 1
    if b_dev:
        b_dev = _device_ptr(b_dev, "b_dev")
    if not fetch and not b_dev:
        raise ValueError("fetch=False needs b_dev")
    if system is not None and not isinstance(system, TbemSystem):
        raise ValueError("system must be a TbemSystem")
    out = np.empty((nrhs, staged.num_dofs), dtype=np.complex128) if fetch else None
    ph = _cphys(physics)
    beta = complex(beta)
    _capi.check(_capi.lib().bemb200_incident_rhs_batch(staged._h, C.byref(ph), beta.real, beta.imag, nrhs, _capi.ptr(src_ptr),
                                                       _capi.ptr(kinds), _capi.ptr(vecs), _capi.ptr(amps),
                                                       system.matrix._h if system is not None else None,
                                                       _capi.ptr(out) if fetch else None, C.c_void_p(b_dev or None)), staged.ctx._h)
    return out


def _solutions_arg(values, staged: StagedMesh, nsol: Optional[int], what: str, allow_none: bool = False):
    """(pointer, on_device, nsol, keep-alive) of surface values given as an (nsol, n) host array (entry j of a row belongs to
    the j-th non-evaluation element, re-addressed to DOF order) or a device pointer to nsol DOF-ordered vectors."""
    if values is None:
        if allow_none:
            return None, nsol, None
        raise ValueError(f"{what} is required")
    if isinstance(values, (int, np.integer)) and not isinstance(values, (bool, np.bool_)):
        if nsol is None or not 1 <= int(nsol) <= 4096:
            raise ValueError(f"{what} as a device pointer needs nsol in 1..4096")
        return C.c_void_p(_device_ptr(values, what)), int(nsol), True
    a = np.ascontiguousarray(values, dtype=np.complex128)
    if a.ndim != 2 or a.shape[1] != staged.num_dofs or not 1 <= a.shape[0] <= 4096:
        raise ValueError(f"{what} must be an (nsol, num_dofs) array with 1 <= nsol <= 4096, got shape {a.shape}")
    if nsol is not None and int(nsol) != a.shape[0]:
        raise ValueError(f"nsol = {nsol} does not match {what} with {a.shape[0]} rows")
    if staged.enum_to_dof is not None:
        b = np.empty_like(a)
        b[:, staged.enum_to_dof] = a
        a = b
    return a, a.shape[0], False


def compute_rcs_batch(surface_pressure, staged: StagedMesh, directions, physics: PhysicsParams, nsol: Optional[int] = None) -> np.ndarray:
    """``compute_rcs`` of nsol solutions over the (M, 3) ``directions`` in one launch -> (nsol, M); row s has the bits of
    ``compute_rcs(surface_pressure[s], ...)``.  ``surface_pressure``: (nsol, n) host array in the order ``compute_rcs`` takes,
    or a device pointer (int) to nsol DOF-ordered vectors, as ``gmres_batched_device`` leaves them, with ``nsol``."""
    ps, nsol, on_dev = _solutions_arg(surface_pressure, staged, nsol, "surface_pressure")
    d = np.ascontiguousarray(directions, dtype=np.float64)
    if d.ndim != 2 or d.shape[1] != 3:
        raise ValueError("directions must be an (M, 3) array")
    out = np.empty((nsol, d.shape[0]), dtype=np.float64)
    ph = _cphys(physics)
    _capi.check(_capi.lib().bemb200_compute_rcs_batch(staged._h, C.byref(ph), nsol, ps if on_dev else _capi.ptr(ps), 1 if on_dev else 0,
                                                      d.shape[0], _capi.ptr(d), _capi.ptr(out)), staged.ctx._h)
    return out


def compute_scattered_field_batch(eval_points, staged: StagedMesh, surface_pressure, surface_velocity, physics: PhysicsParams,
                                  nsol: Optional[int] = None) -> np.ndarray:
    """``compute_scattered_field`` of nsol solutions at the (M, 3) ``eval_points`` in one launch -> (nsol, M) complex; row s has
    the bits of ``compute_scattered_field(eval_points, staged, surface_pressure[s], surface_velocity[s], physics)``.  Surface
    values: (nsol, n) host arrays as ``compute_scattered_field`` takes them, or device pointers (ints, DOF order) with ``nsol``;
    ``surface_velocity`` may be None, and is given the same way as ``surface_pressure``."""
    ps, nsol, on_dev = _solutions_arg(surface_pressure, staged, nsol, "surface_pressure")
    vs, _, v_dev = _solutions_arg(surface_velocity, staged, nsol, "surface_velocity", allow_none=True)
    if vs is not None and v_dev != on_dev:
        raise ValueError("surface_pressure and surface_velocity must both be host arrays or both device pointers")
    pts = np.ascontiguousarray(eval_points, dtype=np.float64)
    if pts.ndim != 2 or pts.shape[1] != 3:
        raise ValueError("eval_points must be an (M, 3) array")
    out = np.empty((nsol, pts.shape[0]), dtype=np.complex128)
    ph = _cphys(physics)
    vptr = None if vs is None else (vs if on_dev else _capi.ptr(vs))
    _capi.check(_capi.lib().bemb200_scattered_field_batch(staged._h, C.byref(ph), nsol, ps if on_dev else _capi.ptr(ps), vptr,
                                                          1 if on_dev else 0, pts.shape[0], _capi.ptr(pts), _capi.ptr(out)),
                staged.ctx._h)
    return out


def compute_scattered_field(eval_points: np.ndarray, staged: StagedMesh, surface_pressure: np.ndarray,
                            surface_velocity: Optional[np.ndarray], physics: PhysicsParams) -> np.ndarray:
    """postprocess/pressure.rs:81-137 on the device.  Surface values as the reference takes them: entry j belongs to the j-th
    non-evaluation element (re-addressed to the ABI's DOF order here when the mesh has a permuted DOF map)."""
    pts = np.ascontiguousarray(eval_points, dtype=np.float64).reshape(-1, 3)
    ps = np.ascontiguousarray(surface_pressure, dtype=np.complex128)
    if ps.shape != (staged.num_dofs,):
        raise ValueError("surface_pressure must have num_dofs entries")
    ps = surface_values_in_dof_order(staged.enum_to_dof, ps)
    vs = None
    if surface_velocity is not None:
        vs = np.ascontiguousarray(surface_velocity, dtype=np.complex128)
        if vs.shape != (staged.num_dofs,):
            raise ValueError("surface_velocity must have num_dofs entries")
        vs = surface_values_in_dof_order(staged.enum_to_dof, vs)
    out = np.empty(pts.shape[0], dtype=np.complex128)
    ph = _cphys(physics)
    _capi.check(_capi.lib().bemb200_scattered_field(staged._h, C.byref(ph), pts.shape[0], _capi.ptr(pts), _capi.ptr(ps),
                                                    _capi.ptr(vs) if vs is not None else None, _capi.ptr(out)), staged.ctx._h)
    return out


def compute_rcs(surface_pressure: np.ndarray, staged: StagedMesh, direction, physics: PhysicsParams):
    """postprocess/pressure.rs:438-478 on the device.  ``direction``: one unit vector (returns a float, as the
    reference) or an (M, 3) array (returns M values, one kernel launch).  The far-field integral has no surface-velocity
    term, so it is the RCS of a rigid body only: a solution with an admittance (``AssemblyOptions``) is not covered."""
    ps = np.ascontiguousarray(surface_pressure, dtype=np.complex128)
    if ps.shape != (staged.num_dofs,):
        raise ValueError("surface_pressure must have num_dofs entries")
    ps = surface_values_in_dof_order(staged.enum_to_dof, ps)  # entry j belongs to the j-th non-evaluation element (pressure.rs:452-458)
    d = np.ascontiguousarray(direction, dtype=np.float64)
    single = d.ndim == 1
    d = d.reshape(-1, 3)
    out = np.empty(d.shape[0], dtype=np.float64)
    ph = _cphys(physics)
    _capi.check(_capi.lib().bemb200_compute_rcs(staged._h, C.byref(ph), d.shape[0], _capi.ptr(d), _capi.ptr(ps), _capi.ptr(out)),
                staged.ctx._h)
    return float(out[0]) if single else out


def compute_far_field(directions, staged: StagedMesh, surface_pressure, surface_velocity, physics: PhysicsParams,
                      nsol: Optional[int] = None) -> np.ndarray:
    """Complex far-field amplitude F in the (M, 3) unit ``directions`` (DESIGN.md 4.9): p_scat(R d) = F(d) exp(i s k R) / R +
    O(1/R^2), s = harmonic_factor, from the representation ``compute_scattered_field`` evaluates, with the surface-velocity
    term and over the whole element (Quad4: its bilinear map).  ``surface_velocity`` is v = dp/dn (None: rigid, v = 0).

    Surface values as ``compute_scattered_field`` takes them: a 1-D ``surface_pressure`` (num_dofs,) returns (M,) complex; an
    (nsol, num_dofs) array, or a device pointer (int) to nsol DOF-ordered vectors with ``nsol``, returns (nsol, M), row s
    with the bits of the single call on solution s.  ``surface_velocity`` is given the same way, or None."""
    single = not isinstance(surface_pressure, (int, np.integer)) and np.ndim(surface_pressure) == 1
    if single:
        surface_pressure = np.reshape(surface_pressure, (1, -1))
        if surface_velocity is not None:
            if isinstance(surface_velocity, (int, np.integer)) or np.ndim(surface_velocity) != 1:
                raise ValueError("a 1-D surface_pressure needs a 1-D surface_velocity (or None)")
            surface_velocity = np.reshape(surface_velocity, (1, -1))
    ps, nsol, on_dev = _solutions_arg(surface_pressure, staged, nsol, "surface_pressure")
    vs, _, v_dev = _solutions_arg(surface_velocity, staged, nsol, "surface_velocity", allow_none=True)
    if vs is not None and v_dev != on_dev:
        raise ValueError("surface_pressure and surface_velocity must both be host arrays or both device pointers")
    d = np.ascontiguousarray(directions, dtype=np.float64)
    if d.ndim != 2 or d.shape[1] != 3 or d.shape[0] == 0:
        raise ValueError("directions must be an (M, 3) array with M >= 1")
    if not np.all(np.isfinite(d)) or np.any(np.abs(np.sqrt((d * d).sum(axis=1)) - 1.0) > 1e-9):
        raise ValueError("directions must be finite unit vectors (| |d| - 1 | <= 1e-9)")
    out = np.empty((nsol, d.shape[0]), dtype=np.complex128)
    ph = _cphys(physics)
    vptr = None if vs is None else (vs if on_dev else _capi.ptr(vs))
    _capi.check(_capi.lib().bemb200_far_field(staged._h, C.byref(ph), nsol, ps if on_dev else _capi.ptr(ps), vptr, 1 if on_dev else 0,
                                              d.shape[0], _capi.ptr(d), _capi.ptr(out)), staged.ctx._h)
    return out[0] if single else out


def evaluate_field(eval_points, staged: StagedMesh, surface_pressure, surface_velocity, physics: PhysicsParams,
                   nsol: Optional[int] = None) -> np.ndarray:
    """Accurate scattered (or radiated) pressure at the (M, 3) ``eval_points`` (DESIGN.md 4.10): the representation
    ``compute_scattered_field`` evaluates, over the whole element (Quad4: its bilinear map), with adaptive subdivision of
    the elements near a point, so it holds close to the surface.  ``compute_far_field`` is its R -> infinity limit.  A point
    on the surface (within about 2^-30 element sizes of it) is NaN for every solution.

    Surface values as ``compute_far_field`` takes them: a 1-D ``surface_pressure`` (num_dofs,) returns (M,) complex; an
    (nsol, num_dofs) array, or a device pointer (int) to nsol DOF-ordered vectors with ``nsol``, returns (nsol, M), row s
    with the bits of the single call on solution s.  ``surface_velocity`` (v = dp/dn) is given the same way, or None."""
    single = not isinstance(surface_pressure, (int, np.integer)) and np.ndim(surface_pressure) == 1
    if single:
        surface_pressure = np.reshape(surface_pressure, (1, -1))
        if surface_velocity is not None:
            if isinstance(surface_velocity, (int, np.integer)) or np.ndim(surface_velocity) != 1:
                raise ValueError("a 1-D surface_pressure needs a 1-D surface_velocity (or None)")
            surface_velocity = np.reshape(surface_velocity, (1, -1))
    ps, nsol, on_dev = _solutions_arg(surface_pressure, staged, nsol, "surface_pressure")
    vs, _, v_dev = _solutions_arg(surface_velocity, staged, nsol, "surface_velocity", allow_none=True)
    if vs is not None and v_dev != on_dev:
        raise ValueError("surface_pressure and surface_velocity must both be host arrays or both device pointers")
    pts = np.ascontiguousarray(eval_points, dtype=np.float64)
    if pts.ndim != 2 or pts.shape[1] != 3 or not 1 <= pts.shape[0] < 2 ** 31:
        raise ValueError("eval_points must be an (M, 3) array with 1 <= M < 2^31")
    if not np.all(np.isfinite(pts)):
        raise ValueError("eval_points must be finite")
    out = np.empty((nsol, pts.shape[0]), dtype=np.complex128)
    ph = _cphys(physics)
    vptr = None if vs is None else (vs if on_dev else _capi.ptr(vs))
    _capi.check(_capi.lib().bemb200_evaluate_field(staged._h, C.byref(ph), nsol, ps if on_dev else _capi.ptr(ps), vptr,
                                                   1 if on_dev else 0, pts.shape[0], _capi.ptr(pts), _capi.ptr(out)), staged.ctx._h)
    return out[0] if single else out


class IdentityPreconditioner:
    """traits.rs:377-385."""

    inv_diag = None

    def apply(self, r: np.ndarray) -> np.ndarray:
        return np.array(r, copy=True)


class DiagonalPreconditioner:
    """math-solvers/src/preconditioners/diagonal.rs:20-80 (Jacobi): M^-1 r = r_i / A_ii."""

    def __init__(self, inv_diag: np.ndarray):
        self.inv_diag = np.ascontiguousarray(inv_diag, dtype=np.complex128)

    @staticmethod
    def from_diagonal(diag: np.ndarray) -> "DiagonalPreconditioner":  # diagonal.rs:40-50
        d = np.asarray(diag, dtype=np.complex128)
        out = np.ones_like(d)
        ok = np.sqrt(d.real ** 2 + d.imag ** 2) > 1e-30
        ns = d.real[ok] ** 2 + d.imag[ok] ** 2
        out[ok] = d.real[ok] / ns - 1j * (d.imag[ok] / ns)  # ComplexField::inv (traits.rs:150-153)
        return DiagonalPreconditioner(out)

    @staticmethod
    def from_inverse_diagonal(inv_diag: np.ndarray) -> "DiagonalPreconditioner":  # diagonal.rs:53-55
        return DiagonalPreconditioner(inv_diag)

    @staticmethod
    def from_operator(operator: "DenseOperator") -> "DiagonalPreconditioner":
        """Jacobi preconditioner of a device-resident operator (diagonal fetched from the GPU)."""
        n = operator.num_rows()
        d = np.empty(n, dtype=np.complex128)
        _capi.check(_capi.lib().bemb200_matrix_diagonal(operator.matrix._h, _capi.ptr(d)), operator.matrix.ctx._h)
        return DiagonalPreconditioner.from_diagonal(d)

    def apply(self, r: np.ndarray) -> np.ndarray:
        return r * self.inv_diag


def schwarz_partition(n: int, num_subdomains: int) -> List[np.ndarray]:
    """The contiguous partition of AdditiveSchwarzPreconditioner::from_csr (schwarz.rs:67-83): ``n / S`` DOFs per
    subdomain, the first ``n % S`` one larger."""
    S = min(max(int(num_subdomains), 1), n)
    base, rem = divmod(n, S)
    out, start = [], 0
    for i in range(S):
        size = base + (1 if i < rem else 0)
        out.append(np.arange(start, start + size, dtype=np.uint64))
        start += size
    return out


def schwarz_partition_aligned(n: int, nranks: int, block_size: int) -> List[np.ndarray]:
    """Contiguous subdomains of about ``block_size`` DOFs that never straddle two ranks' row blocks (bemb200_partition):
    the reference's partition applied inside every rank's rows."""
    chunk = (n + nranks - 1) // nranks
    out = []
    for r in range(nranks):
        b, e = min(chunk * r, n), min(chunk * (r + 1), n)
        if e > b:
            S = max(1, int(round((e - b) / max(1, block_size))))
            out.extend(p + np.uint64(b) for p in schwarz_partition(e - b, S))
    return out


def spatial_subdomains(centers: np.ndarray, nranks: int, block_size: int) -> List[np.ndarray]:
    """Compact clusters of at most ``block_size`` DOFs inside every rank's row block: recursive bisection of the collocation
    points along the longest axis of their bounding box (median split).  The clusters play the role of SLFMM's leaf clusters
    (slfmm.rs:444-460 maps clusters to DOF lists; their self blocks are the near field block-Jacobi inverts); indices inside
    a cluster ascend, as in the reference's subdomains (schwarz.rs:199-202).  ``centers``: (n, 3) in DOF order."""
    centers = np.asarray(centers, dtype=np.float64)
    n = centers.shape[0]
    chunk = (n + nranks - 1) // nranks
    out: List[np.ndarray] = []

    def split(ids: np.ndarray) -> None:
        if len(ids) <= block_size:
            out.append(np.sort(ids).astype(np.uint64))
            return
        c = centers[ids]
        axis = int(np.argmax(c.max(axis=0) - c.min(axis=0)))
        order = ids[np.argsort(c[:, axis], kind="stable")]
        half = len(order) // 2
        split(order[:half])
        split(order[half:])

    for r in range(nranks):
        b, e = min(chunk * r, n), min(chunk * (r + 1), n)
        if e > b:
            split(np.arange(b, e, dtype=np.int64))
    return out


def voronoi_subdomains(centers: np.ndarray, nranks: int, block_size: int, iterations: int = 12) -> List[np.ndarray]:
    """Like ``spatial_subdomains`` but the bisection clusters are relaxed by Lloyd iterations (every DOF joins the nearest
    cluster centroid, centroids are recomputed): Voronoi patches of roughly ``block_size`` DOFs, as round as the mesh allows.
    Deterministic.  Cluster sizes vary; a cluster never leaves its rank's row block."""
    centers = np.asarray(centers, dtype=np.float64)
    n = centers.shape[0]
    chunk = (n + nranks - 1) // nranks
    out: List[np.ndarray] = []
    for r in range(nranks):
        b, e = min(chunk * r, n), min(chunk * (r + 1), n)
        if e <= b:
            continue
        c = centers[b:e]
        seeds = spatial_subdomains(c, 1, block_size)
        cent = np.array([c[s.astype(np.int64)].mean(axis=0) for s in seeds])
        label = np.zeros(e - b, dtype=np.int64)
        for _ in range(iterations):
            d2 = (c * c).sum(1)[:, None] - 2.0 * (c @ cent.T) + (cent * cent).sum(1)[None, :]
            label = np.argmin(d2, axis=1)
            for k in range(len(cent)):
                sel = label == k
                if sel.any():
                    cent[k] = c[sel].mean(axis=0)
        for k in range(len(cent)):
            ids = np.nonzero(label == k)[0]
            if len(ids):
                out.append((ids + b).astype(np.uint64))
    return out


def extend_partition(partition: Sequence[int], adjacency: Sequence[Sequence[int]], overlap: int, n: int) -> np.ndarray:
    """schwarz.rs:177-203: grow a subdomain by ``overlap`` layers of neighbours, result sorted ascending."""
    inside = np.zeros(n, dtype=bool)
    inside[np.asarray(partition, dtype=np.int64)] = True
    frontier = [int(i) for i in partition]
    for _ in range(overlap):
        new = []
        for i in frontier:
            for j in adjacency[i]:
                if not inside[j]:
                    inside[j] = True
                    new.append(int(j))
        frontier = new
    return np.nonzero(inside)[0].astype(np.uint64)


class AdditiveSchwarzPreconditioner:
    """math-solvers/src/preconditioners/schwarz.rs on the device: block-Jacobi (overlap 0) / additive Schwarz built from the
    assembled operator -- local solve = LU without pivoting of the dense diagonal block (ILU(0) of a full pattern)."""

    def __init__(self, operator: DenseOperator, handle):
        self.operator = operator
        self.ctx = operator.matrix.ctx
        self._h = handle
        self.inv_diag = None

    @staticmethod
    def from_operator(operator: DenseOperator, num_subdomains: int = 0, overlap: int = 0,
                      subdomains: Optional[Sequence[np.ndarray]] = None,
                      adjacency: Optional[Sequence[Sequence[int]]] = None) -> "AdditiveSchwarzPreconditioner":
        """``from_csr(matrix, num_subdomains, overlap)`` (schwarz.rs:66-125).  ``subdomains``: explicit index sets instead of
        the contiguous partition (e.g. spatial clusters, rank-aligned blocks).  ``overlap`` > 0 needs ``adjacency`` (the
        reference takes it from the sparsity pattern, schwarz.rs:161-174; a dense operator has none of its own)."""
        n = operator.num_rows()
        if overlap > 0:
            if adjacency is None:
                raise ValueError("overlap > 0 needs an adjacency (a dense operator couples every pair of DOFs)")
            base = subdomains if subdomains is not None else schwarz_partition(n, num_subdomains)
            subdomains = [extend_partition(p, adjacency, overlap, n) for p in base]
        h = C.c_void_p()
        m = operator.matrix
        if subdomains is None:
            _capi.check(_capi.lib().bemb200_schwarz_create(m._h, int(num_subdomains), None, None, C.byref(h)), m.ctx._h)
        else:
            ptr = np.zeros(len(subdomains) + 1, dtype=np.uint64)
            ptr[1:] = np.cumsum([len(p) for p in subdomains])
            idx = (np.concatenate([np.asarray(p, dtype=np.uint64) for p in subdomains]) if len(subdomains)
                   else np.zeros(0, dtype=np.uint64))
            idx = np.ascontiguousarray(idx)
            _capi.check(_capi.lib().bemb200_schwarz_create(m._h, len(subdomains), _capi.ptr(ptr), _capi.ptr(idx), C.byref(h)), m.ctx._h)
        return AdditiveSchwarzPreconditioner(operator, h)

    def apply(self, r: np.ndarray) -> np.ndarray:  # Preconditioner::apply (traits.rs:366-371)
        r = np.ascontiguousarray(r, dtype=np.complex128)
        if r.shape != (self.operator.num_rows(),):
            raise ValueError("preconditioner: wrong vector length")
        z = np.empty_like(r)
        _capi.check(_capi.lib().bemb200_precond_apply(self._h, _capi.ptr(r), _capi.ptr(z)), self.ctx._h)
        return z

    def stats(self) -> dict:  # schwarz.rs:135-158 (+ device figures)
        st = _capi.CPrecondStats()
        _capi.check(_capi.lib().bemb200_precond_stats_get(self._h, C.byref(st)), self.ctx._h)
        return {k: getattr(st, k) for k, _ in st._fields_}

    def close(self) -> None:
        if self._h:
            _capi.lib().bemb200_precond_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _gmres_user_preconditioner(operator: "DenseOperator", precond, b: np.ndarray, x0a: Optional[np.ndarray],
                               config: "GmresConfig") -> "GmresSolution":
    """bemb200_gmres_callback: the caller's ``precond.apply`` behind a C function pointer.  An exception raised by
    ``apply`` (or a result of the wrong shape) ends the solve (BEMB200_ECALLBACK) and is re-raised here."""
    n = operator.num_rows()
    failure = []

    def trampoline(_user, r_ptr, z_ptr, nn):
        try:
            r = np.ctypeslib.as_array(r_ptr, shape=(2 * nn,)).view(np.complex128)
            z = np.asarray(precond.apply(r.copy()), dtype=np.complex128)
            if z.shape != (nn,):
                raise ValueError(f"Preconditioner.apply returned shape {z.shape}, expected ({nn},)")
            np.ctypeslib.as_array(z_ptr, shape=(2 * nn,)).view(np.complex128)[:] = z
            return 0
        except BaseException as e:  # never let an exception cross the C frames
            failure.append(e)
            return 1

    cb = _capi.PRECOND_FN(trampoline)  # kept alive until the call has returned
    x = np.empty(n, dtype=np.complex128)
    info = _capi.CGmresInfo()
    calls = C.c_uint64(0)
    rc = _capi.lib().bemb200_gmres_callback(operator.matrix._h, cb, None, _capi.ptr(b), _capi.ptr(x0a) if x0a is not None else None,
                                            config.max_iterations, config.restart, config.tolerance, _capi.ptr(x), C.byref(info),
                                            C.byref(calls))
    if failure:
        raise failure[0]
    _capi.check(rc, operator.matrix.ctx._h)
    sol = GmresSolution(x=x, iterations=int(info.iterations), restarts=int(info.restarts), residual=float(info.residual),
                        converged=bool(info.converged))
    sol.preconditioner_calls = int(calls.value)
    return sol


def gmres_preconditioned_with_guess(operator: DenseOperator, precond, b: np.ndarray, x0: Optional[np.ndarray],
                                    config: GmresConfig) -> GmresSolution:
    """gmres.rs:434-585: left-preconditioned restarted GMRES on the device.  ``precond`` is an
    IdentityPreconditioner, a DiagonalPreconditioner or an AdditiveSchwarzPreconditioner (block-Jacobi) -- the
    preconditioners of the reference that apply to a dense operator without an O(N^3) factorisation, applied on the
    device -- or ANY other object with the trait's method ``apply(r) -> z`` (traits.rs:366-371), which is called on the
    host once per application while the Arnoldi process stays on the device (bemb200_gmres_callback)."""
    b = np.ascontiguousarray(b, dtype=np.complex128)
    n = operator.num_rows()
    if b.shape != (n,):
        raise ValueError(f"gmres: b has shape {b.shape}, operator has {n} rows")
    x0a = np.ascontiguousarray(x0, dtype=np.complex128) if x0 is not None else None
    if not isinstance(precond, (IdentityPreconditioner, DiagonalPreconditioner, AdditiveSchwarzPreconditioner)):
        if not callable(getattr(precond, "apply", None)):
            raise TypeError("precond must be one of the built-in preconditioners or implement apply(r) -> z (Preconditioner, traits.rs:366)")
        return _gmres_user_preconditioner(operator, precond, b, x0a, config)
    if isinstance(precond, AdditiveSchwarzPreconditioner):
        x = np.empty(n, dtype=np.complex128)
        info = _capi.CGmresInfo()
        _capi.check(_capi.lib().bemb200_gmres_schwarz(operator.matrix._h, precond._h, _capi.ptr(b),
                                                      _capi.ptr(x0a) if x0a is not None else None, config.max_iterations,
                                                      config.restart, config.tolerance, _capi.ptr(x), C.byref(info)),
                    operator.matrix.ctx._h)
        return GmresSolution(x=x, iterations=int(info.iterations), restarts=int(info.restarts), residual=float(info.residual),
                             converged=bool(info.converged))
    idg = precond.inv_diag
    if idg is not None and idg.shape != (n,):
        raise ValueError("preconditioner has the wrong length")
    x = np.empty(n, dtype=np.complex128)
    info = _capi.CGmresInfo()
    _capi.check(_capi.lib().bemb200_gmres_preconditioned(operator.matrix._h, _capi.ptr(idg) if idg is not None else None,
                                                         _capi.ptr(b), _capi.ptr(x0a) if x0a is not None else None,
                                                         config.max_iterations, config.restart, config.tolerance, _capi.ptr(x),
                                                         C.byref(info)), operator.matrix.ctx._h)
    return GmresSolution(x=x, iterations=int(info.iterations), restarts=int(info.restarts), residual=float(info.residual),
                         converged=bool(info.converged))


def gmres_preconditioned(operator: DenseOperator, precond, b: np.ndarray, config: GmresConfig) -> GmresSolution:  # gmres.rs:282
    return gmres_preconditioned_with_guess(operator, precond, b, None, config)


def gmres(operator: DenseOperator, b: np.ndarray, config: GmresConfig) -> GmresSolution:  # gmres.rs:96-102
    return gmres_with_guess(operator, b, None, config)


@dataclass
class BiCgstabConfig:
    """math-solvers/src/iterative/bicgstab.rs:19-37."""

    max_iterations: int = 1000
    tolerance: float = 1e-6
    print_interval: int = 0


@dataclass
class BiCgstabSolution:
    """bicgstab.rs:40-50."""

    x: np.ndarray
    iterations: int
    residual: float
    converged: bool


def bicgstab(operator: DenseOperator, b: np.ndarray, config: BiCgstabConfig) -> BiCgstabSolution:
    """bicgstab.rs:46-187 on the device (x0 = 0; two ZGEMVs per iteration, fused vector kernels)."""
    b = np.ascontiguousarray(b, dtype=np.complex128)
    if b.shape != (operator.num_rows(),):
        raise ValueError("b does not match the operator")
    x = np.empty_like(b)
    info = _capi.CGmresInfo()
    _capi.check(_capi.lib().bemb200_bicgstab(operator.matrix._h, _capi.ptr(b), int(config.max_iterations), float(config.tolerance),
                                             _capi.ptr(x), C.byref(info)), operator.matrix.ctx._h)
    return BiCgstabSolution(x, int(info.iterations), float(info.residual), bool(info.converged))


@dataclass
class CgsConfig:
    """math-solvers/src/iterative/cgs.rs:12-30."""

    max_iterations: int = 1000
    tolerance: float = 1e-6
    print_interval: int = 0


@dataclass
class CgsSolution:
    """cgs.rs:33-43."""

    x: np.ndarray
    iterations: int
    residual: float
    converged: bool


def cgs(operator: DenseOperator, b: np.ndarray, config: CgsConfig) -> CgsSolution:
    """cgs.rs:46-155 on the device (x0 = 0; two ZGEMVs per iteration, fused vector kernels)."""
    b = np.ascontiguousarray(b, dtype=np.complex128)
    if b.shape != (operator.num_rows(),):
        raise ValueError("b does not match the operator")
    x = np.empty_like(b)
    info = _capi.CGmresInfo()
    _capi.check(_capi.lib().bemb200_cgs(operator.matrix._h, _capi.ptr(b), int(config.max_iterations), float(config.tolerance),
                                        _capi.ptr(x), C.byref(info)), operator.matrix.ctx._h)
    return CgsSolution(x, int(info.iterations), float(info.residual), bool(info.converged))


class LuError(RuntimeError):
    """math-solvers/src/direct/lu.rs:15-21."""


def lu_solve(a, b: np.ndarray, ctx: Optional[Context] = None, overwrite: bool = False, stats: Optional[dict] = None) -> np.ndarray:
    """lu.rs:139-161 (LAPACK zgesv in the reference's native build) through cuSOLVER on the device.
    ``a``: host matrix, DeviceMatrix, TbemSystem or DenseOperator.  Raises LuError for a singular matrix /
    dimension mismatch."""
    if isinstance(a, DenseOperator):
        mat = a.matrix
    elif isinstance(a, TbemSystem):
        mat = a.matrix
    elif isinstance(a, DeviceMatrix):
        mat = a
    else:
        arr = np.asarray(a)
        if arr.ndim != 2 or arr.shape[0] != arr.shape[1]:
            raise LuError(f"Matrix dimensions mismatch: expected {arr.shape[0]}, got {arr.shape[-1]}")
        mat = DenseOperator(arr, ctx).matrix
        overwrite = True  # private copy
    b = np.ascontiguousarray(b, dtype=np.complex128)
    if b.shape != (mat.shape[0],):
        raise LuError(f"Matrix dimensions mismatch: expected {mat.shape[0]}, got {b.shape[0]}")
    x = np.empty_like(b)
    ms = C.c_double(0.0)
    try:
        _capi.check(_capi.lib().bemb200_lu_solve(mat._h, _capi.ptr(b), _capi.ptr(x), 1 if overwrite else 0, C.byref(ms)), mat.ctx._h)
    except _capi.Bemb200Error as e:
        if e.code == -7:
            raise LuError("Matrix is singular or nearly singular") from e
        raise
    if stats is not None:
        stats["factor_ms"] = ms.value
    return x


def gmres_batched(operator: DenseOperator, b_all: np.ndarray, config: GmresConfig, precond: "Optional[AdditiveSchwarzPreconditioner]" = None):
    """``[gmres(operator, b, config) for b in b_all]`` (the reference's way to solve several
    right-hand sides) executed in lockstep on the device with one tensor-core block matvec per
    iteration.  ``b_all``: (nrhs, n).  Returns (list of GmresSolution, stats dict).  ``precond``: a block-Jacobi
    AdditiveSchwarzPreconditioner -> ``[gmres_preconditioned(operator, precond, b, config) for b in b_all]``."""
    b_all = np.ascontiguousarray(b_all, dtype=np.complex128)
    n = operator.num_rows()
    if b_all.ndim != 2 or b_all.shape[1] != n:
        raise ValueError(f"gmres_batched: b_all has shape {b_all.shape}, expected (nrhs, {n})")
    nrhs = b_all.shape[0]
    x_all = np.empty_like(b_all)
    infos = (_capi.CGmresInfo * nrhs)()
    ms, cnt = C.c_double(), C.c_uint64()
    if precond is None:
        _capi.check(_capi.lib().bemb200_gmres_batched(operator.matrix._h, _capi.ptr(b_all), nrhs, config.max_iterations, config.restart,
                                                      config.tolerance, _capi.ptr(x_all), infos, C.byref(ms), C.byref(cnt)),
                    operator.matrix.ctx._h)
    else:
        _capi.check(_capi.lib().bemb200_gmres_batched_schwarz(operator.matrix._h, precond._h, _capi.ptr(b_all), nrhs, config.max_iterations,
                                                              config.restart, config.tolerance, _capi.ptr(x_all), infos, C.byref(ms),
                                                              C.byref(cnt)), operator.matrix.ctx._h)
    sols = [GmresSolution(x=x_all[i], iterations=int(infos[i].iterations), restarts=int(infos[i].restarts),
                          residual=float(infos[i].residual), converged=bool(infos[i].converged)) for i in range(nrhs)]
    return sols, dict(block_matvec_ms=float(ms.value), block_matvecs=int(cnt.value))


def gmres_batched_device(operator: DenseOperator, b_dev: int, nrhs: int, config: GmresConfig, x_dev: int,
                         precond: "Optional[AdditiveSchwarzPreconditioner]" = None):
    """``gmres_batched`` on DEVICE vectors: ``b_dev`` / ``x_dev`` point to nrhs (1..32) vectors of num_rows complex128, each
    contiguous, on the operator's device.  Same solutions and infos as ``gmres_batched`` on the same B; returns
    (list of GmresSolution with x=None, stats dict)."""
    b_dev, x_dev = _device_ptr(b_dev, "b_dev"), _device_ptr(x_dev, "x_dev")
    if isinstance(nrhs, (bool, np.bool_)) or not isinstance(nrhs, (int, np.integer)) or not 1 <= int(nrhs) <= 32:
        raise ValueError("nrhs must be an int in 1..32")
    if precond is not None and not isinstance(precond, AdditiveSchwarzPreconditioner):
        raise ValueError("precond must be a block-Jacobi AdditiveSchwarzPreconditioner or None")
    nrhs = int(nrhs)
    infos = (_capi.CGmresInfo * nrhs)()
    ms, cnt = C.c_double(), C.c_uint64()
    _capi.check(_capi.lib().bemb200_gmres_batched_device(operator.matrix._h, precond._h if precond is not None else None,
                                                         C.c_void_p(b_dev), nrhs, config.max_iterations, config.restart,
                                                         config.tolerance, C.c_void_p(x_dev), infos, C.byref(ms), C.byref(cnt)),
                operator.matrix.ctx._h)
    sols = [GmresSolution(x=None, iterations=int(infos[i].iterations), restarts=int(infos[i].restarts),
                          residual=float(infos[i].residual), converged=bool(infos[i].converged)) for i in range(nrhs)]
    return sols, dict(block_matvec_ms=float(ms.value), block_matvecs=int(cnt.value))


def apply_block(operator: DenseOperator, x_all: np.ndarray):
    """A @ x for nrhs vectors at once (tensor-core block matvec) -> (y_all, kernel_ms)."""
    x_all = np.ascontiguousarray(x_all, dtype=np.complex128)
    if x_all.ndim != 2 or x_all.shape[1] != operator.num_cols():
        raise ValueError("apply_block: x_all must be (nrhs, num_cols)")
    y_all = np.empty((x_all.shape[0], operator.num_rows()), dtype=np.complex128)
    ms = C.c_double()
    _capi.check(_capi.lib().bemb200_apply_block(operator.matrix._h, _capi.ptr(x_all), x_all.shape[0], _capi.ptr(y_all), C.byref(ms)),
                operator.matrix.ctx._h)
    return y_all, float(ms.value)


def solve_gmres(operator: DenseOperator, b: np.ndarray, config: GmresConfig) -> GmresSolution:  # fmm_interface.rs:378-384
    return gmres(operator, b, config)


def solve_cgs(operator: DenseOperator, b: np.ndarray, config: CgsConfig) -> CgsSolution:  # fmm_interface.rs:360-366
    return cgs(operator, b, config)


def solve_bicgstab(operator: DenseOperator, b: np.ndarray, config: BiCgstabConfig) -> BiCgstabSolution:  # fmm_interface.rs:369-375
    return bicgstab(operator, b, config)


def solve_with_ilu(matrix, b: np.ndarray, config: CgsConfig, ctx: Optional[Context] = None) -> CgsSolution:
    """fmm_interface.rs:389-417: despite its name the reference builds an ILU factorisation it never
    uses and runs **unpreconditioned** CGS on the dense matrix (it prints a warning saying so).  The
    result is therefore that of `cgs`; the unused factorisation is not reproduced.  ``matrix``: a
    DenseOperator / TbemSystem (device resident) or a host array (uploaded, as `DenseOperator::new`)."""
    op = matrix if isinstance(matrix, DenseOperator) else DenseOperator(matrix, ctx=ctx)
    return cgs(op, b, config)


def solve_tbem_with_ilu(matrix, b: np.ndarray, config: CgsConfig, ctx: Optional[Context] = None) -> CgsSolution:  # fmm_interface.rs:441-447
    return solve_with_ilu(matrix, b, config, ctx=ctx)


# ---- mesh sizing helpers of the same module (fmm_interface.rs:543-602): host scalars --------------------------------
def recommended_mesh_resolution(frequency: float, speed_of_sound: float, elements_per_wavelength: int) -> float:
    """fmm_interface.rs:544-551: elements per metre for `elements_per_wavelength` elements per wavelength."""
    wavelength = speed_of_sound / frequency
    return float(elements_per_wavelength) / wavelength


def mesh_resolution_for_frequency_range(min_freq: float, max_freq: float, speed_of_sound: float, elements_per_wavelength: int) -> float:
    """fmm_interface.rs:554-561: the highest frequency decides (min_freq is unused, as in the reference)."""
    return recommended_mesh_resolution(max_freq, speed_of_sound, elements_per_wavelength)


def estimate_element_count(room_dimensions, mesh_resolution: float) -> int:
    """fmm_interface.rs:564-570: ceil(surface area of the box / element area)."""
    w, d, h = room_dimensions
    surface_area = 2.0 * (w * d + w * h + d * h)
    element_size = 1.0 / mesh_resolution
    return int(np.ceil(surface_area / (element_size * element_size)))


@dataclass
class AdaptiveMeshConfig:
    """fmm_interface.rs:573-602."""

    base_resolution: float
    source_refinement: float
    source_refinement_radius: float

    @staticmethod
    def for_frequency_range(min_freq: float, max_freq: float) -> "AdaptiveMeshConfig":
        return AdaptiveMeshConfig(mesh_resolution_for_frequency_range(min_freq, max_freq, 343.0, 6), 1.5, 0.5)

    @staticmethod
    def from_resolution(resolution: float) -> "AdaptiveMeshConfig":
        return AdaptiveMeshConfig(resolution, 1.0, 0.0)
