"""Frequency-sweep driver: the mesh stays staged on the device and the assembly of frequency
f+1 (FP64-bound) overlaps the GMRES solve of frequency f (HBM-bound) on a second stream with a
second matrix buffer.  SURVEY.md section 8f rank 2; the reference re-runs everything per
frequency (`bem_solver.rs:273-322`, examples/audio_frequency_sweep.rs).

Every frequency still goes through exactly `build_tbem_system_with_beta` + `gmres`; only the
schedule changes.
"""
from __future__ import annotations

import os
import threading
import time
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from . import bem
from .mesh import Mesh
from .types import PhysicsParams


class Sweep:
    """The pipelined frequency sweep behind the C ABI (`bemb200_sweep_*`, csrc/sweep.cu): what a Rust / C caller uses.
    Host buffers in, host buffers out; the schedule (assembly of frequency f + 1 underneath the solve of f, helper
    launch when the solve ends first) lives in the library.

        sw = Sweep(mesh)
        for ph, beta, rhs in cases[:2]: sw.submit(ph, beta, rhs, cfg)      # keep two frequencies in flight
        for i in range(len(cases)):
            sol, stats, b = sw.next()
            if i + 2 < len(cases): sw.submit(*cases[i + 2], cfg)
    """

    def __init__(self, mesh: Mesh, device: int = 0, rank: int = 0, nranks: int = 1, nccl_id: Optional[bytes] = None,
                 overlap: bool = True, background_blocks_per_sm: int = 2):
        import ctypes as C

        from . import _capi

        self._capi, self._C = _capi, C
        self._lib = _capi.lib()
        self._h = C.c_void_p()
        cm = _capi.cmesh(mesh)
        idbuf = (C.c_uint8 * 128).from_buffer_copy(nccl_id) if nccl_id else None
        _capi.check(self._lib.bemb200_sweep_create(device, rank, nranks, idbuf, C.byref(cm), 1 if overlap else 0,
                                                   background_blocks_per_sm, C.byref(self._h)), None)
        self.n = int(self._lib.bemb200_sweep_num_dofs(self._h))
        self._enum_to_dof = bem.enumeration_to_dof(mesh)
        self._bc_type = bem.surface_values_in_dof_order(self._enum_to_dof, np.asarray(mesh.bc_type, dtype=np.int32)[np.asarray(mesh.is_eval) == 0])
        self.mesh_nbytes = _capi.mesh_nbytes(mesh)

    def submit(self, physics: PhysicsParams, beta: complex, rhs_extra: Optional[np.ndarray], config: "bem.GmresConfig") -> None:
        ph = bem._cphys(physics)
        beta = complex(beta)
        extra = None
        if rhs_extra is not None:
            extra = np.ascontiguousarray(rhs_extra, dtype=np.complex128)
            if extra.shape != (self.n,):
                raise ValueError("rhs_extra has the wrong length")
        self._capi.check(self._lib.bemb200_sweep_submit(self._h, self._C.byref(ph), beta.real, beta.imag,
                                                        self._capi.ptr(extra) if extra is not None else None,
                                                        config.max_iterations, config.restart, config.tolerance), None)

    def next(self):
        x = np.empty(self.n, dtype=np.complex128)
        b = np.empty(self.n, dtype=np.complex128)
        info = self._capi.CGmresInfo()
        st = self._capi.CAssemblyStats()
        self._capi.check(self._lib.bemb200_sweep_next(self._h, self._capi.ptr(x), self._C.byref(info), self._C.byref(st),
                                                      self._capi.ptr(b)), None)
        sol = bem.GmresSolution(x=x, iterations=int(info.iterations), restarts=int(info.restarts), residual=float(info.residual),
                                converged=bool(info.converged))
        return sol, {k: getattr(st, k) for k, _ in st._fields_}, b

    def submit_incident(self, physics: PhysicsParams, beta: complex, incidents, config: "bem.GmresConfig") -> None:
        """Queue a frequency with one right-hand side per IncidentField of ``incidents`` (1..32): b = TbemSystem.rhs +
        incident, built on the device right after the frequency's assembly.  ``next_batch`` returns its solutions."""
        src_ptr, kinds, vecs, amps = bem.source_groups(incidents, max_groups=32)
        ph = bem._cphys(physics)
        beta = complex(beta)
        self._capi.check(self._lib.bemb200_sweep_submit_incident(self._h, self._C.byref(ph), beta.real, beta.imag, src_ptr.size - 1,
                                                                 self._capi.ptr(src_ptr), self._capi.ptr(kinds), self._capi.ptr(vecs),
                                                                 self._capi.ptr(amps), config.max_iterations, config.restart,
                                                                 config.tolerance), None)

    def next_batch(self, capacity: int = 32):
        """The oldest queued frequency, submitted by ``submit`` (one solution) or ``submit_incident``: (list of GmresSolution,
        assembly stats).  A frequency with more than ``capacity`` right-hand sides raises and stays queued."""
        if isinstance(capacity, bool) or not isinstance(capacity, (int, np.integer)) or capacity < 1:
            raise ValueError("capacity must be a positive int")
        capacity = int(capacity)
        x = np.empty((capacity, self.n), dtype=np.complex128)
        infos = (self._capi.CGmresInfo * capacity)()
        got = self._C.c_uint32(0)
        st = self._capi.CAssemblyStats()
        self._capi.check(self._lib.bemb200_sweep_next_batch(self._h, capacity, self._capi.ptr(x), infos, self._C.byref(got),
                                                            self._C.byref(st)), None)
        sols = [bem.GmresSolution(x=x[i], iterations=int(infos[i].iterations), restarts=int(infos[i].restarts),
                                  residual=float(infos[i].residual), converged=bool(infos[i].converged)) for i in range(got.value)]
        return sols, {k: getattr(st, k) for k, _ in st._fields_}

    def solve_all(self, cases, config: "bem.GmresConfig") -> list:
        """cases: sequence of (physics, beta, rhs_extra); two frequencies are kept in flight."""
        out = []
        for c in cases[:2]:
            self.submit(c[0], c[1], c[2], config)
        for i in range(len(cases)):
            out.append(self.next())
            if i + 2 < len(cases):
                c = cases[i + 2]
                self.submit(c[0], c[1], c[2], config)
        return out

    def set_block_jacobi(self, num_subdomains: int = 0, subdomains=None) -> None:
        """Solve the frequencies returned from now on with gmres_preconditioned + the block-Jacobi / additive Schwarz
        preconditioner (schwarz.rs) rebuilt from every frequency's matrix: ``num_subdomains`` contiguous blocks, or explicit
        ``subdomains`` (index arrays, e.g. ``bem.voronoi_subdomains``); ``set_block_jacobi(0)`` switches back to plain gmres."""
        if subdomains is None:
            self._capi.check(self._lib.bemb200_sweep_set_block_jacobi(self._h, int(num_subdomains), None, None), None)
            return
        ptr = np.zeros(len(subdomains) + 1, dtype=np.uint64)
        ptr[1:] = np.cumsum([len(p) for p in subdomains])
        idx = np.ascontiguousarray(np.concatenate([np.asarray(p, dtype=np.uint64) for p in subdomains]))
        self._capi.check(self._lib.bemb200_sweep_set_block_jacobi(self._h, len(subdomains), self._capi.ptr(ptr), self._capi.ptr(idx)), None)

    def set_assembly_options(self, options: "Optional[bem.AssemblyOptions]") -> None:
        """Assemble every frequency submitted from now on with ``options`` (``bem.AssemblyOptions``; None restores the
        reference's assembly).  The admittance is copied now, so call this before each submit to give every frequency its
        own Y(f)."""
        if options is None:
            self._capi.check(self._lib.bemb200_sweep_set_assembly_options(self._h, None), None)
            return
        copts, _y = options.to_c(self._bc_type, self._enum_to_dof)
        self._capi.check(self._lib.bemb200_sweep_set_assembly_options(self._h, self._C.byref(copts)), None)

    @property
    def boosts(self) -> int:
        return int(self._lib.bemb200_sweep_boosts(self._h))

    def close(self):
        if self._h:
            self._lib.bemb200_sweep_destroy(self._h)
            self._h = self._C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SweepDriver:
    """The same schedule driven from Python with DEVICE pointers handed to a user callback -- kept for the benchmark's
    device-resident leg (`value`), which must not touch host buffers; everything else uses `Sweep`."""

    def __init__(self, mesh: Mesh, device: int = 0, rank: int = 0, nranks: int = 1, nccl_id: Optional[bytes] = None,
                 solve_stream: int = 0, assembly_stream: int = 0, overlap: bool = True, background_blocks_per_sm: int = 2):
        # the solve context owns the communicator; the assembly context needs none
        self.ctx_solve = bem.Context(device, rank, nranks, nccl_id, cuda_stream=solve_stream)
        self.ctx_asm = bem.Context(device, rank, nranks, None, cuda_stream=assembly_stream) if overlap else self.ctx_solve
        self.overlap = overlap
        self.background_blocks_per_sm = background_blocks_per_sm if overlap else 0
        self.mesh = mesh
        self.staged = bem.StagedMesh(mesh, self.ctx_asm)
        self.n = self.staged.num_dofs
        self.rows = self.ctx_solve.partition(self.n)
        self.buffers: List[Optional[bem.TbemSystem]] = [None, None]
        self.asm_stats: List[dict] = []
        self.sol_stats: List[dict] = []
        self.boosts = 0
        # join a still-running background assembly with full-speed blocks once the solve of the current frequency is done
        self.boost = os.environ.get("BEMB200_SWEEP_BOOST", "1") != "0"
        # BEMB200_SWEEP_TRACE=1: (label, case, seconds since run() started) of every phase boundary, both threads
        self.trace: Optional[list] = [] if os.environ.get("BEMB200_SWEEP_TRACE") else None
        self._t0 = 0.0

    def _mark(self, label: str, i: int) -> None:
        if self.trace is not None:
            self.trace.append((label, i, time.perf_counter() - self._t0))

    def _assemble(self, slot: int, physics: PhysicsParams, beta: complex, mesh_for_stage: Optional[Mesh], err: list, case: int = -1):
        try:
            self._mark("asm_begin", case)
            staged = self.staged if mesh_for_stage is None else bem.StagedMesh(mesh_for_stage, self.ctx_asm)
            self._mark("asm_staged", case)
            first = self.buffers[slot] is None
            self.buffers[slot] = bem.build_tbem_system_with_beta(staged, physics, beta, ctx=self.ctx_asm, rows=self.rows,
                                                                reuse=self.buffers[slot], fetch_rhs=False)
            if first and self.overlap:
                self.buffers[slot].matrix.set_context(self.ctx_solve)
            self._mark("asm_end", case)
        except Exception as e:  # surfaced in the caller thread
            err.append(e)

    def run(self, cases: Sequence[Tuple[PhysicsParams, complex]], config: bem.GmresConfig,
            solve: Callable[[int, bem.TbemSystem, bem.DenseOperator], object], restage_host_mesh: bool = False) -> list:
        """For every (physics, beta) in `cases`: assemble, then call ``solve(i, system, operator)``
        (which builds its right-hand side and calls gmres / gmres_device) -- assembly of case i+1
        runs while case i is being solved.  ``restage_host_mesh``: re-upload the host mesh for every
        frequency (what a caller without a staged mesh pays; used by the end-to-end benchmark)."""
        out = []
        err: list = []
        mesh_arg = self.mesh if restage_host_mesh else None
        if not cases:
            return out
        self._t0 = time.perf_counter()
        self.ctx_asm.set_background(0)  # nothing to hide behind yet: full-speed assembly
        self._assemble(0, cases[0][0], cases[0][1], mesh_arg, err, 0)
        if err:
            raise err[0]
        self.ctx_asm.set_background(self.background_blocks_per_sm)
        self.ctx_solve.set_shared_gpu(self.overlap)  # assembly kernels run beside the solve from here on
        try:
            for i in range(len(cases)):
                t = None
                if i + 1 < len(cases):
                    if self.overlap:
                        t = threading.Thread(target=self._assemble, args=((i + 1) % 2, cases[i + 1][0], cases[i + 1][1], mesh_arg, err, i + 1))
                        t.start()
                elif self.overlap:
                    self.ctx_solve.set_shared_gpu(False)  # last case: nothing left to assemble beside this solve
                system = self.buffers[i % 2]
                self.asm_stats.append(system.matrix.assembly_stats())
                op = bem.DenseOperator(system)
                self._mark("solve_begin", i)
                out.append(solve(i, system, op))
                self._mark("solve_end", i)
                self.sol_stats.append(system.matrix.solver_stats())
                if t is not None:
                    nxt = self.buffers[(i + 1) % 2]
                    if self.boost and nxt is not None and t.is_alive():
                        nxt.matrix.boost_assembly(self.ctx_solve)  # the solver has left the GPU: finish the assembly at full speed
                        self.boosts += 1
                    t.join()
                    self._mark("joined", i)
                elif i + 1 < len(cases):
                    self._assemble((i + 1) % 2, cases[i + 1][0], cases[i + 1][1], mesh_arg, err, i + 1)
                if err:
                    raise err[0]
        finally:
            self.ctx_solve.set_shared_gpu(False)  # the solver owns the GPU again
        return out
