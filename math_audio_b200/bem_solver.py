"""High-level caller of the hot path -- mirror of ``math-bem/src/core/bem_solver.rs``:

* ``SolverMethod`` :51-60, ``AssemblyMethod`` :63-72, ``BoundaryConditionType`` :75-83
* ``BemProblem`` :86-199 (``rigid_sphere_scattering`` :107-139, ``_custom`` :141-161, builders, ``ka``)
* ``BemSolver`` :202-497 (``solve`` :273-317: prepare_elements -> assemble_system (TBEM, beta =
  ``burton_miller_beta_scaled(beta_scale)``) -> add_incident_field_rhs -> solve_dense_system
  (``Direct`` = lu_solve, ``Cgs`` / ``BiCgStab`` = bicgstab on ``DenseMatrixOperator``))
* ``BemSolution`` :500-563, ``BemError`` :567-589

Every stage runs on the device through the C ABI (assembly kernels, cuSOLVER LU or the device
BiCGSTAB, field evaluation).  The FMM assembly methods are out of this repository's scope and
raise ``BemError`` ("NotImplemented"), as ``Mlfmm`` does in the reference.
"""
from __future__ import annotations

import enum
import math
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from . import bem
from .incident import IncidentField
from .postprocess import FieldPoint, compute_far_field, compute_total_field, surface_power
from .mesh import BC_PRESSURE, BC_VELOCITY, Mesh, generate_icosphere_mesh, generate_sphere_mesh
from .types import PhysicsParams


class SolverMethod(enum.Enum):
    Direct = "direct"
    Cgs = "cgs"
    BiCgStab = "bicgstab"


class AssemblyMethod(enum.Enum):
    Tbem = "tbem"
    Slfmm = "slfmm"
    Mlfmm = "mlfmm"


class BoundaryConditionType(enum.Enum):
    Rigid = "rigid"
    Soft = "soft"
    Impedance = "impedance"


class BemError(RuntimeError):
    """bem_solver.rs:567-589 (InvalidMesh / AssemblyFailed / SolverFailed / NotImplemented)."""


@dataclass
class BemProblem:
    mesh: Mesh
    physics: PhysicsParams
    incident_field: IncidentField
    bc_type: BoundaryConditionType = BoundaryConditionType.Rigid
    use_burton_miller: bool = True
    admittance: Optional[np.ndarray] = None  # Y per element (or one for all), see with_admittance
    surface_velocity: Optional[np.ndarray] = None  # prescribed dp/dn per element (or one for all), see with_surface_velocity

    @staticmethod
    def rigid_sphere_scattering(radius: float, frequency: float, speed_of_sound: float, density: float) -> "BemProblem":
        k = 2.0 * math.pi * frequency / speed_of_sound
        ka = k * radius
        subdivisions = 2 if ka < 1.0 else (3 if ka < 5.0 else 4)  # bem_solver.rs:117-125
        return BemProblem(generate_icosphere_mesh(radius, subdivisions), PhysicsParams.new(frequency, speed_of_sound, density, False),
                          IncidentField.plane_wave_z())

    @staticmethod
    def rigid_sphere_scattering_custom(radius: float, frequency: float, speed_of_sound: float, density: float, n_theta: int,
                                       n_phi: int) -> "BemProblem":
        return BemProblem(generate_sphere_mesh(radius, n_theta, n_phi), PhysicsParams.new(frequency, speed_of_sound, density, False),
                          IncidentField.plane_wave_z())

    def with_incident_field(self, incident: IncidentField) -> "BemProblem":
        self.incident_field = incident
        return self

    def with_boundary_condition(self, bc_type: BoundaryConditionType) -> "BemProblem":
        self.bc_type = bc_type
        return self

    def with_admittance(self, admittance) -> "BemProblem":
        """An absorbing surface: v = Y p on every element (v = dp/dn, outward normal), ``admittance`` one complex Y in 1/m
        for all elements or one per element.  Passive surfaces have Im Y <= 0.  Only this builder makes a surface
        absorbing; ``BoundaryConditionType.Impedance`` still solves a rigid body, as the reference does.  Above ka = 0.5
        pair it with ``BemSolver.with_sign_consistent_formulation(True)``: the reference's formulation does not converge
        to the physical solution there (DESIGN.md 4.8)."""
        self.admittance = admittance
        return self

    def with_surface_velocity(self, v_bar) -> "BemProblem":
        """A prescribed surface velocity v_bar = dp/dn (outward normal, as ``Velocity`` values), one complex value for all
        elements or one per element in enumeration order, constant over each element.  With ``with_admittance`` the surface
        satisfies v = v_bar + Y p.  With an empty ``IncidentField()`` this poses a radiation problem.  Above ka = 0.5 pair it
        with ``BemSolver.with_sign_consistent_formulation(True)``: the reference's formulation does not converge to the
        physical solution there (DESIGN.md 4.8)."""
        self.surface_velocity = v_bar
        return self

    def with_burton_miller(self, use_bm: bool) -> "BemProblem":
        self.use_burton_miller = use_bm
        return self

    def mesh_radius(self) -> float:
        return float(np.sqrt((self.mesh.nodes ** 2).sum(axis=1)).max())

    def ka(self) -> float:
        return self.physics.wave_number * self.mesh_radius()


@dataclass
class BemSolution:
    surface_pressure: np.ndarray
    mesh: Mesh                       # elements + nodes with the boundary conditions the solve used
    incident_field: IncidentField
    physics: PhysicsParams
    staged: Optional[bem.StagedMesh] = field(default=None, repr=False)
    admittance: Optional[np.ndarray] = None  # the problem's admittance: the surface velocity is Y p
    v_bar: Optional[np.ndarray] = None       # the problem's prescribed surface velocity

    @property
    def surface_velocity(self) -> np.ndarray:
        """v = dp/dn = v_bar + Y p on the boundary elements (enumeration order); zero for a rigid body."""
        n = len(self.surface_pressure)
        v_bar = None if self.v_bar is None else np.broadcast_to(np.asarray(self.v_bar, dtype=np.complex128), (n,))
        if self.admittance is None:
            return np.zeros(n, dtype=np.complex128) if v_bar is None else np.array(v_bar)
        return bem.surface_velocity(self.mesh, self.admittance, self.surface_pressure, v_bar)

    def _velocity_or_none(self) -> Optional[np.ndarray]:
        return None if self.admittance is None and self.v_bar is None else self.surface_velocity

    def _staged(self) -> bem.StagedMesh:
        if self.staged is None:
            self.staged = bem.StagedMesh(self.mesh)
        return self.staged

    def evaluate_pressure_field(self, points, accurate: bool = False) -> List[FieldPoint]:
        """compute_total_field (pressure.rs:273-309): incident + scattered (device field kernel).  With an admittance or a
        prescribed velocity the scattered field takes the surface velocity v = v_bar + Y p.  ``accurate``: the scattered
        field over whole elements with adaptive quadrature near the surface (``evaluate_field``, DESIGN.md 4.10) instead
        of the reference's rule; points on the surface are NaN."""
        return compute_total_field(points, self._staged(), self.surface_pressure, self._velocity_or_none(), self.incident_field,
                                   self.physics, accurate)

    def far_field(self, directions) -> np.ndarray:
        """Complex far-field amplitude F of the scattered / radiated field in the (M, 3) unit ``directions``:
        p_scat(R d) = F(d) exp(i s k R) / R + O(1/R^2) (device; DESIGN.md 4.9)."""
        return compute_far_field(directions, self._staged(), self.surface_pressure, self._velocity_or_none(), self.physics)

    def radiated_power(self) -> float:
        """Power through the surface, W = -(s / (2 omega rho)) sum_j A_j Im(p_j conj(v_j)): radiated power of a source,
        minus the absorbed power of an absorbing body (host, O(N); DESIGN.md 4.9)."""
        return surface_power(self.mesh, self.surface_pressure, self.surface_velocity, self.physics)

    def evaluate_pressure(self, point, accurate: bool = False) -> complex:
        return self.evaluate_pressure_field(np.asarray(point, dtype=np.float64).reshape(1, 3), accurate)[0].p_total

    def max_surface_pressure(self) -> float:
        return float(np.abs(self.surface_pressure).max())

    def mean_surface_pressure(self) -> float:
        return float(np.abs(self.surface_pressure).sum() / len(self.surface_pressure))

    def num_dofs(self) -> int:
        return int(len(self.surface_pressure))


@dataclass
class BemSolver:
    """bem_solver.rs:202-230 defaults: Direct, Tbem, 1000 iterations, 1e-8, beta_scale 4."""
    solver_method: SolverMethod = SolverMethod.Direct
    assembly_method: AssemblyMethod = AssemblyMethod.Tbem
    max_iterations: int = 1000
    tolerance: float = 1e-8
    verbose: bool = False
    beta_scale: float = 4.0
    sign_consistent: bool = False

    @staticmethod
    def new() -> "BemSolver":
        return BemSolver()

    def with_solver_method(self, method: SolverMethod) -> "BemSolver":
        self.solver_method = method
        return self

    def with_assembly_method(self, method: AssemblyMethod) -> "BemSolver":
        self.assembly_method = method
        return self

    def with_max_iterations(self, max_iter: int) -> "BemSolver":
        self.max_iterations = max_iter
        return self

    def with_tolerance(self, tol: float) -> "BemSolver":
        self.tolerance = tol
        return self

    def with_verbose(self, verbose: bool) -> "BemSolver":
        self.verbose = verbose
        return self

    def with_sign_consistent_formulation(self, on: bool) -> "BemSolver":
        """Assemble with dg_dn_sign = +1 at every frequency and one beta throughout (``bem.AssemblyOptions.sign_consistent``)
        instead of the reference's formulation; needed for physical answers above ka = 0.5 (DESIGN.md 4.8)."""
        self.sign_consistent = on
        return self

    # -- bem_solver.rs:320-350 ------------------------------------------------------------------
    def prepare_elements(self, problem: BemProblem) -> Mesh:
        import copy

        mesh = copy.deepcopy(problem.mesh)
        n = mesh.n_elem
        mesh.bc_val[:] = 0.0
        mesh.bc_len[:] = 1
        if problem.bc_type == BoundaryConditionType.Soft:
            mesh.bc_type[:] = BC_PRESSURE      # Pressure(vec![0])
        else:
            mesh.bc_type[:] = BC_VELOCITY      # Velocity(vec![0]) / VelocityWithAdmittance{velocity: vec![0], ..} (tbem.rs:236-238)
        mesh.dof[:] = np.arange(n, dtype=np.uint32)  # elem.dof_addresses = vec![i]
        if problem.surface_velocity is not None:
            if problem.bc_type == BoundaryConditionType.Soft:
                raise BemError("InvalidMesh: a prescribed surface velocity needs a velocity boundary condition, not Soft")
            v = np.asarray(problem.surface_velocity, dtype=np.complex128)
            if v.ndim > 1 or (v.ndim == 1 and v.shape != (n,)):
                raise BemError(f"InvalidMesh: surface velocity has {v.size} entries, the mesh has {n} elements")
            v = np.broadcast_to(v, (n,))
            # constant over the element: one value per node (a single value would weight the first node's shape function only)
            mesh.bc_len[:] = mesh.etype
            for i in range(4):
                mesh.bc_val[:, i] = np.where(i < mesh.etype, v, 0.0)
        return mesh

    # -- bem_solver.rs:273-317 ------------------------------------------------------------------
    def solve(self, problem: BemProblem, ctx: Optional[bem.Context] = None, stats: Optional[dict] = None) -> BemSolution:
        if self.assembly_method != AssemblyMethod.Tbem:
            raise BemError(f"Not implemented: {self.assembly_method.name} assembly is outside the dense path of this library")
        mesh = self.prepare_elements(problem)
        staged = bem.StagedMesh(mesh, ctx)
        beta = problem.physics.burton_miller_beta_scaled(self.beta_scale)
        options = None
        if self.sign_consistent or problem.admittance is not None:
            options = bem.AssemblyOptions(dg_dn_sign=1 if self.sign_consistent else 0, consistent_beta=self.sign_consistent,
                                          admittance=problem.admittance)
        system = bem.build_tbem_system_with_beta(staged, problem.physics, beta, options=options)
        n = mesh.num_dofs
        rows = mesh.is_eval == 0
        centers, normals = mesh.center[rows], mesh.normal[rows]
        if problem.use_burton_miller:
            inc = problem.incident_field.compute_rhs_with_beta(centers, normals, problem.physics, beta)
        else:
            inc = problem.incident_field.compute_rhs(centers, normals, problem.physics, False)
        rhs = system.rhs_full() + inc
        x = self.solve_dense_system(system, rhs, stats)
        if self.verbose:
            print(f"Solution complete. Max surface pressure: {np.abs(x).max():.6f}")
        return BemSolution(x, mesh, problem.incident_field, problem.physics, staged, problem.admittance, problem.surface_velocity)

    # -- bem_solver.rs:435-463 ------------------------------------------------------------------
    def solve_dense_system(self, system, rhs: np.ndarray, stats: Optional[dict] = None) -> np.ndarray:
        if self.solver_method == SolverMethod.Direct:
            try:
                return bem.lu_solve(system, rhs, stats=stats)
            except bem.LuError as e:
                raise BemError(f"Solver failed: {e}") from e
        sol = bem.bicgstab(bem.DenseOperator(system), rhs, bem.BiCgstabConfig(self.max_iterations, self.tolerance, 0))
        if stats is not None:
            stats.update(iterations=sol.iterations, residual=sol.residual)
        if sol.converged:
            return sol.x
        raise BemError(f"Solver failed: BiCGSTAB did not converge: residual = {sol.residual}")
