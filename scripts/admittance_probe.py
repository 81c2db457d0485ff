"""Cost of admittance boundaries in the device assembly (DESIGN.md section 4.8).

    python scripts/admittance_probe.py --out DIR [--repeats 3] [--level 5]

Workload: the headline mesh, rigid icosphere(5) (20 480 Tri3, radius 0.1 m), at ka = 2 with the adaptive Burton-Miller beta.
Three cases are assembled into one reused matrix, alternating, `repeats` times each:

  rigid   no options: the assembly every existing caller runs;
  patch   a passive admittance Y = (0.3 - 0.3i) k on the 10 % of elements with the largest z (a cap);
  all     the same Y on every element.

Per assembly it records the CUDA-event times of the whole assembly and of the far kernel (bemb200_assembly_stats) and the
host time around the call, which ends in a device synchronise.  It then solves GMRES(50) to 1e-10 with a plane wave along +z
for rigid, for `all` with the reference's sign and beta, and for `all` with the sign-consistent formulation, and records the
iterations.  It checks that the Y = 0 columns of the patch matrix equal the rigid matrix bit for bit on the first 512 rows.
Writes DIR/admittance_probe.json with the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers are then reported without it, and say so
        return {"error": repr(e)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--level", type=int, default=5)
    args = ap.parse_args()

    from math_audio_b200 import bem
    from math_audio_b200.incident import IncidentField
    from math_audio_b200.mesh import generate_icosphere_mesh
    from math_audio_b200.types import PhysicsParams

    a, ka = 0.1, 2.0
    mesh = generate_icosphere_mesh(a, args.level)
    n = mesh.n_elem
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    k = ph.wave_number
    Y = (0.3 - 0.3j) * k
    cap = mesh.center[:, 2] >= np.quantile(mesh.center[:, 2], 0.9)
    cases = {
        "rigid": None,
        "patch": bem.AssemblyOptions(admittance=np.where(cap, Y, 0.0)),
        "all": bem.AssemblyOptions(admittance=np.full(n, Y)),
    }
    st = bem.StagedMesh(mesh)
    system = bem.build_tbem_system_with_beta(st, ph, beta)  # warm-up of the plain kernels and the matrix handle
    for opts in cases.values():
        system = bem.build_tbem_system_with_beta(st, ph, beta, reuse=system, options=opts)  # warm-up of every instantiation
    runs = {name: [] for name in cases}
    for _ in range(args.repeats):
        for name, opts in cases.items():
            t0 = time.perf_counter()
            system = bem.build_tbem_system_with_beta(st, ph, beta, reuse=system, options=opts, fetch_rhs=False)
            t1 = time.perf_counter()
            s = system.matrix.assembly_stats()
            runs[name].append(dict(host_s=t1 - t0, total_ms=s["total_ms"], far_ms=s["far_ms"], near_pairs=s["near_pairs"]))
    med = {name: {key: float(np.median([r[key] for r in rr])) for key in ("host_s", "total_ms", "far_ms")} for name, rr in runs.items()}

    rows = min(512, n)
    rigid = bem.build_tbem_system_with_beta(st, ph, beta, reuse=system).matrix.rows(0, rows)
    patch = bem.build_tbem_system_with_beta(st, ph, beta, reuse=system, options=cases["patch"]).matrix.rows(0, rows)
    zero_cols_bits = bool(np.array_equal(patch[:, ~cap], rigid[:, ~cap]))
    del rigid, patch

    cfg = bem.GmresConfig(max_iterations=2000, restart=50, tolerance=1e-10)
    inc = IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
    solves = {}
    for name, opts in (("rigid", None), ("all_reference_formulation", cases["all"]),
                       ("all_sign_consistent", bem.AssemblyOptions.sign_consistent(np.full(n, Y)))):
        system = bem.build_tbem_system_with_beta(st, ph, beta, reuse=system, options=opts)
        t0 = time.perf_counter()
        sol = bem.gmres(bem.DenseOperator(system), system.rhs + inc, cfg)
        solves[name] = dict(iterations=sol.iterations, restarts=sol.restarts, converged=sol.converged, residual=sol.residual,
                            seconds=time.perf_counter() - t0)

    out = dict(
        card=card(), workload=f"rigid icosphere({args.level}), {n} Tri3, a = {a} m, ka = {ka}, adaptive beta {beta}, Y = {Y}",
        repeats=args.repeats, patch_elements=int(cap.sum()), runs=runs, median=med,
        far_ratio_vs_rigid={name: med[name]["far_ms"] / med["rigid"]["far_ms"] for name in cases},
        total_ratio_vs_rigid={name: med[name]["total_ms"] / med["rigid"]["total_ms"] for name in cases},
        patch_zero_columns_equal_rigid_bits_first_rows=zero_cols_bits, gmres50_1e10=solves)
    Path(args.out).mkdir(parents=True, exist_ok=True)
    (Path(args.out) / "admittance_probe.json").write_text(json.dumps(out, indent=1))
    print(json.dumps(dict(median=med, far_ratio_vs_rigid=out["far_ratio_vs_rigid"], solves=solves, bits=zero_cols_bits)))


if __name__ == "__main__":
    main()
