"""Multi-direction scattering, host path against device path (DESIGN.md section 4.7).

    python scripts/multi_direction_probe.py --out DIR [--repeats 3] [--level 5]

Workload: BASELINE config 5 -- rigid icosphere(5) (20 480 Tri3), ka = 2, adaptive Burton-Miller beta, 32 plane waves from
Fibonacci directions, GMRES(50) to 1e-10 -- followed by the bistatic RCS of every solution on 2048 directions and its
scattered field at 4096 points on a sphere of radius 1 m.  Two arms run alternately in one process:

  (a) host     numpy B, gmres_batched, 32 x compute_rcs, 32 x compute_scattered_field;
  (b) device   incident_rhs_batch -> gmres_batched_device -> compute_rcs_batch / compute_scattered_field_batch.

Every stage ends in a device synchronise.  Writes DIR/multi_direction_probe.json: per-stage times of every repeat, the kernel
times of the single and batch RCS / field kernels (torch.profiler, CUDA activities, in a pass of its own), whether arm (b)'s
batch kernels reproduce arm (a)'s outputs bit for bit on the same x, and the card name and power limit read in the same run.
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


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, type=Path)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--level", type=int, default=5, help="icosphere level (5: 20 480 elements, BASELINE config 5)")
    ap.add_argument("--n-dirs", type=int, default=2048)
    ap.add_argument("--n-points", type=int, default=4096)
    args = ap.parse_args()
    if args.repeats < 1:
        ap.error("--repeats must be >= 1")

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("multi_direction_probe: no CUDA device (this measurement has no CPU form)")
    from math_audio_b200 import bem
    from math_audio_b200.incident import IncidentField
    from math_audio_b200.mesh import fibonacci_directions, generate_icosphere_mesh
    from math_audio_b200.types import PhysicsParams

    args.out.mkdir(parents=True, exist_ok=True)
    info = card()
    a, ka, nrhs = 0.1, 2.0, 32
    mesh = generate_icosphere_mesh(a, args.level)
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    st = bem.StagedMesh(mesh)
    n = st.num_dofs
    system = bem.build_tbem_system_with_beta(st, ph, beta)
    op = bem.DenseOperator(system)
    cfg = bem.GmresConfig(max_iterations=50, restart=50, tolerance=1e-10)
    dirs = fibonacci_directions(nrhs)
    incs = [IncidentField.plane_wave(d) for d in dirs]
    obs = np.ascontiguousarray(fibonacci_directions(args.n_dirs))
    pts = np.ascontiguousarray(fibonacci_directions(args.n_points) * 1.0)
    dev = torch.device("cuda:0")
    bd = torch.empty((nrhs, n), dtype=torch.complex128, device=dev)
    xd = torch.empty((nrhs, n), dtype=torch.complex128, device=dev)

    def sync():
        torch.cuda.synchronize(dev)

    def arm_a():
        t, o = {}, {}
        t0 = time.perf_counter()
        rhs = system.rhs_full()
        B = np.stack([rhs + f.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta) for f in incs])
        t["rhs_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sols, _ = bem.gmres_batched(op, B, cfg)
        sync()
        t["solve_s"] = time.perf_counter() - t0
        X = np.stack([s.x for s in sols])
        t0 = time.perf_counter()
        o["rcs"] = np.stack([bem.compute_rcs(X[s], st, obs, ph) for s in range(nrhs)])
        sync()
        t["rcs_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        o["field"] = np.stack([bem.compute_scattered_field(pts, st, X[s], None, ph) for s in range(nrhs)])
        sync()
        t["field_s"] = time.perf_counter() - t0
        o["B"], o["X"], o["iters"] = B, X, [s.iterations for s in sols]
        return t, o

    def arm_b():
        t, o = {}, {}
        t0 = time.perf_counter()
        bem.incident_rhs_batch(st, ph, beta, incs, system=system, b_dev=bd.data_ptr(), fetch=False)
        sync()
        t["rhs_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sols, _ = bem.gmres_batched_device(op, bd.data_ptr(), nrhs, cfg, xd.data_ptr())
        sync()
        t["solve_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        o["rcs"] = bem.compute_rcs_batch(xd.data_ptr(), st, obs, ph, nsol=nrhs)
        sync()
        t["rcs_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        o["field"] = bem.compute_scattered_field_batch(pts, st, xd.data_ptr(), None, ph, nsol=nrhs)
        sync()
        t["field_s"] = time.perf_counter() - t0
        o["iters"] = [s.iterations for s in sols]
        return t, o

    arm_a(), arm_b()  # warm-up: module loads, pools, the batched solver's Krylov bases
    runs = {"a_host": [], "b_device": []}
    for _ in range(args.repeats):
        ta, oa = arm_a()
        tb, ob = arm_b()
        for t in (ta, tb):
            t["total_s"] = t["rhs_s"] + t["solve_s"] + t["rcs_s"] + t["field_s"]
        runs["a_host"].append(ta)
        runs["b_device"].append(tb)

    def bits(x, y):
        return bool(np.array_equal(np.asarray(x).view(np.uint64), np.asarray(y).view(np.uint64)))

    Bd, Xd = bd.cpu().numpy(), xd.cpu().numpy()
    parity = {
        # the batch kernels on arm (a)'s x (host input) against arm (a)'s 32 single calls
        "rcs_batch_equals_single_calls_bitwise": bits(bem.compute_rcs_batch(oa["X"], st, obs, ph), oa["rcs"]),
        "field_batch_equals_single_calls_bitwise": bits(bem.compute_scattered_field_batch(pts, st, oa["X"], None, ph), oa["field"]),
        # arm (b)'s outputs against the single calls on arm (b)'s own x
        "rcs_b_equals_single_calls_on_b_x_bitwise": bits(ob["rcs"], np.stack([bem.compute_rcs(Xd[s], st, obs, ph) for s in range(nrhs)])),
        "B_device_vs_numpy_max_rel": float(np.abs(Bd - oa["B"]).max() / np.abs(oa["B"]).max()),
        "x_device_vs_host_path_max_rel": float(max(np.linalg.norm(Xd[s] - oa["X"][s]) / np.linalg.norm(oa["X"][s]) for s in range(nrhs))),
        "iterations_equal": oa["iters"] == ob["iters"],
        "rcs_max_rel_between_arms": float(np.max(np.abs(ob["rcs"] - oa["rcs"]) / np.abs(oa["rcs"]))),
        "field_max_rel_between_arms": float(np.abs(ob["field"] - oa["field"]).max() / np.abs(oa["field"]).max()),
    }

    # kernel times: one profiled pass of each post-processing form, separate from the timed repeats
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for s in range(nrhs):
            bem.compute_rcs(oa["X"][s], st, obs, ph)
            bem.compute_scattered_field(pts, st, oa["X"][s], None, ph)
        bem.compute_rcs_batch(xd.data_ptr(), st, obs, ph, nsol=nrhs)
        bem.compute_scattered_field_batch(pts, st, xd.data_ptr(), None, ph, nsol=nrhs)
        bem.incident_rhs_batch(st, ph, beta, incs, b_dev=bd.data_ptr(), fetch=False)
        sync()
    kern = {}
    for ev in prof.events():
        name = ev.name
        for key in ("rcs_batch_kernel", "scattered_field_batch_kernel", "incident_rhs_batch_kernel", "rcs_kernel", "scattered_field_kernel"):
            if key in name and (key.endswith("batch_kernel") or "batch" not in name):
                d = kern.setdefault(key, {"launches": 0, "device_ms": 0.0})
                d["launches"] += 1
                d["device_ms"] += ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
                break

    def med(rows, k):
        return float(np.median([r[k] for r in rows]))

    summary = {arm: {k: med(rows, k) for k in ("rhs_s", "solve_s", "rcs_s", "field_s", "total_s")} for arm, rows in runs.items()}
    out = {
        "probe": "multi_direction_probe",
        "card": info,
        "workload": {"mesh": f"icosphere({args.level})", "n_elements": int(n), "ka": ka, "nrhs": nrhs, "gmres": "GMRES(50), tol 1e-10",
                     "rcs_directions": int(obs.shape[0]), "field_points": int(pts.shape[0]), "field_radius_m": 1.0},
        "repeats": args.repeats,
        "stage_times_median_s": summary,
        "stage_times_s": runs,
        "kernel_device_ms_for_32_solutions": kern,
        "parity": parity,
        "iterations": ob["iters"],
    }
    path = args.out / "multi_direction_probe.json"
    path.write_text(json.dumps(out, indent=1))
    print(json.dumps({"card": info, "stage_times_median_s": summary, "kernels": kern, "parity": parity}, indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
