"""Accurate field evaluation on the device against the reference's field kernel (DESIGN.md section 4.10).

    python scripts/field_eval_probe.py --out DIR [--repeats 3]

Workloads: icosphere(5) (20 480 Tri3, radius 0.1 m, ka = 2) and config 3 (the 0.32 x 0.44 x 0.64 m cabinet, 50 176 Quad4,
1 kHz), each with two sets of 4 096 evaluation points: on a sphere of 10 x the body's radius (every pair regular), and at
delta h above seeded random spots of the surface, delta log-uniform in [1e-3, 1] (h = sqrt(mean element area)), with
nsol = 1, 8 and 32 seeded random surface solutions (p and v; the kernels' work does not depend on the values).  Two forms run
alternately on the same device inputs:

  accurate   evaluate_field (regular pass, near list, near pass, combine)
  reference  compute_scattered_field_batch (scattered_field_batch_kernel: first triangle, 7 points at every distance)

Each call is synchronous (it ends in a stream synchronise); times are host clocks around it after one warm-up call, the
median of --repeats.  A pass of its own under torch.profiler (CUDA activities) splits the accurate form's kernel time into
the regular, near-list, near and combine kernels.  Writes DIR/field_eval_probe.json with the card name and power limit read
in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

KERNELS = ("field_element_kernel", "field_near_count_kernel", "field_near_fill_kernel", "field_near_kernel", "field_regular_kernel",
           "field_combine_kernel", "scattered_field_batch_kernel")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:
        return {"error": repr(e)}


def sphere_points(radius: float, m: int) -> np.ndarray:
    """m points of a Fibonacci lattice on the sphere of the given radius"""
    i = np.arange(m) + 0.5
    z = 1.0 - 2.0 * i / m
    phi = math.pi * (3.0 - math.sqrt(5.0)) * i
    s = np.sqrt(1.0 - z * z)
    return radius * np.stack([s * np.cos(phi), s * np.sin(phi), z], axis=1)


def near_points(mesh, m: int, rng) -> np.ndarray:
    """m points at delta h along the outward normal above random interior spots of random elements, delta log-uniform in
    [1e-3, 1]"""
    h = math.sqrt(float(np.mean(mesh.area)))
    e = rng.integers(0, mesh.n_elem, m)
    delta = 10.0 ** rng.uniform(-3.0, 0.0, m)
    w = rng.uniform(0.1, 0.3, (m, 1))
    x0 = mesh.nodes[mesh.conn[e, 0].astype(np.int64)]
    return (1.0 - w) * mesh.center[e] + w * x0 + (delta * h)[:, None] * mesh.normal[e]


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, type=Path)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    if args.repeats < 1:
        ap.error("--repeats must be >= 1")

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("field_eval_probe: no CUDA device (this measurement has no CPU form)")
    from math_audio_b200 import bem
    from math_audio_b200.mesh import generate_box_mesh_quad, generate_icosphere_mesh
    from math_audio_b200.types import PhysicsParams

    def sync():
        torch.cuda.synchronize()

    def timed(fn):
        fn()
        sync()
        ts = []
        for _ in range(args.repeats):
            t0 = time.perf_counter()
            fn()
            sync()
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts)) * 1e3, [t * 1e3 for t in ts]

    workloads = {
        "icosphere5_ka2": (generate_icosphere_mesh(0.1, 5), PhysicsParams.from_wave_number(20.0), 0.1),
        "config3_1kHz": (generate_box_mesh_quad(0.32, 0.44, 0.64, 64, 88, 128), PhysicsParams.new(1000.0, 343.0, 1.21, False),
                         float(np.linalg.norm([0.16, 0.22, 0.32]))),
    }
    rng = np.random.default_rng(0)
    result = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "repeats": args.repeats, "rows": [], "profile": {}}
    keep = []
    for wname, (mesh, ph, radius) in workloads.items():
        st = bem.StagedMesh(mesh)
        n = st.num_dofs
        P = torch.from_numpy(rng.standard_normal((32, n)) + 1j * rng.standard_normal((32, n))).to("cuda:0")
        V = torch.from_numpy(rng.standard_normal((32, n)) + 1j * rng.standard_normal((32, n))).to("cuda:0")
        sets = {"regular_10a": sphere_points(10.0 * radius, 4096), "near": near_points(mesh, 4096, rng)}
        keep.append((wname, st, ph, P, V, sets))
        for sname, pts in sets.items():
            for nsol in (1, 8, 32):
                row = {"workload": wname, "elements": n, "points": sname, "n_points": len(pts), "nsol": nsol}
                row["accurate_ms"], row["accurate_all_ms"] = timed(
                    lambda: bem.evaluate_field(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol))
                row["reference_ms"], row["reference_all_ms"] = timed(
                    lambda: bem.compute_scattered_field_batch(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol))
                print(json.dumps(row), flush=True)
                result["rows"].append(row)

    from torch.profiler import ProfilerActivity, profile

    for wname, st, ph, P, V, sets in keep:
        for sname, pts in sets.items():
            for nsol in (1, 32):
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    bem.evaluate_field(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol)
                    bem.compute_scattered_field_batch(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol)
                    sync()
                kern = {}
                for ev in prof.events():
                    for key in KERNELS:
                        if key in ev.name:
                            t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                            kern[key] = kern.get(key, 0.0) + t / 1e3
                            break
                result["profile"][f"{wname}/{sname}/nsol{nsol}"] = kern
    result["card_after"] = card()
    args.out.mkdir(parents=True, exist_ok=True)
    (args.out / "field_eval_probe.json").write_text(json.dumps(result, indent=1))
    print(json.dumps(result["profile"], indent=1))
    print(json.dumps(result["card"]))
    return 0


if __name__ == "__main__":
    sys.exit(main())
