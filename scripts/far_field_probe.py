"""Far-field amplitude on the device against today's workarounds (DESIGN.md section 4.9).

    python scripts/far_field_probe.py --out DIR [--repeats 3]

Workloads: icosphere(5) (20 480 Tri3, radius 0.1 m, ka = 2) and config 3 (the 0.32 x 0.44 x 0.64 m cabinet, 50 176 Quad4,
1 kHz), each on a 5 degree balloon (theta 0..180 x phi 0..355: 37 x 72 = 2 664 directions) and a 2 degree balloon (91 x 180 =
16 380), with nsol = 1, 8 and 32 seeded random surface solutions (p and v; the kernel's work does not depend on the values).
Three forms run alternately on the same device inputs:

  far        compute_far_field (far_field_kernel + its split reduction)
  field      compute_scattered_field_batch at R = 1e3 x the body's radius on the same directions (the workaround: F ~ R p)
  rcs        compute_rcs_batch (centroid rule, no velocity term), for scale

Each call is synchronous (it ends in a stream synchronise); times are host clocks around it after one warm-up call, the
median of --repeats.  A pass of its own under torch.profiler (CUDA activities) gives the kernel times of the far field.
Writes DIR/far_field_probe.json with the card name and power limit read in the same run.
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
    except Exception as e:
        return {"error": repr(e)}


def balloon(step_deg: int) -> np.ndarray:
    th = np.radians(np.arange(0, 181, step_deg))
    ph = np.radians(np.arange(0, 360, step_deg))
    T, P = np.meshgrid(th, ph, indexing="ij")
    d = np.stack([np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)], axis=-1).reshape(-1, 3)
    return d / np.linalg.norm(d, axis=1, keepdims=True)


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, type=Path)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    if args.repeats < 1:
        ap.error("--repeats must be >= 1")

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("far_field_probe: no CUDA device (this measurement has no CPU form)")
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
        keep.append((st, P, V))
        for step in (5, 2):
            dirs = balloon(step)
            pts = 1e3 * radius * dirs
            for nsol in (1, 8, 32):
                row = {"workload": wname, "elements": n, "balloon_deg": step, "directions": len(dirs), "nsol": nsol}
                row["far_ms"], row["far_all_ms"] = timed(lambda: bem.compute_far_field(dirs, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol))
                row["field_ms"], row["field_all_ms"] = timed(
                    lambda: bem.compute_scattered_field_batch(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol))
                row["rcs_ms"], row["rcs_all_ms"] = timed(lambda: bem.compute_rcs_batch(P.data_ptr(), st, dirs, ph, nsol=nsol))
                row["pair_evaluations_per_s"] = nsol * len(dirs) * n / (row["far_ms"] * 1e-3)
                print(json.dumps(row), flush=True)
                result["rows"].append(row)

    from torch.profiler import ProfilerActivity, profile

    for (st, P, V), (wname, (_, ph, _)) in zip(keep, workloads.items()):
        for step in (5, 2):
            dirs = balloon(step)
            for nsol in (1, 32):
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    bem.compute_far_field(dirs, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol)
                    sync()
                kern = {}
                for ev in prof.events():
                    for key in ("far_field_reduce_kernel", "far_field_kernel"):
                        if key in ev.name:
                            t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                            kern[key] = kern.get(key, 0.0) + t / 1e3
                            break
                result["profile"][f"{wname}/{step}deg/nsol{nsol}"] = kern
    result["card_after"] = card()
    args.out.mkdir(parents=True, exist_ok=True)
    (args.out / "far_field_probe.json").write_text(json.dumps(result, indent=1))
    print(json.dumps(result["profile"], indent=1))
    print(json.dumps(result["card"]))
    return 0


if __name__ == "__main__":
    sys.exit(main())
