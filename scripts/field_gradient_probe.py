"""Field gradient on the device against the pressure alone and against a central-difference gradient (DESIGN.md section 4.11).

    python scripts/field_gradient_probe.py --out DIR [--repeats 5]

Workloads of scripts/field_eval_probe.py: icosphere(5) (20 480 Tri3, radius 0.1 m, ka = 2) and config 3 (the 0.32 x 0.44 x
0.64 m cabinet, 50 176 Quad4, 1 kHz), each with 4 096 regular points (a sphere of 10 x the body's radius) and 4 096 near points
(delta h above seeded random surface spots, delta log-uniform in [1e-3, 1]), nsol = 1, 8 and 32 seeded random surface
solutions on the device.  Three forms run in alternation, one call of each per round:

  gradient   evaluate_field_gradient with the pressure (out_p)
  field      evaluate_field alone
  fd7        the 7 evaluate_field calls of a central-difference gradient (x and x +- 1e-4 h e_k)

Each call is synchronous (it ends in a stream synchronise); times are host clocks around it after one warm-up round, the
median over --repeats rounds.  A pass of its own under torch.profiler (CUDA activities) splits the gradient's kernel time.
Writes DIR/field_gradient_probe.json with the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "scripts"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

from field_eval_probe import card, near_points, sphere_points  # noqa: E402

KERNELS = ("field_element_kernel", "field_near_count_kernel", "field_near_fill_kernel", "field_gradient_near_kernel",
           "field_gradient_regular_kernel", "field_gradient_combine_kernel", "field_near_kernel", "field_regular_kernel",
           "field_combine_kernel")


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, type=Path)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if args.repeats < 1:
        ap.error("--repeats must be >= 1")

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("field_gradient_probe: no CUDA device (this measurement has no CPU form)")
    from math_audio_b200 import bem
    from math_audio_b200.mesh import generate_box_mesh_quad, generate_icosphere_mesh
    from math_audio_b200.types import PhysicsParams

    def timed_round(fns):
        out = []
        for fn in fns:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            out.append((time.perf_counter() - t0) * 1e3)
        return out

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
        h = math.sqrt(float(np.mean(mesh.area)))
        P = torch.from_numpy(rng.standard_normal((32, n)) + 1j * rng.standard_normal((32, n))).to("cuda:0")
        V = torch.from_numpy(rng.standard_normal((32, n)) + 1j * rng.standard_normal((32, n))).to("cuda:0")
        sets = {"regular_10a": sphere_points(10.0 * radius, 4096), "near": near_points(mesh, 4096, rng)}
        keep.append((wname, st, ph, P, V, sets))
        for sname, pts in sets.items():
            eps = 1e-4 * h
            shifted = [pts] + [pts + sg * eps * e for e in np.eye(3) for sg in (1.0, -1.0)]
            for nsol in (1, 8, 32):
                def gradient():
                    bem.evaluate_field_gradient(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol, with_pressure=True)

                def field():
                    bem.evaluate_field(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol)

                def fd7():
                    for x in shifted:
                        bem.evaluate_field(x, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol)

                timed_round([gradient, field, fd7])  # warm-up
                rounds = np.array([timed_round([gradient, field, fd7]) for _ in range(args.repeats)])
                med = np.median(rounds, axis=0)
                row = {"workload": wname, "elements": n, "points": sname, "n_points": len(pts), "nsol": nsol,
                       "gradient_ms": float(med[0]), "field_ms": float(med[1]), "fd7_ms": float(med[2]),
                       "gradient_over_field": float(med[0] / med[1]), "gradient_over_fd7": float(med[0] / med[2]),
                       "all_ms": rounds.tolist()}
                print(json.dumps({k: v for k, v in row.items() if k != "all_ms"}), flush=True)
                result["rows"].append(row)

    from torch.profiler import ProfilerActivity, profile

    for wname, st, ph, P, V, sets in keep:
        for sname, pts in sets.items():
            for nsol in (1, 32):
                for form in ("gradient", "field"):
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        if form == "gradient":
                            bem.evaluate_field_gradient(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol, with_pressure=True)
                        else:
                            bem.evaluate_field(pts, st, P.data_ptr(), V.data_ptr(), ph, nsol=nsol)
                        torch.cuda.synchronize()
                    kern = {}
                    for ev in prof.events():
                        for key in KERNELS:
                            if key in ev.name:
                                t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                                kern[key] = kern.get(key, 0.0) + t / 1e3
                                break
                    result["profile"][f"{wname}/{sname}/nsol{nsol}/{form}"] = kern
    result["card_after"] = card()
    args.out.mkdir(parents=True, exist_ok=True)
    (args.out / "field_gradient_probe.json").write_text(json.dumps(result, indent=1))
    print(json.dumps(result["profile"], indent=1))
    print(json.dumps(result["card"]))
    return 0


if __name__ == "__main__":
    sys.exit(main())
