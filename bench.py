#!/usr/bin/env python3
"""bench.py -- BEM assemble + GMRES solve, seconds per frequency (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one frequency of the sweep: dense TBEM assembly of the system matrix + restarted
GMRES(50) solve to 1e-10 on that matrix.  Default workload = BASELINE.json configs[1]: rigid
icosphere(5) (20 480 Tri3 elements, 6.7 GB complex128 matrix), 64 frequencies with ka
log-spaced in [0.25, 8], adaptive Burton-Miller beta, plane wave +z.  Step i uses frequency
index (23*i mod 64) so that any number of steps samples the whole band.

N > 1 (torchrun, one process per GPU): the SAME problem is row-block sharded over the ranks
(strong scaling): each rank assembles and stores only its rows, every GMRES iteration
all-gathers the matvec output over NCCL (see csrc/gmres.cu).

value  : device-resident inputs (staged mesh, right-hand sides and solution in HBM), timed with
         CUDA events on the stream the library submits to, max over ranks.
e2e    : the same metric through the public host-buffer API (bem.build_tbem_system_with_beta +
         bem.gmres): mesh H2D staging, rhs D2H, b H2D and x D2H inside the timed region.
--impl reference : the CPU oracle (restatement of the reference; the Rust reference cannot be
         built in this image) on the host cores, bounded samples, rank 0 only.
--dump-outputs DIR : after the timed steps, rank 0 of the native arm writes what the last timed step
         returned as float64 DIR/<name>.npy (see dump_outputs); the inputs depend on the arguments only,
         so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from math_audio_b200.mesh import generate_geodesic_sphere_mesh, generate_icosphere_mesh  # noqa: E402
from math_audio_b200.types import PhysicsParams  # noqa: E402

METRIC = "bem_assemble_plus_gmres_seconds_per_frequency"
UNIT = "s/frequency"
FLOP_PER_QP = 68.0      # SURVEY.md 8d: algorithmic flops per quadrature-point evaluation
FLOP_PER_PAIR = 40.0    # ... and per (row, element) pair
GMRES_RESTART = 50
GMRES_TOL = 1e-10
GMRES_MAX_CYCLES = 1000


def workload(name: str):
    """-> dict(name, mesh, a, ka_list, nq)"""
    if name == "sphere20k_sweep64":
        a = 0.1
        mesh = generate_icosphere_mesh(a, 5)
        ka = np.exp(np.linspace(math.log(0.25), math.log(8.0), 64))
        return dict(name=name, mesh=mesh, a=a, ka=ka, nq=13, desc="rigid icosphere(5), 20480 Tri3, 64 frequencies ka in [0.25, 8]")
    if name == "sphere121k":
        a = 1.0
        mesh = generate_geodesic_sphere_mesh(a, 78)
        return dict(name=name, mesh=mesh, a=a, ka=np.array([16.0]), nq=13, desc="rigid geodesic sphere nu=78, 121680 Tri3, ka=16")
    if name == "sphere1k":  # CPU-test size
        a = 0.1
        mesh = generate_icosphere_mesh(a, 3)
        ka = np.exp(np.linspace(math.log(0.25), math.log(8.0), 64))
        return dict(name=name, mesh=mesh, a=a, ka=ka, nq=13, desc="rigid icosphere(3), 1280 Tri3, 64 frequencies")
    if name == "sphere5k":  # small variant for quick checks
        a = 0.1
        mesh = generate_icosphere_mesh(a, 4)
        ka = np.exp(np.linspace(math.log(0.25), math.log(8.0), 64))
        return dict(name=name, mesh=mesh, a=a, ka=ka, nq=13, desc="rigid icosphere(4), 5120 Tri3, 64 frequencies")
    raise SystemExit(f"unknown workload {name}")


def freq_index(step: int, nfreq: int) -> int:
    return (23 * step) % nfreq


def physics_for(wl, step):
    ka = float(wl["ka"][freq_index(step, len(wl["ka"]))])
    ph = PhysicsParams.from_wave_number(ka / wl["a"])
    beta, _ = ph.burton_miller_beta_adaptive(wl["a"])
    return ka, ph, beta


def base_config(wl) -> dict:
    """The `config` object of the JSON line: identical in the native and the reference arm (run-specific
    detail such as the schedule or the rows per GPU lives under `run`)."""
    return {"workload": wl["name"], "description": wl["desc"], "n_elements": int(wl["mesh"].num_dofs),
            "gmres": f"restart {GMRES_RESTART}, tol {GMRES_TOL}, MGS, max {GMRES_MAX_CYCLES} cycles",
            "beta": "burton_miller_beta_adaptive", "incident": "plane wave +z, amplitude 1",
            "frequency_of_step": "step i solves ka[(23 i) mod nfreq] of the workload's frequency list",
            "l2": "inputs larger than L2: the matrix (16 N^2 bytes) is re-streamed from HBM by every matvec"}


_REAL_STDOUT = None


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
            t0 = time.time()  # nvidia-smi needs a moment before its first sample
            while time.time() - t0 < 3.0 and os.path.getsize(self.f.name) == 0:
                time.sleep(0.05)
            self.skip = len(open(self.f.name).read().splitlines())  # samples taken before the timed region
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines()[getattr(self, "skip", 0):]:
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# -------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle on the host cores, bounded samples
# -------------------------------------------------------------------------------------------
def iteration_table(wl_name: str):
    p = ROOT / "profiles" / f"gmres_iterations_{wl_name}.json"
    if p.exists():
        return json.loads(p.read_text())
    return None


def cpu_sample(wl, step, rows_target_s: float, iters_hint=None):
    """Time the oracle on a bounded sample of one frequency and extrapolate to the whole
    frequency (assembly cost is exactly linear in rows; a matvec is linear in rows)."""
    from oracle import oracle as orc

    mesh = wl["mesh"]
    n = mesh.num_dofs
    ka, ph, beta = physics_for(wl, step)
    threads = orc.num_threads()
    # calibrate
    r_cal = 2 * threads
    t0 = time.perf_counter()
    orc.assemble(mesh, ph.wave_number, beta, row_begin=0, row_end=r_cal)
    t_cal = time.perf_counter() - t0
    rows = int(max(r_cal, min(n, r_cal * rows_target_s / max(t_cal, 1e-6))))
    rows = (rows // threads) * threads or threads
    start = (n // 3) // threads * threads
    if start + rows > n:
        start = 0
    t0 = time.perf_counter()
    A, _, nqp = orc.assemble(mesh, ph.wave_number, beta, row_begin=start, row_end=start + rows)
    t_asm = time.perf_counter() - t0
    x = np.random.default_rng(1234).standard_normal(n) + 1j * np.random.default_rng(4321).standard_normal(n)
    orc.zgemv(A, x)
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        orc.zgemv(A, x)
    t_mv = (time.perf_counter() - t0) / reps
    scale = n / rows
    fi = freq_index(step, len(wl["ka"]))
    if iters_hint is not None and fi in iters_hint:
        matvecs = iters_hint[fi]
        src = "matvec count measured by the native arm in this run"
    else:
        tab = iteration_table(wl["name"])
        if tab and str(fi) in tab:
            matvecs = tab[str(fi)]
            src = "matvec count from profiles/gmres_iterations_*.json (same algorithm, measured on B200)"
        else:
            matvecs = 100
            src = "matvec count assumed 100"
    t_freq = t_asm * scale + matvecs * t_mv * scale
    return dict(seconds_per_frequency=t_freq, asm_s=t_asm * scale, matvec_s=t_mv * scale, matvecs=matvecs, rows=rows,
                threads=threads, ka=ka, asm_gflops=(FLOP_PER_QP * nqp + FLOP_PER_PAIR * rows * (n - 1)) / t_asm / 1e9,
                matvec_gbs=(16.0 * rows * n + 16.0 * n + 16.0 * rows) / t_mv / 1e9, src=src, sample_s=t_asm + (reps + 1) * t_mv + t_cal)


def cpu_full_frequency(wl, step):
    """ONE complete frequency on the host cores, nothing sampled or extrapolated: oracle assembly of
    all N rows (tbem.rs:96-222 restated) + incident right-hand side + oracle GMRES(50) to 1e-10
    (gmres.rs:105-277 restated; every matvec is a threaded row-major zgemv over the whole matrix)."""
    from math_audio_b200.incident import IncidentField
    from oracle import oracle as orc

    mesh = wl["mesh"]
    n = mesh.num_dofs
    ka, ph, beta = physics_for(wl, step)
    t0 = time.perf_counter()
    A, rhs0, nqp = orc.assemble(mesh, ph.wave_number, beta)
    b = rhs0 + IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
    t1 = time.perf_counter()
    x, info = orc.gmres(A, b, max_iterations=GMRES_MAX_CYCLES, restart=GMRES_RESTART, tolerance=GMRES_TOL)
    t2 = time.perf_counter()
    matvecs = info["iterations"] + info["restarts"] + 1
    del A
    return dict(seconds_per_frequency=t2 - t0, asm_s=t1 - t0, gmres_s=t2 - t1, ka=ka, fi=freq_index(step, len(wl["ka"])),
                iterations=info["iterations"], restarts=info["restarts"], residual=info["residual"], converged=info["converged"],
                matvecs=matvecs, threads=orc.num_threads(),
                asm_gflops=(FLOP_PER_QP * nqp + FLOP_PER_PAIR * n * (n - 1)) / (t1 - t0) / 1e9,
                matvec_gbs=(16.0 * n * n + 32.0 * n) * matvecs / (t2 - t1) / 1e9)


def run_reference(args):
    """Reference arm: the CPU restatement of the reference's path (`oracle/`, kind "port": the Rust
    reference cannot be built in this image) on all host threads.  Every timed step is a COMPLETE
    frequency of the workload (full assembly + GMRES to 1e-10), run back to back until --steps is
    reached or the time budget (BENCH_REF_BUDGET_S, default 300 s) would be exceeded -- at least two.
    `steps` of the line is the number of frequencies actually run; `value` is their mean wall time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = workload(args.workload)
    n = wl["mesh"].num_dofs
    if 16.0 * n * n > 0.6 * (os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")):
        raise SystemExit(f"reference arm: the {16.0 * n * n / 1e9:.0f} GB matrix of {wl['name']} does not fit the host memory")
    budget = float(os.environ.get("BENCH_REF_BUDGET_S", "300"))
    t_begin = time.perf_counter()
    for s in range(args.warmup):  # warm-up: thread pool, page cache, libm -- a few rows only
        cpu_sample(wl, s, 0.5)
    res = []
    for s in range(args.steps):
        if len(res) >= 2:
            per = float(np.mean([r["seconds_per_frequency"] for r in res]))
            if (time.perf_counter() - t_begin) + per > budget:
                break
        res.append(cpu_full_frequency(wl, args.warmup + s))
        if os.environ.get("BENCH_DEBUG"):
            print(f"[reference] step {s}: {res[-1]}", file=sys.stderr)
    K = len(res)
    val = float(np.mean([r["seconds_per_frequency"] for r in res]))
    model = cpu_sample(wl, args.warmup, 4.0, {res[0]["fi"]: res[0]["matvecs"]})  # labelled second figure: the sampled model
    sample = (f"oracle port (C++ restatement, std::thread over rows / zgemv rows): {K} complete frequencies of {wl['name']} run in full "
              f"(assembly of all {n} rows + GMRES({GMRES_RESTART}) to {GMRES_TOL}; {args.steps} requested, budget {budget:.0f} s)")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
        "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": val * 1e3, "higher_is_better": False,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": base_config(wl),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": res[0]["threads"], "kind": "port", "sample": sample,
                         "assembly_s": float(np.mean([r["asm_s"] for r in res])), "gmres_s": float(np.mean([r["gmres_s"] for r in res])),
                         "assembly_gflops": float(np.mean([r["asm_gflops"] for r in res])),
                         "matvec_gbs": float(np.mean([r["matvec_gbs"] for r in res])),
                         "iterations": [r["iterations"] for r in res], "frequencies_timed": [r["fi"] for r in res],
                         "all_converged": all(r["converged"] for r in res),
                         "sampled_model": {"value": model["seconds_per_frequency"], "note": f"{model['rows']} rows assembled + 5 zgemv, extrapolated linearly (the round-1 estimate, kept for comparison with the measured figure)"}},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "wall_s": time.perf_counter() - t_begin,
    }
    emit(line)
    return 0


def ride_along(name, fn, world, dev, wait_s=90.0):
    """Run one side block (row-sharded parity, config 3 / 4 / 5) after the headline measurement: its failure must not take the
    headline JSON line with it.  An exception becomes {"error": ...}.  With several ranks the outcome is agreed on with one
    all-reduce; a rank that failed ALONE cannot be joined by the others (they sit in a collective of the block), so it waits
    `wait_s` for them and then ends the job with a non-zero exit instead of leaving it hanging until the driver's limit."""
    err = None
    try:
        out = fn()
    except Exception as e:
        import traceback

        traceback.print_exc(file=sys.stderr)
        err = f"{type(e).__name__}: {e}"
        out = {"error": err}
    if world > 1:
        import torch
        import torch.distributed as dist

        flag = torch.tensor([1.0 if err else 0.0], device=dev)
        work = dist.all_reduce(flag, op=dist.ReduceOp.MAX, async_op=True)
        deadline = time.monotonic() + wait_s
        while not work.is_completed():
            if err and time.monotonic() > deadline:
                print(f"bench.py: {name} failed on this rank only ({err}); the other ranks did not arrive within {wait_s:.0f} s",
                      file=sys.stderr, flush=True)
                os._exit(1)
            time.sleep(0.005)
        work.wait()
        if float(flag.item()) > 0 and not err:
            out = {"error": f"{name} failed on another rank", "this_rank": out}
    return out


def run_sharded_parity(ctx, rank, world, dev):
    """Row-sharded parity inside the bench job (the driver's scaling lease is the only place with several GPUs): the committed
    golden fixtures tests/golden/ico2_ka0p2.npz and ico2_ka6.npz (oracle matrix, right-hand side, GMRES solution and iteration
    count, frozen by tests/golden/make_golden.py) against this job's ranks -- slab entries, solution, iteration / restart counts.
    Collective; returns the block on rank 0.  No oracle import."""
    import torch
    import torch.distributed as dist

    from math_audio_b200 import bem

    out = {}
    for name in ("ico2_ka0p2", "ico2_ka6"):
        gp = ROOT / "tests" / "golden" / f"{name}.npz"
        if not gp.exists():
            continue
        g = np.load(gp)
        mesh = generate_icosphere_mesh(float(g["a"]), int(g["sub"]))
        ph = PhysicsParams.from_wave_number(float(g["k"]))
        system = bem.build_tbem_system_with_beta(mesh, ph, complex(g["beta"]), ctx=ctx)
        r0, r1 = system.matrix.local_rows
        A = system.matrix.rows()
        ent = float(np.max(np.abs(A - g["A"][r0:r1]) / np.abs(g["A"][r0:r1]))) if r1 > r0 else 0.0
        sol = bem.gmres(bem.DenseOperator(system), g["b"], bem.GmresConfig(max_iterations=1000, restart=50, tolerance=1e-10))
        dx = float(np.linalg.norm(sol.x - g["x"]) / np.linalg.norm(g["x"]))
        same = 1.0 if (sol.iterations == int(g["iterations"]) and sol.restarts == int(g["restarts"]) and sol.converged) else 0.0
        t = torch.tensor([ent, dx, -same], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[name] = {"max_entry_rel_err": float(t[0]), "x_rel_err": float(t[1]), "iterations": sol.iterations,
                     "golden_iterations": int(g["iterations"]), "counts_equal_on_every_rank": bool(t[2] <= -1.0),
                     "ok": bool(t[0] < 1e-10 and t[1] < 1e-8 and t[2] <= -1.0)}
    out["ranks"] = world
    return out if rank == 0 else None


def block_jacobi_leg(bem, op, b, cfg, world, dev, block_size, x_plain, plain_iterations, plain_solve_s, centers=None):
    """gmres_preconditioned with the device-built block-Jacobi preconditioner (AdditiveSchwarzPreconditioner, overlap 0,
    math-solvers/src/preconditioners/schwarz.rs) on rank-aligned contiguous diagonal blocks of about `block_size` DOFs, next to
    the plain solve of the same system: set-up time, iterations, solve time, independent true residual, distance to the plain
    solution.  Collective; every rank returns the block."""
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    n = op.num_rows()
    t_cl = time.perf_counter()
    if centers is None:
        parts, kind = bem.schwarz_partition_aligned(n, world, block_size), "contiguous rank-aligned blocks"
    else:  # frequency independent, once per mesh: compact Voronoi clusters inside every rank's row block
        parts, kind = bem.voronoi_subdomains(centers[:n], world, block_size), "rank-aligned Voronoi clusters of the collocation points"
    t_cl = time.perf_counter() - t_cl
    barrier()
    t0 = time.perf_counter()
    pre = bem.AdditiveSchwarzPreconditioner.from_operator(op, subdomains=parts)
    barrier()
    t1 = time.perf_counter()
    sol = bem.gmres_preconditioned(op, pre, b, cfg)
    barrier()
    t2 = time.perf_counter()
    st = pre.stats()
    res = float(np.linalg.norm(op.apply(sol.x) - b) / np.linalg.norm(b))
    dx = float(np.linalg.norm(sol.x - x_plain) / np.linalg.norm(x_plain)) if x_plain is not None else None
    tim = torch.tensor([t1 - t0, t2 - t1, st["factor_ms"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tim, op=dist.ReduceOp.MAX)
    pre.close()
    return {"preconditioner": f"block-Jacobi = AdditiveSchwarzPreconditioner, overlap 0 (schwarz.rs), {kind}; "
                              "explicit inverse blocks applied as one batched block GEMV per Arnoldi step",
            "clustering_s_host_once_per_mesh": t_cl,
            "blocks": int(st["num_subdomains"]), "block_size_max": int(st["max_size"]),
            "inverse_mb_per_gpu": st["inverse_bytes"] / 1e6, "setup_s": float(tim[0]), "setup_ms_device": float(tim[2]),
            "iterations": sol.iterations, "restarts": sol.restarts, "converged": sol.converged,
            "preconditioned_residual": sol.residual, "independent_true_residual": res, "solve_s": float(tim[1]),
            "setup_plus_solve_s": float(tim[0] + tim[1]), "plain_iterations": plain_iterations, "plain_solve_s": plain_solve_s,
            "x_rel_diff_vs_plain": dx, "host_buffers": True}


def run_config4(ctx, rank, world, dev, reps=2):
    """BASELINE.json configs[3] / the north-star target inside the driver-run bench: 121 680-element rigid
    geodesic sphere, ka = 16, adaptive beta, row-sharded over all ranks, one assemble + GMRES(50, 1e-10)
    solve timed end to end (device-resident inputs).  Parity against COMMITTED oracle rows
    (tests/golden/config4_rows.npz, made by tests/golden/make_golden_large.py): 32 sampled rows at the
    256 nearest + every 32nd column, and the whole-row dot products with a seeded vector; the oracle is
    not imported here.  Collective: every rank calls it; returns the block on rank 0."""
    import torch
    import torch.distributed as dist

    from math_audio_b200 import bem
    from math_audio_b200.incident import IncidentField

    gpath = ROOT / "tests" / "golden" / "config4_rows.npz"
    wl = workload("sphere121k")
    mesh = wl["mesh"]
    n = mesh.num_dofs
    r0, r1 = ctx.partition(n)
    nloc = r1 - r0
    free_b, _tot = torch.cuda.mem_get_info(dev)
    need = 16.0 * nloc * n + 52 * 16.0 * n + (1 << 30)
    ok = torch.tensor([1.0 if free_b > need else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if ok.item() < 1.0:
        return {"skipped": f"needs {need / 1e9:.0f} GB per GPU at {world} GPUs"} if rank == 0 else None
    ka, ph, beta = physics_for(wl, 0)
    staged = bem.StagedMesh(mesh, ctx)
    b = IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)  # rigid: TbemSystem.rhs == 0
    b_dev = torch.from_numpy(b).to(dev)
    x_dev = torch.zeros(n, dtype=torch.complex128, device=dev)
    y_dev = torch.zeros(n, dtype=torch.complex128, device=dev)
    cfg = bem.GmresConfig(max_iterations=GMRES_MAX_CYCLES, restart=GMRES_RESTART, tolerance=GMRES_TOL)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    system, best = None, None
    for rep in range(reps):  # rep 0 also allocates the slab and the Krylov workspace
        barrier()
        t0 = time.perf_counter()
        system = bem.build_tbem_system_with_beta(staged, ph, beta, ctx=ctx, rows=(r0, r1), reuse=system, fetch_rhs=False)
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        op = bem.DenseOperator(system)
        sol = bem.gmres_device(op, b_dev.data_ptr(), x_dev.data_ptr(), cfg)
        barrier()
        t2 = time.perf_counter()
        st_a, st_s = system.matrix.assembly_stats(), system.matrix.solver_stats()
        tim = torch.tensor([t2 - t0, t1 - t0, st_a["far_ms"], st_a["total_ms"], st_s["matvec_ms"] / max(1, st_s["matvecs"])],
                           dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tim, op=dist.ReduceOp.MAX)
        cur = dict(s=float(tim[0]), asm_s=float(tim[1]), far_ms=float(tim[2]), asm_ms=float(tim[3]), mv_ms=float(tim[4]), sol=sol,
                   launches=int(st_a["total_launches"] + st_s["kernel_launches"]), solve_s=float(tim[0] - tim[1]))
        if rep > 0 and (best is None or cur["s"] < best["s"]):
            best = cur
    best = best or cur
    op = bem.DenseOperator(system)
    # independent residual through the operator boundary
    bem.apply_device(op, x_dev.data_ptr(), y_dev.data_ptr())
    res = float((torch.linalg.vector_norm(b_dev - y_dev) / torch.linalg.vector_norm(b_dev)).item())
    # the same system through gmres_preconditioned with the device-built block-Jacobi preconditioner (SURVEY 8f rank 4)
    bj = None
    if not os.environ.get("BENCH_NO_BLOCK_JACOBI"):
        try:
            bj = block_jacobi_leg(bem, op, b, cfg, world, dev, int(os.environ.get("BENCH_BJ_BLOCK", "256")), x_dev.cpu().numpy(),
                                  best["sol"].iterations, best["solve_s"],
                                  centers=None if os.environ.get("BENCH_BJ_CONTIGUOUS") else mesh.center)
        except Exception as e:  # the north-star block must survive a failure of the side leg
            bj = {"error": f"{type(e).__name__}: {e}"}
    block = {"workload": wl["name"], "description": wl["desc"], "n_elements": int(n), "n_gpus": world, "rows_per_gpu": int(nloc),
             "matrix_gb_per_gpu": 16.0 * nloc * n / 1e9}
    errs = torch.zeros(3, dtype=torch.float64, device=dev)
    checked = 0
    if gpath.exists():
        g = np.load(gpath)
        xp = np.random.default_rng(1234)
        xprobe = xp.standard_normal(n) + 1j * xp.standard_normal(n)  # == config4_probe_vector() of the generator
        xp_dev = torch.from_numpy(xprobe).to(dev)
        bem.apply_device(op, xp_dev.data_ptr(), y_dev.data_ptr())
        yh = y_dev.cpu().numpy()
        xn = float(np.linalg.norm(xprobe))
        for i, r in enumerate(g["rows"]):
            r = int(r)
            errs[2] = max(float(errs[2]), abs(yh[r] - g["rowdot"][i]) / (float(g["rownorm"][i]) * xn))
            if r0 <= r < r1:
                row = system.matrix.rows(r, r + 1)[0]
                ref = g["vals"][i]
                got = row[g["cols"][i]]
                errs[0] = max(float(errs[0]), float(np.max(np.abs(got - ref) / np.abs(ref))))
                errs[1] = max(float(errs[1]), float(np.max(np.abs(got - ref)) / np.max(np.abs(ref))))
                checked += 1
    cnt = torch.tensor([float(checked)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(errs, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    del system
    if rank != 0:
        return None
    far_flop = (FLOP_PER_QP * wl["nq"] + FLOP_PER_PAIR) * nloc * (n - 1)
    mv_bytes = 16.0 * nloc * n + 16.0 * n + 16.0 * nloc
    fp64_nominal = 148 * 64 * 2 * 1.965e9 / 1e12
    hbm_peak, _src = load_peaks()
    sol = best["sol"]
    block.update({
        "s_per_frequency": best["s"], "assemble_s": best["asm_s"], "assemble_ms_device": best["asm_ms"], "far_ms": best["far_ms"],
        "far_tflops_per_gpu": far_flop / (best["far_ms"] * 1e-3) / 1e12, "far_frac_of_nominal_fp64": far_flop / (best["far_ms"] * 1e-3) / 1e12 / fp64_nominal,
        "matvec_ms": best["mv_ms"], "matvec_gbs_per_gpu": mv_bytes / (best["mv_ms"] * 1e-3) / 1e9,
        "matvec_frac_of_measured_hbm": mv_bytes / (best["mv_ms"] * 1e-3) / 1e9 / hbm_peak,
        "iterations": sol.iterations, "restarts": sol.restarts, "residual": sol.residual, "converged": sol.converged,
        "independent_residual": res, "gpu_launches": best["launches"],
        "parity": ({"golden": "tests/golden/config4_rows.npz (oracle rows, committed)", "rows_checked": int(cnt.item()),
                    "max_entry_rel_err": float(errs[0]), "max_row_normwise_err": float(errs[1]), "max_rowdot_err": float(errs[2]),
                    "bar": 1e-10} if gpath.exists() else {"skipped": "tests/golden/config4_rows.npz missing"}),
    })
    if bj is not None:
        block["block_jacobi"] = bj
    return block


def run_precond_config2(ctx, dev):
    """Block-Jacobi on the headline workload's mesh (icosphere(5), one GPU) at the two ends of its frequency range that need
    the most iterations: plain gmres() against gmres_preconditioned() with 64-DOF diagonal blocks (the icosphere's element
    order is hierarchical, 64 consecutive elements = one level-2 parent triangle).  The headline `value` stays the plain solve."""
    from math_audio_b200 import bem
    from math_audio_b200.incident import IncidentField

    a = 0.1
    mesh = generate_icosphere_mesh(a, 5)
    n = mesh.num_dofs
    cfg = bem.GmresConfig(max_iterations=GMRES_MAX_CYCLES, restart=GMRES_RESTART, tolerance=GMRES_TOL)
    out = {"workload": "sphere20k", "n_elements": int(n), "block_size": 64, "cases": []}
    system = None
    for ka in (2.0, 8.0):
        ph = PhysicsParams.from_wave_number(ka / a)
        beta, _ = ph.burton_miller_beta_adaptive(a)
        system = bem.build_tbem_system_with_beta(mesh, ph, beta, ctx=ctx, reuse=system)
        b = system.rhs_full() + IncidentField.plane_wave_z().compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
        op = bem.DenseOperator(system)
        bem.gmres(op, b, bem.GmresConfig(1, 2, GMRES_TOL))
        t0 = time.perf_counter()
        plain = bem.gmres(op, b, cfg)
        t_plain = time.perf_counter() - t0
        leg = block_jacobi_leg(bem, op, b, cfg, 1, dev, 64, plain.x, plain.iterations, t_plain)
        leg["ka"] = ka
        out["cases"].append(leg)
    system.matrix.close()
    return out


def run_precond_sweep(mesh, cases, b_extra, cfg, e2e_plain_s, background):
    """The headline frequencies once more through the C sweep API (host buffers) with bemb200_sweep_set_block_jacobi: every
    frequency is solved by gmres_preconditioned + block-Jacobi (320 blocks of 64 DOFs) rebuilt from its own matrix."""
    from math_audio_b200.sweep import Sweep

    # with the solve halved the pipelined schedule is bound by its polite one-block-per-SM background assembly (measured
    # 100.5 ms per frequency): assembly at full speed and the solve back to back is the faster schedule here
    mode = os.environ.get("BENCH_PC_SWEEP", "sequential")
    overlap = mode != "sequential"
    if mode.startswith("bg"):
        background = int(mode[2:])
    sw = Sweep(mesh, 0, 0, 1, None, overlap=overlap, background_blocks_per_sm=background)
    sw.set_block_jacobi(mesh.num_dofs // 64)
    jobs = [(ph, beta, b_extra(ph, beta)) for ph, beta in cases]
    sw.solve_all(jobs[:2], cfg)  # untimed: buffers, workspaces
    t0 = time.perf_counter()
    got = sw.solve_all(jobs, cfg)
    dt = (time.perf_counter() - t0) / len(jobs)
    sw.close()
    return {"s_per_frequency_e2e": dt, "plain_s_per_frequency_e2e": e2e_plain_s, "iterations": [g[0].iterations for g in got],
            "all_converged": all(g[0].converged for g in got), "max_preconditioned_residual": max(g[0].residual for g in got),
            "schedule": ("bemb200_sweep_* with host buffers, " + ("assembly of f+1 underneath the preconditioned solve of f"
                                                                   if overlap else "assembly and preconditioned solve back to back"))}


def run_config5(ctx, dev):
    """BASELINE.json configs[4] inside the driver-run bench (one GPU): icosphere(5), ka = 2, adaptive beta, 32 plane-wave
    directions on the Fibonacci sphere; ONE batched GMRES(50, 1e-10) over the FP64 tensor-core block matvec (reference
    semantics: 32 independent gmres() calls).  Parity against the COMMITTED oracle record tests/golden/config5_rhs32.npz
    (per-right-hand-side iteration / restart counts of 32 oracle solves, LAPACK solutions of columns 0, 13, 31).  No oracle import."""
    import torch

    from math_audio_b200 import bem
    from math_audio_b200.incident import IncidentField
    from math_audio_b200.mesh import fibonacci_directions

    a, ka, nrhs = 0.1, 2.0, 32
    mesh = generate_icosphere_mesh(a, 5)
    n = mesh.num_dofs
    ph = PhysicsParams.from_wave_number(ka / a)
    beta, _ = ph.burton_miller_beta_adaptive(a)
    system = bem.build_tbem_system_with_beta(mesh, ph, beta, ctx=ctx)
    op = bem.DenseOperator(system)
    B = np.stack([system.rhs + IncidentField.plane_wave(d).compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
                  for d in fibonacci_directions(nrhs)])
    cfg = bem.GmresConfig(max_iterations=GMRES_MAX_CYCLES, restart=GMRES_RESTART, tolerance=GMRES_TOL)
    bem.gmres_batched(op, B, bem.GmresConfig(1, GMRES_RESTART, GMRES_TOL))  # untimed: allocates the 32 Krylov bases of the batched solver
    X = np.random.default_rng(1).standard_normal((nrhs, n)) + 1j * np.random.default_rng(2).standard_normal((nrhs, n))
    kms = min(bem.apply_block(op, X)[1] for _ in range(3))
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    sols, st = bem.gmres_batched(op, B, cfg)
    torch.cuda.synchronize(dev)
    t_batched = time.perf_counter() - t0
    t0 = time.perf_counter()
    singles = [bem.gmres(op, B[i], cfg) for i in (0, 13, 31)]
    t_single = (time.perf_counter() - t0) / 3
    res = [float(np.linalg.norm(B[i] - op.apply(sols[i].x)) / np.linalg.norm(B[i])) for i in (0, 13, 31)]
    flops = 8.0 * n * n * nrhs
    fp64_nominal = 148 * 64 * 2 * 1.965e9 / 1e12
    block = {"workload": "sphere20k_rhs32", "description": "rigid icosphere(5), 20480 Tri3, ka = 2, 32 plane-wave directions, batched GMRES(50) tol 1e-10",
             "n_elements": int(n), "nrhs": nrhs, "s_per_batch": t_batched, "s_per_rhs": t_batched / nrhs,
             "single_rhs_solve_s": t_single, "speedup_vs_sequential_solves": t_single * nrhs / t_batched,
             "block_matvec": {"kernel": ("zgemm_block_kernel (round-1 kernel, mma.sync m8n8k4 f64 from global fragments)" if os.environ.get("BEMB200_BLOCK_MATVEC") == "legacy"
                                         else "zgemm_streamk_kernel (DMMA.8x8x4 from swizzled shared-memory tiles, cp.async ring, stream-K over 148 CTAs) + block_fixup_kernel"), "ms": kms, "tflops": flops / (kms * 1e-3) / 1e12,
                              "frac_of_nominal_fp64": flops / (kms * 1e-3) / 1e12 / fp64_nominal, "launches": int(st.get("block_matvecs", 0)),
                              "algorithmic_flop_per_launch": flops, "bytes_per_launch": 16.0 * n * n + 32.0 * n * nrhs},
             "iterations": [so.iterations for so in sols], "all_converged": all(so.converged for so in sols),
             "independent_residuals": res,
             "max_dx_vs_single_rhs_device_solve": max(float(np.linalg.norm(sols[i].x - singles[j].x) / np.linalg.norm(singles[j].x))
                                                      for j, i in enumerate((0, 13, 31)))}
    gp = ROOT / "tests" / "golden" / "config5_rhs32.npz"
    if gp.exists():
        g = np.load(gp)
        dx = max(float(np.linalg.norm(sols[int(c)].x - g["x"][j]) / np.linalg.norm(g["x"][j])) for j, c in enumerate(g["x_cols"]))
        same = bool(np.array_equal(np.array([so.iterations for so in sols]), g["iterations"])
                    and np.array_equal(np.array([so.restarts for so in sols]), g["restarts"]))
        block["parity"] = {"golden": "tests/golden/config5_rhs32.npz (32 oracle GMRES solves + LAPACK solutions of 3 columns, committed)",
                           "iteration_and_restart_counts_equal": same, "max_x_rel_err_vs_lapack": dx, "bar_x": 1e-8, "ok": bool(same and dx < 1e-8)}
    else:
        block["parity"] = {"skipped": "tests/golden/config5_rhs32.npz missing"}
    # the same batch as 32 gmres_preconditioned() solves sharing the block-Jacobi preconditioner (320 blocks of 64 DOFs)
    if not os.environ.get("BENCH_NO_BLOCK_JACOBI"):
        try:
            t0 = time.perf_counter()
            pre = bem.AdditiveSchwarzPreconditioner.from_operator(op, n // 64)
            t_setup = time.perf_counter() - t0
            bem.gmres_batched(op, B[:8], bem.GmresConfig(1, 2, GMRES_TOL), precond=pre)  # untimed: first use of the block apply kernel
            t0 = time.perf_counter()
            solp, stp = bem.gmres_batched(op, B, cfg, precond=pre)
            t_pc = time.perf_counter() - t0
            pre.close()
            block["block_jacobi"] = {
                "s_per_batch": t_pc, "setup_s": t_setup, "iterations": [so.iterations for so in solp],
                "all_converged": all(so.converged for so in solp), "block_matvecs": int(stp.get("block_matvecs", 0)),
                "max_x_rel_diff_vs_plain_batch": max(float(np.linalg.norm(solp[i].x - sols[i].x) / np.linalg.norm(sols[i].x)) for i in range(nrhs)),
                "true_residuals": [float(np.linalg.norm(B[i] - op.apply(solp[i].x)) / np.linalg.norm(B[i])) for i in (0, 13, 31)]}
        except Exception as e:
            block["block_jacobi"] = {"error": f"{type(e).__name__}: {e}"}
    system.matrix.close()
    return block


def cabinet_mesh(scale: float):
    """BASELINE.json configs[2] (SURVEY.md 8d row 3): closed 0.32 x 0.44 x 0.64 m Quad4 box, 64 x 88 x 128 subdivisions at
    scale 1 (50 176 elements), piston = full-length velocity BC v = 1 on the front-wall elements within 80 mm of the wall
    centre, rigid elsewhere.  Same construction as tests/golden/make_golden_large.py."""
    from math_audio_b200.mesh import generate_box_mesh_quad

    nx, ny, nz = int(64 * scale), int(88 * scale), int(128 * scale)
    mesh = generate_box_mesh_quad(0.32, 0.44, 0.64, nx, ny, nz)
    front = (np.abs(mesh.center[:, 1] + 0.22) < 1e-9) & (np.hypot(mesh.center[:, 0], mesh.center[:, 2]) < 0.08)
    v = np.zeros((mesh.n_elem, 4), dtype=np.complex128)
    v[front] = 1.0
    mesh.set_velocity_bc(v)
    mesh.bc_len[~front] = 1
    return mesh


def run_config3(ctx, rank, world, dev, reps=2):
    """BASELINE.json configs[2] inside the driver-run bench (2 and 4 GPUs): the 50 176-element Quad4 cabinet with a piston,
    f = 1 kHz, beta = i/k, row-sharded over all ranks: assemble (matrix AND the right-hand side the velocity BC generates) +
    GMRES(50, 1e-10), timed end to end.  Parity against COMMITTED oracle data (tests/golden/make_golden_large.py):
    config3_rows.npz -- 16 sampled rows (entries at the 256 nearest + every 32nd column, whole-row dot products, right-hand-side
    entries) -- and config3_coarse_x.npz -- the 4x-coarsened copy (12 544 elements) assembled and solved in full by this job
    against the oracle's LAPACK solution and GMRES counts.  Collective; returns the block on rank 0.  No oracle import."""
    import torch
    import torch.distributed as dist

    from math_audio_b200 import bem

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    ph = PhysicsParams.new(1000.0, 343.0, 1.21, False)
    beta = ph.burton_miller_beta()
    cfg = bem.GmresConfig(max_iterations=GMRES_MAX_CYCLES, restart=GMRES_RESTART, tolerance=GMRES_TOL)
    block = {"workload": "cabinet50k", "description": "closed Quad4 box 64x88x128 = 50 176 elements, piston velocity BC, f = 1 kHz, beta = i/k",
             "n_gpus": world}
    # ---- the 4x-coarsened copy, solved in full and compared with the oracle's solution ---------------------------------
    gx = ROOT / "tests" / "golden" / "config3_coarse_x.npz"
    if gx.exists():
        g = np.load(gx)
        mesh_c = cabinet_mesh(0.5)
        sys_c = bem.build_tbem_system_with_beta(mesh_c, ph, beta, ctx=ctx)
        b_c = sys_c.rhs_full()
        sol = bem.gmres(bem.DenseOperator(sys_c), b_c, cfg)
        e = allmax([float(np.linalg.norm(b_c - g["b"]) / np.linalg.norm(g["b"])), float(np.linalg.norm(sol.x - g["x"]) / np.linalg.norm(g["x"])),
                    0.0 if (sol.iterations == int(g["iterations"]) and sol.restarts == int(g["restarts"]) and sol.converged) else 1.0])
        block["coarse_copy"] = {"n_elements": int(mesh_c.num_dofs), "golden": "tests/golden/config3_coarse_x.npz (oracle LAPACK solution, committed)",
                                "rhs_rel_err": e[0], "x_rel_err": e[1], "iterations": sol.iterations, "golden_iterations": int(g["iterations"]),
                                "counts_equal_on_every_rank": e[2] == 0.0, "bar_x": 1e-8, "ok": bool(e[0] < 1e-10 and e[1] < 1e-8 and e[2] == 0.0)}
        sys_c.matrix.close()
        del sys_c
    # ---- the full-size problem ------------------------------------------------------------------------------------------
    mesh = cabinet_mesh(1.0)
    n = mesh.num_dofs
    r0, r1 = ctx.partition(n)
    nloc = r1 - r0
    free_b, _tot = torch.cuda.mem_get_info(dev)
    need = 16.0 * nloc * n + 52 * 16.0 * n + (1 << 30)
    if allmax([0.0 if free_b > need else 1.0])[0] > 0.0:
        block["skipped"] = f"needs {need / 1e9:.0f} GB per GPU at {world} GPUs"
        return block if rank == 0 else None
    staged = bem.StagedMesh(mesh, ctx)
    x_dev = torch.zeros(n, dtype=torch.complex128, device=dev)
    y_dev = torch.zeros(n, dtype=torch.complex128, device=dev)
    system, best = None, None
    for rep in range(reps):
        barrier()
        t0 = time.perf_counter()
        system = bem.build_tbem_system_with_beta(staged, ph, beta, ctx=ctx, rows=(r0, r1), reuse=system, fetch_rhs=False)
        b = system.rhs_full()  # the piston's right-hand side: local rows D2H, the other ranks' rows over the communicator
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        sol = bem.gmres(bem.DenseOperator(system), b, cfg)
        barrier()
        t2 = time.perf_counter()
        st_a, st_s = system.matrix.assembly_stats(), system.matrix.solver_stats()
        tim = allmax([t2 - t0, t1 - t0, st_a["far_ms"], st_a["total_ms"], st_s["matvec_ms"] / max(1, st_s["matvecs"])])
        cur = dict(s=tim[0], asm_s=tim[1], far_ms=tim[2], asm_ms=tim[3], mv_ms=tim[4], sol=sol, special=int(st_a["special_pairs"]),
                   launches=int(st_a["total_launches"] + st_s["kernel_launches"]))
        if rep > 0 and (best is None or cur["s"] < best["s"]):
            best = cur
    best = best or cur
    sol = best["sol"]
    op = bem.DenseOperator(system)
    x_dev.copy_(torch.from_numpy(sol.x))
    b_dev = torch.from_numpy(b).to(dev)
    bem.apply_device(op, x_dev.data_ptr(), y_dev.data_ptr())
    res = float((torch.linalg.vector_norm(b_dev - y_dev) / torch.linalg.vector_norm(b_dev)).item())
    gpath = ROOT / "tests" / "golden" / "config3_rows.npz"
    errs, checked = [0.0, 0.0, 0.0, 0.0], 0
    if gpath.exists():
        g = np.load(gpath)
        xp = np.random.default_rng(1234)
        xprobe = xp.standard_normal(n) + 1j * xp.standard_normal(n)
        bem.apply_device(op, torch.from_numpy(xprobe).to(dev).data_ptr(), y_dev.data_ptr())
        yh = y_dev.cpu().numpy()
        xn = float(np.linalg.norm(xprobe))
        bscale = float(np.max(np.abs(g["rhs"])))
        for i, r in enumerate(g["rows"]):
            r = int(r)
            errs[2] = max(errs[2], abs(yh[r] - g["rowdot"][i]) / (float(g["rownorm"][i]) * xn))
            errs[3] = max(errs[3], abs(b[r] - g["rhs"][i]) / bscale)
            if r0 <= r < r1:
                got, ref = system.matrix.rows(r, r + 1)[0][g["cols"][i]], g["vals"][i]
                errs[0] = max(errs[0], float(np.max(np.abs(got - ref) / np.abs(ref))))
                errs[1] = max(errs[1], float(np.max(np.abs(got - ref)) / np.max(np.abs(ref))))
                checked += 1
    errs = allmax(errs)
    cnt = torch.tensor([float(checked)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    # the same system through gmres_preconditioned + block-Jacobi on rank-aligned Voronoi clusters (SURVEY 8f rank 4)
    bj = None
    if not os.environ.get("BENCH_NO_BLOCK_JACOBI"):
        try:
            bj = block_jacobi_leg(bem, op, b, cfg, world, dev, int(os.environ.get("BENCH_BJ_BLOCK", "256")), sol.x, sol.iterations,
                                  best["s"] - best["asm_s"], centers=mesh.center)
        except Exception as e:
            bj = {"error": f"{type(e).__name__}: {e}"}
    del system
    if rank != 0:
        return None
    if bj is not None:
        block["block_jacobi"] = bj
    far_flop = (FLOP_PER_QP * 16 + FLOP_PER_PAIR) * nloc * (n - 1)
    mv_bytes = 16.0 * nloc * n + 16.0 * n + 16.0 * nloc
    fp64_nominal = 148 * 64 * 2 * 1.965e9 / 1e12
    hbm_peak, _src = load_peaks()
    block.update({
        "n_elements": int(n), "rows_per_gpu": int(nloc), "matrix_gb_per_gpu": 16.0 * nloc * n / 1e9,
        "s_per_frequency": best["s"], "assemble_s": best["asm_s"], "assemble_ms_device": best["asm_ms"], "far_ms": best["far_ms"],
        "special_pairs_rank0": best["special"],
        "far_tflops_per_gpu": far_flop / (best["far_ms"] * 1e-3) / 1e12, "far_frac_of_nominal_fp64": far_flop / (best["far_ms"] * 1e-3) / 1e12 / fp64_nominal,
        "matvec_ms": best["mv_ms"], "matvec_gbs_per_gpu": mv_bytes / (best["mv_ms"] * 1e-3) / 1e9,
        "matvec_frac_of_measured_hbm": mv_bytes / (best["mv_ms"] * 1e-3) / 1e9 / hbm_peak,
        "iterations": sol.iterations, "restarts": sol.restarts, "residual": sol.residual, "converged": sol.converged,
        "independent_residual": res, "gpu_launches": best["launches"],
        "parity": ({"golden": "tests/golden/config3_rows.npz (oracle rows, committed)", "rows_checked": int(cnt.item()),
                    "max_entry_rel_err": errs[0], "max_row_normwise_err": errs[1], "max_rowdot_err": errs[2], "max_rhs_err": errs[3],
                    "bar": 1e-10} if gpath.exists() else {"skipped": "tests/golden/config3_rows.npz missing"}),
    })
    return block


DUMP_SEED = 2024
DUMP_MATRIX_BYTES = 32 << 20  # the sampled matrix rows; with x and the GMRES figures well under 64 MB for every workload


def dump_outputs(out_dir: Path, x: np.ndarray, sol: dict, matrix) -> None:
    """--dump-outputs: the arrays a caller of the timed path receives for its last step, as float64 .npy files.
    x.npy                 GMRES solution, n x [re, im]
    gmres.npy             [iterations, restarts, residual, converged]
    matrix_rows.npy       rows of the assembled system matrix, k x n x [re, im]: a fixed seeded sample of this rank's
                          rows (all of them when they fit in DUMP_MATRIX_BYTES)
    matrix_row_index.npy  the k row indices of matrix_rows.npy, ascending"""
    n = x.shape[0]
    r0, r1 = matrix.local_rows
    k = min(r1 - r0, max(1, DUMP_MATRIX_BYTES // (16 * n)))
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(np.arange(r0, r1), size=k, replace=False))
    a = np.stack([matrix.rows(int(r), int(r) + 1)[0] for r in rows])
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "x.npy", x.view(np.float64).reshape(n, 2))
    np.save(out_dir / "gmres.npy", np.array([sol["iterations"], sol["restarts"], sol["residual"], sol["converged"]], dtype=np.float64))
    np.save(out_dir / "matrix_rows.npy", a.view(np.float64).reshape(k, n, 2))
    np.save(out_dir / "matrix_row_index.npy", rows.astype(np.float64))


# -------------------------------------------------------------------------------------------
# native arm
# -------------------------------------------------------------------------------------------
def run_native(args):
    import torch
    import torch.distributed as dist

    from math_audio_b200 import bem
    from math_audio_b200 import dist as bdist
    from math_audio_b200.incident import IncidentField

    rank, local_rank, world = bdist.env_rank()
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for --gpus N > 1 launch with torchrun (one process per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libbemb200 has no CPU fallback (use --impl reference for the CPU arm)")
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
        os.environ.pop("NCCL_DEBUG")  # keep NCCL's version banner off stdout: ONE JSON line only
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        bdist.init_process_group("nccl")
    nccl_id = None
    if world > 1:
        nccl_id = bdist.broadcast_bytes(bem.Context.nccl_unique_id() if rank == 0 else None, 128, 0, device=dev)
    from math_audio_b200.sweep import SweepDriver

    # two streams: the solve (HBM-bound ZGEMV + Arnoldi) gets the higher priority, the assembly of
    # the NEXT frequency (FP64-bound) runs underneath it on the second stream
    s_solve = torch.cuda.Stream(device=dev, priority=-1)
    s_asm = torch.cuda.Stream(device=dev, priority=0)
    wl = workload(args.workload)
    mesh = wl["mesh"]
    n = mesh.num_dofs
    # schedule: on one GPU the FP64 assembly of frequency f+1 hides under the HBM-bound solve of f (101.0 against 103.9 ms
    # sequential); from two GPUs on the solver owns the GPU -- the persistent fused GMRES kernel with its sharded
    # Gram-Schmidt and one peer-memory exchange per iteration -- and assembly and solve run back to back (2 GPUs: 57.3
    # against 61.7 ms pipelined, profiles/r02e_bench_2gpu*.json)
    overlap = (world < 2) if args.schedule == "auto" else (args.schedule == "pipelined")
    if args.no_overlap:
        overlap = False
    driver = SweepDriver(mesh, local_rank, rank, world, nccl_id, solve_stream=s_solve.cuda_stream,
                         assembly_stream=s_asm.cuda_stream, overlap=overlap, background_blocks_per_sm=args.background)
    ctx = driver.ctx_solve
    nsteps = args.warmup + args.steps
    inc = IncidentField.plane_wave_z()
    cfg = bem.GmresConfig(max_iterations=GMRES_MAX_CYCLES, restart=GMRES_RESTART, tolerance=GMRES_TOL)
    r0, r1 = ctx.partition(n)
    nloc = r1 - r0

    # ---- device-resident inputs ------------------------------------------------------------
    b_host, b_dev, cases = [], [], []
    for s in range(nsteps):
        ka, ph, beta = physics_for(wl, s)
        b = inc.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)  # rigid: TbemSystem.rhs == 0
        b_host.append(b)
        b_dev.append(torch.from_numpy(b).to(dev))
        cases.append((ph, beta))
    x_dev = torch.zeros(n, dtype=torch.complex128, device=dev)
    torch.cuda.synchronize(dev)
    dbg = os.environ.get("BENCH_DEBUG")

    def make_solve_device(offset):
        def solve_device(i, system, op):
            s = offset + i
            tq = time.perf_counter()
            sol = bem.gmres_device(op, b_dev[s].data_ptr(), x_dev.data_ptr(), cfg)
            if dbg:
                print(f"[value rank {rank}] step {s}: gmres wall {(time.perf_counter() - tq) * 1e3:.2f} ms it {sol.iterations}", file=sys.stderr)
            return dict(ka=float(wl["ka"][freq_index(s, len(wl["ka"]))]), fi=freq_index(s, len(wl["ka"])), iterations=sol.iterations,
                        restarts=sol.restarts, residual=sol.residual, converged=sol.converged)
        return solve_device

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def fused_phase_times():
        """device-side phase clocks of the persistent fused GMRES kernel accumulated since the last call (rank-local):
        (kernel ms, ms inside its ZGEMV phases, ms inside its reduction rounds, number of rounds = Arnoldi steps)"""
        import ctypes as C

        from math_audio_b200 import _capi

        f = _capi.lib().bemb200_debug_fused_times
        f.restype = None
        a, b_, c, d = C.c_double(), C.c_double(), C.c_double(), C.c_ulonglong()
        f(C.byref(a), C.byref(b_), C.byref(c), C.byref(d))
        return a.value, b_.value, c.value, int(d.value)

    driver.run(cases[: args.warmup], cfg, make_solve_device(0))
    fused_phase_times()  # reset
    driver.asm_stats.clear()
    driver.sol_stats.clear()
    boosts_warm = driver.boosts
    # start the clock sampler BEFORE the barrier: nvidia-smi's start-up stalls CUDA calls for
    # ~100 ms and must not leak into any rank's timed region
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(s_asm)     # the first timed kernel is an assembly kernel on the assembly stream
    if driver.trace is not None:
        driver.trace.clear()
    sols = driver.run(cases[args.warmup:], cfg, make_solve_device(args.warmup))
    ev1.record(s_solve)   # the last one is the solution update on the solve stream
    boosts_timed = driver.boosts - boosts_warm
    fused_ph = fused_phase_times()
    if driver.trace is not None and rank == 0:
        for lab, ci, ts in sorted(driver.trace, key=lambda r: r[2]):
            print(f"[value trace] {ts * 1e3:9.2f} ms  {lab:12s} case {ci}", file=sys.stderr)
    barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # the last timed case was assembled into the driver's buffer (steps - 1) % 2 and solved into x_dev
        dump_outputs(Path(args.dump_outputs), x_dev.cpu().numpy(), sols[-1], driver.buffers[(args.steps - 1) % 2].matrix)
    stats = []
    for i, sd in enumerate(sols):
        stats.append(dict(sd, **{f"asm_{k}": v for k, v in driver.asm_stats[i].items()},
                          **{f"sol_{k}": v for k, v in driver.sol_stats[i].items()}))

    # ---- end-to-end through the host-buffer API -----------------------------------------------
    # the drop-in calls a user of the reference makes, once per frequency, with HOST buffers:
    # build_tbem_system_with_beta(host mesh) [stage H2D, rhs D2H] + gmres(host b) [b H2D, x D2H]
    e2e_steps = max(1, args.steps)
    x_pinned = torch.empty(n, dtype=torch.complex128).pin_memory().numpy()
    sys_e2e = None
    _, ph_w, beta_w = physics_for(wl, 0)
    sys_e2e = bem.build_tbem_system_with_beta(mesh, ph_w, beta_w, ctx=ctx, reuse=sys_e2e)  # untimed warm-up of the host path
    sys_e2e.rhs_full()
    bem.gmres(bem.DenseOperator(sys_e2e), b_host[0], bem.GmresConfig(max_iterations=1, restart=2, tolerance=GMRES_TOL))
    h2d = d2h = 0
    e2e_far_ms = []  # the FP64 far kernel in the foreground (the e2e calls are sequential: nothing overlaps it)
    barrier()
    t0 = time.perf_counter()
    for s in range(args.warmup, args.warmup + e2e_steps):
        ph, beta = cases[s]
        sys_e2e = bem.build_tbem_system_with_beta(mesh, ph, beta, ctx=ctx, reuse=sys_e2e)
        b = sys_e2e.rhs_full() + inc.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
        sol = bem.gmres(bem.DenseOperator(sys_e2e), b, cfg)
        x_pinned[:] = sol.x
        e2e_far_ms.append(sys_e2e.matrix.assembly_stats()["far_ms"])
        if dbg:
            print(f"[e2e rank {rank}] step {s}: cumulative {(time.perf_counter() - t0) * 1e3:.2f} ms", file=sys.stderr)
        h2d += driver.staged.nbytes_host + b.nbytes
        d2h += nloc * 16 + n * 16 + sol.x.nbytes
    barrier()
    e2e_seq_s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_seq_s, op=dist.ReduceOp.MAX)
    # ---- the same frequencies through the sweep API of the C ABI (bemb200_sweep_*, what a Rust / C caller of a sweep uses): the
    # mesh is staged once by the sweep object, every frequency passes HOST buffers -- physics, the incident right-hand side
    # computed on the host, b H2D inside bemb200_gmres, TbemSystem.rhs and x D2H -- and the library pipelines the assembly of
    # frequency f + 1 underneath the solve of f (1 GPU) or runs them back to back with the fused solver (2 GPUs on)
    from math_audio_b200.sweep import Sweep

    nid2 = None
    if world > 1:
        nid2 = bdist.broadcast_bytes(bem.Context.nccl_unique_id() if rank == 0 else None, 128, 0, device=dev)
    csw = Sweep(mesh, local_rank, rank, world, nid2, overlap=overlap, background_blocks_per_sm=args.background)
    e2e_cases = cases[args.warmup: args.warmup + e2e_steps]

    def run_csweep(cs):
        outs = []

        def sub(c):
            ph, beta = c
            csw.submit(ph, beta, inc.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta), cfg)

        for c in cs[:2]:
            sub(c)
        for i in range(len(cs)):
            sol, _st, _b = csw.next()
            x_pinned[:] = sol.x
            outs.append(sol)
            if i + 2 < len(cs):
                sub(cs[i + 2])
        return outs

    run_csweep(e2e_cases[:2])  # untimed: buffers of the sweep object, first use of its solver workspace
    barrier()
    t0 = time.perf_counter()
    sols_e2e = run_csweep(e2e_cases)
    barrier()
    e2e_s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    assert all(so.converged for so in sols_e2e)
    h2d_sw = n * 16                 # b
    d2h_sw = nloc * 16 + n * 16     # TbemSystem.rhs (local rows; the other ranks' rows arrive over NVLink) + x
    e2e_schedule = ("bemb200_sweep_* (C ABI) with host buffers: mesh staged once at sweep creation; per frequency the incident right-hand "
                    "side is computed on the host, b goes up, TbemSystem.rhs and x come down; "
                    + ("assembly of frequency f+1 overlaps the solve of f" if overlap else "assembly and solve back to back"))
    csw.close()

    # ---- the ZGEMV alone (nothing else on the GPU): 20 launches through the operator boundary
    iso_ms = None
    try:
        op_iso = bem.DenseOperator(sys_e2e)
        y_dev = torch.zeros(n, dtype=torch.complex128, device=dev)
        tot, cnt = 0.0, 0
        for it in range(23):
            bem.apply_device(op_iso, b_dev[0].data_ptr(), y_dev.data_ptr())
            if it >= 3:
                st_iso = sys_e2e.matrix.solver_stats()
                tot += st_iso["matvec_ms"]
                cnt += st_iso["matvecs"]
        iso_ms = tot / max(1, cnt)
    except Exception as e:  # diagnostics only
        print(f"isolated zgemv measurement failed: {e}", file=sys.stderr)

    # ---- row-sharded parity against the committed golden fixtures (several GPUs exist only in the driver's scaling lease)
    sharded_parity = ride_along("sharded_parity", lambda: run_sharded_parity(ctx, rank, world, dev), world, dev) if world > 1 else None
    # ---- 32 right-hand sides on the tensor-core block matvec (config 5) ride along on one GPU
    config5 = None
    if world == 1 and not os.environ.get("BENCH_NO_CONFIG5"):
        try:
            config5 = run_config5(ctx, dev)
        except Exception as e:  # the headline line must survive a failure of the side block
            config5 = {"error": f"{type(e).__name__}: {e}"}
    # ---- block-Jacobi preconditioned solves of the same mesh (SURVEY 8f rank 4) ride along on one GPU
    precond = None
    if world == 1 and not os.environ.get("BENCH_NO_BLOCK_JACOBI") and not os.environ.get("BENCH_NO_CONFIG5"):
        try:
            precond = run_precond_config2(ctx, dev)
            precond["sweep"] = run_precond_sweep(mesh, e2e_cases, lambda ph, beta: inc.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta),
                                                 cfg, float(e2e_s.item()), args.background)
        except Exception as e:
            precond = {"error": f"{type(e).__name__}: {e}"}
    # ---- the Quad4 cabinet (config 3) rides along at 2 and 4 GPUs (the sizes BASELINE.json quotes it on)
    config3 = None
    if (world in (2, 4) or os.environ.get("BENCH_CONFIG3")) and not os.environ.get("BENCH_NO_CONFIG3"):
        try:
            del sys_e2e, op_iso
            driver.buffers = [None, None]
        except Exception:
            pass
        config3 = ride_along("config3", lambda: run_config3(ctx, rank, world, dev), world, dev)
    # ---- the north-star target (config 4) rides along whenever all 8 GPUs of the box are in the job
    config4 = None
    if (world >= 8 or os.environ.get("BENCH_CONFIG4")) and not os.environ.get("BENCH_NO_CONFIG4"):
        try:
            del sys_e2e, op_iso
            driver.buffers = [None, None]
        except Exception:
            pass
        config4 = ride_along("config4", lambda: run_config4(ctx, rank, world, dev), world, dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- report -------------------------------------------------------------------------------
    K = args.steps
    value = total_ms * 1e-3 / K
    hbm_peak, peak_src = load_peaks()
    mv_ms = sum(st["sol_matvec_ms"] for st in stats)
    mv_cnt = sum(st["sol_matvecs"] for st in stats)
    mv_bytes = 16.0 * nloc * n + 16.0 * n + 16.0 * nloc      # per launch on this rank (SURVEY 8d)
    mv_gbs = mv_bytes * mv_cnt / (mv_ms * 1e-3) / 1e9 if mv_ms > 0 else 0.0
    far_ms = sum(st["asm_far_ms"] for st in stats)
    asm_ms = sum(st["asm_total_ms"] for st in stats)
    far_flop = (FLOP_PER_QP * wl["nq"] + FLOP_PER_PAIR) * nloc * (n - 1)   # every off-diagonal pair once through the 13-pt rule
    far_tf = far_flop * K / (far_ms * 1e-3) / 1e12 if far_ms > 0 else 0.0
    fp64_meas = ctx.measure_fp64_peak()
    fp64_nominal = 148 * 64 * 2 * 1.965e9 / 1e12
    launches = int(sum(st["asm_total_launches"] + st["sol_kernel_launches"] for st in stats))
    fused_used = all(st["sol_kernel_launches"] == 1 for st in stats)  # the persistent kernel is ONE launch per solve
    traffic = None
    tp = ROOT / "profiles" / "ncu_traffic.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get(f"zgemv_{wl['name']}_{world}")
        except Exception:
            traffic = None
    # FP64 far kernel.  `achieved` = the kernel as a foreground launch (the sequential host-buffer calls of this very run time it
    # with nothing beside it); in the pipelined sweep it deliberately runs as a polite one-block-per-SM grid underneath the
    # solve, which `in_sweep` reports (there its duration is hidden, not minimised).
    fg_ms = float(np.mean(e2e_far_ms)) if e2e_far_ms else None
    fa = {"kernel": "far_kernel<13>", "bound": "fp64", "peak": fp64_nominal, "unit": "TFLOP/s",
          "peak_measured_dfma": fp64_meas, "algorithmic_flop_per_launch": far_flop,
          "peak_source": "nominal 148 SM x 64 DFMA/clk x 2 x 1.965 GHz; measured = register-resident DFMA loop on this GPU"}
    in_sweep = {"achieved": far_tf, "frac": far_tf / fp64_nominal, "avg_launch_ms": far_ms / K, "share_of_step": far_ms / total_ms,
                "assembly_share_of_step": asm_ms / total_ms,
                "note": (f"background grid ({148 * args.background} persistent blocks pulling work items from a device counter) underneath the solve of the previous frequency"
                         if overlap else "foreground launch of the timed sweep (sequential schedule)")}
    if fg_ms:
        fg_tf = far_flop / (fg_ms * 1e-3) / 1e12
        fa.update(achieved=fg_tf, frac=fg_tf / fp64_nominal, frac_of_measured=(fg_tf / fp64_meas if fp64_meas > 0 else None),
                  avg_launch_ms=fg_ms, launches=len(e2e_far_ms),
                  note="foreground launches of this run (the sequential host-buffer calls; nothing overlaps the kernel)", in_sweep=in_sweep)
        mhz = (clocks or {}).get("sm_mhz")
        if mhz:
            # the board runs this run's sustained FP64 load under its power cap: the same kernel against the DFMA peak at the SM
            # clock nvidia-smi reported during the timed sweep (burst launches at 1.96 GHz: profiles/r01e_ncu_far_summary.json)
            pk = 148 * 64 * 2 * mhz * 1e6 / 1e12
            fa["at_sampled_clock"] = {"sm_mhz": mhz, "peak": pk, "frac": fg_tf / pk}
    else:
        fa.update(in_sweep, frac_of_measured=(far_tf / fp64_meas if fp64_meas > 0 else None))
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": total_ms / K, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": base_config(wl),
        "run": {"rows_per_gpu": int(nloc), "matrix_bytes_per_gpu": int(16 * nloc * n), "parallelism": f"row-block x{world}",
                "schedule": ("sweep pipeline: assembly of frequency f+1 on a second stream/buffer overlaps the solve of f"
                             if overlap else "sequential: assemble then solve"),
                "exchange": ("single GPU" if world == 1 else
                             ("persistent fused GMRES kernel per rank: Krylov vector and reduction partials through peer memory (flag-in-data)"
                              if fused_used else
                              ("peer memory: ZGEMV epilogue stores A v into every rank's work vector (NVLink), consumer waits on in-data flags"
                               if ctx.peer_exchange_active() and not overlap else "NCCL all-gather of A v per Arnoldi step"))),
                "solver": ("gmres_fused_kernel (one launch per solve)" if fused_used else "zgemv_kernel + one Gram-Schmidt kernel per Arnoldi step"),
                "frequencies_timed": [st["fi"] for st in stats]},
        "roofline": {"kernel": "zgemv_kernel", "bound": "hbm", "achieved": mv_gbs, "peak": hbm_peak, "unit": "GB/s",
                     "frac": mv_gbs / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                     "launches": int(mv_cnt), "avg_launch_ms": mv_ms / max(1, mv_cnt), "share_of_step": mv_ms / total_ms,
                     "frac_of_nominal_8TBs": mv_gbs / 8000.0,
                     "isolated": (None if not iso_ms else {"avg_launch_ms": iso_ms, "achieved": mv_bytes / (iso_ms * 1e-3) / 1e9,
                                                           "frac": mv_bytes / (iso_ms * 1e-3) / 1e9 / hbm_peak,
                                                           "note": "same kernel with nothing else running (no overlapped assembly)"})},
        "roofline_assembly": fa,
        "e2e": {"value": float(e2e_s.item()), "unit": UNIT, "h2d_bytes_per_step": int(h2d_sw),
                "d2h_bytes_per_step": int(d2h_sw), "steps": e2e_steps, "schedule": e2e_schedule,
                "sequential_value": float(e2e_seq_s.item()),
                "sequential": {"schedule": "drop-in calls one after the other: build_tbem_system_with_beta(HOST mesh, re-staged every frequency) then gmres(host b)",
                               "h2d_bytes_per_step": int(h2d // e2e_steps), "d2h_bytes_per_step": int(d2h // e2e_steps)}},
        "gpu_launches": launches,
        "clocks": clocks,
        "gmres": {"matvecs_per_step": mv_cnt / K, "iterations": [st["iterations"] for st in stats],
                  "matvecs": [st["sol_matvecs"] for st in stats],
                  "all_converged": all(st["converged"] for st in stats),
                  "max_residual": max(st["residual"] for st in stats)},
        "breakdown_ms_per_step": {"assembly": asm_ms / K, "far_kernel": far_ms / K, "matvec": mv_ms / K,
                                  "wall": total_ms / K, "boosted_assemblies": int(boosts_timed),
                                  "note": "kernel times are per-kernel CUDA-event durations; with the sweep pipeline assembly overlaps the solve, so they do not add up to wall"},
    }
    if fused_used and fused_ph[3] > 0:
        tot, mvp, rnd, nr = fused_ph
        line["fused_kernel"] = {"kernel_ms_per_step": tot / K, "zgemv_phase_ms_per_step": mvp / K, "reduction_round_ms_per_step": rnd / K,
                                "arnoldi_steps": nr, "non_matvec_us_per_arnoldi_step": (tot - mvp) / nr * 1e3,
                                "reduction_round_us_per_arnoldi_step": rnd / nr * 1e3,
                                "note": "device-side clocks (%globaltimer) of CTA 0 on rank 0 inside gmres_fused_kernel over the timed solves; waiting for slower CTAs or ranks counts as non-matvec time"}
    if sharded_parity is not None:
        line["sharded_parity"] = sharded_parity
    if config5 is not None:
        line["config5"] = config5
    if precond is not None:
        line["block_jacobi"] = precond
    if config3 is not None:
        line["config3"] = config3
    if config4 is not None:
        line["config4"] = config4
    if world == 1 and not args.no_cpu_baseline:
        hint = {st["fi"]: st["sol_matvecs"] for st in stats}
        cs = cpu_sample(wl, args.warmup, 12.0, hint)
        line["cpu_baseline"] = {
            "value": cs["seconds_per_frequency"], "unit": UNIT, "cores": cs["threads"], "kind": "port",
            "sample": (f"oracle port: {cs['rows']} of {n} rows assembled ({cs['asm_s']:.1f} s/frequency extrapolated) + zgemv on that slab "
                       f"({cs['matvec_s'] * 1e3:.1f} ms/matvec extrapolated) x {cs['matvecs']} matvecs at ka={cs['ka']:.3f}; {cs['src']}"),
            "assembly_gflops": cs["asm_gflops"], "matvec_gbs": cs["matvec_gbs"]}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    # ONE JSON line on stdout: everything else any library prints (NCCL banner, warnings) is sent
    # to stderr by pointing fd 1 at fd 2 and keeping a private handle on the real stdout.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="sphere20k_sweep64")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--background", type=int, default=2, help="blocks/SM of the background assembly kernel in the sweep pipeline")
    ap.add_argument("--no-overlap", action="store_true", help="do not overlap assembly(f+1) with solve(f)")
    ap.add_argument("--schedule", choices=["auto", "pipelined", "sequential"], default="auto",
                    help="auto: pipelined sweep on 1 GPU, sequential (persistent fused solver) from 2 GPUs on")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (native arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native arm")
    if args.warmup < 3 and args.impl == "native":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        return run_reference(args)
    return run_native(args)


if __name__ == "__main__":
    sys.exit(main())
