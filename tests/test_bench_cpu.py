"""CPU checks of bench.py's reference arm and of the committed large-configuration fixtures
(tests/golden/make_golden_large.py)."""
import json
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"
sys.path.insert(0, str(GOLD))

from make_golden_large import exact_dot  # noqa: E402  (the summation rowdot_fsum.npz was made with)


def _run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, env=e, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "bench.py must print exactly ONE JSON line on stdout"
    return json.loads(lines[0])


def test_reference_arm_runs_complete_frequencies():
    """--impl reference runs COMPLETE frequencies (all rows assembled, GMRES to 1e-10 on the CPU) and reports a
    value that fits inside its own wall time (the driver's fits_in_driver_run check)."""
    line = _run_bench("--impl", "reference", "--workload", "sphere1k", "--steps", "3", "--warmup", "1")
    assert line["impl"] == "reference" and line["unit"] == "s/frequency" and line["higher_is_better"] is False
    assert line["steps"] == 3 and line["steps_requested"] == 3
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["all_converged"]
    assert len(cb["iterations"]) == 3 and all(20 <= it <= 200 for it in cb["iterations"])
    assert line["value"] * line["steps"] <= line["wall_s"]
    assert line["e2e"] == {"value": line["value"], "unit": "s/frequency", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_respects_its_budget():
    line = _run_bench("--impl", "reference", "--workload", "sphere1k", "--steps", "50", "--warmup", "0",
                      env={"BENCH_REF_BUDGET_S": "0.5"})
    assert line["steps"] == 2 and line["steps_requested"] == 50  # never fewer than two complete frequencies


def test_bench_rejects_no_steps_and_a_dump_of_the_reference_arm(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "out")]):
        p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "sphere1k", *args], capture_output=True, text=True, timeout=300)
        assert p.returncode == 2 and p.stdout == "" and "error:" in p.stderr, args
    assert not (tmp_path / "out").exists()


def test_both_arms_share_the_config_object():
    sys.path.insert(0, str(ROOT))
    import bench

    wl = bench.workload("sphere1k")
    a, b = bench.base_config(wl), bench.base_config(wl)
    assert a == b and a["workload"] == "sphere1k" and a["n_elements"] == 1280
    src = (ROOT / "bench.py").read_text()
    assert src.count('"config": base_config(wl)') == 2  # native and reference line


def test_config4_golden_rows_match_the_oracle():
    """The committed rows of the 121 680-element configuration are what the oracle computes today (two of the 32)."""
    from math_audio_b200.mesh import generate_geodesic_sphere_mesh
    from math_audio_b200.types import PhysicsParams
    from oracle import oracle as orc

    g = np.load(GOLD / "config4_rows.npz")
    mesh = generate_geodesic_sphere_mesh(float(g["a"]), int(g["nu"]))
    assert mesh.num_dofs == int(g["n"]) == 121680
    ph = PhysicsParams.from_wave_number(float(g["k"]))
    beta, _ = ph.burton_miller_beta_adaptive(float(g["a"]))
    assert abs(beta - complex(g["beta"])) == 0.0
    rng = np.random.default_rng(1234)
    xprobe = rng.standard_normal(mesh.num_dofs) + 1j * rng.standard_normal(mesh.num_dofs)
    rowdot = np.load(GOLD / "rowdot_fsum.npz")["config4"]
    for i in (5, 31):
        r = int(g["rows"][i])
        A, _, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=r, row_end=r + 1)
        assert np.array_equal(A[0, g["cols"][i]], g["vals"][i])
        assert exact_dot(A[0], xprobe) == rowdot[i]
        assert r in g["cols"][i][:256]  # the self term is among the nearest columns


@pytest.mark.parametrize("tag", ["0p25", "2", "8"])
def test_config2_solution_fixture_is_consistent(tag):
    p = GOLD / f"config2_x_ka{tag}.npz"
    if not p.exists():
        pytest.skip("fixture not generated (tests/golden/make_golden_large.py config2)")
    g = np.load(p)
    assert g["x"].shape == (20480,) and g["x"].dtype == np.complex128
    assert float(g["gmres_vs_lu"]) < 1e-8 and float(g["residual"]) < 1e-10
    assert 20 <= int(g["iterations"]) <= 300


def test_config3_golden_rows_match_the_oracle():
    """bench.py builds the same cabinet as the fixture generator, and the committed rows of the 50 176-element Quad4 box are what
    the oracle computes today (entries, whole-row dot product and the piston's right-hand-side term of two of the 16 rows)."""
    sys.path.insert(0, str(ROOT))
    import bench
    from math_audio_b200.types import PhysicsParams
    from oracle import oracle as orc

    g = np.load(GOLD / "config3_rows.npz")
    mesh = bench.cabinet_mesh(1.0)
    assert mesh.num_dofs == int(g["n"]) == 50176
    assert int(np.count_nonzero(np.abs(mesh.bc_val[:, 0]) > 0)) > 100  # the piston
    ph = PhysicsParams.new(1000.0, 343.0, 1.21, False)
    beta = ph.burton_miller_beta()
    assert abs(beta - complex(g["beta"])) == 0.0 and ph.wave_number == float(g["k"])
    rng = np.random.default_rng(1234)
    xprobe = rng.standard_normal(mesh.num_dofs) + 1j * rng.standard_normal(mesh.num_dofs)
    assert np.max(np.abs(g["rhs"])) > 0.0
    rowdot = np.load(GOLD / "rowdot_fsum.npz")["config3"]
    for i in (1, len(g["rows"]) - 1):
        r = int(g["rows"][i])
        A, rhs, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=r, row_end=r + 1)
        assert np.array_equal(A[0, g["cols"][i]], g["vals"][i])
        assert exact_dot(A[0], xprobe) == rowdot[i] and rhs[0] == g["rhs"][i]


def test_config3_and_config5_solution_fixtures_are_consistent():
    g = np.load(GOLD / "config3_coarse_x.npz")
    assert int(g["n"]) == 12544 and g["x"].shape == (12544,) and g["b"].shape == (12544,)
    assert float(g["gmres_vs_lu"]) < 1e-8 and float(g["residual"]) < 1e-10 and int(g["iterations"]) == 195
    g = np.load(GOLD / "config5_rhs32.npz")
    assert g["iterations"].shape == (32,) and g["restarts"].shape == (32,) and g["x"].shape == (3, 20480)
    assert list(g["x_cols"]) == [0, 13, 31] and float(np.max(g["residual"])) < 1e-10
    assert 90 <= int(g["iterations"].min()) and int(g["iterations"].max()) <= 100


def test_side_blocks_are_wired_into_the_native_line():
    """The configurations BASELINE.json names beside the headline ride along in the driver-run bench: config 5 on one GPU,
    config 3 at 2 and 4 GPUs, config 4 at 8 -- and none of them imports the oracle."""
    src = (ROOT / "bench.py").read_text()
    for key in ('line["config3"]', 'line["config4"]', 'line["config5"]'):
        assert key in src
    for fn in ("run_config3", "run_config4", "run_config5", "run_sharded_parity"):
        body = src[src.index(f"def {fn}("):]
        body = body[: body.index("\ndef ", 10)]
        assert not re.search(r"^\s*(from\s+oracle|import\s+oracle)", body, re.M), fn


def test_reference_arm_under_torchrun_only_rank0_works():
    """Launched like the repo's own arm for N > 1 (one process per GPU): rank 0 alone runs and prints the line, the other
    ranks exit 0 at once without output and without touching a process group."""
    e = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29541")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "sphere1k",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, env=e, timeout=120)
    assert p.returncode == 0 and p.stdout.strip() == ""
    line = _run_bench("--impl", "reference", "--gpus", "2", "--workload", "sphere1k", "--steps", "2", "--warmup", "1",
                      env={"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29541"})
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["steps"] == 2 and line["gpu_launches"] == 0
