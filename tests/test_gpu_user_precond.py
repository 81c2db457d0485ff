"""gmres_preconditioned with a caller-supplied `Preconditioner` (math-solvers/src/traits.rs:366-371) behind the C ABI:
bemb200_gmres_callback.  The check runs in its own process (tests/drivers/user_precond.py: a caller's Python code runs inside a
library call there); first green run on a B200: profiles/r02zz_user_precond.json."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.gpu
def test_gmres_with_user_preconditioner_callback():
    p = subprocess.run([sys.executable, str(ROOT / "tests" / "drivers" / "user_precond.py")], capture_output=True, text=True, timeout=240)
    assert p.returncode == 0, p.stderr[-3000:]
    out = json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])
    i = out["identity"]
    assert i["converged"] and i["iterations"][0] == i["iterations"][1] and i["restarts"][0] == i["restarts"][1]
    assert i["max_abs_dx"] < 1e-13                                    # the callback only hands the vector back
    assert i["calls"][0] == i["calls"][1] == i["iterations"][0] + i["restarts"][0] + 2   # M^-1 b, one per cycle, one per Arnoldi step
    assert i["true_residual"] < 1e-8
    j = out["jacobi"]
    assert j["converged"] and abs(j["iterations"][0] - j["iterations"][1]) <= 1 and j["x_rel_diff"] < 1e-8 and j["true_residual"] < 1e-8
    b = out["block"]
    assert b["converged"] and b["restarts"] >= 1 and b["true_residual"] < 1e-8
    assert b["calls"] == b["reported_calls"] == b["iterations"] + b["restarts"] + 2
    assert out["guess"] == {"iterations": 0, "converged": True}
    assert out["exception"] == "KeyError: user preconditioner failed" and out["wrong_shape"] == "ValueError"
    assert out["after_failure"]["converged"] and out["after_failure"]["true_residual"] < 1e-8
    assert out["rc_on_nonzero_return"] == -8                          # BEMB200_ECALLBACK


def _build_cpp(tmp_path):
    from math_audio_b200 import _capi

    exe = tmp_path / "test_user_precond"
    libdir = _capi.LIB_PATH.parent
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "test_user_precond.cpp"), "-o", str(exe),
           f"-L{libdir}", "-lbemb200", f"-Wl,-rpath,{libdir}", "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"]
    subprocess.run(cmd, check=True)
    return exe


def test_cpp_user_preconditioner_compiles(tmp_path):
    assert _build_cpp(tmp_path).exists()


@pytest.mark.gpu
def test_cpp_user_preconditioner_on_gpu(tmp_path):
    """bemb200::Preconditioner (include/bemb200.hpp) on the device solver: the C++ twin of the Python wrapper test above."""
    out = subprocess.run([str(_build_cpp(tmp_path))], capture_output=True, text=True, timeout=240)
    assert out.returncode == 0 and "PASS" in out.stdout, out.stdout + out.stderr
