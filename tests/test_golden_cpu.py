"""CPU suite: the oracle against the committed golden fixtures, the host-side logic, and the
C-ABI library surface (load + exported symbols; no compute without a GPU)."""
import ctypes as C
import os
import re
from pathlib import Path

import numpy as np
import pytest

from math_audio_b200.mesh import (fibonacci_directions, generate_box_mesh_quad, generate_geodesic_sphere_mesh,
                                  generate_icosphere_mesh, generate_sphere_mesh)
from math_audio_b200.types import PhysicsParams

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"


def reference_tree():
    """The Rust math-audio source tree this port restates, if MATH_AUDIO_REFERENCE names a checkout of it.  It is not part of
    this repository, so the checks that read it skip without one."""
    p = os.environ.get("MATH_AUDIO_REFERENCE")
    return Path(p) if p and Path(p).is_dir() else None


NO_REFERENCE = "set MATH_AUDIO_REFERENCE to a checkout of the math-audio Rust sources"


def box_piston_mesh():
    mesh = generate_box_mesh_quad(0.32, 0.44, 0.64, 4, 6, 8)
    front = (np.abs(mesh.center[:, 1] + 0.22) < 1e-9) & (np.hypot(mesh.center[:, 0], mesh.center[:, 2]) < 0.12)
    v = np.zeros((mesh.n_elem, 4), dtype=np.complex128)
    v[front] = 1.0
    mesh.set_velocity_bc(v)
    mesh.bc_len[~front] = 1
    return mesh, front


# ---- oracle vs frozen fixtures -------------------------------------------------------
@pytest.mark.parametrize("name", ["ico1_ka0p5", "ico2_ka0p2", "ico2_ka6"])
def test_oracle_matches_golden_sphere(orc, name):
    g = np.load(GOLD / f"{name}.npz")
    mesh = generate_icosphere_mesh(float(g["a"]), int(g["sub"]))
    A, rhs0, nq = orc.assemble(mesh, float(g["k"]), complex(g["beta"]))
    # same compiler flags, same libm => bit-identical; allow 1e-13 for a different libm
    assert np.max(np.abs(A - g["A"]) / np.abs(g["A"])) < 1e-13
    assert nq == int(g["nqp"])
    x, info = orc.gmres(g["A"], g["b"], max_iterations=1000, restart=50, tolerance=1e-10)
    assert info["iterations"] == int(g["iterations"]) and info["restarts"] == int(g["restarts"])
    assert np.linalg.norm(x - g["x"]) / np.linalg.norm(g["x"]) < 1e-12
    # independent check of the frozen solution (LAPACK)
    xl = np.linalg.solve(g["A"], g["b"])
    assert np.linalg.norm(g["x"] - xl) / np.linalg.norm(xl) < 1e-8


def test_oracle_matches_golden_box(orc):
    g = np.load(GOLD / "box_4x6x8_piston.npz")
    mesh, front = box_piston_mesh()
    assert (front == g["front"]).all() and front.sum() == 4
    A, rhs, nq = orc.assemble(mesh, float(g["k"]), complex(g["beta"]))
    assert np.max(np.abs(A - g["A"])) / np.max(np.abs(g["A"])) < 1e-13
    assert np.max(np.abs(rhs - g["rhs"])) / np.max(np.abs(g["rhs"])) < 1e-13
    assert np.abs(g["rhs"]).min() > 0  # every row sees the piston (tbem.rs:164,342-344)


def test_oracle_row_blocks_equal_full(orc):
    mesh = generate_icosphere_mesh(0.1, 1)
    ph = PhysicsParams.from_wave_number(5.0)
    beta = ph.burton_miller_beta_scaled(4.0)
    A, rhs, _ = orc.assemble(mesh, ph.wave_number, beta)
    A1, r1, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=0, row_end=33)
    A2, r2, _ = orc.assemble(mesh, ph.wave_number, beta, row_begin=33, row_end=80)
    assert (np.vstack([A1, A2]) == A).all() and (np.concatenate([r1, r2]) == rhs).all()
    # thread count must not change a single bit (rows are independent)
    A3, _, _ = orc.assemble(mesh, ph.wave_number, beta, nthreads=1)
    assert (A3 == A).all()


def test_oracle_eval_elements_and_dof_permutation(orc):
    mesh = generate_icosphere_mesh(0.1, 1)
    ph = PhysicsParams.from_wave_number(5.0)
    beta = ph.burton_miller_beta()
    A, _, _ = orc.assemble(mesh, ph.wave_number, beta)
    perm = np.random.default_rng(7).permutation(mesh.n_elem).astype(np.uint32)
    mesh.dof[:] = perm
    Ap, _, _ = orc.assemble(mesh, ph.wave_number, beta)
    # A[dof_i, dof_j] = entry of (element i, element j)
    assert (Ap[np.ix_(perm, perm)] == A).all()
    # evaluation elements are skipped as sources and as field elements (tbem.rs:128-131,152-155)
    mesh = generate_icosphere_mesh(0.1, 1)
    mesh.is_eval[-5:] = 1
    assert mesh.num_dofs == 75
    Ae, _, _ = orc.assemble(mesh, ph.wave_number, beta)
    assert Ae.shape == (75, 75)
    # NB the dg_dn_sign heuristic still reads the first 100 elements, evaluation or not
    assert np.max(np.abs(Ae - A[:75, :75])) == 0.0


# ---- host logic --------------------------------------------------------------------------
def test_physics_params_beta_variants():
    ph = PhysicsParams.new(1000.0, 343.0, 1.21, False)  # types.rs:745-751
    assert abs(ph.wave_number - 2 * np.pi * 1000 / 343) < 1e-10 and abs(ph.wave_length - 0.343) < 1e-10 and ph.tau == 1.0
    k = ph.wave_number
    assert ph.burton_miller_beta() == complex(0, 1 / k)
    assert ph.burton_miller_beta_scaled(4.0) == complex(0, 4 / k)
    assert ph.burton_miller_beta_optimal(0.01) == complex(0, 1 / (k + 100.0))
    a = 0.1
    for ka, scale in [(0.49, 1.0), (0.5, 4.0), (1.19, 4.0), (1.2, 8.0), (1.79, 8.0), (1.8, 16.0), (8.0, 16.0)]:
        p = PhysicsParams.from_wave_number(ka / a)
        b, s = p.burton_miller_beta_adaptive(a)
        assert s == scale and abs(b - complex(0, scale / p.wave_number)) < 1e-15
    pin = PhysicsParams.new(100.0, 343.0, 1.21, True)
    assert pin.tau == -1.0 and pin.burton_miller_beta() == 0 and pin.burton_miller_beta_adaptive(1.0) == (0j, 1.0)


def test_mesh_generators_counts():
    assert generate_sphere_mesh(0.1, 32, 32).n_elem == 1984  # config 1 (SURVEY 8d)
    m = generate_icosphere_mesh(0.1, 3)
    assert m.n_elem == 1280 and m.n_nodes == 642
    g = generate_geodesic_sphere_mesh(1.0, 6)
    assert g.n_elem == 20 * 36 and g.n_nodes == 10 * 36 + 2
    assert np.abs(np.linalg.norm(g.nodes, axis=1) - 1).max() < 1e-12 and g.meta["n_flipped"] == 0
    # class-I geodesic with nu = 2^s has the icosphere's element count
    assert generate_geodesic_sphere_mesh(1.0, 4).n_elem == generate_icosphere_mesh(1.0, 2).n_elem
    b = generate_box_mesh_quad(0.32, 0.44, 0.64, 4, 6, 8)
    assert b.n_elem == 2 * (4 * 6 + 4 * 8 + 6 * 8) and (b.etype == 4).all()
    assert b.meta["n_flipped"] == 0 and ((b.normal * b.center).sum(1) > 0).all()  # outward winding
    assert abs(b.area.sum() - 2 * (0.32 * 0.44 + 0.32 * 0.64 + 0.44 * 0.64)) < 1e-12
    d = fibonacci_directions(32)
    assert d.shape == (32, 3) and np.abs(np.linalg.norm(d, axis=1) - 1).max() < 1e-12
    for mm in (m, g, b):
        mm.validate()


def test_incident_rhs_matches_oracle(orc):
    from math_audio_b200.incident import IncidentField

    mesh = generate_icosphere_mesh(0.1, 2)
    ph = PhysicsParams.from_wave_number(12.0)
    beta = ph.burton_miller_beta_scaled(4.0)
    for kind, vec in [(0, [0, 0, 1.0]), (0, [0.6, 0.0, 0.8]), (1, [0.3, 0.1, -0.4])]:
        inc = IncidentField.plane_wave(vec) if kind == 0 else IncidentField.point_source(vec)
        got = inc.compute_rhs_with_beta(mesh.center, mesh.normal, ph, beta)
        ref, pinc = orc.incident_rhs(kind, vec, 1.0, mesh.center, mesh.normal, ph.wave_number, beta)
        assert np.max(np.abs(got - ref)) / np.max(np.abs(ref)) < 1e-13
        assert np.max(np.abs(inc.evaluate_pressure(mesh.center, ph) - pinc)) < 1e-13


# ---- the C-ABI library: loads, exports everything the header declares, fails loudly --------
def test_capi_exports_every_declared_symbol():
    from math_audio_b200 import _capi

    header = (ROOT / "include" / "bemb200.h").read_text()
    declared = set(re.findall(r"\b(bemb200_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 30
    assert declared == set(_capi.SYMBOLS), declared ^ set(_capi.SYMBOLS)
    lib = C.CDLL(str(_capi.LIB_PATH))
    for name in declared:
        assert hasattr(lib, name), name


def test_capi_partition_and_loud_failure_without_gpu():
    from math_audio_b200 import _capi, bem

    lib = _capi.lib()
    for n, p in [(20480, 8), (121680, 8), (10, 3), (5, 8)]:
        covered = []
        for r in range(p):
            b, e = C.c_uint64(), C.c_uint64()
            lib.bemb200_partition(n, p, r, C.byref(b), C.byref(e))
            covered += list(range(b.value, e.value)) if n < 100 else []
            assert b.value <= e.value <= n
        if n < 100:
            assert covered == list(range(n))
    if lib.bemb200_device_count() == 0:
        with pytest.raises(_capi.Bemb200Error) as ei:
            bem.Context(0)
        assert ei.value.code == -2 and "no CPU fallback" in str(ei.value)


def test_rust_shim_matches_the_build_and_the_header():
    """The Rust FFI crate cannot be compiled here (no cargo): keep at least its build recipe and its extern
    block in step with what this repository builds and exports."""
    import re

    from math_audio_b200 import _capi
    from math_audio_b200.build import UNITS

    root = Path(__file__).resolve().parent.parent
    rs = (root / "rust" / "bem-b200-sys" / "build.rs").read_text()
    units = {m.group(1): re.findall(r'"([^"]+)"', m.group(2)) for m in re.finditer(r'\("(\w+\.cu)", &\[(.*?)\]\)', rs)}
    assert units == {k: list(v) for k, v in UNITS.items()}          # same translation units, same per-unit flags
    assert "arch=compute_100a,code=sm_100a" in rs
    lib_rs = (root / "rust" / "bem-b200-sys" / "src" / "lib.rs").read_text()
    declared = set(re.findall(r"pub fn (bemb200_\w+)\(", lib_rs))
    assert declared and declared <= set(_capi.SYMBOLS), declared - set(_capi.SYMBOLS)
    header = (root / "include" / "bemb200.h").read_text()
    for name in declared:
        assert re.search(rf"\b{name}\(", header), name
    # every FFI symbol the safe crate calls is declared by the sys crate
    safe = (root / "rust" / "math-bem-b200" / "src" / "lib.rs").read_text()
    used = set(re.findall(r"\b(bemb200_\w+)\(", safe))
    assert used and used <= declared, used - declared


def test_rust_manifests_resolve_against_the_reference_workspace():
    """Cargo resolves dependencies by PACKAGE name (math-solvers, math-bem) while the code imports the LIB names
    (math_audio_solvers, math_audio_bem); the FFI crate must not depend on the workspace (no cycle), and math-bem must
    not be asked to depend on the GPU crates."""
    import re
    import tomllib

    root = Path(__file__).resolve().parent.parent
    sysm = tomllib.loads((root / "rust" / "bem-b200-sys" / "Cargo.toml").read_text())
    safem = tomllib.loads((root / "rust" / "math-bem-b200" / "Cargo.toml").read_text())
    assert sysm["package"]["name"] == "bem-b200-sys" and sysm["package"]["links"] == "bemb200"
    assert not sysm.get("dependencies")                      # raw FFI: nothing of the workspace, no cycle possible
    deps = safem["dependencies"]
    assert set(deps) == {"bem-b200-sys", "math-solvers", "math-bem", "ndarray", "num-complex"}
    assert deps["bem-b200-sys"]["path"] == "../bem-b200-sys"
    expected = {"math-solvers": "math_audio_solvers", "math-bem": "math_audio_bem"}
    src = (root / "rust" / "math-bem-b200" / "src" / "lib.rs").read_text() + (root / "rust" / "math-bem-b200" / "examples" / "frequency_sweep_b200.rs").read_text()
    reference = reference_tree()
    for pkg, libname in expected.items():
        assert deps[pkg]["path"].endswith(pkg)
        assert re.search(rf"\buse {libname}::", src), libname
        if reference is not None:  # the package / lib names are the reference's own
            ref = reference / pkg / "Cargo.toml"
            m = tomllib.loads(ref.read_text())
            assert m["package"]["name"] == pkg and m["lib"]["name"] == libname
            assert "math-bem-b200" not in ref.read_text() and "bem-b200-sys" not in ref.read_text()
    assert "use bem_b200_sys::" in src and "use math_bem_b200::" in src
    integ = (root / "INTEGRATION.md").read_text()
    assert 'cfg(feature = "b200")' not in integ              # the switch is made by the caller, not inside math-bem


def test_binding_arities_match_the_header():
    """ctypes table (math_audio_b200/_capi.py) and the Rust extern block: same number of arguments as include/bemb200.h."""
    import re

    from math_audio_b200 import _capi

    root = Path(__file__).resolve().parent.parent
    header = re.sub(r"/\*.*?\*/", "", (root / "include" / "bemb200.h").read_text(), flags=re.S)

    def nargs(s):
        s = s.strip()
        return 0 if s in ("", "void") else len([a for a in s.split(",") if a.strip()])

    decl = {m.group(1): nargs(m.group(2)) for m in re.finditer(r"\b(bemb200_\w+)\s*\(([^)]*)\)\s*;", header)}
    assert len(decl) > 40
    for name, (_, argtypes) in _capi.SYMBOLS.items():
        if name in decl:
            assert len(argtypes) == decl[name], (name, len(argtypes), decl[name])
    lib_rs = (root / "rust" / "bem-b200-sys" / "src" / "lib.rs").read_text()
    for m in re.finditer(r"pub fn (bemb200_\w+)\(([^)]*)\)", lib_rs, flags=re.S):
        assert nargs(m.group(2)) == decl[m.group(1)], m.group(1)


def test_rust_imports_resolve_to_public_items_of_the_reference():
    """Every `use math_audio_{bem,solvers}::path::{Items}` of the safe crate and its example names a public item of the reference
    source tree (MATH_AUDIO_REFERENCE).  Without a Rust compiler this is the nearest thing to name resolution the crates get."""
    import re

    ref = reference_tree()
    if ref is None:
        pytest.skip(NO_REFERENCE)
    root = Path(__file__).resolve().parent.parent
    src = (root / "rust" / "math-bem-b200" / "src" / "lib.rs").read_text() + (root / "rust" / "math-bem-b200" / "examples" / "frequency_sweep_b200.rs").read_text()
    crates = {"math_audio_bem": ref / "math-bem" / "src", "math_audio_solvers": ref / "math-solvers" / "src"}
    seen = 0
    for m in re.finditer(r"\buse (math_audio_\w+)((?:::\w+)+)::(\{[^}]*\}|\w+);", src):
        base = crates[m.group(1)]
        mods = m.group(2).strip(":").split("::")
        items = [i.strip() for i in m.group(3).strip("{}").split(",") if i.strip()]
        cand = [base.joinpath(*mods).with_suffix(".rs"), base.joinpath(*mods) / "mod.rs"]
        files = [c for c in cand if c.exists()]
        assert files, (m.group(0), "no such module in the reference")
        text = files[0].read_text()
        for it in items:
            public = re.search(rf"pub (?:fn|struct|enum|trait|type|const) {it}\b", text) or re.search(rf"pub use [^;]*\b{it}\b", text, flags=re.S)
            assert public, (m.group(0), it)
            seen += 1
    assert seen >= 12
    # the two reference calls the example makes with non-trivial argument types
    inc = (ref / "math-bem" / "src" / "core" / "incident.rs").read_text()
    sig = re.search(r"pub fn compute_rhs_with_beta\(\s*&self,\s*element_centers: &(\w+)<f64>,\s*element_normals: &(\w+)<f64>", inc)
    assert sig and sig.group(1) == sig.group(2) == "Array2"
    ex = (root / "rust" / "math-bem-b200" / "examples" / "frequency_sweep_b200.rs").read_text()
    assert "Array2::<f64>::zeros((n, 3))" in ex and "Vec<Array1<f64>>" not in ex
    # tuple structs are addressed by position
    safe = (root / "rust" / "math-bem-b200" / "src" / "lib.rs").read_text()
    for name in re.findall(r"struct (\w+)\([^)]*\);", safe):
        body = re.findall(rf"impl(?: \w+ for)? {name} \{{.*?\n\}}|impl Drop for {name} \{{[^\n]*\}}", safe, flags=re.S)
        for b in body:
            assert not re.search(r"self\.[a-z_]+\b(?!\()", re.sub(r"self\.\d", "", b)) or name not in ("CtxInner", "GpuContext"), (name, b[:120])


def test_oracle_is_test_infrastructure_only():
    """oracle/ is the checker, never the product: nothing under math_audio_b200/ or include/ imports, links or names it; the
    library's dynamic dependencies do not include it; bench.py imports it only inside the two functions of the CPU legs
    (cpu_baseline sample, --impl reference) and __graft_entry__ only in build() (compiling the checker) and smoke()."""
    import ast
    import re
    import subprocess

    from math_audio_b200 import _capi

    root = Path(__file__).resolve().parent.parent

    def oracle_imports(path):
        tree = ast.parse(path.read_text())
        parents = {}
        for node in ast.walk(tree):
            for child in ast.iter_child_nodes(node):
                parents[child] = node
        found = []
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                names = [node.module or ""]
            if any(n == "oracle" or n.startswith("oracle.") for n in names):
                fn = node
                while fn in parents and not isinstance(fn, (ast.FunctionDef, ast.AsyncFunctionDef)):
                    fn = parents[fn]
                found.append(fn.name if isinstance(fn, ast.FunctionDef) else "<module>")
        return found

    for py in (root / "math_audio_b200").rglob("*.py"):
        assert oracle_imports(py) == [], py
    for src in list((root / "math_audio_b200" / "csrc").iterdir()) + list((root / "include").iterdir()):
        if src.is_file():
            assert not re.search(r"\boracle\b|bem_oracle", src.read_text(errors="replace")), src
    needed = subprocess.run(["readelf", "-d", str(_capi.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    assert "NEEDED" in needed and "oracle" not in needed
    assert set(oracle_imports(root / "bench.py")) == {"cpu_sample", "cpu_full_frequency"}
    assert set(oracle_imports(root / "__graft_entry__.py")) == {"build", "smoke"}


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """The drop-in boundary is a C ABI: include/bemb200.h must compile as C99 with pedantic warnings as errors (no C++ in the
    signatures, no torch types), and a C program using it must link against libbemb200.so and get a clean error -- not a crash --
    for a NULL mesh without ever touching a GPU."""
    import subprocess

    from math_audio_b200 import _capi

    root = Path(__file__).resolve().parent.parent
    src = tmp_path / "use_from_c.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "bemb200.h"
static int jacobi(void* user, const double* r, double* z, uint64_t n) { (void)user; memcpy(z, r, 16 * n); return 0; }
int main(void) {
    uint64_t b = 7, e = 7;
    bemb200_partition(10, 4, 1, &b, &e);                 /* [3, 6) */
    bemb200_precond_fn fn = jacobi;                      /* the callback type is a plain C function pointer */
    bemb200_sweep* sw = NULL;
    int rc = bemb200_sweep_create(0, 0, 1, NULL, NULL, 1, 2, &sw);   /* NULL mesh: EINVAL before any device work */
    printf("%llu %llu %d %d\n", (unsigned long long)b, (unsigned long long)e, rc, fn != NULL);
    return (b == 3 && e == 6 && rc == BEMB200_EINVAL && sw == NULL) ? 0 : 1;
}
''')
    exe = tmp_path / "use_from_c"
    libdir = _capi.LIB_PATH.parent
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Wpedantic", "-Werror", "-I", str(root / "include"), str(src), "-o", str(exe),
                    f"-L{libdir}", "-lbemb200", f"-Wl,-rpath,{libdir}"], check=True)
    p = subprocess.run([str(exe)], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr


def test_qualified_reference_paths_in_the_docs_resolve():
    """Every fully qualified `math_audio_bem::...` / `math_audio_solvers::...` path quoted in INTEGRATION.md, DESIGN.md, README.md
    and the Rust sources names a module file and a public item of the reference (MATH_AUDIO_REFERENCE)."""
    import re

    ref = reference_tree()
    if ref is None:
        pytest.skip(NO_REFERENCE)
    root = Path(__file__).resolve().parent.parent
    crates = {"math_audio_bem": ref / "math-bem" / "src", "math_audio_solvers": ref / "math-solvers" / "src"}
    texts = [(root / n).read_text() for n in ("INTEGRATION.md", "DESIGN.md", "README.md")]
    texts += [p.read_text() for p in (root / "rust").rglob("*.rs")]
    seen = set()
    for text in texts:
        for m in re.finditer(r"\b(math_audio_(?:bem|solvers))((?:::[A-Za-z_]\w*)+)", text):
            parts = m.group(2).strip(":").split("::")
            if len(parts) < 2 or (m.group(1), tuple(parts)) in seen:
                continue  # `use crate::{...}` lists and bare crate::Item re-exports are covered by the import test
            seen.add((m.group(1), tuple(parts)))
            mods, item = parts[:-1], parts[-1]
            base = crates[m.group(1)]
            cand = [base.joinpath(*mods).with_suffix(".rs"), base.joinpath(*mods) / "mod.rs"]
            files = [c for c in cand if c.exists()]
            if not files:  # the last component may itself be a module (a `use a::b::c::{...}` prefix)
                cand = [base.joinpath(*parts).with_suffix(".rs"), base.joinpath(*parts) / "mod.rs"]
                assert any(c.exists() for c in cand), m.group(0)
                continue
            src = files[0].read_text()
            ok = (re.search(rf"pub (?:fn|struct|enum|trait|type|const|mod) {item}\b", src)
                  or re.search(rf"pub use [^;]*\b{item}\b", src, flags=re.S))
            assert ok, m.group(0)
    assert len(seen) >= 8


def test_reference_citations_resolve():
    """Every `path/file.rs:line[-line]` citation in the headers, the CUDA sources, the Python / C++ / Rust mirrors, the oracle, the
    tests and the documents names a file of the reference that has that many lines (MATH_AUDIO_REFERENCE).  Parity is checked
    through these citations; a stale one is a wrong map."""
    import re

    ref = reference_tree()
    if ref is None:
        pytest.skip(NO_REFERENCE)
    root = Path(__file__).resolve().parent.parent
    by_name, nlines = {}, {}
    for p in ref.rglob("*.rs"):
        by_name.setdefault(p.name, []).append(p)
    docs = [root / "include" / "bemb200.h", root / "include" / "bemb200.hpp", root / "DESIGN.md", root / "INTEGRATION.md", root / "README.md",
            root / "oracle" / "bem_oracle.cpp", root / "oracle" / "independent" / "bem_numpy.py", root / "bench.py"]
    docs += list((root / "math_audio_b200").glob("*.py")) + list((root / "math_audio_b200" / "csrc").glob("*.cu"))
    docs += list((root / "math_audio_b200" / "csrc").glob("*.h")) + list((root / "rust").rglob("*.rs"))
    docs += list((root / "tests").glob("*.py")) + list((root / "tests" / "cpp").glob("*.cpp")) + list((root / "oracle").glob("*.py"))
    total, bad = 0, []
    for d in docs:
        for m in re.finditer(r"((?:[\w\-]+/)*[\w\-]+\.rs):(\d+)(?:-(\d+))?", d.read_text(errors="replace")):
            path, l0, l1 = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            total += 1
            cands = [p for p in by_name.get(Path(path).name, []) if str(p).endswith("/" + path)]
            for p in cands:
                if p not in nlines:
                    nlines[p] = sum(1 for _ in open(p, errors="replace"))
            if not cands or l0 > l1 or not any(nlines[p] >= l1 for p in cands):
                bad.append((d.name, m.group(0)))
    assert total > 500 and not bad, bad[:10]
