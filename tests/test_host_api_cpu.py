"""CPU-only checks of the host layer: the C-ABI library loads and exports every declared symbol, argument
validation mirrors the reference's Cython errors, and the product path fails loudly without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def test_library_exports_every_declared_symbol():
    from astro_sph_tools_b200 import _lib
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "astro_sph_b200.h")).read()
    declared = set(re.findall(r"^(?:int|const char \*)\s*(ast_[a-z0-9_]+)\s*\(", hdr, re.M))
    assert declared == set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.ast_abi_version() == 1 and lib.ast_tile_size() == 32


def test_struct_layout_matches_header():
    from astro_sph_tools_b200 import _lib
    assert C.sizeof(_lib.Project2DParams) == 8 + 6 * 4 + 6 * 8 + 4 * 8 + 8 + 2 * 4
    assert C.sizeof(_lib.Project2DStats) == 4 * 8 + 8 * 4 + 2 * 4         # ... stage_ms[8], reordered, reserved


def test_c_abi_argument_validation_without_gpu():
    """validation happens before any CUDA call, so it can be exercised on a CPU box"""
    from astro_sph_tools_b200 import _lib
    lib = _lib.load()
    p = _lib.Project2DParams()
    need = C.c_size_t(0)
    p.n = 10; p.axis = 5; p.nx = p.ny = 8; p.n_prop = 1; p.x_max = p.y_max = 1.0
    assert lib.ast_project2d_workspace_bytes(C.byref(p), C.byref(need)) == _lib.AST_EINVAL
    assert b"axis" in lib.ast_last_error()
    p.axis = 2; p.kernel_id = 17
    assert lib.ast_project2d_workspace_bytes(C.byref(p), C.byref(need)) == _lib.AST_EINVAL
    p.kernel_id = 0; p.pair_capacity = 1000; p.huge_capacity = 10
    assert lib.ast_project2d_workspace_bytes(C.byref(p), C.byref(need)) == _lib.AST_OK and need.value > 1000 * 16
    with pytest.raises(ValueError):
        _lib.check(_lib.AST_EINVAL)


def test_create_image_validation_mirrors_reference_errors():
    from astro_sph_tools_b200 import CoordinateAxes
    from astro_sph_tools_b200.tools.projections import create_image
    pos = np.zeros((4, 3)); h = np.ones(4); a = np.ones(4)
    args = ((8, 8), 4, CoordinateAxes.Z, 0.0, 1.0, 0.0, 1.0)
    with pytest.raises(ValueError, match="Buffer dtype mismatch, expected 'double' but got 'float'"):
        create_image(pos.astype(np.float32), h, a, *args)
    with pytest.raises(ValueError, match="wrong number of dimensions"):
        create_image(pos[:, 0], h, a, *args)
    with pytest.raises(NotImplementedError, match="self-similar"):
        create_image(pos, h, a, *args, kernel_func=lambda r, hh: r + hh)          # not f(r/h)/h^dim: cannot be tabulated


def test_python_callable_kernels_are_tabulated_on_the_host():
    from astro_sph_tools_b200.tools.projections import kernel_id_of, TabulatedKernel, quartic_spline_kernel
    assert kernel_id_of(quartic_spline_kernel) == "cubic_spline_3d" and kernel_id_of("wendland_c2_2d") == "wendland_c2_2d"
    gauss2d = lambda r, h: np.exp(-(r / h) ** 2) / (np.pi * h ** 2)
    t = kernel_id_of(gauss2d)
    assert isinstance(t, TabulatedKernel) and t.dim == 2 and t.pairs.shape == (TabulatedKernel.N, 2)
    assert kernel_id_of(gauss2d) is t                                             # cached per callable
    top3d = lambda r, h: np.where(r < 2 * h, 3.0 / (32 * np.pi * h ** 3), 0.0)
    assert kernel_id_of(top3d).dim == 3


def test_no_cpu_fallback():
    """run in a child interpreter that sees no CUDA device, so that the check also runs on a machine with a GPU"""
    import subprocess
    import sys
    code = (f"import sys; sys.path.insert(0, {ROOT!r})\n"
            "import numpy as np, pytest\n"
            "from astro_sph_tools_b200 import CoordinateAxes\n"
            "from astro_sph_tools_b200.tools.projections import create_image, quartic_spline_kernel\n"
            "with pytest.raises(RuntimeError, match='no CPU fallback'):\n"
            "    create_image(np.zeros((4, 3)), np.ones(4), np.ones(4), (8, 8), 4, CoordinateAxes.Z, 0.0, 1.0, 0.0, 1.0)\n"
            "with pytest.raises(RuntimeError, match='no CPU fallback'):\n"
            "    quartic_spline_kernel(np.ones(3), np.ones(3))\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr


def test_coordinate_axes_mirror():
    from astro_sph_tools_b200 import CoordinateAxes
    assert [a.value for a in CoordinateAxes] == [0, 1, 2]
    assert [str(a) for a in CoordinateAxes] == ["x", "y", "z"]
    assert CoordinateAxes.from_string(" Y ") is CoordinateAxes.Y
    with pytest.raises(ValueError):
        CoordinateAxes.from_string("w")
    assert CoordinateAxes.X.plane_columns == (1, 2) and CoordinateAxes.Y.plane_columns == (0, 2) and CoordinateAxes.Z.plane_columns == (0, 1)


def test_product_never_imports_oracle():
    """the oracle is test infrastructure: nothing under the package may reference it"""
    pkg = os.path.join(ROOT, "astro-sph-tools_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "liboracle" not in src, f


def test_strip_units_is_a_view_without_importing_unyt():
    from astro_sph_tools_b200.tools.projections import strip_units

    class U(np.ndarray):
        pass

    a = np.arange(6.0).reshape(2, 3).view(U)
    a.units = "Mpc"
    v = strip_units(a)
    assert type(v) is np.ndarray and np.shares_memory(v, a)

    class Q:                      # unyt_quantity-like: only .value
        value = np.ones(3)
    assert np.array_equal(strip_units(Q()), np.ones(3))


def test_host_batch_schedule():
    from astro_sph_tools_b200.tools.projections._engine import batch_cuts
    for n, nb, ramp in [(7001, 8, True), (7001, 8, False), (16777216, 4, True), (10, 16, True), (5, 2, True), (1, 1, True)]:
        bn, cuts = batch_cuts(n, nb, ramp)
        assert cuts[0] == 0 and cuts[-1] == n and all(b > a for a, b in zip(cuts, cuts[1:]))
        sizes = np.diff(cuts)
        assert sizes.max() <= bn
        if ramp and nb >= 2 and n > 4 * nb:
            assert sizes[0] == bn // 4 and sizes[1] == bn // 2         # short first copies
            assert all(sizes[i + 1] <= 2 * sizes[i] + 1 for i in range(len(sizes) - 1))   # each copy hides behind the batch before
    assert batch_cuts(7001, 8, True)[1][:3] == [0, 219, 657] and len(batch_cuts(7001, 8, True)[1]) - 1 == 10


def test_header_is_plain_c(tmp_path):
    """the drop-in boundary is a C ABI: include/astro_sph_b200.h must compile as C99 (no C++ or CUDA types in it)"""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    src = tmp_path / "hdr.c"
    src.write_text('#include "astro_sph_b200.h"\n'
                   "int main(void) { ast_project2d_params a; ast_grid3d_params g; ast_knn_params k; ast_table_params t;\n"
                   "  (void)a; (void)g; (void)k; (void)t; return AST_KNN_FULL_BUILD + AST_TABLE_POW10 + AST_FLAG_PERIODIC; }\n")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                        "-fsyntax-only", str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
