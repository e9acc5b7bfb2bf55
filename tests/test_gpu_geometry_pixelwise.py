"""-m gpu: every voxel and pixel against the float64 oracle, within the per-cell bound of tests/pixel_bound.py and the global
gates, on the geometry the other per-pixel tests leave out (scenes in tests/geometry_scenes.py):
  - periodic boxes whose three sides differ, 3-D, on every path and with and without the spatial pre-ordering: the window
    equal to the box, inside it, and reaching past it; supports wider than half the shortest side; particles at 0 and just
    below L.  Plus the 3-D index work bit-exact against the oracle in such a box;
  - 2-D projections given the 3-component box of the snapshot, on each axis;
  - anisotropic cells (97:1 voxels and 128:1 pixels), where a particle can have a bbox of many short cells and still an h far
    below half a long cell;
  - grid shapes the brick kernel masks at its edges (1-voxel axes, nz < 4, 8k+1, 4k+2);
  - Wendland C2 in 3-D, and tabulated kernels (Python restatements of the built-in kernels) in 2-D and 3-D;
  - one scene that runs every branch of the brick kernel, checked to have run them.
The forced tile and brick paths keep only particles with h >= half of the largest cell side, as everywhere else."""
import functools

import numpy as np
import pytest

from geometry_scenes import (ANISO2, ANISO3, BOX3, BOX3_2D, BOX_WINDOWS, BRANCH_BAND_GAP, BRANCH_GRID, BRANCH_KW, ODD_SHAPES,
                             PLANE, PRESORT_MIN_N, aniso_scene2d, aniso_scene3d, box_scene2d, box_scene3d, branch_scene3d,
                             keep_forced, odd_scene3d, outer_annulus_columns, pad_for_presort, python_kernels, table_scene2d,
                             table_scene3d)
from pixel_bound import assert_pixelwise, envelope2d, envelope3d

pytestmark = pytest.mark.gpu

PATHS2 = {"default": {}, "all_direct": dict(small_max_px=1 << 40), "all_tiled": dict(small_max_px=1, huge_min_tiles=1 << 40),
          "all_global": dict(small_max_px=1, huge_min_tiles=0)}
PATHS3 = {"default": {}, "all_direct": dict(small_max_vox=1 << 40), "all_bricks": dict(small_max_vox=1, huge_min_bricks=1 << 40),
          "all_global": dict(small_max_vox=1, huge_min_bricks=0)}
FORCED = ("all_tiled", "all_global", "all_bricks")
KERNELS = ["cubic_spline_3d", "cubic_spline_2d", "wendland_c2_2d", "wendland_c2_3d"]


def global_gates(m, ref):
    """relative L2 <= 1e-5 and total within 1e-6"""
    assert m.shape == ref.shape and m.dtype == np.float64
    nb = np.linalg.norm(ref)
    assert (np.linalg.norm(m - ref) / nb if nb > 0 else np.linalg.norm(m)) <= 1e-5
    assert abs(m.sum() - ref.sum()) <= 1e-6 * np.abs(ref).sum()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def grid(pos, h, prop, size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, presort="never", **kw):
    import torch
    from astro_sph_tools_b200.tools.projections import Gridder3D
    from astro_sph_tools_b200.tools.projections._kernels import kernel_id_of
    g = Gridder3D(**kw)
    out = g.grid(dev(pos), dev(h), dev(prop), size, lo, hi, kernel_id_of(kernel), periodic, box, presort=presort)
    torch.cuda.synchronize()
    return out.cpu().numpy(), g.last_stats


def project(pos, h, prop, size, axis, bounds, kernel="cubic_spline_3d", periodic=False, box=None, presort="never", **kw):
    import torch
    from astro_sph_tools_b200.tools.projections import Projector2D
    from astro_sph_tools_b200.tools.projections._kernels import kernel_id_of
    eng = Projector2D(**kw)
    out = eng.project(dev(pos), dev(h), dev(prop), size, axis, bounds, kernel_id_of(kernel), periodic, box, presort=presort)
    torch.cuda.synchronize()
    return out.cpu().numpy(), eng.last_stats


# oracle and envelope of a scene, once per scene and particle subset (the envelope is a Python loop over particle images)
_REF = {}


def reference3d(key, pos, h, prop, size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, env_kernel=None):
    import oracle
    if key not in _REF:
        ref = oracle.grid3d(pos, h, prop, size, lo, hi, kernel=kernel, periodic=periodic, box=box)
        env = envelope3d(pos, h, prop, size, lo, hi, env_kernel or kernel, periodic, box)
        _REF[key] = (ref, env)
    return _REF[key]


def reference2d(key, pos, h, prop, size, axis, bounds, kernel="cubic_spline_3d", periodic=False, box=None, env_kernel=None):
    import oracle
    if key not in _REF:
        ref = oracle.project2d(pos, h, prop, size, axis, *bounds, kernel=kernel, periodic=periodic, box=box)
        env = envelope2d(pos, h, prop, size, axis, bounds, env_kernel or kernel, periodic, box)
        _REF[key] = (ref, env)
    return _REF[key]


def subset(path, h, size, lo, hi):
    return keep_forced(h, size, lo, hi) if path in FORCED else np.ones(len(h), dtype=bool)


def check3d(key, path, pos, h, prop, size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, presort="never",
            ref_kernel=None, **kw):
    """gate one grid; kernel may be a Python callable (tabulated on the device), the oracle then runs ref_kernel"""
    keep = subset(path, h, size, lo, hi)
    assert keep.sum() >= 50
    pos, h, prop = pos[keep], h[keep], prop[keep]
    ref, env = reference3d((key, path in FORCED), pos, h, prop, size, lo, hi, ref_kernel or kernel, periodic, box,
                           env_kernel=kernel if callable(kernel) else None)
    g, st = grid(pos, h, prop, size, lo, hi, kernel, periodic, box, presort, **PATHS3[path], **kw)
    assert_pixelwise(g, ref, env, what=f"{key} path {path}: ")
    global_gates(g, ref)
    assert (env > 0).sum() > 0.02 * env.size
    return g, st


def check2d(key, path, pos, h, prop, size, axis, bounds, kernel="cubic_spline_3d", periodic=False, box=None, ref_box=None,
            ref_kernel=None, **kw):
    """ref_box: the in-plane box the oracle gets, written out by the caller (box may be the 3-component box)"""
    keep = subset(path, h, size, (bounds[0], bounds[2]), (bounds[1], bounds[3]))
    assert keep.sum() >= 50
    pos, h, prop = pos[keep], h[keep], prop[keep]
    ref, env = reference2d((key, path in FORCED), pos, h, prop, size, axis, bounds, ref_kernel or kernel, periodic,
                           ref_box if ref_box is not None else box, env_kernel=kernel if callable(kernel) else None)
    m, st = project(pos, h, prop, size, axis, bounds, kernel, periodic, box, **PATHS2[path], **kw)
    assert_pixelwise(m, ref, env, what=f"{key} path {path}: ")
    global_gates(m, ref)
    assert (env > 0).sum() > 0.02 * env.size
    return m, st


# ---- 1. periodic boxes whose sides differ, 3-D -----------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _box3(window):
    pos, h, prop, size, lo, hi = box_scene3d(window)
    return pad_for_presort(pos, h, prop, 1) + (size, lo, hi)


@pytest.mark.parametrize("presort", ["never", "always"])
@pytest.mark.parametrize("path", list(PATHS3))
@pytest.mark.parametrize("window", list(BOX_WINDOWS))
def test_noncubic_periodic_box_3d(window, path, presort):
    pos, h, prop, size, lo, hi = _box3(window)
    assert len(h) >= PRESORT_MIN_N
    _, st = check3d(("box3", window), path, pos, h, prop, size, lo, hi, periodic=True, box=BOX3, presort=presort)
    assert st["reordered"] == (presort == "always")
    if path != "all_direct":
        assert st["n_pairs"] > 0


@pytest.mark.parametrize("window", ["box", "past_low"])
def test_bin3d_bit_exact_in_a_noncubic_box(oracle, window):
    """bbox, class, sorted pairs and the large-h list of ast_bin3d equal oracle.bin3d with the same box"""
    from test_gpu_grid3d import gpu_bin3d
    pos, h, _, size, lo, hi = _box3(window)
    h = h.copy()
    h[5::41] = 0.0; h[7::43] = np.nan
    o = oracle.bin3d(pos, h, size, lo, hi, small_max_vox=20, huge_min_bricks=12, periodic=True, box=BOX3)
    ob = oracle.bbox3d(pos, h, size, lo, hi, periodic=True, box=BOX3)
    g = gpu_bin3d(pos, h, size, lo, hi, True, BOX3, small=20, huge=12)
    assert np.array_equal(g["bbox"], ob)
    assert np.array_equal(g["cls"], o["cls"])
    assert np.array_equal(g["sorted"], o["sorted"])
    assert np.array_equal(g["huge"], o["huge"])
    assert len(o["sorted"]) > 1000 and len(o["huge"]) > 0 and set(np.unique(o["cls"])) == {0, 1, 2, 3}
    # every image index occurs: the shifts along all three axes are exercised
    assert len(np.unique((o["sorted"] >> np.uint64(32)) & np.uint64(31))) == 27


# ---- 2. 3-component boxes in 2-D -------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", list(PATHS2))
@pytest.mark.parametrize("axis", [0, 1, 2])
def test_three_component_box_2d(axis, path):
    pos, h, prop, size, b, pair = box_scene2d(axis)
    a, c = PLANE[axis]
    assert pair == (BOX3_2D[a], BOX3_2D[c])                      # the in-plane sides, written out for the oracle
    check2d(("box2", axis), path, pos, h, prop, size, axis, b, periodic=True, box=BOX3_2D, ref_box=pair)


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_three_component_box_create_image(axis):
    from astro_sph_tools_b200 import CoordinateAxes
    from astro_sph_tools_b200.tools.projections import create_image
    pos, h, prop, size, b, pair = box_scene2d(axis)
    ref, env = reference2d((("box2", axis), False), pos, h, prop, size, axis, b, periodic=True, box=pair)
    got = create_image(pos, h, prop, size, 32, CoordinateAxes(axis), *b, periodic=True, box_size=BOX3_2D)
    assert_pixelwise(got, ref, env)
    global_gates(got, ref)


# ---- 3. anisotropic cells --------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _aniso3(name):
    return aniso_scene3d(name)


@functools.lru_cache(maxsize=None)
def _aniso2(name):
    return aniso_scene2d(name)


@pytest.mark.parametrize("path", list(PATHS3))
@pytest.mark.parametrize("name", list(ANISO3))
def test_anisotropic_voxels(name, path):
    pos, h, prop, size, lo, hi = _aniso3(name)
    check3d(("aniso3", name), path, pos, h, prop, size, lo, hi)


@pytest.mark.parametrize("path", list(PATHS2))
@pytest.mark.parametrize("name", list(ANISO2))
def test_anisotropic_pixels(name, path):
    pos, h, prop, size, b = _aniso2(name)
    check2d(("aniso2", name), path, pos, h, prop, size, 2, b)


# ---- 4. odd grid shapes ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", list(PATHS3))
@pytest.mark.parametrize("size", ODD_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_odd_grid_shapes(size, path):
    pos, h, prop, size, lo, hi = odd_scene3d(size)
    check3d(("odd", size), path, pos, h, prop, size, lo, hi)


# ---- 5. Wendland C2 in 3-D -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", list(PATHS3))
@pytest.mark.parametrize("scene", ["grid_vs_oracle", "noncubic_box"])
def test_wendland_c2_3d_per_voxel(scene, path):
    from conftest import random_cloud
    if scene == "grid_vs_oracle":                                # the scene of test_gpu_grid3d.py::test_grid_vs_oracle
        pos, h, prop = random_cloud(41, 3000, L=1.0, h_lo=0.0, h_hi=0.09, signed=True)
        size, lo, hi = (48, 40, 56), (0.0, 0.1, 0.0), (1.0, 0.9, 1.0)
        check3d(("wc2", scene), path, pos, h, prop, size, lo, hi, "wendland_c2_3d")
    else:
        pos, h, prop, size, lo, hi = _box3("past_low")
        check3d(("wc2", scene), path, pos, h, prop, size, lo, hi, "wendland_c2_3d", periodic=True, box=BOX3)


# ---- 6. tabulated kernels --------------------------------------------------------------------------------------------
TABLES = python_kernels()                  # one callable per kernel for the whole module: its device table is built once


@pytest.mark.parametrize("path", list(PATHS2))
@pytest.mark.parametrize("name", KERNELS)
def test_tabulated_kernels_2d(name, path):
    from astro_sph_tools_b200.tools.projections._kernels import TabulatedKernel, kernel_id_of
    assert isinstance(kernel_id_of(TABLES[name]), TabulatedKernel)
    pos, h, prop, size, b = table_scene2d()
    check2d(("table2", name), path, pos, h, prop, size, 2, b, TABLES[name], ref_kernel=name)


@pytest.mark.parametrize("path", list(PATHS3))
@pytest.mark.parametrize("name", KERNELS)
def test_tabulated_kernels_3d(name, path):
    pos, h, prop, size, lo, hi = table_scene3d()
    check3d(("table3", name), path, pos, h, prop, size, lo, hi, TABLES[name], ref_kernel=name)


@pytest.mark.parametrize("path", list(PATHS3))
def test_tabulated_kernel_in_a_noncubic_periodic_box(path):
    pos, h, prop, size, lo, hi = table_scene3d(periodic=True)
    check3d(("table3p", "cubic_spline_3d"), path, pos, h, prop, size, lo, hi, TABLES["cubic_spline_3d"], periodic=True,
            box=BOX3, ref_kernel="cubic_spline_3d")


# ---- 7. every branch of the brick kernel -----------------------------------------------------------------------------
@pytest.mark.parametrize("presort", ["never", "always"])
def test_brick_kernel_branches(oracle, presort):
    pos, h, prop, nc, ns, nl = branch_scene3d()
    pos, h, prop = pad_for_presort(pos, h, prop, 2)
    size, lo, hi = BRANCH_GRID
    _, st = check3d(("branches",), "default", pos, h, prop, size, lo, hi, presort=presort, **BRANCH_KW)
    # the windows: pairs walked in three rounds or more, the large-h list longer than its window
    assert st["n_rounds"] >= 3 and st["n_huge"] > BRANCH_KW["huge_capacity"], st
    assert st["reordered"] == (presort == "always")
    # per-brick list lengths from the oracle's index work (with the large-h member bricks)
    o = oracle.bin3d(pos, h, size, lo, hi, small_max_vox=27, huge_min_bricks=BRANCH_KW["huge_min_bricks"])
    per_brick = np.bincount((o["sorted"] >> np.uint64(32)).astype(np.int64))
    assert st["n_pairs"] == len(o["sorted"]) and st["n_huge"] == len(o["huge"])
    # a list longer than the 1024-entry minimum segment: split into interleaved work items that add with float64 atomics.
    # It still holds more than 1024 entries in one round: the clump's pairs are consecutive in emit order (by particle, and
    # by brick when pre-ordered) and number more than twice 1024, and a round holds pair_capacity > 1024 consecutive pairs,
    # so one round holds more than 1024 of them
    assert per_brick.max() > 2 * 1024 and BRANCH_KW["pair_capacity"] > 1024
    # lists with fewer than 10 entries: their batches are evaluated without the distance tables
    assert ((per_brick > 0) & (per_brick < 10)).sum() >= 5
    # whole 4x4x8 columns in the outer annulus of the large-h particles (cubic spline: the second loop)
    assert outer_annulus_columns(pos[h > 5.5 / 48], h[h > 5.5 / 48], size, lo, hi) >= 50
    # weights of the brick path span more than one band
    norm = np.abs(prop) / (np.pi * h ** 3)
    e = np.frexp(norm[h > 0.6 / 48])[1]
    assert e.max() - e.min() > BRANCH_BAND_GAP - 10 > 100
