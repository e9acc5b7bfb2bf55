"""The oracle and the per-cell gate of tests/pixel_bound.py on the geometry of tests/test_gpu_geometry_pixelwise.py (no device
needed): periodic boxes whose sides differ against replicated particles and the literal per-voxel rule, the envelope on
anisotropic cells and non-cubic boxes, and the gate's power to fail there -- a box with its sides permuted, or a kernel
table read one node off, must break it on many cells.  Without that, a green GPU run would prove nothing about swapped box
components or off-by-one table indexing."""
import re

import numpy as np
import pytest

from conftest import rel_l2
from geometry_scenes import (ANISO2, ANISO3, BOX3, BOX3_2D, BOX_WINDOWS, PLANE, box_scene2d, box_scene3d, aniso_scene2d,
                             aniso_scene3d, table_kernel, table_scene2d, table_scene3d)
from literal3d import grid3d_literal, project2d_literal
from pixel_bound import assert_pixelwise, envelope2d, envelope3d

SHIFTS3 = [(i, j, k) for i in (-1, 0, 1) for j in (-1, 0, 1) for k in (-1, 0, 1)]


def n_outside(got, ref, env):
    """cells assert_pixelwise rejects (0 when it passes)"""
    try:
        assert_pixelwise(got, ref, env)
    except AssertionError as e:
        return int(re.search(r"(\d+) of \d+ pixels outside", str(e)).group(1))
    return 0


def box_permutations(box):
    perms = [(0, 2, 1), (1, 0, 2), (2, 1, 0), (1, 2, 0), (2, 0, 1)]
    return [tuple(box[i] for i in p) for p in perms]


# ---- the periodic oracle on boxes whose sides differ ---------------------------------------------------------------
def test_oracle_grid3d_noncubic_box_equals_literal_and_replicated_particles(oracle):
    rng = np.random.default_rng(11)
    n = 250
    L = np.array(BOX3)
    pos = rng.uniform(0.0, 1.0, (n, 3)) * L
    h = rng.choice([0.02, 0.06, 0.15, 0.4], n)                  # 0.4: images of one particle overlap
    h[::13] = 0.0
    pos[0] = (0.0, np.nextafter(0.7, 0.0), 0.0)
    pos[1] = (np.nextafter(1.0, 0.0), 0.0, np.nextafter(1.3, 0.0))
    prop = rng.normal(size=n)
    size, lo, hi = (10, 7, 13), (0.0, 0.0, 0.0), BOX3
    orc = oracle.grid3d(pos, h, prop, size, lo, hi, periodic=True, box=BOX3)
    shifts = [tuple(s[c] * L[c] for c in range(3)) for s in SHIFTS3]
    lit = grid3d_literal(pos, h, prop, size, lo, hi, shifts=shifts)
    assert np.array_equal(lit != 0, orc != 0) and rel_l2(orc, lit) < 1e-13
    rep = np.concatenate([pos + np.array(s) for s in shifts])
    flat = oracle.grid3d(rep, np.tile(h, 27), np.tile(prop, 27), size, lo, hi)
    assert np.array_equal(flat != 0, orc != 0) and rel_l2(orc, flat) < 1e-13
    # a window that reaches past the box on the low side and one inside it
    for lo2, hi2 in ((tuple(-0.2 * v for v in L), tuple(0.8 * v for v in L)), ((0.15, 0.1, 0.3), (0.75, 0.55, 1.0))):
        orc = oracle.grid3d(pos, h, prop, size, lo2, hi2, periodic=True, box=BOX3)
        flat = oracle.grid3d(rep, np.tile(h, 27), np.tile(prop, 27), size, lo2, hi2)
        assert (orc != 0).sum() > 300
        assert np.array_equal(flat != 0, orc != 0) and rel_l2(orc, flat) < 1e-13


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_oracle_project2d_nonsquare_box_equals_replicated_particles(oracle, axis):
    pos, h, prop, size, b, pair = box_scene2d(axis, n=600)
    a, c = PLANE[axis]
    orc = oracle.project2d(pos, h, prop, size, axis, *b, periodic=True, box=pair)
    rep = np.concatenate([pos + np.array([(ia * BOX3_2D[a] if k == a else ib * BOX3_2D[c] if k == c else 0.0) for k in range(3)])
                          for ia in (-1, 0, 1) for ib in (-1, 0, 1)])
    flat = oracle.project2d(rep, np.tile(h, 9), np.tile(prop, 9), size, axis, *b)
    assert np.array_equal(flat != 0, orc != 0) and rel_l2(orc, flat) < 1e-13
    assert pair[0] != pair[1]


# ---- the envelope on these scenes ------------------------------------------------------------------------------------
def _mask3(oracle, pos, h, size, lo, hi, periodic=False, box=None):
    """contributor mask: unit weights with the cubic spline, which is positive on its whole support"""
    return oracle.grid3d(pos, h, np.ones(len(h)), size, lo, hi, kernel="cubic_spline_3d", periodic=periodic, box=box) > 0


@pytest.mark.parametrize("window", list(BOX_WINDOWS))
def test_envelope3d_covers_the_oracle_in_noncubic_boxes(oracle, window):
    pos, h, prop, size, lo, hi = box_scene3d(window, n=700)
    ref = oracle.grid3d(pos, h, prop, size, lo, hi, periodic=True, box=BOX3)
    env = envelope3d(pos, h, prop, size, lo, hi, periodic=True, box=BOX3)
    assert np.all(env >= np.abs(ref))
    exact = envelope3d(pos, h, prop, size, lo, hi, periodic=True, box=BOX3, widen=0.0)
    assert np.array_equal(exact > 0, _mask3(oracle, pos, h, size, lo, hi, True, BOX3))


@pytest.mark.parametrize("name", list(ANISO3))
def test_envelope3d_covers_the_oracle_on_anisotropic_cells(oracle, name):
    pos, h, prop, size, lo, hi = aniso_scene3d(name, n=800)
    ref = oracle.grid3d(pos, h, prop, size, lo, hi)
    env = envelope3d(pos, h, prop, size, lo, hi)
    assert np.all(env >= np.abs(ref))
    exact = envelope3d(pos, h, prop, size, lo, hi, widen=0.0)
    assert np.array_equal(exact > 0, _mask3(oracle, pos, h, size, lo, hi))
    assert (exact > 0).sum() > 0.05 * exact.size


@pytest.mark.parametrize("name", list(ANISO2))
def test_envelope2d_covers_the_oracle_on_anisotropic_pixels(oracle, name):
    pos, h, prop, size, b = aniso_scene2d(name)
    ref = oracle.project2d(pos, h, prop, size, 2, *b)
    env = envelope2d(pos, h, prop, size, 2, b)
    cnt = oracle.contrib_count2d(pos, h, size, 2, *b)
    assert np.all(env >= np.abs(ref))
    assert np.array_equal(envelope2d(pos, h, prop, size, 2, b, widen=0.0) > 0, cnt > 0)
    assert (cnt > 0).sum() > 0.05 * cnt.size


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_envelope2d_covers_the_oracle_in_nonsquare_boxes(oracle, axis):
    pos, h, prop, size, b, pair = box_scene2d(axis, n=800)
    ref = oracle.project2d(pos, h, prop, size, axis, *b, periodic=True, box=pair)
    env = envelope2d(pos, h, prop, size, axis, b, periodic=True, box=pair)
    cnt = oracle.contrib_count2d(pos, h, size, axis, *b, periodic=True, box=pair)
    assert np.all(env >= np.abs(ref))
    assert np.array_equal(envelope2d(pos, h, prop, size, axis, b, periodic=True, box=pair, widen=0.0) > 0, cnt > 0)


def test_peaks_accept_a_kernel_callable(oracle):
    from geometry_scenes import python_kernels
    pos, h, prop, size, b = table_scene2d(n=400)
    for name, f in python_kernels().items():
        by_name = envelope2d(pos, h, prop, size, 2, b, name)
        by_func = envelope2d(pos, h, prop, size, 2, b, f)
        assert np.allclose(by_func, by_name, rtol=1e-13, atol=0) and by_name.any()


# ---- sensitivity: the gate fails when the box is permuted or the table is off by one node -------------------------
@pytest.mark.parametrize("window", list(BOX_WINDOWS))
def test_gate_catches_permuted_box_3d(oracle, window):
    pos, h, prop, size, lo, hi = box_scene3d(window, n=700)
    ref = oracle.grid3d(pos, h, prop, size, lo, hi, periodic=True, box=BOX3)
    env = envelope3d(pos, h, prop, size, lo, hi, periodic=True, box=BOX3)
    assert n_outside(ref, ref, env) == 0
    for perm in box_permutations(BOX3):
        wrong = oracle.grid3d(pos, h, prop, size, lo, hi, periodic=True, box=perm)
        assert n_outside(wrong, ref, env) >= 100, perm


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_gate_catches_swapped_box_2d(oracle, axis):
    pos, h, prop, size, b, pair = box_scene2d(axis, n=800)
    ref = oracle.project2d(pos, h, prop, size, axis, *b, periodic=True, box=pair)
    env = envelope2d(pos, h, prop, size, axis, b, periodic=True, box=pair)
    assert n_outside(ref, ref, env) == 0
    wrong = oracle.project2d(pos, h, prop, size, axis, *b, periodic=True, box=pair[::-1])
    assert n_outside(wrong, ref, env) >= 100
    # the projection's third box side in place of an in-plane one
    other = BOX3_2D[axis]
    for w in ((other, pair[1]), (pair[0], other)):
        wrong = oracle.project2d(pos, h, prop, size, axis, *b, periodic=True, box=w)
        assert n_outside(wrong, ref, env) >= 100, w


@pytest.mark.parametrize("name", ["cubic_spline_3d", "cubic_spline_2d", "wendland_c2_2d", "wendland_c2_3d"])
def test_gate_holds_for_tables_and_catches_a_table_one_node_off_2d(oracle, name):
    pos, h, prop, size, b = table_scene2d(n=1500)
    n = 64                                                       # the literal rule takes square maps
    ref = oracle.project2d(pos, h, prop, (n, n), 2, *b, kernel=name)
    env = envelope2d(pos, h, prop, (n, n), 2, b, name)
    exact = project2d_literal(pos, h, prop, n, 2, b, table_kernel(name))
    assert n_outside(exact, ref, env) == 0
    off = project2d_literal(pos, h, prop, n, 2, b, table_kernel(name, shift=1))
    assert n_outside(off, ref, env) >= 100


@pytest.mark.parametrize("periodic", [False, True])
@pytest.mark.parametrize("name", ["cubic_spline_3d", "wendland_c2_3d"])
def test_gate_holds_for_tables_and_catches_a_table_one_node_off_3d(oracle, name, periodic):
    pos, h, prop, size, lo, hi = table_scene3d(periodic, n=400)
    size = tuple(max(4, s // 2) for s in size)                   # the literal rule walks voxels one at a time
    box = BOX3 if periodic else None
    L = np.array(BOX3)
    shifts = [tuple(s[c] * L[c] for c in range(3)) for s in SHIFTS3] if periodic else ((0.0, 0.0, 0.0),)
    ref = oracle.grid3d(pos, h, prop, size, lo, hi, kernel=name, periodic=periodic, box=box)
    env = envelope3d(pos, h, prop, size, lo, hi, name, periodic, box)
    exact = grid3d_literal(pos, h, prop, size, lo, hi, table_kernel(name), shifts=shifts)
    assert n_outside(exact, ref, env) == 0
    off = grid3d_literal(pos, h, prop, size, lo, hi, table_kernel(name, shift=1), shifts=shifts)
    assert n_outside(off, ref, env) >= 50
