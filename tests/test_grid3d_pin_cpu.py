"""The 3-D oracle (oracle.grid3d, oracle/sph_oracle.c) against an independent literal numpy restatement of the reference's
per-pixel rule carried to three dimensions (tests/literal3d.py), with the reference's own compiled kernel function when
oracle/_ref is present.  Pins the extension's oracle on something other than itself (VERDICT r1, missing item 7)."""
import numpy as np
import pytest

from conftest import load_golden, rel_l2
from literal3d import grid3d_literal, project2d_literal, quartic_spline_numpy, reference_kernel


def cloud(seed, n):
    rng = np.random.default_rng(seed)
    pos = rng.uniform(-0.05, 1.05, (n, 3))
    h = rng.choice([0.01, 0.03, 0.06, 0.15], n)
    h[::17] = 0.0
    prop = rng.normal(size=n)
    return pos, h, prop


def test_reference_kernel_is_the_numpy_restatement_of_kernels_pyx():
    rng = np.random.default_rng(0)
    r = rng.uniform(0, 2.5, 5000); h = rng.uniform(0.5, 1.5, 5000)
    k = reference_kernel()
    assert np.allclose(k(r, h), quartic_spline_numpy(r, h), rtol=1e-14, atol=0)
    # without oracle/_ref, k is the restatement itself: pin it, with the literal 2-D pixel rule, on the reference's stored maps
    for name in ("single_particle", "single_particle_axis0", "single_particle_axis1", "cloud_axis0", "cloud_axis1",
                 "cloud_axis2", "cloud_tiny_and_huge_h"):
        g = load_golden(name)
        assert str(g["kernel"]) == "cubic_spline_3d"
        lit = project2d_literal(g["pos"], g["h"], g["prop"], int(g["npix"]), int(g["axis"]), g["bounds"], quartic_spline_numpy)
        assert np.array_equal(lit != 0, g["ref_map"] != 0) and rel_l2(lit, g["ref_map"]) < 1e-13


@pytest.mark.parametrize("size,lo,hi", [((14, 14, 14), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)), ((9, 16, 12), (0.1, 0.0, 0.2), (0.9, 1.2, 0.8))])
def test_oracle_grid3d_equals_literal_restatement(oracle, size, lo, hi):
    pos, h, prop = cloud(4, 600)
    lit = grid3d_literal(pos, h, prop, size, lo, hi)
    orc = oracle.grid3d(pos, h, prop, size, lo, hi)
    assert np.array_equal(lit != 0, orc != 0)                     # identical support: the strict r2 < (2h)^2 mask
    assert rel_l2(orc, lit) < 1e-13
    assert abs(orc.sum() - lit.sum()) <= 1e-12 * np.abs(lit).sum()


def test_oracle_grid3d_periodic_equals_replicated_particles(oracle):
    pos, h, prop = cloud(7, 300)
    pos = np.mod(pos, 1.0)
    shifts = [(i, j, k) for i in (-1.0, 0.0, 1.0) for j in (-1.0, 0.0, 1.0) for k in (-1.0, 0.0, 1.0)]
    lit = grid3d_literal(pos, h, prop, (10, 10, 10), (0.0,) * 3, (1.0,) * 3, shifts=shifts)
    orc = oracle.grid3d(pos, h, prop, (10, 10, 10), (0.0,) * 3, (1.0,) * 3, periodic=True, box=(1.0, 1.0, 1.0))
    assert np.array_equal(lit != 0, orc != 0) and rel_l2(orc, lit) < 1e-13
