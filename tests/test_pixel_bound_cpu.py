"""The per-pixel bound of tests/pixel_bound.py against the C oracle (no device needed): the envelope covers every oracle
pixel, is non-zero exactly on the contributor mask when it is not widened, and assert_pixelwise catches one faint pixel
that is wrong by twice its bound."""
import numpy as np
import pytest

from conftest import random_cloud
from pixel_bound import TAU, assert_pixelwise, envelope2d, envelope3d

KERNELS = ["cubic_spline_3d", "wendland_c2_2d", "wendland_c2_3d", "cubic_spline_2d"]


def _scene2d(kernel, periodic):
    import zlib
    pos, h, prop = random_cloud(zlib.crc32(repr((kernel, periodic)).encode()) % 1000, 700, h_lo=0.0, h_hi=1.4, signed=True)
    h[::40] = 4.0
    h[3::97] = 0.0
    if periodic:
        return pos, h, prop, (37, 29), 2, (0.5, 7.9, 1.0, 9.7), (10.0, 10.0)
    return pos, h, prop, (37, 29), 1, (-0.5, 8.0, 1.5, 21.0), None     # the top rows see no particle


@pytest.mark.parametrize("periodic", [False, True])
@pytest.mark.parametrize("kernel", KERNELS)
def test_envelope2d_covers_the_oracle(oracle, kernel, periodic):
    pos, h, prop, size, axis, b, box = _scene2d(kernel, periodic)
    ref = oracle.project2d(pos, h, prop, size, axis, *b, kernel=kernel, periodic=periodic, box=box)
    cnt = oracle.contrib_count2d(pos, h, size, axis, *b, periodic=periodic, box=box)
    env = envelope2d(pos, h, prop, size, axis, b, kernel, periodic, box)
    assert (cnt > 0).sum() > 200 and ((cnt == 0).any() or periodic)
    assert np.all(env >= np.abs(ref))
    assert np.all(env[cnt > 0] > 0)
    exact = envelope2d(pos, h, prop, size, axis, b, kernel, periodic, box, widen=0.0)
    assert np.array_equal(exact > 0, cnt > 0)
    assert np.all(exact <= env)
    # two fields at once: each has its own envelope
    env2 = envelope2d(pos, h, np.stack([prop, 1e-30 * prop]), size, axis, b, kernel, periodic, box)
    assert env2.shape == (2,) + size and np.array_equal(env2[0], env) and np.allclose(env2[1], 1e-30 * env, rtol=1e-13, atol=0)


@pytest.mark.parametrize("periodic", [False, True])
@pytest.mark.parametrize("kernel", KERNELS)
def test_assert_pixelwise_passes_the_oracle_and_catches_one_faint_pixel(oracle, kernel, periodic):
    pos, h, prop, size, axis, b, box = _scene2d(kernel, periodic)
    ref = oracle.project2d(pos, h, prop, size, axis, *b, kernel=kernel, periodic=periodic, box=box)
    env = envelope2d(pos, h, prop, size, axis, b, kernel, periodic, box)
    assert_pixelwise(ref, ref, env)
    assert_pixelwise(ref + 0.5 * TAU * env, ref, env)
    faint = np.unravel_index(np.argmin(np.where(env > 0, env, np.inf)), env.shape)
    assert env[faint] < 0.2 * env.max()
    bad = ref.copy()
    bad[faint] += 2 * TAU * env[faint]
    with pytest.raises(AssertionError, match="1 of"):
        assert_pixelwise(bad, ref, env)
    # a non-zero value where no particle reaches, and a NaN, fail too
    if (env == 0).any():
        bad = ref.copy()
        bad[np.unravel_index(np.argmax(env == 0), env.shape)] = 1e-300
        with pytest.raises(AssertionError):
            assert_pixelwise(bad, ref, env)
    bad = ref.copy()
    bad[np.unravel_index(np.argmax(env), env.shape)] = np.nan
    with pytest.raises(AssertionError):
        assert_pixelwise(bad, ref, env)


@pytest.mark.parametrize("periodic", [False, True])
@pytest.mark.parametrize("kernel", ["cubic_spline_3d", "wendland_c2_3d"])
def test_envelope3d_covers_the_oracle(oracle, kernel, periodic):
    rng = np.random.default_rng(3 + periodic)
    n = 400
    pos = rng.uniform(0.0, 1.0, (n, 3))
    h = rng.uniform(0.005, 0.08, n)
    prop = rng.normal(size=n)
    size, lo, hi = (17, 13, 21), (0.05, 0.0, -0.1), (0.95, 0.8, 1.0)
    box = (1.0, 1.0, 1.0) if periodic else None
    ref = oracle.grid3d(pos, h, prop, size, lo, hi, kernel=kernel, periodic=periodic, box=box)
    env = envelope3d(pos, h, prop, size, lo, hi, kernel, periodic, box)
    assert np.all(env >= np.abs(ref))
    assert np.array_equal(env > 0, envelope3d(pos, h, prop, size, lo, hi, kernel, periodic, box) > 0)
    # the contributor mask: the oracle grid of unit weights with a kernel that is positive on its whole support is
    # non-zero exactly where a particle reaches (cubic spline: W > 0 for r < 2h)
    cnt = oracle.grid3d(pos, h, np.ones(n), size, lo, hi, kernel="cubic_spline_3d", periodic=periodic, box=box)
    exact = envelope3d(pos, h, prop, size, lo, hi, kernel, periodic, box, widen=0.0)
    assert np.array_equal(exact > 0, cnt > 0)
    assert_pixelwise(ref, ref, env)
    faint = np.unravel_index(np.argmin(np.where(env > 0, env, np.inf)), env.shape)
    bad = ref.copy()
    bad[faint] -= 2 * TAU * env[faint]
    with pytest.raises(AssertionError, match="1 of"):
        assert_pixelwise(bad, ref, env)
