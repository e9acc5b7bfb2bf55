"""-m gpu: every pixel of 2-D maps and every voxel of 3-D grids against the float64 oracle, within the per-pixel bound of
tests/pixel_bound.py (|got - ref| <= tau * sum_i |prop_i| W(0, h_i), zero where no particle reaches), on top of the global
gates (relative L2 <= 1e-5, total within 1e-6).  The scenes: the golden maps and random clouds of the other GPU tests, weights
spread over a huge dynamic range inside one call (ion column densities: 10^-45 ion fractions next to ordinary gas), outliers
far above the rest, image sizes that are not multiples of a tile, windows that end inside the cloud, periodic boxes that
are not square and windows smaller than the box."""
import zlib

import numpy as np
import pytest

from conftest import golden_cases, load_golden, random_cloud
from pixel_bound import assert_pixelwise, envelope2d, envelope3d

pytestmark = pytest.mark.gpu

# log2 of the weight span one float32 band of the tile and brick paths covers (kWeightBand in project2d.cu / grid3d.cu)
BAND = 100

PATHS2 = {"default": {}, "all_direct": dict(small_max_px=1 << 40), "all_tiled": dict(small_max_px=1, huge_min_tiles=1 << 40),
          "all_global": dict(small_max_px=1, huge_min_tiles=0)}
PATHS3 = {"default": {}, "all_direct": dict(small_max_vox=1 << 40), "all_bricks": dict(small_max_vox=1, huge_min_bricks=1 << 40),
          "all_global": dict(small_max_vox=1, huge_min_bricks=0)}
FORCED = ("all_tiled", "all_global", "all_bricks")


def global_gates(m, ref):
    """relative L2 <= 1e-5 and total within 1e-6, after an exact power-of-two rescale (weights near 2^1000 overflow a norm)"""
    assert m.shape == ref.shape and m.dtype == np.float64
    top = np.abs(ref).max()
    s = 2.0 ** -int(np.frexp(top)[1]) if top > 0 else 1.0
    a, b = m * s, ref * s
    nb = np.linalg.norm(b)
    assert (np.linalg.norm(a - b) / nb if nb > 0 else np.linalg.norm(a)) <= 1e-5
    assert abs(a.sum() - b.sum()) <= 1e-6 * np.abs(b).sum()


def project(pos, h, prop, size, axis, bounds, kernel="cubic_spline_3d", periodic=False, box=None, **kw):
    from gpu_util import gpu_project
    return gpu_project(pos, h, prop, size, axis, bounds, kernel=kernel, periodic=periodic, box=box, **kw)


def grid(pos, h, prop, size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, **kw):
    import torch
    from astro_sph_tools_b200.tools.projections import Gridder3D
    g = Gridder3D(**kw)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    out = g.grid(d(pos), d(h), d(prop), size, lo, hi, kernel, periodic, box)
    torch.cuda.synchronize()
    return out.cpu().numpy(), g.last_stats


def check2d(oracle, pos, h, prop, size, axis, bounds, kernel="cubic_spline_3d", periodic=False, box=None, path="default",
            ref=None, **kw):
    if ref is None:
        ref = oracle.project2d(pos, h, prop, size, axis, *bounds, kernel=kernel, periodic=periodic, box=box)
    env = envelope2d(pos, h, prop, size, axis, bounds, kernel, periodic, box)
    m, st = project(pos, h, list(prop) if np.ndim(prop) == 2 else prop, size, axis, bounds, kernel, periodic, box,
                    **PATHS2[path], **kw)
    for k in range(m.shape[0] if m.ndim == 3 else 1):
        mk, rk, ek = (m[k], ref[k], env[k]) if m.ndim == 3 else (m, ref, env)
        assert_pixelwise(mk, rk, ek, what=f"path {path}, field {k}: ")
        global_gates(mk, rk)
    return m, st


def check3d(oracle, pos, h, prop, size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, path="default", **kw):
    ref = oracle.grid3d(pos, h, prop, size, lo, hi, kernel=kernel, periodic=periodic, box=box)
    env = envelope3d(pos, h, prop, size, lo, hi, kernel, periodic, box)
    g, st = grid(pos, h, prop, size, lo, hi, kernel, periodic, box, **PATHS3.get(path, {}), **kw)
    assert_pixelwise(g, ref, env, what=f"path {path}: ")
    global_gates(g, ref)
    return g, st


def not_subhalf(h, pixel):
    """the forced tile / brick paths need h >= half a pixel (voxel) for their float32 relative coordinates"""
    return ~(h < 0.5 * pixel)


# ---- existing scenes, gated per pixel --------------------------------------------------------------------------------
@pytest.mark.parametrize("name", golden_cases())
@pytest.mark.parametrize("path", list(PATHS2))
def test_golden_maps_per_pixel(oracle, name, path):
    g = load_golden(name)
    n = int(g["npix"])
    b = tuple(float(v) for v in g["bounds"])
    pos, h, prop = g["pos"], g["h"], g["prop"]
    ref = g["ref_map"]
    if path in FORCED:
        keep = not_subhalf(h, max((b[1] - b[0]) / n, (b[3] - b[2]) / n))
        if not keep.all():
            pos, h, prop, ref = pos[keep], h[keep], prop[keep], None
    check2d(oracle, pos, h, prop, (n, n), int(g["axis"]), b, str(g["kernel"]), path=path, ref=ref)


@pytest.mark.parametrize("kernel", ["cubic_spline_3d", "wendland_c2_2d", "wendland_c2_3d", "cubic_spline_2d"])
@pytest.mark.parametrize("shape,bounds", [((100, 100), (0.0, 10.0, 0.0, 10.0)), ((70, 45), (2.0, 9.0, -1.0, 6.5)),
                                          ((33, 129), (0.0, 10.0, 0.0, 10.0))])
def test_random_clouds_per_pixel(oracle, kernel, shape, bounds):
    seed = zlib.crc32(repr((kernel, shape)).encode()) % 1000
    pos, h, prop = random_cloud(seed, 5000, h_lo=0.0, h_hi=1.3, signed=True)
    h[::50] = 6.0
    check2d(oracle, pos, h, prop, shape, 2, bounds, kernel)
    big = h > 0.5 * max((bounds[1] - bounds[0]) / shape[0], (bounds[3] - bounds[2]) / shape[1])
    for path in ("all_tiled", "all_global"):
        check2d(oracle, pos[big], h[big], prop[big], shape, 2, bounds, kernel, path=path)


def _random_window_scene(seed):
    """the scene of test_gpu_grid3d.py::test_random_grids_through_random_windows"""
    rng = np.random.default_rng(500 + seed)
    n = int(rng.integers(200, 2500))
    size = tuple(int(v) for v in rng.integers(9, 40, 3))
    lo = tuple(rng.uniform(-0.1, 0.2, 3)); hi = tuple(np.array(lo) + rng.uniform(0.6, 1.1, 3))
    pos = rng.uniform(0.0, 1.0, (n, 3))
    vox = max((hi[c] - lo[c]) / size[c] for c in range(3))
    h = np.exp(rng.uniform(np.log(0.1 * vox), np.log(8 * vox), n))
    h[rng.random(n) < 0.03] = 0.0
    prop = rng.normal(size=n)
    periodic = bool(rng.random() < 0.4)
    box = (1.0, 1.0, 1.0) if periodic else None
    kw = dict(pair_capacity=int(rng.choice([300, 5000, 200_000])), huge_capacity=int(rng.choice([1, 5, 500])),
              huge_min_bricks=int(rng.choice([0, 2, 30, 512])), small_max_vox=int(rng.choice([1, 27, 200])))
    return pos, h, prop, size, lo, hi, periodic, box, kw


@pytest.mark.parametrize("seed", [s for s in range(12) if _random_window_scene(s)[-1]["small_max_vox"] >= 8])
def test_random_grid_windows_per_voxel(oracle, seed):
    pos, h, prop, size, lo, hi, periodic, box, kw = _random_window_scene(seed)
    check3d(oracle, pos, h, prop, size, lo, hi, periodic=periodic, box=box, path="given", **kw)


# ---- dynamic range within one call -----------------------------------------------------------------------------------
# A clump of small-h particles with weights ~2^top on one side, a diffuse phase of large-h particles on the other whose
# weights fall from 2^top to 2^(top - span) along y (z in 3-D): the pixels at the far end see only the faintest weights.
SPANS = {"span140": (140, 0), f"span{BAND - 1}": (BAND - 1, 0), f"span{BAND + 1}": (BAND + 1, 0), "span2000": (2000, 1000),
         "zeros": (140, 0)}


def dyn_scene2d(span, top, seed=1, zeros=False):
    rng = np.random.default_rng(seed)
    nc, nd = 1500, 2500
    pos = np.empty((nc + nd, 3))
    pos[:nc] = rng.uniform([0.3, 0.3, 0.0], [4.0, 9.7, 10.0], (nc, 3))
    pos[nc:] = rng.uniform([5.5, 0.0, 0.0], [9.7, 10.0, 10.0], (nd, 3))
    h = np.concatenate([rng.uniform(0.05, 0.3, nc), rng.uniform(0.3, 1.2, nd)])     # pixel 10/128 = 0.078
    h[nc::97] = 3.0
    w = np.concatenate([rng.uniform(0.5, 1.5, nc), rng.uniform(0.5, 1.5, nd) * 2.0 ** (-span * pos[nc:, 1] / 10.0)])
    prop = w * 2.0 ** top
    if zeros:
        prop[rng.random(nc + nd) < 0.15] = 0.0
    return pos, h, prop


def dyn_scene3d(span, top, seed=1, zeros=False):
    rng = np.random.default_rng(seed)
    nc, nd = 1200, 1800
    pos = np.empty((nc + nd, 3))
    pos[:nc] = rng.uniform([0.03, 0.03, 0.03], [0.4, 0.97, 0.97], (nc, 3))
    pos[nc:] = rng.uniform([0.55, 0.0, 0.0], [0.97, 1.0, 1.0], (nd, 3))
    h = np.concatenate([rng.uniform(0.0125, 0.04, nc), rng.uniform(0.04, 0.1, nd)])  # voxel 1/40 = 0.025
    h[nc::61] = 0.2
    w = np.concatenate([rng.uniform(0.5, 1.5, nc), rng.uniform(0.5, 1.5, nd) * 2.0 ** (-span * pos[nc:, 2])])
    prop = w * 2.0 ** top
    if zeros:
        prop[rng.random(nc + nd) < 0.15] = 0.0
    return pos, h, prop


B2 = (0.0, 10.0, 0.0, 10.0)
G3 = ((40, 40, 40), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))


@pytest.mark.parametrize("path", list(PATHS2))
@pytest.mark.parametrize("scene", list(SPANS))
def test_dynamic_range_2d(oracle, scene, path):
    span, top = SPANS[scene]
    pos, h, prop = dyn_scene2d(span, top, zeros=scene == "zeros")
    check2d(oracle, pos, h, prop, (128, 128), 2, B2, path=path)


@pytest.mark.parametrize("path", list(PATHS3))
@pytest.mark.parametrize("scene", list(SPANS))
def test_dynamic_range_3d(oracle, scene, path):
    span, top = SPANS[scene]
    pos, h, prop = dyn_scene3d(span, top, zeros=scene == "zeros")
    check3d(oracle, pos, h, prop, *G3, path=path)


@pytest.mark.parametrize("path", list(PATHS2))
def test_dynamic_range_two_fields(oracle, path):
    """one wide-range field and one ordinary field in the same pass: each keeps its own bands"""
    pos, h, wide = dyn_scene2d(300, 200, seed=2)
    plain = np.random.default_rng(3).uniform(0.5, 1.5, len(h))
    for props in (np.stack([wide, plain]), np.stack([plain, wide])):
        check2d(oracle, pos, h, props, (96, 112), 2, B2, path=path)


@pytest.mark.parametrize("path", ["default", "all_tiled", "all_global"])
def test_dynamic_range_accumulates_onto_a_map(oracle, path):
    import torch
    from astro_sph_tools_b200.tools.projections import Projector2D
    pa, ha, wa = dyn_scene2d(140, 0, seed=4)
    pb, hb, wb = dyn_scene2d(180, -30, seed=5)
    pb[:, 1] = 10.0 - pb[:, 1]                                 # the two faint ends on opposite sides
    ref_a = oracle.project2d(pa, ha, wa, (128, 128), 2, *B2)
    ref_b = oracle.project2d(pb, hb, wb, (128, 128), 2, *B2)
    env = envelope2d(pa, ha, wa, (128, 128), 2, B2) + envelope2d(pb, hb, wb, (128, 128), 2, B2)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    out = d(ref_a.reshape(1, 128, 128))
    Projector2D(**PATHS2[path]).project(d(pb), d(hb), d(wb), (128, 128), 2, B2, out=out, accumulate=True)
    got = out.cpu().numpy()[0]
    assert_pixelwise(got, ref_a + ref_b, env)
    global_gates(got, ref_a + ref_b)


@pytest.mark.parametrize("path", ["default", "all_bricks", "all_global"])
def test_dynamic_range_accumulates_onto_a_grid(oracle, path):
    import torch
    from astro_sph_tools_b200.tools.projections import Gridder3D
    pa, ha, wa = dyn_scene3d(140, 0, seed=4)
    pb, hb, wb = dyn_scene3d(180, -30, seed=5)
    ref_a = oracle.grid3d(pa, ha, wa, *G3)
    ref_b = oracle.grid3d(pb, hb, wb, *G3)
    env = envelope3d(pa, ha, wa, *G3) + envelope3d(pb, hb, wb, *G3)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    out = d(ref_a)
    Gridder3D(**PATHS3[path]).grid(d(pb), d(hb), d(wb), *G3, out=out, accumulate=True)
    got = out.cpu().numpy()
    assert_pixelwise(got, ref_a + ref_b, env)
    global_gates(got, ref_a + ref_b)


# ---- outliers ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["default", "all_tiled", "all_global"])
def test_one_tiled_particle_far_above_the_rest_2d(oracle, path):
    rng = np.random.default_rng(21)
    n = 3000
    pos = rng.uniform(0.0, 10.0, (n, 3))
    h = rng.uniform(0.15, 0.5, n)                              # 2-6 pixels of 10/128: tiled by default
    prop = rng.uniform(0.5, 1.5, n)
    pos[0] = (2.0, 2.0, 5.0); h[0] = 0.3; prop[0] = 2.0 ** 140
    check2d(oracle, pos, h, prop, (128, 128), 2, B2, path=path)


def test_one_direct_particle_far_above_the_rest_3d(oracle):
    """3000 brick-path particles on a 40^3 grid and one sub-voxel particle next to a voxel corner whose prop * norm(h) is
    2^140 times the largest of the others: deposited directly, it must not decide the float32 scale of the bricks"""
    rng = np.random.default_rng(22)
    n = 3000
    d = 1.0 / 40
    pos = rng.uniform(0.0, 1.0, (n + 1, 3))
    h = rng.uniform(d, 3 * d, n + 1)
    prop = rng.uniform(0.5, 1.5, n + 1)
    pos[n] = (20 * d + 0.1 * d, 20 * d + 0.05 * d, 20 * d + 0.1 * d)
    h[n] = 0.3 * d
    norm = lambda hh: 1.0 / (np.pi * hh ** 3)
    prop[n] = 2.0 ** 140 * (prop[:n] * norm(h[:n])).max() / norm(h[n])
    g, st = check3d(oracle, pos, h, prop, *G3)
    assert st["n_pairs"] > 0
    assert (g != 0).sum() > 60000


# ---- ion column density ----------------------------------------------------------------------------------------------
def test_ion_map_with_trace_fractions(oracle):
    """log10 ion fraction falling to about -45 in hot gas, whose particles also have the largest h: the void pixels are
    filled by weights ~1e-50 of the clump's"""
    from astro_sph_tools_b200 import CoordinateAxes
    from astro_sph_tools_b200.tools.ionisation import IonisationTableBase, create_ion_image
    from table_util import synthetic_table
    base, axes = synthetic_table(shape=(41, 141, 49))
    T = np.meshgrid(*axes, indexing="ij")[1]
    table = base - 45.0 * np.clip((T - 5.5) / 1.5, 0.0, 1.0)
    t = IonisationTableBase(table, *axes, redshift_input_index=2)
    rng = np.random.default_rng(23)
    nc, nh = 3000, 5000
    pos = np.concatenate([rng.uniform([0.02, 0.02, 0], [0.45, 0.98, 1], (nc, 3)), rng.uniform([0.5, 0, 0], [1, 1, 1], (nh, 3))])
    h = np.concatenate([rng.uniform(0.006, 0.02, nc), rng.uniform(0.02, 0.07, nh)])        # pixel 1/256
    m = rng.uniform(0.5, 1.5, nc + nh)
    lognh = np.concatenate([rng.uniform(-4.0, -2.0, nc), rng.uniform(-6.0, -3.0, nh)])
    logt = np.concatenate([rng.uniform(3.0, 5.0, nc), rng.uniform(4.0 + 4.5 * pos[nc:, 1], 4.5 + 4.5 * pos[nc:, 1])])
    z = 1.3
    w = m * 10.0 ** oracle.table_interp_scipy(table, axes, np.stack([lognh, logt, np.full(nc + nh, z)], axis=1))
    assert w[nc:].min() < 1e-45 * w[:nc].min() and w.min() > 0
    b = (0.0, 1.0, 0.0, 1.0)
    got = create_ion_image(t, pos, h, m, lognh, logt, z, (256, 256), 32, CoordinateAxes.Z, *b)
    ref = oracle.project2d(pos, h, w, (256, 256), 2, *b)
    assert_pixelwise(got, ref, envelope2d(pos, h, w, (256, 256), 2, b))
    global_gates(got, ref)


# ---- edges the global gates blur -------------------------------------------------------------------------------------
EDGES = {
    "1x97": ((1, 97), (0.0, 10.0, 0.0, 10.0), False, None),
    "31x33": ((31, 33), (0.0, 10.0, 0.0, 10.0), False, None),
    "65x64": ((65, 64), (0.0, 10.0, 0.0, 10.0), False, None),
    "window_inside_cloud": ((70, 90), (2.3, 7.9, 1.1, 8.6), False, None),
    "periodic_box_10x7": ((80, 56), (0.0, 10.0, 0.0, 7.0), True, (10.0, 7.0)),
    "periodic_subwindow": ((48, 40), (0.5, 3.5, 5.0, 6.9), True, (10.0, 7.0)),
}


@pytest.mark.parametrize("path", ["default", "all_tiled", "all_global"])
@pytest.mark.parametrize("edge", list(EDGES))
def test_edges_per_pixel(oracle, edge, path):
    size, b, periodic, box = EDGES[edge]
    pos, h, prop = random_cloud(zlib.crc32(edge.encode()) % 1000, 3000, h_lo=0.0, h_hi=1.3, signed=True)
    if box is not None:
        pos[:, 1] *= box[1] / 10.0
    h[::60] = 6.0                                               # some survive the forced paths' h >= half a pixel on 1 x 97
    if path in FORCED:
        keep = not_subhalf(h, max((b[1] - b[0]) / size[0], (b[3] - b[2]) / size[1]))
        pos, h, prop = pos[keep], h[keep], prop[keep]
    m, _ = check2d(oracle, pos, h, prop, size, 2, b, periodic=periodic, box=box, path=path)
    if edge == "periodic_subwindow":
        # particles of the far side of the box reach the window only through their periodic images
        far = (pos[:, 0] > 8.5) | (pos[:, 1] < 1.0)
        alone = oracle.project2d(pos[far], h[far], np.abs(prop[far]), size, 2, *b, periodic=True, box=box)
        assert (alone > 0).sum() > 100
