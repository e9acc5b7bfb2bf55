"""-m gpu: 3-D gridding on x-windows of the grid and on x-slabs owned by ranks (distributed.grid_sharded), with the real CUDA
kernels; multi-rank runs use in-process ranks on one GPU (tests/inprocess_dist.py).

  * Gridder3D.grid with x_window=(0, nx) is the whole-grid call bit for bit;
  * ast_bin3d on windows: bboxes, classes, sorted pairs and the large-h list equal the window reference built on the oracle
    (tests/grid_window_ref.py), whose bboxes are the whole grid's clipped to the window;
  * window grids on every path, per voxel against the slice of the whole oracle grid: a non-cubic periodic box, a tabulated
    kernel, weights 2^140 apart;
  * the routing kernel's rows and counts equal the numpy definition from oracle.bbox3d, in row order, on periodic wrap, slab
    faces hit exactly and one ulp either side, supports spanning several slabs, zero and NaN h;
  * grid_sharded on 1 to 8 ranks and create_grid_sharded: every slab per voxel against the oracle slice, the assembled grid
    against the global gates."""
import numpy as np
import pytest
import torch

from conftest import random_cloud
from geometry_scenes import BOX3, box_scene3d, keep_forced, python_kernels, table_scene3d
from grid_window_ref import bin3d_window, route_reference
from inprocess_dist import thread_ranks  # noqa: F401  (fixture)
from pixel_bound import assert_pixelwise, envelope3d

pytestmark = pytest.mark.gpu

PATHS3 = {"default": {}, "all_direct": dict(small_max_vox=1 << 40), "all_bricks": dict(small_max_vox=1, huge_min_bricks=1 << 40),
          "all_global": dict(small_max_vox=1, huge_min_bricks=0)}


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def global_gates(m, ref):
    """relative L2 <= 1e-5 and total within 1e-6"""
    assert m.shape == ref.shape and m.dtype == np.float64
    nb = np.linalg.norm(ref)
    assert (np.linalg.norm(m - ref) / nb if nb > 0 else np.linalg.norm(m)) <= 1e-5
    assert abs(m.sum() - ref.sum()) <= 1e-6 * np.abs(ref).sum()


def grid(pos, h, prop, size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, x_window=None, **kw):
    from astro_sph_tools_b200.tools.projections import Gridder3D
    from astro_sph_tools_b200.tools.projections._kernels import kernel_id_of
    out = Gridder3D(**kw).grid(dev(pos), dev(h), dev(prop), size, lo, hi, kernel_id_of(kernel), periodic, box, presort="never",
                               x_window=x_window)
    torch.cuda.synchronize()
    return out.cpu().numpy()


# ---- x_window = (0, nx) is the whole grid ------------------------------------------------------------------------------
def scene_random():
    pos, h, prop = random_cloud(41, 3000, L=1.0, h_lo=0.0, h_hi=0.09, signed=True)
    return pos, h, prop, (48, 40, 56), (0.0, 0.1, 0.0), (1.0, 0.9, 1.0), False, None


def scene_periodic():
    from astro_sph_tools_b200 import synthetic
    s = synthetic.s1(12, k=32)
    return s["pos"], s["h"], s["mass"], (32, 32, 32), (0, 0, 0), (1, 1, 1), True, 1.0


# (the brick paths write every voxel once per call on these small scenes; the direct deposits use float64 atomics, whose order
# is not fixed between two calls)
@pytest.mark.parametrize("path", ["all_bricks", "all_global"])
@pytest.mark.parametrize("scene", [scene_random, scene_periodic])
def test_full_window_is_the_whole_grid(scene, path):
    pos, h, prop, size, lo, hi, periodic, box = scene()
    whole = grid(pos, h, prop, size, lo, hi, periodic=periodic, box=box, **PATHS3[path])
    win = grid(pos, h, prop, size, lo, hi, periodic=periodic, box=box, x_window=(0, size[0]), **PATHS3[path])
    assert np.array_equal(win, whole)
    assert np.abs(whole).sum() > 0


def test_window_is_validated():
    from astro_sph_tools_b200.tools.projections import Gridder3D
    g = Gridder3D()
    for w in ((-1, 4), (4, 4), (6, 3), (0, 9)):
        with pytest.raises(ValueError):
            g.grid(dev(np.zeros((1, 3))), dev(np.ones(1)), dev(np.ones(1)), (8, 8, 8), (0, 0, 0), (1, 1, 1), x_window=w)


# ---- ast_bin3d on windows ---------------------------------------------------------------------------------------------
def gpu_bin3d_window(pos, h, size, lo, hi, window, periodic=False, box=None, small=20, huge=60, cap=1 << 22):
    import ctypes as C
    from astro_sph_tools_b200 import _lib
    from astro_sph_tools_b200.tools.projections import Gridder3D
    g = Gridder3D(pair_capacity=cap, huge_capacity=1 << 18, small_max_vox=small, huge_min_bricks=huge)
    n = len(h); n_img = 27 if periodic else 1
    p = g.params(n, size, lo, hi, "cubic_spline_3d", periodic, box, x_window=window)
    ws = g.workspace(p)
    bbox = torch.empty((n_img * n, 6), dtype=torch.int32, device="cuda")
    cls = torch.empty(n_img * n, dtype=torch.uint8, device="cuda")
    ps = torch.zeros(cap, dtype=torch.int64, device="cuda"); hg = torch.zeros(1 << 18, dtype=torch.int64, device="cuda")
    counts = (C.c_int64 * 2)()
    pos_d, h_d = dev(pos), dev(h)                                 # (kept alive across the call)
    _lib.check(g.lib.ast_bin3d(C.byref(p), _lib.ptr(pos_d), _lib.ptr(h_d), _lib.ptr(bbox), _lib.ptr(cls), _lib.ptr(ps), _lib.ptr(hg),
                               counts, _lib.ptr(ws), C.c_size_t(ws.numel()), _lib.stream_ptr()))
    torch.cuda.synchronize()
    return dict(bbox=bbox.cpu().numpy(), cls=cls.cpu().numpy().reshape(n_img, n), sorted=ps.cpu().numpy()[:counts[0]].view(np.uint64),
                huge=hg.cpu().numpy()[:counts[1]].view(np.uint64))


@pytest.mark.parametrize("window", [(8, 24), (5, 6), (39, 40)])
@pytest.mark.parametrize("periodic", [False, True])
def test_bin3d_window_bit_exact(oracle, periodic, window):
    from test_grid_sharded_cpu import LO, HI, SIZE, bin_scene
    pos, h = bin_scene(3000)
    box = (1.0, 1.0, 1.0) if periodic else None
    ref = bin3d_window(oracle, pos, h, SIZE, LO, HI, window, small_max_vox=20, huge_min_bricks=60, periodic=periodic, box=box)
    g = gpu_bin3d_window(pos, h, SIZE, LO, HI, window, periodic, box)
    assert np.array_equal(g["bbox"], ref["bbox"])
    assert np.array_equal(g["cls"], ref["cls"])
    assert np.array_equal(g["sorted"], ref["sorted"])
    assert np.array_equal(g["huge"], ref["huge"])
    assert (ref["cls"] > 0).sum() > 50


# ---- window grids against the slice of the whole oracle grid ----------------------------------------------------------
def window_scene(name):
    """-> pos, h, prop, size, lo, hi, periodic, box, kernel for the device, kernel name for the oracle"""
    if name == "box3":
        pos, h, prop, size, lo, hi = box_scene3d("box")
        return pos, h, prop, size, lo, hi, True, BOX3, "cubic_spline_3d", "cubic_spline_3d"
    if name == "table":
        pos, h, prop, size, lo, hi = table_scene3d()
        return pos, h, prop, size, lo, hi, False, None, python_kernels()["cubic_spline_3d"], "cubic_spline_3d"
    rng = np.random.default_rng(140)                              # "span140": two weight phases 2^140 apart
    pos = rng.uniform(0.0, 1.0, (3000, 3))
    h = rng.uniform(0.02, 0.08, 3000)
    prop = rng.uniform(0.5, 1.5, 3000) * np.where(np.arange(3000) % 2 == 0, 1.0, 2.0 ** 140)
    return pos, h, prop, (40, 40, 40), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), False, None, "cubic_spline_3d", "cubic_spline_3d"


@pytest.mark.parametrize("path", list(PATHS3))
@pytest.mark.parametrize("name", ["box3", "table", "span140"])
def test_window_grid_per_voxel(oracle, name, path):
    pos, h, prop, size, lo, hi, periodic, box, kernel, ref_kernel = window_scene(name)
    if path in ("all_bricks", "all_global"):
        keep = keep_forced(h, size, lo, hi)
        pos, h, prop = pos[keep], h[keep], prop[keep]
    ref = oracle.grid3d(pos, h, prop, size, lo, hi, kernel=ref_kernel, periodic=periodic, box=box)
    env = envelope3d(pos, h, prop, size, lo, hi, ref_kernel, periodic, box)
    for w in ((8, 16), (5, size[0] - 3), (size[0] - 1, size[0])):
        got = grid(pos, h, prop, size, lo, hi, kernel, periodic, box, x_window=w, **PATHS3[path])
        assert_pixelwise(got, ref[w[0]:w[1]], env[w[0]:w[1]], what=f"{name} {path} window {w}: ")


# ---- the routing kernel -----------------------------------------------------------------------------------------------
def route_scene(periodic):
    """particles on slab-face corner planes and one ulp either side, wrapping across x = 0 and x = L, supports spanning
    several slabs, zero and NaN h"""
    rng = np.random.default_rng(77 + periodic)
    size, lo, hi = (40, 12, 10), (0.0, 0.0, 0.0), (1.0, 0.6, 0.5)
    n = 4000
    pos = rng.uniform(-0.05, 1.05, (n, 3)) * np.array(hi)
    if periodic:
        pos = np.mod(pos, np.array(hi))
    d = 1.0 / 40
    h = rng.choice([0.1 * d, 0.5 * d, d, 3 * d, 9 * d, 25 * d], n)
    k = 0
    for plane in (0, 8, 16, 24, 32, 39, 40):
        x = plane * d
        for v in (np.nextafter(x, -1.0), x, np.nextafter(x, 2.0)):
            for hh in (0.25 * d, 0.5 * d, 0.5 * d * (1 + 1e-15), 4.0 * d):
                pos[k, 0] = v; h[k] = hh; k += 1
    pos[k:k + 20, 0] = rng.uniform(0.0, 0.02, 20); pos[k + 20:k + 40, 0] = rng.uniform(0.98, 1.0, 20)   # wrap across 0 / L
    h[::37] = 0.0
    h[5::41] = np.nan
    prop = rng.normal(size=n)
    return pos, h, prop, size, lo, hi, (hi if periodic else None)


@pytest.mark.parametrize("world,nx", [(5, 40), (8, 40), (8, 20), (1, 40), (32, 40)])
@pytest.mark.parametrize("periodic", [False, True])
def test_route_kernel_matches_the_bbox_definition(oracle, periodic, world, nx):
    from astro_sph_tools_b200 import distributed as astd
    pos, h, prop, size, lo, hi, box = route_scene(periodic)
    size = (nx,) + size[1:]
    edges = astd.grid_slab_planes(nx, world)
    want, want_counts = route_reference(oracle, pos, h, prop, edges, size, lo, hi, periodic, box)
    send, counts, overflow = astd._GridRouter(torch.device("cuda")).route(dev(pos), dev(h), dev(prop), edges, size, lo, hi, periodic, box)
    assert np.array_equal(counts.numpy(), want_counts)
    got = send.cpu().numpy()
    assert got.shape == want.shape and np.array_equal(np.isnan(got), np.isnan(want))
    assert np.array_equal(np.nan_to_num(got), np.nan_to_num(want))
    assert int(overflow.item()) == 0
    assert (want_counts > 0).sum() == sum(1 for g in range(world) if edges[g + 1] > edges[g])


def test_route_write_stops_at_the_counted_rows():
    """a write pass told that the buffer holds fewer rows than it has to write leaves the rows beyond alone and sets the
    flag (the buffer here is big enough either way)"""
    import ctypes as C
    from astro_sph_tools_b200 import _lib, distributed as astd
    pos, h, prop, size, lo, hi, box = route_scene(True)
    edges = astd.grid_slab_planes(size[0], 4)
    r = astd._GridRouter(torch.device("cuda"))
    send, counts, _ = r.route(dev(pos), dev(h), dev(prop), edges, size, lo, hi, True, box)
    total = int(counts.sum())
    p = _lib.GridRouteParams()
    p.n = len(h); p.world = 4; p.periodic = 1; p.nx, p.ny, p.nz = size
    for c in range(3):
        p.lo[c] = lo[c]; p.hi[c] = hi[c]; p.box[c] = box[c]
    for g, e in enumerate(edges):
        p.edges[g] = e
    buf = torch.full((total, 5), -7.0, dtype=torch.float64, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    pos_d, h_d, prop_d = dev(pos), dev(h), dev(prop)
    # the table of the count pass (the route above) is still in r._ws
    _lib.check(r.lib.ast_grid_route_count(C.byref(p), _lib.ptr(pos_d), _lib.ptr(h_d), _lib.ptr(torch.empty(4, dtype=torch.int64, device="cuda")),
                                          _lib.ptr(r._ws), C.c_size_t(r._ws.numel()), _lib.stream_ptr()))
    _lib.check(r.lib.ast_grid_route_write(C.byref(p), _lib.ptr(pos_d), _lib.ptr(h_d), _lib.ptr(prop_d), _lib.ptr(buf), C.c_int64(total - 3),
                                          _lib.ptr(flag), _lib.ptr(r._ws), C.c_size_t(r._ws.numel()), _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert int(flag.item()) == 1
    assert torch.equal(buf[:total - 3], send[:total - 3]) and bool((buf[total - 3:] == -7.0).all())


def test_route_inputs_are_checked_before_any_launch():
    """float32, host, mis-sized, mixed-device and non-contiguous inputs raise ValueError; the router never gets as far as
    allocating its workspace"""
    from astro_sph_tools_b200 import distributed as astd
    from astro_sph_tools_b200.tools.projections import Gridder3D
    n = 64
    pos, h, prop = dev(np.random.default_rng(0).uniform(0, 1, (n, 3))), dev(np.full(n, 0.05)), dev(np.ones(n))
    wide = torch.zeros((n, 6), dtype=torch.float64, device="cuda")
    wide[:, :3] = pos
    bad = {"float32": (pos.float(), h, prop), "host": (pos.cpu(), h.cpu(), prop.cpu()), "short h": (pos, h[:-1], prop),
           "2-D prop": (pos, h, prop.reshape(n, 1)), "h on the host": (pos, h.cpu(), prop), "pos (N,2)": (pos[:, :2].contiguous(), h, prop),
           "non-contiguous pos": (wide[:, :3], h, prop), "non-contiguous h": (pos, wide[:, 0], prop)}
    for what, (p, hh, pp) in bad.items():
        r = astd._GridRouter(torch.device("cuda", torch.cuda.current_device()))
        with pytest.raises(ValueError):
            r.route(p, hh, pp, [0, 4, 8], (8, 8, 8), (0, 0, 0), (1, 1, 1), False, None)
        assert r._ws is None, what
        with pytest.raises(ValueError):
            astd.grid_sharded(Gridder3D(), p, hh, pp, (8, 8, 8), (0, 0, 0), (1, 1, 1))


# ---- grid_sharded on in-process ranks ---------------------------------------------------------------------------------
def random_shards(n, fractions, seed):
    perm = np.random.default_rng(seed).permutation(n)
    cuts = [0] + [int(f * n) for f in fractions] + [n]
    return [np.sort(perm[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]


def sharded_scene(name):
    """-> pos, h, prop, size, lo, hi, periodic, box, kernel"""
    if name == "random":
        pos, h, prop = random_cloud(7, 6000, L=1.0, h_lo=0.0, h_hi=0.12, signed=True)
        return pos, h, prop, (40, 24, 28), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), False, None, "cubic_spline_3d"
    if name == "box3":
        pos, h, prop, size, lo, hi = box_scene3d("box")
        return pos, h, prop, size, lo, hi, True, BOX3, "cubic_spline_3d"
    if name == "nfw":
        from astro_sph_tools_b200 import synthetic
        s = synthetic.s2(6000, k=32, n_haloes=8, seed=3)
        h = s["h"].copy()
        h[::300] = 0.3                                            # large-h entries spanning several slabs
        return s["pos"], h, s["mass"], (48, 32, 32), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), True, (1.0, 1.0, 1.0), "cubic_spline_3d"
    if name == "nx20":
        pos, h, prop = random_cloud(8, 3000, L=1.0, h_lo=0.01, h_hi=0.15)
        return pos, h, prop, (20, 24, 16), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), False, None, "cubic_spline_3d"
    pos, h, prop = random_cloud(9, 4000, L=1.0, h_lo=0.01, h_hi=0.1)   # "wendland"
    return pos, h, prop, (32, 32, 32), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), True, (1.0, 1.0, 1.0), "wendland_c2_3d"


CASES = {"random-1": ("random", 1, None), "random-2": ("random", 2, "random"), "random-3": ("random", 3, "unequal"),
         "random-8": ("random", 8, "random"), "box3-4": ("box3", 4, "random"), "nfw-8": ("nfw", 8, "unequal"),
         "nx20-4": ("nx20", 4, "random"), "empty-rank-3": ("random", 3, "empty"), "wendland-2": ("wendland", 2, "unequal")}


def shards_of(kind, n, world):
    if kind is None:
        return [np.arange(n)]
    if kind == "unequal":                                         # contiguous index ranges growing with the rank
        cuts = [0] + [n * (g + 1) ** 2 // world ** 2 for g in range(world)]
        return [np.arange(a, b) for a, b in zip(cuts[:-1], cuts[1:])]
    if kind == "empty":
        return [np.arange(0, n // 3), np.arange(0, 0), np.arange(n // 3, n)]
    return random_shards(n, [(g + 1) / world - 0.3 / world * (g % 2) for g in range(world - 1)], world)


# the NFW case puts its h = 0.3 entries on the large-h list (huge_bricks_kernel) of every slab they reach
GRIDDER_KW = {"nfw-8": dict(huge_min_bricks=4)}


@pytest.mark.parametrize("case", list(CASES))
def test_grid_sharded_per_voxel(oracle, thread_ranks, case):
    from astro_sph_tools_b200 import distributed as astd
    from astro_sph_tools_b200.tools.projections import Gridder3D
    name, world, kind = CASES[case]
    pos, h, prop, size, lo, hi, periodic, box = sharded_scene(name)[:8]
    kernel = sharded_scene(name)[8]
    shards = shards_of(kind, len(h), world)
    assert len(shards) == world and sum(len(s) for s in shards) == len(h)
    ref = oracle.grid3d(pos, h, prop, size, lo, hi, kernel=kernel, periodic=periodic, box=box)
    env = envelope3d(pos, h, prop, size, lo, hi, kernel, periodic, box)

    def body(r):
        g = Gridder3D(**GRIDDER_KW.get(case, {}))
        s = shards[r]
        slab, x0, st = astd.grid_sharded(g, dev(pos[s]), dev(h[s]), dev(prop[s]), size, lo, hi, kernel, periodic, box, return_stats=True)
        whole = astd.collect_slabs(slab, size[0], all_ranks=True)
        torch.cuda.synchronize()
        return slab.cpu().numpy(), x0, st, whole.cpu().numpy()

    res = thread_ranks(world, body) if world > 1 else [body(0)]
    e = astd.grid_slab_planes(size[0], world)
    for r, (slab, x0, st, whole) in enumerate(res):
        assert x0 == e[r] and slab.shape == (e[r + 1] - e[r],) + tuple(size[1:])
        assert_pixelwise(slab, ref[e[r]:e[r + 1]], env[e[r]:e[r + 1]], what=f"{case} rank {r}: ")
        global_gates(whole, ref)
    if case == "nx20-4":
        assert e[4] == e[3]                                       # the last rank owns no planes
    if case in GRIDDER_KW:
        assert all(st["n_huge"] > 0 for _, _, st, _ in res if st["x_end"] > st["x_begin"])
    assert sum(st["received"] for _, _, st, _ in res) == sum(sum(st["sent"]) for _, _, st, _ in res)
    for r, (_, _, st, _) in enumerate(res):
        assert st["fan_out"] == sum(st["sent"]) / max(len(shards[r]), 1)


@pytest.mark.parametrize("periodic", [False, True])
def test_create_grid_sharded(oracle, thread_ranks, periodic):
    from astro_sph_tools_b200 import distributed as astd
    from astro_sph_tools_b200.tools.projections import quartic_spline_kernel
    pos, h, prop = random_cloud(11, 5000, L=1.0, h_lo=0.005, h_hi=0.1, signed=True)
    size, box = (36, 20, 28), ((1.0, 1.0, 1.0) if periodic else None)
    ref = oracle.grid3d(pos, h, prop, size, (0, 0, 0), (1, 1, 1), periodic=periodic, box=box)
    env = envelope3d(pos, h, prop, size, (0, 0, 0), (1, 1, 1), "cubic_spline_3d", periodic, box)
    cuts = [0, 700, 3100, 5000]

    def body(r):
        s = slice(cuts[r], cuts[r + 1])
        args = (pos[s], h[s], prop[s], size, 0.0, 1.0, 0.0, 1.0, 0.0, 1.0, quartic_spline_kernel)
        one = astd.create_grid_sharded(*args, periodic=periodic, box_size=1.0 if periodic else None, dst=1)
        every = astd.create_grid_sharded(*args, periodic=periodic, box_size=1.0 if periodic else None, all_ranks=True)
        return one, every

    res = thread_ranks(3, body)
    for r, (one, every) in enumerate(res):
        assert (one is None) == (r != 1)
        for g in ([one] if one is not None else []) + [every]:
            assert g.shape == size and g.dtype == np.float64
            assert_pixelwise(g, ref, env, what=f"rank {r}: ")
            global_gates(g, ref)
