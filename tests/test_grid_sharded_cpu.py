"""CPU checks of multi-GPU 3-D gridding on x-slabs (distributed.grid_sharded) and of the window rules it rests on, with the
float64 oracle standing in for the CUDA kernels (tests/grid_window_ref.py):

  * the window reference of bin3d with the window (0, nx) is oracle.bin3d bit for bit; window bboxes equal a brute-force scan
    of the window's own voxel corners lo + (x_begin + i) * d;
  * plane edges: monotone, whole bricks, cover [0, nx), empty ranks when nx < 8 * world;
  * grid_sharded on in-process ranks with CPU tensors, an oracle router and an oracle gridder: every slab is bit-equal to the
    slice of the whole oracle grid (routed rows arrive in global index order, so every voxel sums in the same order), and
    collect_slabs assembles the whole grid on dst or on every rank."""
import numpy as np
import pytest
import torch

from grid_window_ref import OracleGridder, OracleRouter, bbox3d_window, bin3d_window
from inprocess_dist import thread_ranks  # noqa: F401  (fixture)

SIZE, LO, HI = (40, 48, 33), (0.0, 0.0, 0.0), (1.0, 1.2, 0.825)


def bin_scene(n=3000):
    """test_gpu_grid3d.test_bin3d_bit_exact's scene: voxel-corner particles, h from 0.2 to 9 voxels, zero and NaN h"""
    rng = np.random.default_rng(31)
    pos = rng.uniform(-0.05, 1.05, (n, 3))
    d = 1.0 / 40
    on = rng.random(n) < 0.3
    pos[on] = np.round(pos[on] / d) * d
    h = rng.choice([0.2 * d, 0.5 * d, d, 2 * d, 3.7 * d, 9 * d], n)
    h[::19] = 0.0
    h[3::23] = np.nan
    return pos, h


@pytest.mark.parametrize("periodic", [False, True])
def test_whole_window_is_the_oracle_bin3d(oracle, periodic):
    pos, h = bin_scene(1200)
    box = (1.0, 1.0, 1.0) if periodic else None
    o = oracle.bin3d(pos, h, SIZE, LO, HI, small_max_vox=20, huge_min_bricks=60, periodic=periodic, box=box)
    w = bin3d_window(oracle, pos, h, SIZE, LO, HI, (0, SIZE[0]), small_max_vox=20, huge_min_bricks=60, periodic=periodic, box=box)
    assert np.array_equal(w["bbox"], oracle.bbox3d(pos, h, SIZE, LO, HI, periodic=periodic, box=box))
    assert np.array_equal(w["cls"], o["cls"])
    assert np.array_equal(w["sorted"], o["sorted"])
    assert np.array_equal(w["huge"], o["huge"])
    assert len(o["sorted"]) > 300 and len(o["huge"]) > 0


@pytest.mark.parametrize("periodic", [False, True])
@pytest.mark.parametrize("window", [(8, 24), (5, 6), (SIZE[0] - 1, SIZE[0])])
def test_window_bbox_is_a_scan_of_the_window_corners(oracle, periodic, window):
    pos, h = bin_scene(600)
    box = (1.0, 1.0, 1.0) if periodic else None
    got = bbox3d_window(oracle, pos, h, SIZE, LO, HI, window, periodic, box)
    n_img, s3 = oracle.images3(periodic, box)
    s3 = np.asarray(s3).reshape(-1, 3)
    d = [(HI[c] - LO[c]) / SIZE[c] for c in range(3)]
    idx = [np.arange(window[0], window[1]), np.arange(SIZE[1]), np.arange(SIZE[2])]
    N = len(h)
    for m in range(n_img):
        for i in range(N):
            R = 2.0 * h[i]
            R2 = R * R
            want = [0, -1, 0, -1, 0, -1]
            if h[i] > 0.0:
                hits = []
                for c in range(3):
                    t = (pos[i, c] + s3[m, c]) - (LO[c] + idx[c].astype(np.float64) * d[c])
                    hits.append(np.flatnonzero(t * t < R2))
                if all(len(k) for k in hits):
                    want = [int(v) for k in hits for v in (k[0], k[-1])]
            assert list(got[m * N + i]) == want, (m, i)


@pytest.mark.parametrize("nx,world", [(512, 8), (64, 1), (20, 4), (7, 3), (100, 3), (8, 2), (1, 1), (33, 32)])
def test_plane_edges(nx, world):
    from astro_sph_tools_b200.distributed import grid_slab_planes
    e = grid_slab_planes(nx, world)
    assert len(e) == world + 1 and e[0] == 0 and e[-1] == nx
    assert all(a <= b for a, b in zip(e[:-1], e[1:]))
    assert all(v % 8 == 0 or v == nx for v in e[:-1])                # whole bricks, the last one clipped to nx
    if -(-nx // 8) < world:                                        # fewer bricks than ranks
        assert any(a == b for a, b in zip(e[:-1], e[1:]))
    assert e == grid_slab_planes(nx, world)                       # every rank derives the same edges


def sharded_scene(periodic):
    rng = np.random.default_rng(5 if periodic else 6)
    n = 700
    L = np.array([1.0, 0.7, 1.3]) if periodic else np.ones(3)
    pos = rng.uniform(0.0, 1.0, (n, 3)) * L if periodic else rng.uniform(-0.1, 1.1, (n, 3))
    h = rng.choice([0.01, 0.03, 0.08, 0.3], n, p=[0.4, 0.3, 0.2, 0.1])
    h[::41] = 0.0
    prop = rng.normal(size=n)
    size, lo, hi = ((20, 14, 26), (0.0, 0.0, 0.0), tuple(L)) if periodic else ((28, 12, 10), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))
    box = tuple(L) if periodic else None
    return pos, h, prop, size, lo, hi, box


@pytest.mark.parametrize("periodic", [False, True])
def test_grid_sharded_slabs_are_bit_equal_to_the_whole_oracle_grid(oracle, thread_ranks, periodic):
    from astro_sph_tools_b200 import distributed as astd
    pos, h, prop, size, lo, hi, box = sharded_scene(periodic)
    world = 3
    ref = oracle.grid3d(pos, h, prop, size, lo, hi, periodic=periodic, box=box, nthreads=1)
    cuts = [0, 100, 450, len(h)]                                  # unequal contiguous index shards

    def body(r):
        a, b = cuts[r], cuts[r + 1]
        t = lambda x: torch.from_numpy(np.ascontiguousarray(x[a:b]))
        slab, x0, st = astd.grid_sharded(OracleGridder(oracle), t(pos), t(h), t(prop), size, lo, hi, "cubic_spline_3d", periodic, box,
                                         return_stats=True, router=OracleRouter(oracle))
        whole = astd.collect_slabs(slab, size[0], dst=1)
        every = astd.collect_slabs(slab, size[0], all_ranks=True)
        return slab.numpy(), x0, st, None if whole is None else whole.numpy(), every.numpy()

    res = thread_ranks(world, body)
    e = astd.grid_slab_planes(size[0], world)
    for r, (slab, x0, st, whole, every) in enumerate(res):
        assert x0 == e[r] and slab.shape == (e[r + 1] - e[r],) + tuple(size[1:])
        assert np.array_equal(slab, ref[e[r]:e[r + 1]]), f"rank {r}"
        assert (whole is not None) == (r == 1)
        assert np.array_equal(every, ref)
        assert len(st["sent"]) == world and st["fan_out"] >= 0.0
    assert np.array_equal(res[1][3], ref)
    assert sum(st["received"] for _, _, st, _, _ in res) == sum(sum(st["sent"]) for _, _, st, _, _ in res)


@pytest.mark.parametrize("nx,world", [(28, 3), (100, 3), (20, 4), (64, 8), (9, 2)])
def test_collect_slabs_on_dst_and_on_every_rank(thread_ranks, nx, world):
    """slabs of unequal thickness (and empty ones) come back as the whole grid, plane for plane, on dst or on every rank"""
    from astro_sph_tools_b200 import distributed as astd
    e = astd.grid_slab_planes(nx, world)
    whole = torch.arange(nx * 3 * 2, dtype=torch.float64).reshape(nx, 3, 2)
    dst = world - 1

    def body(r):
        slab = whole[e[r]:e[r + 1]].clone()
        one = astd.collect_slabs(slab, nx, dst=dst)
        every = astd.collect_slabs(slab, nx, all_ranks=True)
        return one, every

    for r, (one, every) in enumerate(thread_ranks(world, body)):
        assert (one is None) == (r != dst)
        assert torch.equal(every, whole)
        if one is not None:
            assert torch.equal(one, whole)


def test_grid_sharded_refuses_host_tensors_before_routing():
    """the default router hands raw pointers to a CUDA kernel: host tensors are refused before anything is launched"""
    from astro_sph_tools_b200 import distributed as astd
    pos, h, prop = torch.zeros((4, 3), dtype=torch.float64), torch.ones(4, dtype=torch.float64), torch.ones(4, dtype=torch.float64)
    before = dict(astd._grid_routers)
    with pytest.raises(ValueError, match="CUDA"):
        astd.grid_sharded(OracleGridder(None), pos, h, prop, (8, 8, 8), (0, 0, 0), (1, 1, 1))
    assert astd._grid_routers == before                            # no router (and no workspace) was made
