"""-m gpu: the multi-GPU paths of distributed.py with their real CUDA kernels, on one GPU, with ranks that are threads of this
process (tests/inprocess_dist.py).

  * smoothing_lengths_slabs (the 1024^3, k = 48 k-NN of bench.py on 8 GPUs, scaled down) with the default solver and the
    slab packing kernel: every rank's h bit-equal to scipy's cKDTree over the whole set.  The inputs ast_knn_h gets there and
    nowhere else: one slab plus ghost layers (wrapping across x = 0 in a periodic box), a cell grid over the whole box at
    cell_target = 1.75 * fill, queries that are the prefix [0, n_owned) in "owned from rank 0, 1, ..." order, and after
    the ghost zone has widened more ghosts than owned particles (the reach-limited build inside ast_knn_h);
  * smoothing_lengths_sharded (replicated positions, q_begin / q_count per rank), bit-equal to scipy;
  * create_images_sharded with the default projector, every map gated per pixel against the float64 oracle;
  * ShardedArrayReorder with the default GPU matcher and row gather, on the golden cases of the reference's class."""
import functools

import numpy as np
import pytest
import torch

from conftest import random_cloud
from inprocess_dist import thread_ranks  # noqa: F401  (fixture)
from reorder_util import golden_reorder_cases, load_reorder

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@functools.lru_cache(maxsize=None)
def _scipy_h(name, k, box):
    import oracle
    return oracle.knn_scipy(SCENES[name]()[0], k, box, workers=-1)[0]


def run_slabs(run, name, world, k, box, shards=None, **kw):
    """smoothing_lengths_slabs on `world` thread-ranks, rank r holding pos[shards[r]] (default: contiguous shard_bounds);
    asserts every rank's h is bit-equal to scipy over the whole set and returns the per-rank stats"""
    from astro_sph_tools_b200 import distributed as astd
    pos = SCENES[name]()[0]
    if shards is None:
        shards = [np.arange(*astd.shard_bounds(len(pos), world, r)) for r in range(world)]
    assert len(shards) == world and sum(len(s) for s in shards) == len(pos)

    def body(r):
        h, st = astd.smoothing_lengths_slabs(dev(pos[shards[r]]), k, box, return_stats=True, **kw)
        return h.cpu().numpy(), st

    res = run(world, body)
    ref = _scipy_h(name, k, box)
    for r, (h, st) in enumerate(res):
        want = ref[shards[r]]
        bad = np.flatnonzero(h != want)
        assert h.shape == want.shape and bad.size == 0, \
            f"rank {r}: {bad.size} of {len(want)} h differ from scipy, e.g. {h[bad[:4]]} vs {want[bad[:4]]}"
    stats = [st for _, st in res]
    assert sum(st["owned"] for st in stats) == len(pos)
    return stats


def random_shards(n, fractions, seed):
    """a random index subset per rank (not a contiguous range), sizes from the cumulative fractions"""
    perm = np.random.default_rng(seed).permutation(n)
    cuts = [0] + [int(f * n) for f in fractions] + [n]
    return [np.sort(perm[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]


# ---- scenes: (positions, _) like synthetic.s1_positions, cached with their scipy reference -------------------------------
@functools.lru_cache(maxsize=None)
def lattice48():
    from astro_sph_tools_b200 import synthetic
    return synthetic.s1_positions(48)


@functools.lru_cache(maxsize=None)
def lattice64():
    from astro_sph_tools_b200 import synthetic
    return synthetic.s1_positions(64)


@functools.lru_cache(maxsize=None)
def clustered():
    from astro_sph_tools_b200 import synthetic
    return synthetic.s2_positions(120_000, 1.0, n_haloes=16, seed=7)


@functools.lru_cache(maxsize=None)
def open_aniso():
    """open box with extents 3 : 1 : 0.5, offset from the origin"""
    rng = np.random.default_rng(31)
    return rng.uniform(0.0, 1.0, (60_000, 3)) * np.array([3.0, 1.0, 0.5]) + np.array([-1.5, 2.0, 0.1]), None


@functools.lru_cache(maxsize=None)
def uniform80k():
    return np.random.default_rng(41).uniform(0.0, 1.0, (80_000, 3)), None


@functools.lru_cache(maxsize=None)
def uniform30k():
    return np.random.default_rng(43).uniform(0.0, 1.0, (30_000, 3)), None


@functools.lru_cache(maxsize=None)
def sheet():
    """60 % of the particles in a sheet thinner than one histogram bin of the slab plan: the equal-count boundaries of
    ranks 1 and 2 of 4 fall into that bin, so those slabs are empty and their ranks own nothing"""
    rng = np.random.default_rng(47)
    pos = rng.uniform(0.0, 1.0, (40_000, 3))
    pos[:24_000, 0] = 0.5 + rng.uniform(0.0, 1.0 / 8192, 24_000)
    return pos, None


BOUNDARY_L = 3.0


@functools.lru_cache(maxsize=None)
def boundary():
    """periodic box of side 3 on 4 ranks, 8 particles in each of the 4096 histogram bins of the slab plan, plus particles
    exactly on the slab faces 0.75, 1.5 and 2.25, one ulp below them at the same (y, z), at 0 and at nextafter(3, 0), each of
    them twice.  The extra particles sit in pairs of neighbouring bins, so the equal-count faces stay at 1024 g bins."""
    rng = np.random.default_rng(53)
    L, nb = BOUNDARY_L, 4096
    b = np.repeat(np.arange(nb), 8)
    base = np.column_stack([(b + rng.uniform(0.1, 0.9, len(b))) / nb * L, rng.uniform(0.0, L, (len(b), 2))])
    extra = []
    for face in (0.75, 1.5, 2.25):
        yz = rng.uniform(0.0, L, (4, 2))
        for x in (face, np.nextafter(face, 0.0)):
            extra.append(np.repeat(np.column_stack([np.full(4, x), yz]), 2, axis=0))
    for x in (0.0, np.nextafter(L, 0.0)):
        extra.append(np.repeat(np.column_stack([np.full(4, x), rng.uniform(0.0, L, (4, 2))]), 2, axis=0))
    return np.concatenate([base] + extra), None


SCENES = dict(lattice48=lattice48, lattice64=lattice64, clustered=clustered, open_aniso=open_aniso, uniform80k=uniform80k,
              uniform30k=uniform30k, sheet=sheet, boundary=boundary)


# ---- smoothing_lengths_slabs ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world,name,order", [(2, "lattice48", "contiguous"), (4, "lattice48", "random"), (8, "lattice64", "contiguous")])
def test_slabs_lattice_periodic_k48(thread_ranks, world, name, order):
    """configs[4] scaled down: jittered lattice, periodic, k = 48; the ghost layers of the first and last slab wrap across
    x = 0; with random shards every rank holds particles of every slab"""
    n = len(SCENES[name]()[0])
    shards = random_shards(n, np.arange(1, world) / world, world) if order == "random" else None
    stats = run_slabs(thread_ranks, name, world, 48, 1.0, shards)
    assert all(st["local_set"] < 0.95 * n for st in stats)                  # slab + ghosts, not the whole set


@pytest.mark.parametrize("ghost_width", [0.002, 0.25])
def test_slabs_clustered_periodic_k48(thread_ranks, ghost_width):
    """NFW-clustered set on 4 ranks.  0.002: the ghost zone is too thin for the crowded-out queries and doubles (the widening
    loop with the real solver).  0.25: every rank holds more ghosts than owned particles, so ast_knn_h builds its cell list
    from the particles within reach of the queries only"""
    stats = run_slabs(thread_ranks, "clustered", 4, 48, 1.0, ghost_width=ghost_width)
    if ghost_width < 0.01:
        assert all(st["iterations"] >= 2 for st in stats)
    else:
        assert all(st["local_set"] > 2 * st["owned"] for st in stats)


def test_slabs_open_anisotropic_box_random_subsets(thread_ranks):
    """open box 3 : 1 : 0.5, k = 32 (the reference's default), 3 ranks that hold random index subsets of unequal size"""
    n = len(open_aniso()[0])
    run_slabs(thread_ranks, "open_aniso", 3, 32, None, random_shards(n, [0.2, 0.55], 3))


@pytest.mark.parametrize("ghost_width", [0.3, 0.5])
def test_slabs_ghost_zone_wider_than_a_slab(thread_ranks, ghost_width):
    """8 ranks, slabs about 1/8 wide.  0.3: every rank's ghosts come from at least three other slabs.  0.5 = L / 2: every
    particle goes everywhere (covers_all)"""
    stats = run_slabs(thread_ranks, "uniform80k", 8, 48, 1.0, ghost_width=ghost_width)
    n, owned_max = len(uniform80k()[0]), max(st["owned"] for st in stats)
    for st in stats:
        if ghost_width >= 0.5:
            assert st["local_set"] == n
        else:
            assert st["local_set"] - st["owned"] > 2 * owned_max


def test_slabs_rank_without_particles_and_ranks_without_a_slab(thread_ranks):
    """rank 1 of 4 holds no particles; the slabs of ranks 1 and 2 are empty, so they own nothing and answer no query"""
    n = len(sheet()[0])
    shards = random_shards(n, [0.3, 0.3, 0.6], 5)
    assert len(shards[1]) == 0
    stats = run_slabs(thread_ranks, "sheet", 4, 32, 1.0, shards)
    assert [st["owned"] == 0 for st in stats] == [False, True, True, False]


@pytest.mark.parametrize("k", [1, 2, 96, 128])
def test_slabs_k_edges(thread_ranks, k):
    """k = 1 (h = 0), 2, 96 (above 67: the selection kernel is off on a slab's grid) and 128 (the largest k)"""
    run_slabs(thread_ranks, "uniform30k", 4, k, 1.0, random_shards(30_000, [0.25, 0.5, 0.75], k))


def test_slabs_particles_on_slab_faces_and_box_edges(thread_ranks):
    """particles exactly on the faces _slab_plan returns, one ulp below them, at 0 and at nextafter(L, 0), every one of them
    twice (ties: h stays bit-equal), shuffled over the ranks so that duplicates are held by different ranks"""
    from astro_sph_tools_b200 import distributed as astd
    pos = boundary()[0]
    shards = random_shards(len(pos), [0.25, 0.5, 0.75], 11)
    faces = thread_ranks(4, lambda r: astd._slab_plan(dev(pos[shards[r], 0]), 0.0, BOUNDARY_L, 4)[1].cpu().numpy())
    for f in faces:
        assert np.array_equal(f, [0.0, 0.75, 1.5, 2.25, 3.0])
    run_slabs(thread_ranks, "boundary", 4, 32, BOUNDARY_L, shards)
    run_slabs(thread_ranks, "boundary", 4, 48, BOUNDARY_L, shards, ghost_width=0.01)


# ---- smoothing_lengths_sharded ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k,box,cuts", [("lattice48", 48, 1.0, None), ("open_aniso", 32, None, [0, 9_000, 41_000, 60_000])])
def test_sharded_smoothing_lengths(thread_ranks, name, k, box, cuts):
    """positions all-gathered (unequal shards are padded), every rank answers its own index range of the replicated set"""
    from astro_sph_tools_b200 import distributed as astd
    pos = SCENES[name]()[0]
    world = 4 if cuts is None else len(cuts) - 1
    if cuts is None:
        cuts = [astd.shard_bounds(len(pos), world, r)[0] for r in range(world)] + [len(pos)]
    res = thread_ranks(world, lambda r: astd.smoothing_lengths_sharded(dev(pos[cuts[r]:cuts[r + 1]]), k, box).cpu().numpy())
    ref = _scipy_h(name, k, box)
    for r, h in enumerate(res):
        assert np.array_equal(h, ref[cuts[r]:cuts[r + 1]]), f"rank {r}"


# ---- create_images_sharded --------------------------------------------------------------------------------------------------
def _image_scene(periodic):
    if periodic:
        from geometry_scenes import BOX3_2D, box_scene2d
        pos, h, prop, size, bounds, pair = box_scene2d(1)
        props = np.stack([prop, np.abs(prop) * 1e-30])
        return pos, h, props, size, 1, bounds, dict(periodic=True, box_size=BOX3_2D), dict(periodic=True, box=pair)
    pos, h, prop = random_cloud(61, 20_000, h_hi=0.8)
    props = np.stack([prop, np.random.default_rng(62).normal(size=len(h))])
    return pos, h, props, (128, 96), 2, (0.0, 10.0, 1.0, 9.0), {}, {}


@pytest.mark.parametrize("periodic,all_ranks", [(False, False), (False, True), (True, False)])
def test_create_images_sharded_pixelwise(thread_ranks, oracle, periodic, all_ranks):
    """3 ranks with unequal index shards deposit their particles and the partial maps are summed on dst = 1 (or on every
    rank); each returned map is gated per pixel against the oracle's map of the whole set, the other ranks get None"""
    from astro_sph_tools_b200 import CoordinateAxes, distributed as astd
    from pixel_bound import assert_pixelwise, envelope2d
    from test_gpu_pixelwise import global_gates
    pos, h, props, size, axis, b, kw, okw = _image_scene(periodic)
    n = len(h)
    cuts = [0, n // 7, (n * 3) // 5, n]

    def body(r):
        s = slice(cuts[r], cuts[r + 1])
        return astd.create_images_sharded(pos[s], h[s], list(props[:, s]), size, 32, CoordinateAxes(axis), *b, dst=1,
                                          all_ranks=all_ranks, **kw)

    maps = thread_ranks(3, body)
    ref = oracle.project2d(pos, h, props, size, axis, *b, **okw)
    env = envelope2d(pos, h, props, size, axis, b, periodic=periodic, box=okw.get("box"))
    for r, m in enumerate(maps):
        if not all_ranks and r != 1:
            assert m is None
            continue
        assert m.shape == ref.shape
        for f in range(len(props)):
            assert_pixelwise(m[f], ref[f], env[f], what=f"rank {r}, field {f}: ")
            global_gates(m[f], ref[f])


# ---- ShardedArrayReorder ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name", golden_reorder_cases())
def test_sharded_reorder_with_the_gpu_matcher(thread_ranks, name, world):
    """the golden results of the reference's ArrayReorder, with sources and targets split unequally over the ranks: each
    rank's output and target_filter equal its slice of the golden result"""
    from astro_sph_tools_b200 import distributed as astd
    g = load_reorder(name)
    src, tgt, data, sf, tf = g["source_ids"], g["target_ids"], g["data"], g["source_order_filter"], g["target_order_filter"]
    if src.dtype != tgt.dtype:
        pytest.skip("ShardedArrayReorder raises TypeError for source and target IDs of different types, as the reference does")
    # ID 2^63 would alias the hash join's empty-slot key after the cast to int64
    assert src.min() > np.iinfo(np.int64).min and tgt.min() > np.iinfo(np.int64).min
    scut = [0] + [int(len(src) * f) for f in ((0.6,) if world == 2 else (0.1, 0.7))] + [len(src)]
    tcut = [0] + [int(len(tgt) * f) for f in ((0.3,) if world == 2 else (0.45, 0.5))] + [len(tgt)]
    part = lambda a, c, r: None if a is None else a[c[r]:c[r + 1]]

    def body(r):
        # (the cases without a default value match every target)
        ro = astd.ShardedArrayReorder.create(part(src, scut, r), part(tgt, tcut, r), part(sf, scut, r), part(tf, tcut, r))
        return ro(part(data, scut, r), default_value=g["default_value"]), ro.target_filter

    res = thread_ranks(world, body)
    for r, (out, mine) in enumerate(res):
        want = part(g["result"], tcut, r)
        assert np.array_equal(mine, part(g["target_filter"], tcut, r)), f"rank {r}"
        assert out.dtype == want.dtype and np.array_equal(out, want), f"rank {r}"
