"""Scenes of the geometry tests (test infrastructure, plain numpy): periodic boxes whose sides differ, 2-D projections of a
3-D box on each axis, anisotropic cells, odd grid shapes, a scene for every branch of the 3-D brick kernel, and Python
kernel functions that restate the built-in kernels (so that kernel_id_of tabulates them).  Shared by
tests/test_geometry_pin_cpu.py (the oracle and the per-cell gate, no device) and tests/test_gpu_geometry_pixelwise.py."""
import zlib

import numpy as np

BOX3 = (1.0, 0.7, 1.3)                     # every side different
BOX3_2D = (10.0, 7.0, 13.0)                # the box of the 2-D projections
PLANE = {0: (1, 2), 1: (0, 2), 2: (0, 1)}  # in-plane position columns of each projection axis


def seed_of(*key):
    return zlib.crc32(repr(key).encode()) % 100_000


def cells(size, lo, hi):
    return [(hi[c] - lo[c]) / size[c] for c in range(len(size))]


def log_h(rng, n, lo, hi):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), n))


PRESORT_MIN_N = 65536                      # the spatial pre-ordering leaves smaller sets alone (presort.cuh)


def pad_for_presort(pos, h, prop, seed):
    """insert particles with h = NaN (they never contribute, and the forced paths keep them) at random places, keeping the
    order of the others, so that the set is large enough for the spatial pre-ordering to act on it (with room for the
    particles the forced paths drop)"""
    n = len(h)
    m = max(PRESORT_MIN_N + 4096 - n, 0)
    rng = np.random.default_rng(seed)
    at = np.sort(rng.integers(0, n + 1, m))
    pos = np.insert(pos, at, rng.uniform(0.0, 1.0, (m, 3)), axis=0)
    return pos, np.insert(h, at, np.nan), np.insert(prop, at, rng.normal(size=m))


def keep_forced(h, size, lo, hi):
    """the forced tile / brick paths need h >= half of the LARGEST cell side for their float32 relative coordinates"""
    return ~(h < 0.5 * max(cells(size, lo, hi)))


# ---- non-cubic periodic boxes, 3-D -----------------------------------------------------------------------------------
# window: (grid size, lo, hi).  Voxels are within a few per cent of cubic (d ~ 0.042).
BOX_WINDOWS = {
    "box": ((24, 17, 31), (0.0, 0.0, 0.0), BOX3),
    "inside": ((15, 11, 17), (0.15, 0.1, 0.3), (0.75, 0.55, 1.0)),
    "past_low": ((24, 17, 31), tuple(-0.2 * L for L in BOX3), tuple(0.8 * L for L in BOX3)),
}


def box_scene3d(window, n=2500):
    """particles in [0, L) of BOX3: h from 0.3 to 8 voxels, a few whose support exceeds half the shortest side (their
    images overlap each other), and particles exactly at 0 and just below L on every axis"""
    rng = np.random.default_rng(seed_of("box3", window))
    L = np.array(BOX3)
    pos = rng.uniform(0.0, 1.0, (n, 3)) * L
    d = 0.042
    h = log_h(rng, n, 0.3 * d, 8 * d)
    h[::150] = rng.uniform(0.2, 0.3, len(h[::150]))         # 2h > 0.35 = half of the shortest side
    prop = rng.normal(size=n)
    k = 0
    for c in range(3):
        for v in (0.0, np.nextafter(L[c], 0.0)):
            for hh in (0.5 * d, 2.5 * d):
                pos[k, c] = v
                h[k] = hh
                k += 1
    size, lo, hi = BOX_WINDOWS[window]
    return pos, h, prop, size, lo, hi


# ---- 3-component boxes in 2-D --------------------------------------------------------------------------------------
def box_scene2d(axis, n=3000):
    """particles in BOX3_2D projected along `axis` onto the whole in-plane face of the box (pixels near-square)"""
    rng = np.random.default_rng(seed_of("box2", axis))
    L = np.array(BOX3_2D)
    pos = rng.uniform(0.0, 1.0, (n, 3)) * L
    a, b = PLANE[axis]
    size = (int(round(L[a] / 0.2)), int(round(L[b] / 0.2)))
    h = log_h(rng, n, 0.3 * 0.2, 8 * 0.2)
    h[::100] = rng.uniform(2.0, 3.0, len(h[::100]))         # support beyond half the shortest side
    prop = rng.normal(size=n)
    for k, c in enumerate((a, b)):
        pos[4 * k, c] = 0.0
        pos[4 * k + 1, c] = np.nextafter(L[c], 0.0)
    bounds = (0.0, L[a], 0.0, L[b])
    return pos, h, prop, size, bounds, (L[a], L[b])


# ---- anisotropic cells -----------------------------------------------------------------------------------------------
ANISO3 = {"64x64x2": (64, 64, 2), "256x256x2": (256, 256, 2), "16x16x64": (16, 16, 64), "48x6x48": (48, 6, 48)}
ANISO2 = {"512x8": ((512, 8), (0.0, 10.0, 0.0, 10.0)), "16x2048": ((16, 2048), (0.0, 10.0, 0.0, 10.0)),
          "256sq_100x1": ((256, 256), (0.0, 100.0, 0.0, 1.0))}


def aniso_scene3d(name, n=3000):
    """unit cube; h from 0.3 to 8 SHORT voxels (so the default classes send particles with h << half a long voxel through
    the brick path), and 2 % with h of half to one long voxel, which the forced brick paths keep"""
    size = ANISO3[name]
    lo, hi = (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)
    rng = np.random.default_rng(seed_of("aniso3", name))
    ds, dl = min(cells(size, lo, hi)), max(cells(size, lo, hi))
    pos = rng.uniform(0.0, 1.0, (n, 3))
    h = log_h(rng, n, 0.3 * ds, 8 * ds)
    big = rng.random(n) < 0.02
    h[big] = rng.uniform(0.5 * dl, dl, int(big.sum()))
    prop = rng.normal(size=n)
    return pos, h, prop, size, lo, hi


def aniso_scene2d(name, n=3000):
    size, b = ANISO2[name]
    rng = np.random.default_rng(seed_of("aniso2", name))
    d = cells(size, (b[0], b[2]), (b[1], b[3]))
    ds, dl = min(d), max(d)
    pos = np.empty((n, 3))
    pos[:, 0] = rng.uniform(b[0], b[1], n)
    pos[:, 1] = rng.uniform(b[2], b[3], n)
    pos[:, 2] = rng.uniform(0.0, 1.0, n)
    h = log_h(rng, n, 0.3 * ds, 8 * ds)
    big = rng.random(n) < 0.02
    h[big] = rng.uniform(0.5 * dl, dl, int(big.sum()))
    prop = rng.normal(size=n)
    return pos, h, prop, size, b


# ---- odd grid shapes, 3-D --------------------------------------------------------------------------------------------
ODD_SHAPES = [(1, 1, 64), (1, 37, 5), (8, 8, 1), (7, 9, 3), (9, 17, 33), (33, 8, 2), (65, 1, 12)]


def odd_scene3d(size, n=1500):
    """cubic voxels of 1/24 over a window of `size` voxels; particles reach up to 8 voxels past every face"""
    rng = np.random.default_rng(seed_of("odd", size))
    d = 1.0 / 24
    lo = (0.1, -0.2, 0.05)
    hi = tuple(lo[c] + size[c] * d for c in range(3))
    pos = rng.uniform(np.array(lo) - 8 * d, np.array(hi) + 8 * d, (n, 3))
    h = log_h(rng, n, 0.3 * d, 8 * d)
    prop = rng.normal(size=n)
    return pos, h, prop, size, lo, hi


# ---- the brick kernel's branches -------------------------------------------------------------------------------------
BRANCH_GRID = ((48, 48, 48), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))
BRANCH_KW = dict(pair_capacity=1500, huge_capacity=3, huge_min_bricks=20)
BRANCH_BAND_GAP = 130                      # binary orders between the two weight phases (one band covers 100)


def branch_scene3d():
    """a dense clump inside one brick (more than 1024 pairs there: its list is split into interleaved work items that add
    with float64 atomics, and every warp folds its float32 sums after 96 hits), sparse isolated particles (fewer than 10
    hits per batch: the batches without distance tables), large-h particles whose supports put whole 4x4x8 columns in the
    outer annulus 1 <= q < 2 and that go on the large-h list, and weights of two phases 2^130 apart (two bands)"""
    rng = np.random.default_rng(77)
    d = 1.0 / 48
    nc, ns, nl = 2600, 250, 6
    clump = rng.uniform(18.5 * d, 21.5 * d, (nc, 3))         # supports reach voxels 17..23 only: brick (2, 2, 2) = 16..23
    sparse = rng.uniform(0.0, 1.0, (ns, 3))
    large = rng.uniform(0.3, 0.7, (nl, 3))
    pos = np.concatenate([clump, sparse, large])
    h = np.concatenate([rng.uniform(0.8 * d, 1.0 * d, nc), rng.uniform(0.6 * d, 1.5 * d, ns), rng.uniform(6 * d, 9 * d, nl)])
    prop = np.concatenate([rng.uniform(0.5, 1.5, nc), rng.uniform(0.5, 1.5, ns) * 2.0 ** -BRANCH_BAND_GAP,
                           rng.normal(size=nl)])
    return pos, h, prop, nc, ns, nl


def outer_annulus_columns(pos, h, size, lo, hi):
    """number of (particle, 4x4x8 column) pairs with every voxel sample of the column at 1 <= q < 2 and the nearest one
    inside the support (the brick kernel's second, outer-annulus loop)"""
    d = np.array(cells(size, lo, hi))
    n = 0
    cx = np.arange(0, size[0], 4); cy = np.arange(0, size[1], 4); cz = np.arange(0, size[2], 8)
    X0, Y0, Z0 = np.meshgrid(cx, cy, cz, indexing="ij")
    box_lo = np.stack([X0, Y0, Z0], -1).reshape(-1, 3)
    box_hi = np.minimum(box_lo + np.array([3, 3, 7]), np.array(size) - 1)
    for p, hh in zip(pos, h):
        f = (p - np.array(lo)) / d
        dd = np.maximum(np.maximum(box_lo - f, f - box_hi), 0.0) * d
        q = np.sqrt((dd * dd).sum(1)) / hh
        n += int(((q >= 1.0) & (q < 2.0)).sum())
    return n


# ---- kernel functions that restate the built-in kernels (tabulated by kernel_id_of) ---------------------------------
def _cubic_shape(q):
    return np.where(q < 1.0, 1.0 - 1.5 * q * q + 0.75 * q * q * q, np.where(q < 2.0, 0.25 * (2.0 - q) ** 3, 0.0))


def _wendland_shape(q):
    u = 0.5 * q
    return np.where(u < 1.0, (1.0 - u) ** 4 * (1.0 + 4.0 * u), 0.0)


def python_kernels():
    """name of the built-in kernel -> a new Python callable of the same W(r, h) (new objects: kernel_id_of keys its table
    cache on the callable, and the built-in callables themselves are recognised and not tabulated)"""
    return {
        "cubic_spline_3d": lambda r, h: _cubic_shape(r / h) / (np.pi * h ** 3),
        "cubic_spline_2d": lambda r, h: _cubic_shape(r / h) * 10.0 / (7.0 * np.pi * h ** 2),
        "wendland_c2_2d": lambda r, h: _wendland_shape(r / h) * 7.0 / (4.0 * np.pi * h ** 2),
        "wendland_c2_3d": lambda r, h: _wendland_shape(r / h) * 21.0 / (16.0 * np.pi * h ** 3),
    }


KERNEL_DIM = {"cubic_spline_3d": 3, "cubic_spline_2d": 2, "wendland_c2_2d": 2, "wendland_c2_3d": 3}
TABLE_N = 8192                             # TabulatedKernel.N: intervals on q in [0, 2]


def table_kernel(name, shift=0):
    """the device's table rule in float64: linear interpolation between the float32 nodes f(2j / N) of the built-in kernel
    `name`, evaluated at q + shift * dq (shift = 1: the table read one node off)"""
    f = np.asarray(python_kernels()[name](np.linspace(0.0, 2.0, TABLE_N + 1), np.ones(TABLE_N + 1)), dtype=np.float32)
    f = f.astype(np.float64)
    dim = KERNEL_DIM[name]

    def W(r, h):
        q = r / h
        x = (q + shift * 2.0 / TABLE_N) * (TABLE_N / 2)
        j = np.minimum(np.floor(x).astype(np.int64), TABLE_N - 1)
        j = np.clip(j, 0, TABLE_N - 1)
        v = f[j] + (x - j) * (f[j + 1] - f[j])
        return np.where(q < 2.0, v, 0.0) / h ** dim
    return W


def table_scene3d(periodic=False, n=2500):
    rng = np.random.default_rng(seed_of("table3", periodic))
    if periodic:
        size, lo, hi = (20, 14, 26), (0.0, 0.0, 0.0), BOX3
        pos = rng.uniform(0.0, 1.0, (n, 3)) * np.array(BOX3)
    else:
        size, lo, hi = (28, 24, 30), (0.05, 0.0, -0.1), (0.95, 0.8, 0.9)
        pos = rng.uniform(-0.05, 1.0, (n, 3))
    d = max(cells(size, lo, hi))
    h = log_h(rng, n, 0.3 * d, 6 * d)
    prop = rng.normal(size=n)
    return pos, h, prop, size, lo, hi


def table_scene2d(n=3000):
    rng = np.random.default_rng(seed_of("table2"))
    pos = rng.uniform(0.0, 10.0, (n, 3))
    size, b = (90, 110), (0.5, 9.5, -0.5, 10.5)
    h = log_h(rng, n, 0.03, 0.6)
    prop = rng.normal(size=n)
    return pos, h, prop, size, b
