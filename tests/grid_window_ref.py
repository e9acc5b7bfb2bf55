"""Reference definitions of the x-window and slab-routing rules of 3-D gridding, written on top of the oracle's whole-grid
output (oracle.bbox3d, oracle.grid3d) and plain float64 numpy.  Test infrastructure only.

  * window bbox: the whole grid's bbox with x clipped to [x_begin, x_end) and shifted by -x_begin; empty (0,-1,0,-1,0,-1)
    when the clipped x range is empty;
  * window bin3d: classes, (brick, particle) pairs and the large-h list from those bboxes and the window's bricks (brick bx
    covers window planes [8 bx, 8 bx + 7]), with the membership test of oracle.bin3d evaluated at the whole grid's voxel
    corners lo + (x_begin + i) * d;
  * routing: particle i goes to rank g iff some image's whole-grid bbox row is non-empty and its [x0, x1] meets
    [e_g, e_{g+1}); rows (x, y, z, h, prop) in ascending particle index per destination."""
import numpy as np


def _box3(periodic, box):
    if not periodic:
        return None
    return (float(box),) * 3 if np.isscalar(box) else tuple(float(v) for v in box)


def bbox3d_window(oracle, pos, h, size, lo, hi, window, periodic=False, box=None):
    bb = oracle.bbox3d(pos, h, size, lo, hi, periodic=periodic, box=_box3(periodic, box))
    x0, x1 = window
    a = np.maximum(bb[:, 0], x0)
    b = np.minimum(bb[:, 1], x1 - 1)
    keep = (bb[:, 1] >= bb[:, 0]) & (a <= b)
    out = np.tile(np.array([0, -1, 0, -1, 0, -1], dtype=np.int32), (bb.shape[0], 1))
    out[keep, 0] = a[keep] - x0
    out[keep, 1] = b[keep] - x0
    out[keep, 2:] = bb[keep, 2:]
    return out


def _brick_min_dist2(p, vmin, d, lo_, hi_, off, brick):
    """per brick b0..b1 of the local voxel range [lo_, hi_]: min over its voxels of (p - (vmin + (off + i) * d))^2"""
    res = []
    for b in range(lo_ // brick, hi_ // brick + 1):
        idx = np.arange(max(b * brick, lo_), min(b * brick + brick - 1, hi_) + 1) + off
        t = p - (vmin + idx.astype(np.float64) * d)
        res.append((b, float(np.min(t * t))))
    return res


def bin3d_window(oracle, pos, h, size, lo, hi, window, brick=8, small_max_vox=64, huge_min_bricks=512, periodic=False, box=None):
    """oracle.bin3d's outputs (cls, sorted, huge) and the window bboxes, for the x window [x_begin, x_end)"""
    pos = np.ascontiguousarray(pos, dtype=np.float64); h = np.ascontiguousarray(h, dtype=np.float64)
    N = len(h)
    n3 = [int(v) for v in size]
    x0, x1 = window
    nw = [x1 - x0, n3[1], n3[2]]
    d = [(hi[c] - lo[c]) / n3[c] for c in range(3)]
    n_img, s3 = oracle.images3(periodic, _box3(periodic, box))
    s3 = np.asarray(s3, dtype=np.float64).reshape(-1, 3)
    img_mul = 1 if n_img == 1 else 32
    nby, nbz = -(-nw[1] // brick), -(-nw[2] // brick)
    bb = bbox3d_window(oracle, pos, h, size, lo, hi, window, periodic, box)
    cls = np.zeros(n_img * N, dtype=np.uint8)
    tiled, huge_entries = [], []

    def members(i, m, row):
        p = [pos[i, c] + s3[m, c] for c in range(3)]
        R = 2.0 * h[i]
        R2 = R * R
        md = [_brick_min_dist2(p[c], lo[c], d[c], row[2 * c], row[2 * c + 1], x0 if c == 0 else 0, brick) for c in range(3)]
        out = []
        for bx, mx in md[0]:
            for by, my in md[1]:
                mxy = mx + my
                for bz, mz in md[2]:
                    if mxy + mz < R2:
                        out.append((((bx * nby + by) * nbz + bz) * img_mul + m) << 32 | i)
        return out

    for i in range(N):
        for m in range(n_img):
            j = m * N + i
            row = bb[j]
            if row[1] < row[0]:
                continue
            ext = [int(row[2 * c + 1] - row[2 * c] + 1) for c in range(3)]
            if ext[0] * ext[1] * ext[2] <= small_max_vox:
                cls[j] = 1
                continue
            nb = 1
            for c in range(3):
                nb *= row[2 * c + 1] // brick - row[2 * c] // brick + 1
            if nb > huge_min_bricks:
                cls[j] = 3
                huge_entries.append((i, m, row))
                continue
            cls[j] = 2
            tiled.extend(members(i, m, row))
    pairs = tiled + [e for i, m, row in huge_entries for e in members(i, m, row)]
    pairs = np.array(pairs, dtype=np.uint64)
    shift = np.uint64(32 + (5 if n_img > 1 else 0))
    order = np.argsort(pairs >> shift, kind="stable")
    huge = np.array([(m << 32) | i for i, m, _ in huge_entries], dtype=np.uint64)
    return dict(bbox=bb, cls=cls.reshape(n_img, N), sorted=pairs[order], huge=huge)


def route_reference(oracle, pos, h, prop, edges, size, lo, hi, periodic=False, box=None):
    """-> (send rows (S, 5), counts per destination): the definition the routing kernel is tested against"""
    pos = np.ascontiguousarray(pos, dtype=np.float64)
    N = len(h)
    world = len(edges) - 1
    if N == 0:
        return np.zeros((0, 5)), np.zeros(world, dtype=np.int64)
    bb = oracle.bbox3d(pos, h, size, lo, hi, periodic=periodic, box=_box3(periodic, box)).reshape(-1, N, 6)
    ok = bb[:, :, 1] >= bb[:, :, 0]
    rows = np.column_stack([pos, np.asarray(h, dtype=np.float64), np.asarray(prop, dtype=np.float64)])
    parts, counts = [], []
    for g in range(world):
        e0, e1 = edges[g], edges[g + 1]
        hit = (ok & (bb[:, :, 0] < e1) & (bb[:, :, 1] >= e0)).any(axis=0) if e1 > e0 else np.zeros(N, dtype=bool)
        idx = np.flatnonzero(hit)
        parts.append(rows[idx])
        counts.append(len(idx))
    return np.concatenate(parts), np.array(counts, dtype=np.int64)


class OracleRouter:
    """route() of distributed._GridRouter on CPU tensors, from route_reference"""

    def __init__(self, oracle):
        self.oracle = oracle

    def route(self, pos, h, prop, edges, grid_size, lo, hi, periodic, box):
        import torch
        send, counts = route_reference(self.oracle, pos.numpy(), h.numpy(), prop.numpy(), edges, grid_size, lo, hi, periodic, box)
        return torch.from_numpy(np.ascontiguousarray(send)), torch.from_numpy(counts), None


class OracleGridder:
    """grid() of Gridder3D on CPU tensors: the whole oracle grid of the particles given, sliced to the x window"""

    def __init__(self, oracle):
        self.oracle = oracle
        self.last_stats = None

    def grid(self, pos, h, prop, grid_size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, x_window=None):
        import torch
        g = self.oracle.grid3d(pos.numpy(), h.numpy(), prop.numpy(), grid_size, lo, hi, kernel=kernel, periodic=periodic,
                               box=_box3(periodic, box), nthreads=1)
        x0, x1 = x_window if x_window is not None else (0, g.shape[0])
        self.last_stats = dict(n_pairs=0, n_huge=0)
        return torch.from_numpy(np.ascontiguousarray(g[x0:x1]))
