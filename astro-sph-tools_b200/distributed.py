"""Multi-GPU projection: particles shard by index across ranks (one process per GPU), every rank deposits its
shard onto a full-size partial map, and the partial maps are summed with ONE collective.

This mirrors how the reference distributes particles (each MPI rank reads a disjoint particle subset,
io/EAGLE/_SnapshotEAGLE.py:120-130); the reference has no map reduction because its projector is single-process.
Deposition is linear in the particles, so sum_g map(shard_g) == map(all particles) up to float summation order.
The collective is torch.distributed (NCCL over NVLink on GPUs; gloo in the CPU tests of the host logic).
"""
import numpy as np


def shard_bounds(n, world_size, rank):
    """contiguous index range [lo, hi) of rank `rank` when n particles are split over world_size ranks"""
    base, rem = divmod(int(n), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def reduce_maps(partial, dst=0, group=None, all_ranks=False):
    """Sum the per-rank partial maps (a torch tensor, in place).  all_ranks=False: result valid on `dst` only."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return partial
    if all_ranks:
        dist.all_reduce(partial, op=dist.ReduceOp.SUM, group=group)
    else:
        dist.reduce(partial, dst=dst, op=dist.ReduceOp.SUM, group=group)
    return partial


def project_sharded(projector, pos, h, props, image_size, axis, bounds, kernel="cubic_spline_3d", periodic=False, box=None,
                    dst=0, group=None, all_ranks=False, out=None):
    """Device-resident sharded projection: this rank's particles in, summed map(s) out (valid on dst / all ranks)."""
    part = projector.project(pos, h, props, image_size, axis, bounds, kernel, periodic, box, out=out)
    return reduce_maps(part, dst, group, all_ranks)


def create_images_sharded(positions, smoothing_lengths, particle_properties, image_size, chunk_size, projection_axis,
                          x_min, x_max, y_min, y_max, kernel_func=None, *, periodic=False, box_size=None, dst=0, group=None,
                          all_ranks=False):
    """Host-buffer entry for one rank of a multi-GPU job: same arguments as create_images, but the arrays hold only
    THIS rank's particles.  Returns the summed (P,nx,ny) float64 numpy maps on `dst` (or every rank), else None."""
    import torch
    import torch.distributed as dist
    from .tools.projections._projector import _validate, default_projector
    from .tools.projections._kernels import kernel_id_of, quartic_spline_kernel
    kernel = kernel_id_of(kernel_func if kernel_func is not None else quartic_spline_kernel)
    positions, smoothing_lengths, props = _validate(positions, smoothing_lengths, list(particle_properties))
    eng = default_projector()
    from . import _lib
    parts = []
    for s0 in range(0, len(props), _lib.MAX_PROPS):              # more weight fields than one pass takes: several passes, like create_images
        parts.append(eng.project_host(positions, smoothing_lengths, props[s0:s0 + _lib.MAX_PROPS], image_size, projection_axis,
                                      (x_min, x_max, y_min, y_max), kernel, periodic, box_size, return_device=True))
    part = parts[0] if len(parts) == 1 else torch.cat(parts, dim=0)
    part = reduce_maps(part, dst, group, all_ranks)
    rank = dist.get_rank(group) if dist.is_available() and dist.is_initialized() else 0
    if all_ranks or rank == dst:
        host = torch.empty(part.shape, dtype=part.dtype, pin_memory=True)
        host.copy_(part)
        return host.numpy()
    return None


def gather_positions(pos_local, group=None):
    """All ranks hold consecutive index ranges of the particle set (the reference's per-rank read,
    io/EAGLE/_SnapshotEAGLE.py:120-130): returns (all positions (N,3) on this rank's device, offset of this rank's range).
    ONE collective (all-gather; NCCL over NVLink on GPUs), shards may differ in length (padded to the longest)."""
    import torch
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return pos_local, 0
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n_local = torch.tensor([pos_local.shape[0]], dtype=torch.int64, device=pos_local.device)
    sizes = [torch.zeros_like(n_local) for _ in range(world)]
    dist.all_gather(sizes, n_local, group=group)
    sizes = [int(t.item()) for t in sizes]
    n_max = max(sizes)
    padded = pos_local
    if pos_local.shape[0] < n_max:
        padded = torch.zeros((n_max, 3), dtype=pos_local.dtype, device=pos_local.device)
        padded[:pos_local.shape[0]] = pos_local
    parts = [torch.empty((n_max, 3), dtype=pos_local.dtype, device=pos_local.device) for _ in range(world)]
    dist.all_gather(parts, padded.contiguous(), group=group)
    return torch.cat([p[:m] for p, m in zip(parts, sizes)], dim=0), sum(sizes[:rank])


def smoothing_lengths_sharded(pos_local, k=32, box_size=None, group=None, solver=None):
    """Multi-GPU smoothing lengths: this rank's particles in (a (n_g,3) float64 tensor on its GPU), this rank's h out (n_g,).
    Positions are all-gathered once (1024^3 x 24 B = 25.8 GB fits every 180 GB GPU); every rank then answers its own index
    range on a cell list built from the particles within reach of it (ast_knn_h with q_begin / q_count).  `solver` is any
    object with SmoothingLengthSolver.solve's signature (the CPU tests of this host logic inject a scipy-based one)."""
    if solver is None:
        from .tools.smoothing import SmoothingLengthSolver
        solver = SmoothingLengthSolver()
    pos_all, offset = gather_positions(pos_local, group)
    n_local = pos_local.shape[0]
    if n_local == pos_all.shape[0]:
        return solver.solve(pos_all, k, box_size)
    return solver.solve(pos_all, k, box_size, q_begin=offset, q_count=n_local)


# ---- ID matching across ranks (SURVEY 8(f) N4) ---------------------------------------------------------------------------
def gather_rows(local, group=None):
    """All-gather of per-rank arrays that differ in their first dimension (padded to the longest; ONE data collective plus
    the sizes).  Returns (concatenation in rank order, list of per-rank row counts)."""
    import torch
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return local, [local.shape[0]]
    world = dist.get_world_size(group)
    n_local = torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device)
    sizes = [torch.zeros_like(n_local) for _ in range(world)]
    dist.all_gather(sizes, n_local, group=group)
    sizes = [int(t.item()) for t in sizes]
    n_max = max(sizes)
    padded = local
    if local.shape[0] < n_max:
        padded = torch.zeros((n_max,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        padded[:local.shape[0]] = local
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded.contiguous(), group=group)
    return torch.cat([p[:m] for p, m in zip(parts, sizes)], dim=0), sizes


class ShardedArrayReorder:
    """The reference's MPI reorder (tools/_ArrayReorder.py:88-258 ArrayReorder_MPI_2: every rank holds a piece of the source
    IDs / data and a piece of the target IDs; IDs and data are gathered on the root rank, matched there on one core, and the
    reordered rows scattered back) with the root bottleneck removed: the (filtered) source IDs are all-gathered once at
    create(), every rank joins its OWN target IDs against them on its GPU (hash join, ast_match_ids), and a call all-gathers the
    source rows and gathers this rank's rows locally (ast_gather_rows).  Same contract per rank: output[i] is the source row
    whose ID equals this rank's target ID i, `default_value` where no rank holds it.

    `matcher(source_ids, target_ids, source_filter, target_filter) -> int64 index of the source element per target (-1: none)`
    and `row_gather(rows, index, default) -> rows[index]` default to the CUDA entry points; the CPU tests of this host logic
    inject numpy stand-ins (there is no CPU fallback on the product path)."""

    def __init__(self, t2s, n_source_local, source_filter_local, group, row_gather):
        self._t2s = t2s                                   # index into the gathered FILTERED source rows, -1 = no match
        self._n_source_local = n_source_local
        self._source_filter_local = source_filter_local
        self._group = group
        self._row_gather = row_gather
        self.target_filter = t2s >= 0
        self.matched_items = int(self.target_filter.sum())

    @staticmethod
    def create(source_order, target_order, source_order_filter=None, target_order_filter=None, group=None, matcher=None,
               row_gather=None, device=None):
        import torch
        if source_order.dtype != target_order.dtype:          # tools/_ArrayReorder.py:229-231
            raise TypeError(f"Input source and target order arrays have different datatypes ({source_order.dtype} and "
                            f"{target_order.dtype}).\nThese input arrays MUST declare matching datatypes.")
        if matcher is None:
            from .tools._ArrayReorder import _match as matcher
        if row_gather is None:
            from .tools._ArrayReorder import gather_rows_device as row_gather
        sf = np.ones(source_order.shape[0], dtype=bool) if source_order_filter is None else np.asarray(source_order_filter, dtype=bool)
        ids_local = torch.from_numpy(np.ascontiguousarray(source_order[sf]).astype(np.int64, copy=False))
        if device is not None:
            ids_local = ids_local.to(device)
        ids_all, _ = gather_rows(ids_local, group)
        t2s = np.asarray(matcher(ids_all.cpu().numpy(), np.asarray(target_order), None, target_order_filter))
        return ShardedArrayReorder(t2s, source_order.shape[0], sf, group, row_gather)

    def __call__(self, source_data, default_value=None):
        import torch
        if source_data.shape[0] != self._n_source_local:
            raise IndexError("One or more ranks provided the wrong number of input data elements.")     # :147-148
        if default_value is None and self.matched_items != self._t2s.shape[0]:
            raise ValueError("More output elements expected than matches but no default value provided and no output target "
                             "array to write matches to.")
        rows = torch.from_numpy(np.ascontiguousarray(source_data[self._source_filter_local]))
        rows_all, _ = gather_rows(rows, self._group)
        return self._row_gather(rows_all.numpy(), self._t2s, default_value)


# ---- smoothing lengths on slabs with ghost zones (SURVEY 8(e): the k-NN path has ONE exchange step) ------------------------
def _slab_plan(x, lo, length, world, n_bins=4096, group=None):
    """Equal-count slab boundaries along one axis from a global histogram (ONE small all-reduce).  Ownership is decided on the
    integer bin of a particle, so every rank derives the same owner for the same coordinate.  Returns (owner per local particle,
    boundaries (world + 1,) as float64 tensor)."""
    import torch
    import torch.distributed as dist
    bins = torch.clamp(((x - lo) / length * n_bins).floor().long(), 0, n_bins - 1)
    hist = torch.bincount(bins, minlength=n_bins).to(torch.int64)
    dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=group)
    cum = hist.cumsum(0)
    targets = (torch.arange(1, world, device=x.device, dtype=torch.int64) * cum[-1]) // world
    edges = torch.searchsorted(cum, targets, right=False) + 1                   # slab g owns bins [edges[g-1], edges[g])
    edges = torch.clamp(edges, 0, n_bins)
    owner = torch.bucketize(bins, edges, right=True)                             # number of edges <= bin
    full = torch.cat([torch.zeros(1, dtype=torch.int64, device=x.device), edges, torch.full((1,), n_bins, dtype=torch.int64, device=x.device)])
    return owner, lo + length * full.to(torch.float64) / n_bins


def _route_torch(pos_local, x, owner, b_lo, b_hi, w, length, periodic, covers_all, world):
    """destinations of every local particle, one pass of torch index operations per destination rank (CPU tensors: the gloo
    tests of the host logic; also the definition the packing kernel is tested against).
    Returns (send rows [owned -> 0 | owned -> 1 | ... | ghosts -> 0 | ...] (S,3), src_index (S,), counts (2, world) int64 on the host)."""
    import torch
    own_idx, ghost_idx = [], []
    for g in range(world):
        own = owner == g
        if periodic:
            t = torch.remainder(x - b_lo[g], length)
            seg = b_hi[g] - b_lo[g]
            d = torch.where(t <= seg, torch.zeros_like(t), torch.minimum(t - seg, length - t))
        else:
            d = torch.clamp(torch.maximum(b_lo[g] - x, x - b_hi[g]), min=0.0)
        ghost = (~own) & ((d <= w) | covers_all)
        own_idx.append(torch.nonzero(own).flatten())
        ghost_idx.append(torch.nonzero(ghost).flatten())
    counts = torch.tensor([[t.numel() for t in own_idx], [t.numel() for t in ghost_idx]], dtype=torch.int64)
    src = torch.cat(own_idx + ghost_idx)
    return pos_local[src].contiguous(), src, counts


class _SlabRouter:
    """the packing kernel behind ast_slab_route_count / _write (csrc/slabroute.cu): two passes over the local particles in all"""

    def __init__(self, device):
        from . import _lib
        self._lib = _lib
        self.lib = _lib.load()
        self.device = device
        self._ws = None

    def route(self, pos_local, owner, bounds, w, length, periodic, covers_all, world):
        import ctypes as C
        import torch
        _lib = self._lib
        p = _lib.SlabRouteParams()
        p.n = pos_local.shape[0]; p.world = world; p.periodic = 1 if periodic else 0; p.covers_all = 1 if covers_all else 0
        p.length = float(length); p.w = float(w)
        for g, b in enumerate(bounds.tolist()):
            p.bounds[g] = b
        need = C.c_size_t(0)
        _lib.check(self.lib.ast_slab_route_workspace_bytes(C.byref(p), C.byref(need)))
        if self._ws is None or self._ws.numel() < need.value:
            self._ws = None
            self._ws = torch.empty(need.value, dtype=torch.uint8, device=self.device)
        stream = _lib.stream_ptr(None)
        counts_d = torch.empty(2 * world, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.ast_slab_route_count(C.byref(p), _lib.ptr(pos_local), _lib.ptr(owner), _lib.ptr(counts_d), _lib.ptr(self._ws),
                                                 C.c_size_t(self._ws.numel()), stream))
        counts = counts_d.cpu().view(2, world)
        total = int(counts.sum())
        send = torch.empty((total, 3), dtype=torch.float64, device=self.device)
        src = torch.empty(total, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.ast_slab_route_write(C.byref(p), _lib.ptr(pos_local), _lib.ptr(owner), _lib.ptr(send), _lib.ptr(src),
                                                 _lib.ptr(self._ws), C.c_size_t(self._ws.numel()), stream))
        return send, src, counts


def smoothing_lengths_slabs(pos_local, k=32, box_size=None, group=None, solver=None, ghost_width=None, return_stats=False):
    """Multi-GPU smoothing lengths WITHOUT replicating the positions: every rank passes the particles it holds (any index
    range, any spatial distribution: the reference's per-rank read, io/EAGLE/_SnapshotEAGLE.py:120-130) and gets their h back.

      1. slabs of equal particle count along x from a global histogram (one small all-reduce);
      2. ONE all-to-all of positions: a particle goes to the rank that owns its slab, and as a ghost to every rank whose slab
         lies within `ghost_width` of it (periodic distance when box_size is given);
      3. each rank answers its owned queries on owned + ghost particles (ast_knn_h, same float64 arithmetic as scipy, so the
         distances are bit-equal to a search over the whole set);
      4. a query is complete when its K-th distance does not reach beyond the ghost zone; if any query of any rank is not (one
         all-reduce), the ghost width doubles and steps 2-3 repeat (clustered sets with near-empty regions);
      5. ONE all-to-all returns h to the ranks and positions the particles came from.

    Memory per GPU is N/G plus the ghost layers instead of N (1024^3 on 8 GPUs: 3.2 GB of positions + ~15 % ghosts instead of
    25.8 GB).  `solver`: any object with SmoothingLengthSolver.solve's signature (the CPU tests inject a scipy-based one)."""
    import torch
    import torch.distributed as dist
    if solver is None:
        from .tools.smoothing import SmoothingLengthSolver
        solver = SmoothingLengthSolver()
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        h = solver.solve(pos_local, k, box_size)
        return (h, dict(iterations=1, ghost_fraction=0.0)) if return_stats else h
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = pos_local.device
    n_loc = pos_local.shape[0]
    x = pos_local[:, 0].contiguous()
    # global extent (periodic: the box) and the mean K-th neighbour distance it implies
    ext = torch.empty(6, dtype=torch.float64, device=dev)
    if n_loc:
        mn, mx = torch.aminmax(pos_local, dim=0)                  # one pass over the positions
        ext[:3] = mn
        ext[3:] = -mx
    else:
        ext[:] = float("inf")
    dist.all_reduce(ext, op=dist.ReduceOp.MIN, group=group)
    n_tot = torch.tensor([n_loc], dtype=torch.int64, device=dev)
    dist.all_reduce(n_tot, op=dist.ReduceOp.SUM, group=group)
    n_tot = int(n_tot.item())
    if box_size:
        lo, length = 0.0, float(box_size)
        volume = float(box_size) ** 3
    else:
        lo, length = float(ext[0]), max(float(-ext[3] - ext[0]), 1e-300)
        volume = max(length * max(float(-ext[4] - ext[1]), 1e-300) * max(float(-ext[5] - ext[2]), 1e-300), 1e-300)
    owner, bounds = _slab_plan(x, lo, length, world, group=group)
    b_lo, b_hi = bounds[:-1], bounds[1:]
    r_k = (3.0 * k * volume / (4.0 * np.pi * max(n_tot, 1))) ** (1.0 / 3.0)
    w = float(ghost_width) if ghost_width else 1.5 * r_k
    router = None
    if pos_local.is_cuda and world <= 32 and pos_local.dtype == torch.float64 and pos_local.is_contiguous():
        router = _SlabRouter(dev)                                 # (CPU tensors -- the gloo tests of this logic -- take the torch route)
    iterations = 0
    while True:
        iterations += 1
        covers_all = bool(box_size) and w >= 0.5 * length
        # ---- step 2: destinations (distance from x to slab g's interval, along the circle when periodic) and the send buffer
        # [owned -> 0 | owned -> 1 | ... | ghosts -> 0 | ghosts -> 1 | ...]: the packing kernel on the GPU, torch index ops on the CPU
        if router is not None:
            send, src, counts = router.route(pos_local, owner, bounds, w, length, bool(box_size), covers_all, world)
        else:
            send, src, counts = _route_torch(pos_local, x, owner, b_lo, b_hi, w, length, bool(box_size), covers_all, world)
        counts_d = counts.to(dev)
        recv_counts = torch.empty_like(counts_d)
        for row in range(2):
            dist.all_to_all_single(recv_counts[row], counts_d[row].contiguous(), group=group)
        send_owned, send_ghost = counts[0].tolist(), counts[1].tolist()
        rc = recv_counts.cpu()
        own_from, ghost_from = rc[0].tolist(), rc[1].tolist()
        n_owned, n_ghost = sum(own_from), sum(ghost_from)
        n_send_owned = sum(send_owned)
        # two exchanges (owned rows, then ghost rows) leave [owned from all ranks | ghosts from all ranks]: no reorder
        pos_slab = torch.empty((n_owned + n_ghost, 3), dtype=pos_local.dtype, device=dev)
        dist.all_to_all_single(pos_slab[:n_owned], send[:n_send_owned], output_split_sizes=own_from, input_split_sizes=send_owned, group=group)
        dist.all_to_all_single(pos_slab[n_owned:], send[n_send_owned:], output_split_sizes=ghost_from, input_split_sizes=send_ghost, group=group)
        src_owned = src[:n_send_owned]
        del send
        if n_owned:
            # the slab + ghosts fill only a fraction of the box the cell grid spans: size the cells for ~1.75 particles per OCCUPIED
            # cell (with the default, 8 slabs would put 14 particles in every occupied cell and 2000 candidates in front of a query)
            # (an open box is gridded over the bounding box of the local set itself: nothing to correct there)
            fill = min(1.0, float((b_hi[rank] - b_lo[rank]).item() + 2.0 * w) / length) if box_size else 1.0
            h_owned = solver.solve(pos_slab, k, box_size, q_begin=0, q_count=n_owned if n_owned < pos_slab.shape[0] else 0,
                                   cell_target=max(1.75 * fill, 0.02))
        else:
            h_owned = torch.empty(0, dtype=pos_local.dtype, device=dev)
        # ---- step 4: every neighbour within h of an owned query at x lies in [b_lo - w, b_hi + w]
        if covers_all or (not box_size and w >= length):
            unsafe = torch.zeros(1, dtype=torch.int64, device=dev)
        else:
            xo = pos_slab[:n_owned, 0]
            inf = torch.full_like(xo, float("inf"))
            # (no particle lies below the first slab or above the last one of an open box)
            below = inf if (not box_size and rank == 0) else w + (xo - b_lo[rank]).clamp(min=0.0)
            above = inf if (not box_size and rank == world - 1) else w + (b_hi[rank] - xo).clamp(min=0.0)
            reach = torch.minimum(below, above)
            unsafe = (~(h_owned <= reach)).sum().to(torch.int64).reshape(1)
        dist.all_reduce(unsafe, op=dist.ReduceOp.SUM, group=group)
        if int(unsafe.item()) == 0:
            break
        w *= 2.0
    # ---- step 5: h back to where the particles came from
    back = torch.empty(sum(send_owned), dtype=pos_local.dtype, device=dev)
    dist.all_to_all_single(back, h_owned.contiguous(), output_split_sizes=send_owned, input_split_sizes=own_from, group=group)
    h_local = torch.empty(n_loc, dtype=pos_local.dtype, device=dev)
    h_local[src_owned] = back
    if return_stats:
        return h_local, dict(iterations=iterations, ghost_width=w, ghost_fraction=(pos_slab.shape[0] - n_owned) / max(n_owned, 1),
                             owned=n_owned, local_set=int(pos_slab.shape[0]))
    return h_local


# ---- 3-D gridding on x-slabs of the grid: each rank holds 1/G of the grid, particles go to the slabs their support reaches --
def grid_slab_planes(nx, world):
    """Plane edges e[0..world] of the x-slabs: rank g owns planes [e[g], e[g+1]) of an nx-plane grid.  Slabs are whole bricks
    of 8 planes (the last one clipped to nx), split like shard_bounds, so every rank derives the same edges without a
    collective; when nx < 8 * world the last ranks own no planes."""
    nbx = -(-int(nx) // 8)
    return [min(8 * shard_bounds(nbx, world, g)[0], int(nx)) for g in range(world)] + [int(nx)]


def _check_route_inputs(pos, h, prop):
    """the routing kernel reads pos[3 i], h[i], prop[i] through raw device pointers: anything but contiguous float64 CUDA
    tensors of shapes (N, 3), (N,), (N,) on one device is refused before a launch"""
    import torch
    n = pos.shape[0] if isinstance(pos, torch.Tensor) and pos.dim() == 2 else -1
    for name, t, shape in (("pos", pos, (n, 3)), ("h", h, (n,)), ("prop", prop, (n,))):
        if not isinstance(t, torch.Tensor):
            raise ValueError(f"grid routing: {name} must be a torch tensor")
        if t.dtype != torch.float64 or tuple(t.shape) != shape or not t.is_cuda or not t.is_contiguous() or t.device != pos.device:
            raise ValueError("grid routing needs contiguous float64 CUDA tensors on one device, pos (N,3), h (N,), prop (N,); "
                             f"{name} is {t.dtype} {tuple(t.shape)} on {t.device}{'' if t.is_contiguous() else ', not contiguous'}")


class _GridRouter:
    """the routing kernel behind ast_grid_route_count / _write (csrc/slabroute.cu): two passes over the local particles"""

    def __init__(self, device):
        import threading
        from . import _lib
        import torch
        self._lib = _lib
        self.lib = _lib.load()
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self._ws = None
        self._lock = threading.RLock()        # one workspace: the count and the write pass of a call must not interleave with another's

    def route(self, pos, h, prop, edges, grid_size, lo, hi, periodic, box):
        """-> (send rows (S, 5) = x, y, z, h, prop [-> rank 0 | -> rank 1 | ...], counts per destination (world,) int64 on the
        host, overflow flag (1,) int32 on the device: 1 if the write pass met a row beyond the counted total)"""
        _check_route_inputs(pos, h, prop)
        if pos.device != self.device:
            raise ValueError(f"grid routing: tensors on {pos.device}, router on {self.device}")
        with self._lock:
            return self._route(pos, h, prop, edges, grid_size, lo, hi, periodic, box)

    def _route(self, pos, h, prop, edges, grid_size, lo, hi, periodic, box):
        import ctypes as C
        import torch
        _lib = self._lib
        world = len(edges) - 1
        p = _lib.GridRouteParams()
        p.n = pos.shape[0]; p.world = world; p.periodic = 1 if periodic else 0
        p.nx, p.ny, p.nz = (int(v) for v in grid_size)
        b = (0.0, 0.0, 0.0)
        if periodic:
            b = (float(box),) * 3 if np.isscalar(box) else tuple(float(v) for v in box)
        for c in range(3):
            p.lo[c] = float(lo[c]); p.hi[c] = float(hi[c]); p.box[c] = b[c]
        for g, e in enumerate(edges):
            p.edges[g] = int(e)
        need = C.c_size_t(0)
        _lib.check(self.lib.ast_grid_route_workspace_bytes(C.byref(p), C.byref(need)))
        if self._ws is None or self._ws.numel() < need.value:
            self._ws = None
            self._ws = torch.empty(need.value, dtype=torch.uint8, device=self.device)
        stream = _lib.stream_ptr(None)
        counts_d = torch.empty(world, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.ast_grid_route_count(C.byref(p), _lib.ptr(pos), _lib.ptr(h), _lib.ptr(counts_d), _lib.ptr(self._ws),
                                                 C.c_size_t(self._ws.numel()), stream))
        counts = counts_d.cpu()
        total = int(counts.sum())
        send = torch.empty((total, 5), dtype=torch.float64, device=self.device)
        overflow = torch.empty(1, dtype=torch.int32, device=self.device)
        _lib.check(self.lib.ast_grid_route_write(C.byref(p), _lib.ptr(pos), _lib.ptr(h), _lib.ptr(prop), _lib.ptr(send),
                                                 C.c_int64(total), _lib.ptr(overflow), _lib.ptr(self._ws), C.c_size_t(self._ws.numel()),
                                                 stream))
        return send, counts, overflow


_grid_routers = {}


def default_grid_router(device):
    """one _GridRouter (and its workspace) per device, reused by every grid_sharded call that injects none"""
    import torch
    device = torch.device(device)
    key = torch.device(device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _grid_routers:
        _grid_routers[key] = _GridRouter(key)
    return _grid_routers[key]


def grid_sharded(gridder, pos, h, prop, grid_size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, group=None,
                 return_stats=False, router=None):
    """Multi-GPU 3-D gridding without a full-size grid on any rank: rank r owns planes [e_r, e_{r+1}) of the grid
    (grid_slab_planes) and gets back that slab, a (e_{r+1} - e_r, ny, nz) float64 tensor, with e_r: (slab, x_begin).
    Every rank passes the particles it holds (any index range, any spatial spread):

      1. the routing kernel sends every particle to each rank whose planes its support reaches (rows x, y, z, h, prop, in
         ascending local index per destination);
      2. ONE all-to-all of the per-destination row counts (the split sizes: one host synchronisation), each with the sender's
         routing flag, so that if any rank's write pass met a row beyond its counted total every rank raises RuntimeError
         here (that only happens through a bug; no rank enters the row exchange);
      3. ONE all-to-all of the rows;
      4. the rank grids what it received on its x window of the whole grid (gridder.grid(..., x_window=...)), whose voxel
         corners are the whole grid's, bit for bit.

    No collective is grid-sized.  `gridder` is a Gridder3D (or any object with its grid() signature) and `router` any object
    with _GridRouter.route's signature: the CPU tests of this host logic inject oracle-backed stand-ins.  The default router
    takes pos (N,3), h (N,), prop (N,) contiguous float64 CUDA tensors on one device and raises ValueError otherwise.  return_stats adds a
    dict: rows sent to each rank, rows received, fan-out (rows sent / local particles) and the grid call's n_pairs / n_huge."""
    import torch
    import torch.distributed as dist
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    world, rank = (dist.get_world_size(group), dist.get_rank(group)) if multi else (1, 0)
    nx, ny, nz = (int(v) for v in grid_size)
    edges = grid_slab_planes(nx, world)
    dev = pos.device
    if router is None:
        _check_route_inputs(pos, h, prop)
        router = default_grid_router(dev)
    send, counts, overflow = router.route(pos, h, prop, edges, grid_size, lo, hi, periodic, box)
    counts = counts.to(torch.int64)
    # row g = (rows for rank g, this rank's routing flag): after the exchange row g = (rows from rank g, rank g's flag)
    flag = torch.zeros(1, dtype=torch.int64, device=dev) if overflow is None else overflow.to(device=dev, dtype=torch.int64)
    out_d = torch.stack([counts.to(dev), flag.expand(world)], dim=1).contiguous()
    if multi:
        recv_d = torch.empty_like(out_d)
        dist.all_to_all_single(recv_d, out_d, group=group)
    else:
        recv_d = out_d
    host = recv_d.cpu()                                         # the split sizes and every rank's flag in one copy
    recv = host[:, 0].tolist()
    bad = [g for g in range(world) if host[g, 1]]
    if bad:
        raise RuntimeError(f"grid routing on rank(s) {bad} met a row beyond the counted total (count and write passes disagree)")
    sent = counts.tolist()
    if multi:
        rows = torch.empty((sum(recv), 5), dtype=torch.float64, device=dev)
        dist.all_to_all_single(rows, send, output_split_sizes=recv, input_split_sizes=sent, group=group)
    else:
        rows = send
    del send
    x0, x1 = edges[rank], edges[rank + 1]
    stats = None
    if x1 > x0:
        slab = gridder.grid(rows[:, :3].contiguous(), rows[:, 3].contiguous(), rows[:, 4].contiguous(), grid_size, lo, hi, kernel,
                            periodic, box, x_window=(x0, x1))
        stats = getattr(gridder, "last_stats", None)
    else:
        slab = torch.zeros((0, ny, nz), dtype=torch.float64, device=dev)
    if return_stats:
        st = dict(sent=sent, received=sum(recv), fan_out=sum(sent) / max(pos.shape[0], 1), x_begin=x0, x_end=x1,
                  n_pairs=stats["n_pairs"] if stats else 0, n_huge=stats["n_huge"] if stats else 0)
        return slab, x0, st
    return slab, x0


def collect_slabs(slab, nx, dst=0, group=None, all_ranks=False):
    """The whole (nx, ny, nz) grid from the x-slabs of grid_sharded, on `dst` (or every rank); None elsewhere.  Slabs are
    contiguous plane blocks of the C-order grid, so collecting them on dst is one all-to-all whose only non-empty splits go
    to dst, with no reorder.  all_ranks all-gathers the slabs, padded to the thickest, straight into one buffer of
    world * thickest planes (at most 8 * world planes more than the grid) and moves each slab down to its planes in place,
    so a rank holds one grid, not a gathered copy plus a concatenation."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
        return slab
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    edges = grid_slab_planes(nx, world)
    planes = [edges[g + 1] - edges[g] for g in range(world)]
    if all_ranks:
        tp = max(planes)
        buf = torch.empty((world * tp,) + tuple(slab.shape[1:]), dtype=slab.dtype, device=slab.device)
        mine = slab.contiguous()
        if planes[rank] < tp:
            mine = torch.zeros((tp,) + tuple(slab.shape[1:]), dtype=slab.dtype, device=slab.device)
            mine[:planes[rank]] = slab
        dist.all_gather([buf[g * tp:(g + 1) * tp] for g in range(world)], mine, group=group)
        # slab g sits at g * tp and belongs at edges[g] <= g * tp: move it down in blocks no longer than the shift, in
        # ascending order, so that no block overwrites planes not yet moved
        for g in range(1, world):
            src, dst, shift = g * tp, edges[g], g * tp - edges[g]
            for k in range(0, planes[g] if shift else 0, max(shift, 1)):
                m = min(shift, planes[g] - k)
                buf[dst + k:dst + k + m].copy_(buf[src + k:src + k + m])
        return buf[:nx]
    send_splits = [planes[rank] if g == dst else 0 for g in range(world)]
    recv_splits = planes if rank == dst else [0] * world
    whole = torch.empty((sum(recv_splits),) + tuple(slab.shape[1:]), dtype=slab.dtype, device=slab.device)
    dist.all_to_all_single(whole, slab.contiguous(), output_split_sizes=recv_splits, input_split_sizes=send_splits, group=group)
    return whole if rank == dst else None


def create_grid_sharded(positions, smoothing_lengths, particle_properties, grid_size, x_min, x_max, y_min, y_max, z_min, z_max,
                        kernel_func=None, *, periodic=False, box_size=None, dst=0, group=None, all_ranks=False):
    """Host-buffer entry for one rank of a multi-GPU job: create_grid's arguments, but the arrays hold only THIS rank's
    particles.  Each rank grids its x-slab (grid_sharded); the slabs are collected on `dst` (or on every rank) and the
    whole (nx, ny, nz) float64 numpy grid is returned there, None elsewhere.  kernel_func=None is quartic_spline_kernel."""
    import torch
    from .tools.projections._gridder import default_gridder
    from .tools.projections._kernels import kernel_id_of, quartic_spline_kernel
    from .tools.projections._projector import _check_buffer
    kernel = kernel_id_of(kernel_func if kernel_func is not None else quartic_spline_kernel)
    positions = _check_buffer(positions, 2, "positions")
    smoothing_lengths = _check_buffer(smoothing_lengths, 1, "smoothing_lengths")
    particle_properties = _check_buffer(particle_properties, 1, "particle_properties")
    if positions.shape[1] != 3 or not (positions.shape[0] == smoothing_lengths.shape[0] == particle_properties.shape[0]):
        raise ValueError("positions (N,3), smoothing_lengths (N,), particle_properties (N,) expected")
    eng = default_gridder()
    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(eng.device)
    nx, ny, nz = (int(v) for v in grid_size)
    slab, _ = grid_sharded(eng, to_dev(positions), to_dev(smoothing_lengths), to_dev(particle_properties), (nx, ny, nz),
                           (x_min, y_min, z_min), (x_max, y_max, z_max), kernel, periodic, box_size, group)
    whole = collect_slabs(slab, nx, dst, group, all_ranks)
    if whole is not None:
        host = torch.empty(whole.shape, dtype=whole.dtype, pin_memory=whole.is_cuda)
        host.copy_(whole)
        return host.numpy()
    return None
