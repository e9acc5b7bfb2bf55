"""create_grid: SPH deposition onto a 3-D voxel grid.  EXTENSION (BASELINE.json config 4); the reference has no 3-D
function, so the rules are those of its 2-D pixel routine (tools/projections/_pixel_calculations.pyx:11-14,30-34)
carried to three axes: grid[xi,yi,zi] = sum_i A_i W(|p_i - corner(xi,yi,zi)|, h_i) over r^2 < (2 h_i)^2 with
corner = min + index*delta.  Arguments follow create_image's style (reference _projector.py:75-87)."""
import ctypes as C
import threading
from typing import Callable

import numpy as np

from ... import _lib
from ._kernels import kernel_id_of, quartic_spline_kernel
from ._projector import _check_buffer


class Gridder3D:
    """Reusable 3-D gridding context on one CUDA device (keeps its workspace)."""

    def __init__(self, device=None, pair_capacity=None, huge_capacity=1 << 20, small_max_vox=-1, huge_min_bricks=-1):
        self.torch = _lib.require_cuda()
        self.lib = _lib.load()
        torch = self.torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.pair_capacity = pair_capacity
        self.huge_capacity = int(huge_capacity)
        self.small_max_vox = int(small_max_vox)
        self.huge_min_bricks = int(huge_min_bricks)
        self._ws = None
        self.last_stats = None
        self._lock = threading.RLock()        # one workspace: calls on this engine serialise

    def params(self, n, grid_size, lo, hi, kernel, periodic=False, box=None, timing=False, accumulate=False, x_window=None):
        p = _lib.Grid3DParams()
        p.n = int(n)
        p.nx, p.ny, p.nz = (int(v) for v in grid_size)
        if x_window is not None:
            p.x_begin, p.x_end = (int(v) for v in x_window)
            if not 0 <= p.x_begin < p.x_end <= p.nx:
                raise ValueError(f"x_window {tuple(x_window)} is not inside [0, {p.nx})")
        if isinstance(kernel, str):
            p.kernel_id = _lib.KERNEL_IDS[kernel]
        elif hasattr(kernel, "device_table"):                      # TabulatedKernel: arbitrary kernel_func callable
            tab = kernel.device_table(self.torch, self.device)
            self._kernel_table = tab
            p.kernel_id = _lib.KERNEL_TABLE
            p.kernel_table = tab.data_ptr()
            p.kernel_table_n = tab.shape[0]
            p.kernel_dim = kernel.dim
        else:
            p.kernel_id = int(kernel)
        p.flags = (_lib.FLAG_PERIODIC if periodic else 0) | (_lib.FLAG_TIMING if timing else 0) | \
                  (_lib.FLAG_ACCUMULATE if accumulate else 0)
        for c in range(3):
            p.lo[c] = float(lo[c]); p.hi[c] = float(hi[c])
        if periodic:
            if box is None:
                raise ValueError("periodic=True needs box_size")
            b = (float(box),) * 3 if np.isscalar(box) else tuple(float(v) for v in box)
            for c in range(3):
                p.box[c] = b[c]
        p.small_max_vox = self.small_max_vox
        p.huge_min_bricks = self.huge_min_bricks
        cap = self.pair_capacity
        if cap is None:
            cap = min(max(32 * int(n), 1 << 20), 1 << 30)
        p.pair_capacity = int(cap)
        p.huge_capacity = int(self.huge_capacity)
        return p

    def workspace(self, p):
        need = C.c_size_t(0)
        _lib.check(self.lib.ast_grid3d_workspace_bytes(C.byref(p), C.byref(need)))
        if self._ws is None or self._ws.numel() < need.value:
            self._ws = None
            self._ws = self.torch.empty(need.value, dtype=self.torch.uint8, device=self.device)
        return self._ws

    def grid(self, pos, h, prop, grid_size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, out=None, timing=False,
             accumulate=False, stream=None, presort="auto", x_window=None):
        """pos (N,3), h (N,), prop (N,) float64 CUDA tensors -> (nx,ny,nz) float64 CUDA tensor.
        x_window=(x_begin, x_end): planes [x_begin, x_end) of that grid only, a (x_end - x_begin, ny, nz) tensor whose voxels
        are bit for bit the whole grid's voxel corners (so a slab has the same contributors as in the whole grid)."""
        torch = self.torch
        n = pos.shape[0]
        for t, shape in ((pos, (n, 3)), (h, (n,)), (prop, (n,))):
            if t.dtype != torch.float64 or tuple(t.shape) != shape or not t.is_cuda or not t.is_contiguous():
                raise ValueError("device inputs must be contiguous float64 CUDA tensors of shapes (N,3), (N,), (N,)")
        p = self.params(n, grid_size, lo, hi, kernel, periodic, box, timing, accumulate, x_window)
        # optional spatial pre-ordering: 'auto' = the library looks at a sample of the input order (the deposition is 27 % faster
        # on the randomly ordered NFW set of config 4 when the particles are first ordered by brick), 'always', 'never'
        if presort in (True, "always"):
            p.flags |= _lib.FLAG_ORDER_ALWAYS
        elif presort in ("auto", "sample"):
            p.flags |= _lib.FLAG_ORDER_AUTO
        elif presort not in (None, False, "never"):
            raise ValueError("presort must be 'auto', 'always' or 'never'")
        if out is None:
            out = torch.empty((p.x_end - p.x_begin if x_window is not None else p.nx, p.ny, p.nz), dtype=torch.float64, device=self.device)
        stats = _lib.Project2DStats()
        with torch.cuda.device(self.device), self._lock:
            # pair_capacity / huge_capacity are windows (the library walks any number of pairs and large-h entries through them
            # in passes): no capacity can fail once the direct deposits have started, nothing is retried
            ws = self.workspace(p)
            _lib.check(self.lib.ast_grid3d(C.byref(p), _lib.ptr(pos), _lib.ptr(h), _lib.ptr(prop), _lib.ptr(out), _lib.ptr(ws),
                                           C.c_size_t(ws.numel()), _lib.stream_ptr(stream), C.byref(stats)))
        self.last_stats = dict(n_pairs=stats.n_pairs, n_huge=stats.n_huge, n_rounds=stats.n_rounds,
                               n_launches=stats.n_launches, stage_ms=list(stats.stage_ms), reordered=bool(stats.reordered))
        return out


_default = {}


def default_gridder(device=None):
    torch = _lib.require_cuda()
    key = torch.cuda.current_device() if device is None else torch.device(device).index
    if key not in _default:
        _default[key] = Gridder3D(device)
    return _default[key]


def create_grid(
    positions: np.ndarray,
    smoothing_lengths: np.ndarray,
    particle_properties: np.ndarray,
    grid_size: tuple,
    x_min: float, x_max: float, y_min: float, y_max: float, z_min: float, z_max: float,
    kernel_func: Callable = quartic_spline_kernel,
    *,
    periodic: bool = False,
    box_size=None,
    device=None,
) -> np.ndarray:
    """numpy in / numpy out: (nx, ny, nz) float64 grid, grid[xi, yi, zi]."""
    kernel = kernel_id_of(kernel_func)
    positions = _check_buffer(positions, 2, "positions")
    smoothing_lengths = _check_buffer(smoothing_lengths, 1, "smoothing_lengths")
    particle_properties = _check_buffer(particle_properties, 1, "particle_properties")
    if positions.shape[1] != 3 or not (positions.shape[0] == smoothing_lengths.shape[0] == particle_properties.shape[0]):
        raise ValueError("positions (N,3), smoothing_lengths (N,), particle_properties (N,) expected")
    eng = default_gridder(device)
    torch = eng.torch
    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(eng.device, non_blocking=True)
    out = eng.grid(to_dev(positions), to_dev(smoothing_lengths), to_dev(particle_properties), grid_size,
                   (x_min, y_min, z_min), (x_max, y_max, z_max), kernel, periodic, box_size)
    return out.cpu().numpy()
