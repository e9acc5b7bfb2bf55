"""A literal numpy restatement, in three dimensions, of the reference's pixel routine
(/root/reference/src/astro_sph_tools/tools/projections/_pixel_calculations.pyx:11-14, 20-34) -- written independently of
oracle/sph_oracle.c so that the 3-D oracle (for which the reference has no function) is pinned by something other than
itself.  One voxel at a time, exactly as calculate_pixel_value does one pixel at a time:

    x = x_min + xi * pixel_size_x ...                       (:13-14, lower corner)
    dx = positions[:, 0] - x ...                            (:20-28)
    r2 = dx**2 + dy**2 (+ dz**2)                            (:30)
    mask = r2 < (2.0 * smoothing_lengths)**2                (:31)
    r = np.sqrt(r2[mask]); weights = kernel_func(r, smoothing_lengths[mask])   (:32-33)
    return np.sum(particle_properties[mask] * weights)      (:34)

The kernel is the reference's own compiled quartic_spline_kernel when oracle/_ref is present (it travels to the GPU box),
else the numpy restatement of _kernels.pyx:15-19 below.  Test infrastructure only."""
import numpy as np


def quartic_spline_numpy(r, h):
    q = r / h
    out = np.zeros_like(q)
    inner = q < 1.0
    outer = (q >= 1.0) & (q < 2.0)
    out[inner] = (1.0 - 1.5 * q[inner] ** 2 + 0.75 * q[inner] ** 3) / (np.pi * h[inner] ** 3)
    out[outer] = 0.25 * (2.0 - q[outer]) ** 3 / (np.pi * h[outer] ** 3)
    return out


def reference_kernel():
    try:
        import oracle
        if oracle.reference_available():
            mod, _ = oracle.reference_module()
            return lambda r, h: np.asarray(mod.quartic_spline_kernel(np.ascontiguousarray(r), np.ascontiguousarray(h)))
    except Exception:
        pass
    return quartic_spline_numpy


def grid3d_literal(pos, h, prop, grid_size, lo, hi, kernel_func=None, shifts=((0.0, 0.0, 0.0),)):
    """grid[xi, yi, zi] by the literal per-voxel rule; `shifts`: periodic images = replicated particles (SURVEY App. D)"""
    kernel_func = kernel_func or reference_kernel()
    nx, ny, nz = grid_size
    d = [(hi[c] - lo[c]) / grid_size[c] for c in range(3)]
    P = np.concatenate([pos + np.asarray(s) for s in shifts]); H = np.tile(h, len(shifts)); A = np.tile(prop, len(shifts))
    ok = H > 0                                                    # documented deviation: h <= 0 never contributes
    P, H, A = P[ok], H[ok], A[ok]
    R2 = (2.0 * H) ** 2
    out = np.zeros((nx, ny, nz))
    for xi in range(nx):
        x = lo[0] + xi * d[0]
        dx = P[:, 0] - x
        near = dx ** 2 < R2                                       # only skips work: dx**2 >= R2 implies r2 >= R2
        if not near.any():
            continue
        Pn, Hn, An, R2n, dxn = P[near], H[near], A[near], R2[near], dx[near]
        for yi in range(ny):
            y = lo[1] + yi * d[1]
            dy = Pn[:, 1] - y
            for zi in range(nz):
                z = lo[2] + zi * d[2]
                dz = Pn[:, 2] - z
                r2 = dxn ** 2 + dy ** 2 + dz ** 2
                mask = r2 < R2n
                if mask.any():
                    r = np.sqrt(r2[mask])
                    out[xi, yi, zi] = np.sum(An[mask] * kernel_func(r, Hn[mask]))
    return out


def project2d_literal(pos, h, prop, npix, axis, bounds, kernel_func=None):
    """the reference's 2-D pixel rule itself: grid3d_literal on a one-voxel-thick grid at z = 0, fed the particles'
    in-plane coordinates (columns of CoordinateAxes.plane_columns) and z = 0, so that r2 = dx**2 + dy**2 + 0"""
    a, b = {0: (1, 2), 1: (0, 2), 2: (0, 1)}[axis]
    flat = np.zeros_like(pos)
    flat[:, 0], flat[:, 1] = pos[:, a], pos[:, b]
    x0, x1, y0, y1 = bounds
    return grid3d_literal(flat, h, prop, (npix, npix, 1), (x0, y0, 0.0), (x1, y1, 1.0), kernel_func)[:, :, 0]
