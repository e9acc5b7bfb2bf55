"""Per-pixel error bound for 2-D maps and 3-D grids against the float64 oracle (test infrastructure, plain numpy).

The global gates (relative L2, total weight) are dominated by the brightest pixels: a map that is wrong, or empty, wherever
the weights are faint passes them.  Maps of this kind are usually read on a log scale, so every pixel is checked here
against its own bound

    |got - ref| <= tau * env,    env = sum_i |prop_i| W(0, h_i)

over the particle images whose squared distance to the pixel's sample point (its lower corner, the oracle's) is below
(2 h_i)^2 (1 + 2^-16), and got == 0 exactly where env == 0.  W(0, h) is the kernel's peak, so env bounds the sum of the
magnitudes of a pixel's terms.  The mask is widened by 2^-16 because the float32 paths may give a pixel just outside the
float64 support a contribution of ~1e-21 of the peak: such a pixel must have a non-zero envelope.

Why tau = 2^-15 (3.05e-5).  Per pixel, relative to env:
  - weight mantissa rounded to float32: 2^-24 = 6e-8;
  - shape factor: the tile (brick) relative float32 coordinates carry an error in q of at most ~2^-18 for h >= 0.5 pixel
    (voxel), and the largest shape slope is |df/dq| <= 1.05 (Wendland C2): <= 4e-6;
  - float32 partial sums: the tile kernel (rowcol_accum_kernel) and the brick kernel (brick_accum_kernel) both fold their
    float32 accumulators into float64 once at least 96 hits have been added since the last fold; a batch adds at most 32,
    so a float32 run holds at most 127 terms and its rounding error is at most 126 * 2^-24 = 7.5e-6 of the sum of |terms|;
  - the float64 fold, the float64 direct deposits and the oracle itself: ~1e-15.
Sum: ~1.2e-5, below tau with a factor 2.6 to spare.  The direct-deposit paths (float64 mask and weights, float32 shape
only) are well inside the same bound.  Weights flushed to zero because they lie far below the largest weight of the call
are errors of up to env itself, i.e. tau^-1 = 32768 times the bound.

Outside this bound, on purpose: scenes that force sub-half-pixel h through the tile path (the q error grows as 1/h there),
and AST_KERNEL_TABLE, whose table interpolation error is a separate, separately tested matter.
"""
import numpy as np

import oracle

TAU = 2.0 ** -15
WIDEN = 2.0 ** -16

_PLANE = {0: (1, 2), 1: (0, 2), 2: (0, 1)}


def _peaks(prop, h, kernel):
    """|prop| W(0, h) as (P, N), and the particles that have a support at all"""
    ok = (h > 0) & np.isfinite(2.0 * h)
    w0 = np.zeros(h.shape)
    if ok.any():
        w0[ok] = oracle.kernel_eval(kernel, np.zeros(int(ok.sum())), h[ok])
    return np.abs(prop) * w0, ok


def _window(p, R, vmin, d, n):
    """candidate sample range of one axis (generous by two samples; the exact test follows)"""
    with np.errstate(invalid="ignore"):
        lo = np.floor((p - R - vmin) / d) - 2
        hi = np.ceil((p + R - vmin) / d) + 2
    good = np.isfinite(lo) & np.isfinite(hi) & (hi >= 0) & (lo <= n - 1)
    lo = np.where(good, np.clip(lo, 0, n - 1), 0).astype(np.int64)
    hi = np.where(good, np.clip(hi, 0, n - 1), -1).astype(np.int64)
    return lo, hi, good


def envelope2d(pos, h, prop, image_size, axis, bounds, kernel="cubic_spline_3d", periodic=False, box=None, widen=WIDEN):
    """Per-pixel envelope of a 2-D map.  prop (N,) -> (nx, ny); (P, N) -> (P, nx, ny)."""
    pos = np.asarray(pos, dtype=np.float64); h = np.asarray(h, dtype=np.float64); prop = np.asarray(prop, dtype=np.float64)
    N = len(h)
    single = prop.ndim == 1
    amp, ok = _peaks(prop.reshape(-1, N), h, kernel)
    nx, ny = int(image_size[0]), int(image_size[1])
    x_min, x_max, y_min, y_max = bounds
    dx, dy = (x_max - x_min) / nx, (y_max - y_min) / ny
    X = x_min + np.arange(nx) * dx                 # the oracle's sample(vmin, d, i) = vmin + i * d
    Y = y_min + np.arange(ny) * dy
    a, b = _PLANE[axis]
    n_img, sa, sb = oracle.images(periodic, box)
    R = 2.0 * h
    R2 = R * R * (1.0 + widen)
    env = np.zeros((amp.shape[0], nx, ny))
    for m in range(n_img):
        pa = pos[:, a] + sa[m]; pb = pos[:, b] + sb[m]
        xlo, xhi, gx = _window(pa, R, x_min, dx, nx)
        ylo, yhi, gy = _window(pb, R, y_min, dy, ny)
        for i in np.nonzero(ok & gx & gy)[0]:
            ex = pa[i] - X[xlo[i]:xhi[i] + 1]; ey = pb[i] - Y[ylo[i]:yhi[i] + 1]
            inside = (ex * ex)[:, None] + (ey * ey)[None, :] < R2[i]
            env[:, xlo[i]:xhi[i] + 1, ylo[i]:yhi[i] + 1] += amp[:, i, None, None] * inside
    return env[0] if single else env


def envelope3d(pos, h, prop, grid_size, lo, hi, kernel="cubic_spline_3d", periodic=False, box=None, widen=WIDEN):
    """Per-voxel envelope of a 3-D grid (sample point = voxel lower corner, r^2 = (dx^2 + dy^2) + dz^2 as in the oracle)."""
    pos = np.asarray(pos, dtype=np.float64); h = np.asarray(h, dtype=np.float64); prop = np.asarray(prop, dtype=np.float64)
    amp, ok = _peaks(prop.reshape(1, -1), h, kernel)
    amp = amp[0]
    n3 = [int(v) for v in grid_size]
    d = [(hi[c] - lo[c]) / n3[c] for c in range(3)]
    S = [lo[c] + np.arange(n3[c]) * d[c] for c in range(3)]
    n_img, s3 = oracle.images3(periodic, box)
    s3 = np.asarray(s3, dtype=np.float64).reshape(-1, 3)
    R = 2.0 * h
    R2 = R * R * (1.0 + widen)
    env = np.zeros(n3)
    for m in range(n_img):
        p = [pos[:, c] + s3[m, c] for c in range(3)]
        win = [_window(p[c], R, lo[c], d[c], n3[c]) for c in range(3)]
        sel = ok & win[0][2] & win[1][2] & win[2][2]
        for i in np.nonzero(sel)[0]:
            sl = [slice(win[c][0][i], win[c][1][i] + 1) for c in range(3)]
            e = [p[c][i] - S[c][sl[c]] for c in range(3)]
            inside = ((e[0] * e[0])[:, None, None] + (e[1] * e[1])[None, :, None]) + (e[2] * e[2])[None, None, :] < R2[i]
            env[sl[0], sl[1], sl[2]] += amp[i] * inside
    return env


def assert_pixelwise(got, ref, env, tau=TAU, what=""):
    """|got - ref| <= tau * env everywhere (NaN fails), got == 0 exactly where env == 0; reports the worst pixels."""
    got = np.asarray(got, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64); env = np.asarray(env, dtype=np.float64)
    assert got.shape == ref.shape == env.shape, (got.shape, ref.shape, env.shape)
    err = np.abs(got - ref)
    bound = tau * env
    bad = ~(err <= bound) | ((env == 0) & (got != 0))
    if not bad.any():
        return
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(env > 0, err / bound, np.inf)
    ratio = np.where(np.isnan(ratio), np.inf, ratio)
    idx = np.argsort(np.where(bad, ratio, -1.0), axis=None)[::-1][:8]
    lines = [f"{tuple(int(v) for v in np.unravel_index(j, got.shape))}: got {got.flat[j]:.6e} ref {ref.flat[j]:.6e} "
             f"env {env.flat[j]:.6e} |err|/(tau env) {ratio.flat[j]:.3g}" for j in idx]
    n_zero = int(((env > 0) & (got == 0) & (ref != 0) & bad).sum())
    raise AssertionError(f"{what}{int(bad.sum())} of {bad.size} pixels outside the per-pixel bound (tau = {tau:.3g}; "
                         f"{n_zero} of them are zero where the reference is not); worst:\n  " + "\n  ".join(lines))
