// ast_geom.h -- float64 index work shared by every kernel: sample points, the canonical 1-D contributor
// range of a particle, tile membership, particle classes.  Host+device so the same source can be unit
// tested on the CPU (csrc/host_geom.cpp) before it ever runs on a GPU.
//
// Semantics come from the reference's pixel routine (tools/projections/_pixel_calculations.pyx:11-14,30-31):
//   X(i) = vmin + (double)i * d            sample point = pixel LOWER corner
//   contributor  <=>  (pa - X(xi))^2 + (pb - Y(yi))^2 < (2.0*h)^2        (strict, float64, no FMA)
// Every product below uses __dmul_rn/__dadd_rn on the device so that nvcc cannot contract a*b+c into an
// FMA: the results are bit-identical to a host compiler running with -ffp-contract=off, which is what
// "index work bit-exact" is measured against (oracle/sph_oracle.c).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define AST_HD __host__ __device__ __forceinline__
#else
#define AST_HD static inline
#endif

#if defined(__CUDA_ARCH__)
#define AST_DMUL(a, b) __dmul_rn((a), (b))
#define AST_DADD(a, b) __dadd_rn((a), (b))
#define AST_DSUB(a, b) __dsub_rn((a), (b))
#else
#define AST_DMUL(a, b) ((a) * (b))
#define AST_DADD(a, b) ((a) + (b))
#define AST_DSUB(a, b) ((a) - (b))
#endif

namespace ast {

enum : int { CLS_EMPTY = 0, CLS_SMALL = 1, CLS_TILED = 2, CLS_HUGE = 3 };

// one image axis: n samples X(i) = vmin + i*d
struct Axis1 {
    double vmin, d, inv_d;
    int n;
};

AST_HD Axis1 make_axis(double vmin, double vmax, int n)
{
    Axis1 a;
    a.vmin = vmin;
    a.d = (vmax - vmin) / (double)n;        // _projector.py:34-35 pixel_size = (max - min) / image_size
    a.inv_d = 1.0 / a.d;
    a.n = n;
    return a;
}

AST_HD double sample(const Axis1 &a, int i) { return AST_DADD(a.vmin, AST_DMUL((double)i, a.d)); }

// (p - X(i))^2
AST_HD double dist2(const Axis1 &a, double p, int i)
{
    double t = AST_DSUB(p, sample(a, i));
    return AST_DMUL(t, t);
}

AST_HD double radius2(double h)
{
    double R = AST_DMUL(2.0, h);             // (2.0 * smoothing_lengths)**2, _pixel_calculations.pyx:31
    return AST_DMUL(R, R);
}

// Canonical 1-D contributor range {i in [0,n) : dist2(p,i) < R2}.  |p - X(i)| is unimodal in i, so the set is
// an interval; the multiplication by inv_d only seeds the search, the edges are settled by the exact
// predicate, hence the result does not depend on how the seed was rounded.
AST_HD bool range1(const Axis1 &a, double p, double h, double R2, int &lo, int &hi)
{
    // h <= 0, NaN or inf never contributes (documented deviation: the reference would use (2h)^2 for h < 0)
    if (!(h > 0.0) || !(R2 > 0.0) || !(R2 < INFINITY) || !(fabs(p) < INFINITY)) return false;
    double h2 = AST_DMUL(2.0, h);
    double tl = floor(AST_DMUL(AST_DSUB(AST_DSUB(p, h2), a.vmin), a.inv_d));
    double th = ceil(AST_DMUL(AST_DSUB(AST_DADD(p, h2), a.vmin), a.inv_d));
    if (!(tl == tl) || !(th == th)) return false;
    const int n = a.n;
    int c = tl < 0.0 ? 0 : (tl > (double)n ? n : (int)tl);
    int e = th < -1.0 ? -1 : (th > (double)(n - 1) ? n - 1 : (int)th);
    while (c > 0 && dist2(a, p, c - 1) < R2) --c;
    while (c < n && !(dist2(a, p, c) < R2) && sample(a, c) <= p) ++c;
    if (c >= n || !(dist2(a, p, c) < R2)) return false;
    while (e < n - 1 && dist2(a, p, e + 1) < R2) ++e;
    while (e >= 0 && !(dist2(a, p, e) < R2) && sample(a, e) >= p) --e;
    if (e < 0 || !(dist2(a, p, e) < R2)) return false;
    lo = c;
    hi = e;
    return true;
}

// Cheap conservative pre-test used to skip periodic images: false only when no sample of the axis can lie within 2h of p
// (one sample spacing of slack against rounding), i.e. only when range1 would return false anyway.  NaN -> false.
AST_HD bool may_touch(const Axis1 &a, double p, double h2)
{
    return (p + h2 >= a.vmin - a.d) && (p - h2 <= a.vmin + ((double)a.n) * a.d);
}

// index of the sample at or just below p (seed only; callers look at e-1, e, e+1)
AST_HD int floor_index(const Axis1 &a, double p, int lo, int hi)
{
    double t = floor(AST_DMUL(AST_DSUB(p, a.vmin), a.inv_d));
    return t < (double)lo ? lo : (t > (double)hi ? hi : (int)t);
}

// min over i in [lo,hi] of dist2(p,i).  |p - X(i)| is unimodal in i with its minimum at m* in {f, f+1}, f the true floor
// of (p - vmin)/d; the seed e (computed with a multiply) satisfies |e - m*| <= 1.  Hence: e < lo -> the minimum over the
// interval is at lo; e > hi -> at hi; otherwise among e-1, e, e+1 (clamped).  One or three evaluations, same value as
// scanning the whole interval (oracle: brute force).
AST_HD double min_dist2(const Axis1 &a, double p, int lo, int hi)
{
    const double t = floor(AST_DMUL(AST_DSUB(p, a.vmin), a.inv_d));
    if (t < (double)lo) return dist2(a, p, lo);
    if (t > (double)hi) return dist2(a, p, hi);
    const int e = (int)t;
    double m = dist2(a, p, e);
    if (e > lo) { const double v = dist2(a, p, e - 1); m = v < m ? v : m; }
    if (e < hi) { const double v = dist2(a, p, e + 1); m = v < m ? v : m; }
    return m;
}

struct Box2 {
    int x0, x1, y0, y1;
};

// classification of one particle image on the 2-D screen
struct Bin2 {
    Box2 bb;
    int cls;
    int tx0, tx1, ty0, ty1;
};

template <int TILE>
AST_HD Bin2 classify2(const Axis1 &ax, const Axis1 &ay, double pa, double pb, double h, double R2,
                      int64_t small_max_px, int64_t huge_min_tiles)
{
    Bin2 b;
    b.cls = CLS_EMPTY;
    b.bb.x0 = 0; b.bb.x1 = -1; b.bb.y0 = 0; b.bb.y1 = -1;
    b.tx0 = b.ty0 = 0; b.tx1 = b.ty1 = -1;
    int x0, x1, y0, y1;
    if (!range1(ax, pa, h, R2, x0, x1)) return b;
    if (!range1(ay, pb, h, R2, y0, y1)) return b;
    b.bb.x0 = x0; b.bb.x1 = x1; b.bb.y0 = y0; b.bb.y1 = y1;
    int64_t area = (int64_t)(x1 - x0 + 1) * (int64_t)(y1 - y0 + 1);
    if (area <= small_max_px) { b.cls = CLS_SMALL; return b; }
    b.tx0 = x0 / TILE; b.tx1 = x1 / TILE; b.ty0 = y0 / TILE; b.ty1 = y1 / TILE;
    int64_t nt = (int64_t)(b.tx1 - b.tx0 + 1) * (int64_t)(b.ty1 - b.ty0 + 1);
    b.cls = nt > huge_min_tiles ? CLS_HUGE : CLS_TILED;
    return b;
}

// Enumerate the tiles of a CLS_TILED particle image in emit order (tx ascending, then ty ascending) and call
// f(tile_key) for every tile that holds at least one pixel satisfying the 2-D mask.  Returns the count.
// (the callback of the _xy form gets the tile coordinates instead of the key)
template <int TILE, class F>
AST_HD int for_each_tile2_xy(const Axis1 &ax, const Axis1 &ay, double pa, double pb, double R2, const Bin2 &b, F &&f)
{
    int cnt = 0;
    for (int tx = b.tx0; tx <= b.tx1; ++tx) {
        int xa = tx * TILE > b.bb.x0 ? tx * TILE : b.bb.x0;
        int xb = tx * TILE + TILE - 1 < b.bb.x1 ? tx * TILE + TILE - 1 : b.bb.x1;
        double mdx = min_dist2(ax, pa, xa, xb);
        for (int ty = b.ty0; ty <= b.ty1; ++ty) {
            int ya = ty * TILE > b.bb.y0 ? ty * TILE : b.bb.y0;
            int yb = ty * TILE + TILE - 1 < b.bb.y1 ? ty * TILE + TILE - 1 : b.bb.y1;
            double mdy = min_dist2(ay, pb, ya, yb);
            if (AST_DADD(mdx, mdy) < R2) {
                f(tx, ty);
                ++cnt;
            }
        }
    }
    return cnt;
}

template <int TILE, class F>
AST_HD int for_each_tile2(const Axis1 &ax, const Axis1 &ay, double pa, double pb, double R2, const Bin2 &b,
                          int nty, F &&f)
{
    return for_each_tile2_xy<TILE>(ax, ay, pa, pb, R2, b, [&](int tx, int ty) { f((uint32_t)(tx * nty + ty)); });
}

// ---- 3-D voxel grid: bricks of BRICK^3 voxels, same canonical ranges per axis ----------------------------------
struct Bin3 {
    int lo[3], hi[3];      // voxel bbox, inclusive (empty: hi < lo)
    int b0[3], b1[3];      // brick bbox
    int cls;
};

// x window of a grid: planes [x0, x0 + n) of the whole grid's x axis.  The axes stay the whole grid's, so every sample
// point and every contributor range is the whole grid's value; bboxes and bricks are numbered from x0.
struct Win1 {
    int x0, n;
};

template <int BRICK>
AST_HD Bin3 classify3(const Axis1 *ax /* [3] */, Win1 w, const double *p /* [3] */, double h, double R2, int64_t small_max_vox,
                      int64_t huge_min_bricks)
{
    Bin3 b;
    b.cls = CLS_EMPTY;
    for (int c = 0; c < 3; ++c) { b.lo[c] = 0; b.hi[c] = -1; b.b0[c] = 0; b.b1[c] = -1; }
    int lo[3], hi[3];
    for (int c = 0; c < 3; ++c)
        if (!range1(ax[c], p[c], h, R2, lo[c], hi[c])) return b;
    lo[0] = (lo[0] > w.x0 ? lo[0] : w.x0) - w.x0;                      // clip the whole grid's x range to the window
    hi[0] = (hi[0] < w.x0 + w.n - 1 ? hi[0] : w.x0 + w.n - 1) - w.x0;
    if (lo[0] > hi[0]) return b;
    int64_t vol = 1, nb = 1;
    for (int c = 0; c < 3; ++c) {
        b.lo[c] = lo[c]; b.hi[c] = hi[c];
        vol *= (int64_t)(hi[c] - lo[c] + 1);
    }
    if (vol <= small_max_vox) { b.cls = CLS_SMALL; return b; }
    for (int c = 0; c < 3; ++c) {
        b.b0[c] = lo[c] / BRICK; b.b1[c] = hi[c] / BRICK;
        nb *= (int64_t)(b.b1[c] - b.b0[c] + 1);
    }
    b.cls = nb > huge_min_bricks ? CLS_HUGE : CLS_TILED;
    return b;
}

// bricks in emit order (bx, by, bz ascending) that hold at least one voxel with (dx^2 + dy^2) + dz^2 < R2; b from classify3
// on the window that starts at plane x0
template <int BRICK, class F>
AST_HD int for_each_brick3(const Axis1 *ax, int x0, const double *p, double R2, const Bin3 &b, int nby, int nbz, F &&f)
{
    int cnt = 0;
    for (int bx = b.b0[0]; bx <= b.b1[0]; ++bx) {
        int xa = bx * BRICK > b.lo[0] ? bx * BRICK : b.lo[0];
        int xb = bx * BRICK + BRICK - 1 < b.hi[0] ? bx * BRICK + BRICK - 1 : b.hi[0];
        double mdx = min_dist2(ax[0], p[0], x0 + xa, x0 + xb);
        for (int by = b.b0[1]; by <= b.b1[1]; ++by) {
            int ya = by * BRICK > b.lo[1] ? by * BRICK : b.lo[1];
            int yb = by * BRICK + BRICK - 1 < b.hi[1] ? by * BRICK + BRICK - 1 : b.hi[1];
            double mdxy = AST_DADD(mdx, min_dist2(ax[1], p[1], ya, yb));
            for (int bz = b.b0[2]; bz <= b.b1[2]; ++bz) {
                int za = bz * BRICK > b.lo[2] ? bz * BRICK : b.lo[2];
                int zb = bz * BRICK + BRICK - 1 < b.hi[2] ? bz * BRICK + BRICK - 1 : b.hi[2];
                double mdz = min_dist2(ax[2], p[2], za, zb);
                if (AST_DADD(mdxy, mdz) < R2) {
                    f((uint32_t)((bx * nby + by) * nbz + bz));
                    ++cnt;
                }
            }
        }
    }
    return cnt;
}

// in-plane columns of the (N,3) position rows: X->(1,2), Y->(0,2), Z->(0,1)  (_pixel_calculations.pyx:20-28)
AST_HD void plane_columns(int axis, int &a, int &b)
{
    a = axis == 0 ? 1 : 0;
    b = axis == 2 ? 1 : 2;
}

}  // namespace ast
