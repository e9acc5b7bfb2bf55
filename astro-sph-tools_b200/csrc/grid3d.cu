// grid3d.cu -- SPH deposition onto a 3-D voxel grid, sm_100a.  EXTENSION named by BASELINE.json (config 4); the
// reference has no 3-D function.  Rules are the 2-D path's (tools/projections/_pixel_calculations.pyx:11-14,30-34)
// carried to three axes: sample point = voxel lower corner min + index*delta, contributor iff
// (dx^2 + dy^2) + dz^2 < (2h)^2 in float64, value = sum A_i W(r, h_i) with a 3-D normalised kernel.
//
// Same pipeline as project2d.cu on bricks of 8^3 voxels: bin (+ direct deposit of few-voxel particles with float64
// atomics) -> scan -> emit (brick key << 32 | particle) -> stable radix sort -> brick ranges -> one CTA per brick:
// 4 warps, each owning a 4x4x8 column of the brick, 4 voxels (contiguous in z) per thread in registers.
#include <string.h>

#include "ast_geom.h"
#include "ast_math.h"
#include "block_utils.cuh"
#include "common.cuh"
#include "presort.cuh"
#include "scan_sort.cuh"
#include "work_items.cuh"

namespace ast {

constexpr int BRICK = AST_BRICK;
constexpr int kBin3Threads = 256;
constexpr int kAcc3Threads = 128;

struct __align__(32) Rec3 {
    double x, y, z;
    float inv_h, c;            // 1/h and prop * norm(h), narrowed once per particle
};
static_assert(sizeof(Rec3) == 32, "record is one 32-byte sector");

struct P3 {
    const double *pos, *h, *prop;
    double *out;
    int64_t n;
    int kernel_id, shape;
    Axis1 ax[3];
    int nb[3];                       // bricks per axis
    int n_img, img_shift;
    double box[3];                   // periodic image m = 9*(ia+1) + 3*(ib+1) + (ic+1), shift = (ia,ib,ic) * box
    ShapeTab tab;
    double norm_c;
    int norm_dim;
    int64_t small_max_vox, huge_min_bricks;
    // written by bin3_kernel for the blocks that have pairs or large-h entries, read by emit3_kernel (one enumeration there)
    uint32_t *pcount;                // pairs of particle i
    uint64_t *pmask;                 // bit m: image m is tiled, bit 27 + m: image m is on the large-h list
    const int *wexp;                 // [2] largest binary exponent of prop * norm(h) over the particles that may take the brick
                                     // path + kExpBias3, and kExpBias3 - the smallest (0: none); see wexp3_kernel
};

// The brick kernels work on float32 weights, the 2-D reference rules on float64 in any unit system (ADVICE r1: 1e48 or 1e-59
// are legitimate weights), and one call may mix weights hundreds of binary orders apart.  Rec3 has no room for a
// per-particle exponent, so one pre-pass takes the largest and the smallest binary exponent of prop * norm(h) over the
// particles that may take the brick path (16 bytes per particle: 0.05 ms at 256^3 against a 70 ms step; the direct deposits
// of few-voxel particles use the float64 weight and take no part).  The weights are staged in exponent BANDS of kWeightBand
// binary orders: band j holds prop * norm(h) * 2^-T_j for exponents T_j - kWeightBand < e <= T_j (T_0 = the largest,
// T_j = T_0 - j kWeightBand; the last band takes everything below) and 0 otherwise, bricks sum in those units and multiply
// by 2^T_j in float64 when they write.  A staged weight is at least 2^-kWeightBand, so even times a shape factor near the
// support edge it stays a normal float.  Nearly every call spans fewer orders than one band: bin3_kernel stages it and
// the bricks are summed once, as they always were; each further band rewrites the record weights from prop and h in
// float64 (rec3_weights_kernel, O(n)) and sums the bricks again over the same sorted pairs.
constexpr int kExpBias3 = 1 << 20;
constexpr int kWeightBand = 100;

// band j of the call from the two words of wexp3_kernel: exponents bot <= e <= hi are staged relative to 2^top (hi = top
// except in band 0, which takes everything above as well)
struct Band3 { int top, bot, hi; };
__host__ __device__ __forceinline__ Band3 band3(int wmax, int wmin, int j)
{
    if (wmax <= 0) return { 0, -(1 << 30), 1 << 30 };             // no finite non-zero weight may take the brick path
    const int emax = wmax - kExpBias3, emin = kExpBias3 - wmin, top = emax - j * kWeightBand;
    return { top, top - kWeightBand < emin ? -(1 << 30) : top - kWeightBand + 1, j == 0 ? 1 << 30 : top };
}
__host__ __device__ __forceinline__ int n_bands3(int wmax, int wmin)
{
    return wmax <= 0 ? 1 : ((wmax - kExpBias3) - (kExpBias3 - wmin)) / kWeightBand + 1;
}

// float32 record weight of band b (0 outside it; 0, inf and NaN as they are)
__device__ __forceinline__ float band_weight3(double w, Band3 b)
{
    if (w != 0.0 && fabs(w) < INFINITY) {
        int ex;
        frexp(w, &ex);
        if (ex < b.bot || ex > b.hi) return 0.f;
    }
    return (float)scalbn(w, -b.top);
}


// periodic image shift along axis c of image m (0 when there is a single image).  Computed arithmetically: a table in
// kernel-parameter space indexed by the loop counter made ptxas keep the counter in a uniform register across the
// divergent early returns of classify3 and the kernel faulted on some inputs.
__host__ __device__ __forceinline__ double image_shift3(int n_img, const double *box, int m, int c)
{
    const int t = c == 0 ? m / 9 : (c == 1 ? (m / 3) % 3 : m % 3);
    return n_img == 1 ? 0.0 : (double)(t - 1) * box[c];
}

__device__ __forceinline__ double norm3(const P3 &p, double h)
{
    const double ih = 1.0 / h;
    const double t = p.norm_c * ih * ih;
    return p.norm_dim == 3 ? t * ih : t;
}

// wexp[0] = largest exponent + kExpBias3, wexp[1] = kExpBias3 - smallest exponent, over the particles that may get a record.
// A particle whose support spans at most small_max_vox voxels even unclipped (at most floor(4h / d) + 1 samples per axis lie
// within 2h) is deposited directly in every periodic image and is left out: a heavy or tiny-h particle deposited directly
// must not push the brick path's weights into a lower band.
__global__ void __launch_bounds__(256) wexp3_kernel(P3 p, int *__restrict__ wexp)
{
    int emax = 0, emin = 0;                                       // biased, 0 = nothing seen
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += (int64_t)gridDim.x * blockDim.x) {
        const double h = p.h[i];
        if (!(h > 0.0 && 2.0 * h < INFINITY)) continue;
        const double span = 4.0 * h * (1.0 + 1e-9);
        double vox = 1.0;
#pragma unroll
        for (int c = 0; c < 3; ++c) vox *= floor(span * p.ax[c].inv_d) + 1.0;
        if (vox <= (double)p.small_max_vox) continue;
        const double c = p.prop[i] * norm3(p, h);
        if (c != 0.0 && fabs(c) < INFINITY) {
            int ex;
            frexp(c, &ex);
            emax = max(emax, ex + kExpBias3);
            emin = max(emin, kExpBias3 - ex);
        }
    }
    emax = __reduce_max_sync(0xffffffffu, emax);
    emin = __reduce_max_sync(0xffffffffu, emin);
    if ((threadIdx.x & 31) == 0 && emax > 0) { atomicMax(wexp, emax); atomicMax(wexp + 1, emin); }
}

// record weights of band b for every particle (the entries of particles without a record are never read)
__global__ void __launch_bounds__(256) rec3_weights_kernel(P3 p, Rec3 *__restrict__ rec, Band3 b)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < p.n) rec[i].c = band_weight3(p.prop[i] * norm3(p, p.h[i]), b);
}

template <int SHAPE>
__device__ __forceinline__ void deposit_small3(const P3 &p, const Bin3 &b, const double *q, double h, double R2, double coef)
{
    const double inv_h2 = 1.0 / (h * h);
    const size_t ny = p.ax[1].n, nz = p.ax[2].n;
    for (int xi = b.lo[0]; xi <= b.hi[0]; ++xi) {
        const double dx2 = dist2(p.ax[0], q[0], xi);
        for (int yi = b.lo[1]; yi <= b.hi[1]; ++yi) {
            const double dxy = AST_DADD(dx2, dist2(p.ax[1], q[1], yi));
            double *row = p.out + ((size_t)xi * ny + yi) * nz;
            for (int zi = b.lo[2]; zi <= b.hi[2]; ++zi) {
                const double r2 = AST_DADD(dxy, dist2(p.ax[2], q[2], zi));
                if (r2 < R2) atomicAdd(row + zi, coef * (double)shape_eval<SHAPE>(fast_sqrt((float)(r2 * inv_h2)), p.tab));
            }
        }
    }
}

template <int SHAPE, bool DEPOSIT>
__global__ void __launch_bounds__(kBin3Threads) bin3_kernel(P3 p, Rec3 *__restrict__ rec, uint64_t *__restrict__ block_pairs,
                                                            uint64_t *__restrict__ block_huge)
{
    __shared__ uint32_t red[34];
    const int64_t i = (int64_t)blockIdx.x * kBin3Threads + threadIdx.x;
    uint32_t npairs = 0, nhuge = 0;
    uint64_t mask = 0;
    if (i < p.n) {
        const double x0[3] = { p.pos[3 * i], p.pos[3 * i + 1], p.pos[3 * i + 2] };
        const double h = p.h[i], R2 = radius2(h), h2 = 2.0 * h;
        bool need_rec = false;
        // images m = 9 ia + 3 ib + ic in ascending order; an axis shift that cannot reach the grid prunes its 9 or 3 images at once
        const int nt = p.n_img == 1 ? 1 : 3;
        for (int ia = 0; ia < nt; ++ia) {
            double q[3];
            q[0] = AST_DADD(x0[0], p.n_img == 1 ? 0.0 : (double)(ia - 1) * p.box[0]);
            if (!may_touch(p.ax[0], q[0], h2)) continue;
            for (int ib = 0; ib < nt; ++ib) {
                q[1] = AST_DADD(x0[1], p.n_img == 1 ? 0.0 : (double)(ib - 1) * p.box[1]);
                if (!may_touch(p.ax[1], q[1], h2)) continue;
                for (int ic = 0; ic < nt; ++ic) {
                    q[2] = AST_DADD(x0[2], p.n_img == 1 ? 0.0 : (double)(ic - 1) * p.box[2]);
                    if (!may_touch(p.ax[2], q[2], h2)) continue;
                    const int m = 9 * ia + 3 * ib + ic;
                    Bin3 b = classify3<BRICK>(p.ax, q, h, R2, p.small_max_vox, p.huge_min_bricks);
                    if (b.cls == CLS_SMALL) {
                        if (DEPOSIT) deposit_small3<SHAPE>(p, b, q, h, R2, p.prop[i] * norm3(p, h));
                    } else if (b.cls == CLS_TILED) {
                        npairs += (uint32_t)for_each_brick3<BRICK>(p.ax, q, R2, b, p.nb[1], p.nb[2], [](uint32_t) {});
                        mask |= 1ull << m;
                        need_rec = true;
                    } else if (b.cls == CLS_HUGE) {
                        ++nhuge;
                        mask |= 1ull << (27 + m);
                        need_rec = true;
                    }
                }
            }
        }
        if (need_rec && DEPOSIT) {
            Rec3 r;
            r.x = x0[0]; r.y = x0[1]; r.z = x0[2];
            r.inv_h = (float)(1.0 / h);
            r.c = band_weight3(p.prop[i] * norm3(p, h), band3(__ldg(p.wexp), __ldg(p.wexp + 1), 0));     // band 0
            rec[i] = r;
        }
    }
    uint32_t tp = block_sum_u32(npairs, red);
    uint32_t th = block_sum_u32(nhuge, red);
    if ((tp | th) != 0u && i < p.n) { p.pcount[i] = npairs; p.pmask[i] = mask; }     // emit3 only visits blocks with entries
    if (threadIdx.x == 0) {
        block_pairs[blockIdx.x] = tp;
        block_huge[blockIdx.x] = th;
    }
}

__global__ void __launch_bounds__(kBin3Threads, 3) emit3_kernel(P3 p, const uint64_t *__restrict__ pairs_excl,
                                                             const uint64_t *__restrict__ huge_excl, uint64_t w0, uint64_t w1,
                                                             uint64_t *__restrict__ pairs, uint64_t *__restrict__ huge,
                                                             uint64_t h0, uint64_t h1)
{
    __shared__ uint32_t sm[34];
    const uint64_t pbase = pairs_excl[blockIdx.x], pnext = pairs_excl[blockIdx.x + 1];
    const uint64_t hbase = huge_excl[blockIdx.x], hnext = huge_excl[blockIdx.x + 1];
    const bool any_pairs = pnext > pbase && pnext > w0 && pbase < w1;
    const bool any_huge = hnext > hbase && hnext > h0 && hbase < h1;     // large-h entries with list index in [h0, h1) -> huge[gh - h0]
    if (!any_pairs && !any_huge) return;
    const int64_t i = (int64_t)blockIdx.x * kBin3Threads + threadIdx.x;
    // counts and image masks come from bin3_kernel: one enumeration of the bricks here, and only for the images that have any
    uint32_t npairs = 0, nhuge = 0;
    uint64_t mask = 0;
    if (i < p.n) {
        npairs = p.pcount[i];
        mask = p.pmask[i];
        nhuge = (uint32_t)__popcll(mask >> 27);
    }
    uint32_t tot;
    uint64_t g = pbase + block_excl_scan_u32(npairs, sm, &tot);
    uint64_t gh = hbase + block_excl_scan_u32(nhuge, sm, &tot);
    if (i >= p.n || (npairs == 0 && nhuge == 0)) return;
    const double x0[3] = { p.pos[3 * i], p.pos[3 * i + 1], p.pos[3 * i + 2] };
    const double h = p.h[i], R2 = radius2(h);
    for (int m = 0; m < p.n_img; ++m) {
        if (!((mask >> m) & 0x8000001ull)) continue;                       // image m has neither pairs nor a large-h entry
        const double q[3] = { AST_DADD(x0[0], image_shift3(p.n_img, p.box, m, 0)), AST_DADD(x0[1], image_shift3(p.n_img, p.box, m, 1)), AST_DADD(x0[2], image_shift3(p.n_img, p.box, m, 2)) };
        Bin3 b = classify3<BRICK>(p.ax, q, h, R2, p.small_max_vox, p.huge_min_bricks);
        if (b.cls == CLS_TILED) {
            if (!any_pairs) continue;
            for_each_brick3<BRICK>(p.ax, q, R2, b, p.nb[1], p.nb[2], [&](uint32_t key) {
                if (g >= w0 && g < w1)
                    pairs[g - w0] = ((uint64_t)((key << p.img_shift) | (uint32_t)m) << 32) | (uint64_t)(uint32_t)i;
                ++g;
            });
        } else if (b.cls == CLS_HUGE) {
            if (gh >= h0 && gh < h1) huge[gh - h0] = ((uint64_t)m << 32) | (uint64_t)(uint32_t)i;
            ++gh;
        }
    }
}

// Large-h split (round 2, same as huge_tiles_kernel of project2d.cu): one WARP per entry of the large-h list enumerates the
// entry's brick bbox 32 bricks at a time in emit order (bx, by, bz ascending) with the membership test of for_each_brick3.
// WRITE = false: hoff[e] = number of member bricks.  WRITE = true: hoff holds the exclusive scan; pair number
// g = base + hoff[e] + rank goes to pairs[g - w0] when it falls into the window [w0, w1).  Round 1 let EVERY brick walk and cull
// the whole list (O(bricks x entries)).
template <bool WRITE>
__global__ void __launch_bounds__(256) huge_bricks_kernel(P3 p, const uint64_t *__restrict__ huge, uint32_t n_entries,
                                                          uint64_t *__restrict__ hoff, uint64_t base, uint64_t w0, uint64_t w1,
                                                          uint64_t *__restrict__ pairs)
{
    const uint32_t e = (uint32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (e >= n_entries) return;                             // uniform for the warp
    uint64_t g = 0;
    if (WRITE) {
        g = base + hoff[e];
        const uint64_t gend = base + hoff[e + 1];
        if (gend <= w0 || g >= w1) return;
    }
    const uint64_t ent = huge[e];
    const int64_t i = (int64_t)(uint32_t)ent;
    const int m = (int)(ent >> 32);
    const double h = p.h[i], R2 = radius2(h);
    const double q[3] = { AST_DADD(p.pos[3 * i], image_shift3(p.n_img, p.box, m, 0)), AST_DADD(p.pos[3 * i + 1], image_shift3(p.n_img, p.box, m, 1)),
                          AST_DADD(p.pos[3 * i + 2], image_shift3(p.n_img, p.box, m, 2)) };
    const Bin3 b = classify3<BRICK>(p.ax, q, h, R2, p.small_max_vox, p.huge_min_bricks);
    const int ny_b = b.b1[1] - b.b0[1] + 1, nz_b = b.b1[2] - b.b0[2] + 1;
    const int64_t nt = (int64_t)(b.b1[0] - b.b0[0] + 1) * ny_b * nz_b;
    uint32_t cnt = 0;
    const unsigned lt = (1u << lane) - 1u;
    for (int64_t t0 = 0; t0 < nt; t0 += 32) {
        const int64_t t = t0 + lane;
        bool in = false;
        uint32_t key = 0;
        if (t < nt) {
            const int bz = b.b0[2] + (int)(t % nz_b), by = b.b0[1] + (int)((t / nz_b) % ny_b), bx = b.b0[0] + (int)(t / ((int64_t)nz_b * ny_b));
            const int bc[3] = { bx, by, bz };
            double md[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const int a0 = bc[c] * BRICK > b.lo[c] ? bc[c] * BRICK : b.lo[c];
                const int a1 = bc[c] * BRICK + BRICK - 1 < b.hi[c] ? bc[c] * BRICK + BRICK - 1 : b.hi[c];
                md[c] = min_dist2(p.ax[c], q[c], a0, a1);
            }
            in = AST_DADD(AST_DADD(md[0], md[1]), md[2]) < R2;
            key = (uint32_t)((bx * p.nb[1] + by) * p.nb[2] + bz);
        }
        const unsigned ball = __ballot_sync(0xffffffffu, in);
        if (WRITE) {
            const uint64_t gg = g + (uint64_t)__popc(ball & lt);
            if (in && gg >= w0 && gg < w1)
                pairs[gg - w0] = ((uint64_t)((key << p.img_shift) | (uint32_t)m) << 32) | (uint64_t)(uint32_t)i;
            g += (uint64_t)__popc(ball);
        } else {
            cnt += (uint32_t)__popc(ball);
        }
    }
    if (!WRITE && lane == 0) hoff[e] = (uint64_t)cnt;
}

static __global__ void brick_range_kernel(const uint64_t *__restrict__ sorted, int64_t n, int img_shift, uint32_t *__restrict__ tbeg,
                                          uint32_t *__restrict__ tend)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t t = (uint32_t)(sorted[i] >> 32) >> img_shift;
    if (i == 0 || ((uint32_t)(sorted[i - 1] >> 32) >> img_shift) != t) tbeg[t] = (uint32_t)i;
    if (i == n - 1 || ((uint32_t)(sorted[i + 1] >> 32) >> img_shift) != t) tend[t] = (uint32_t)(i + 1);
}

struct Acc3 {
    const uint64_t *sorted;
    const uint32_t *tbeg, *tend;
    const uint64_t *huge;
    uint32_t n_huge;
    const Rec3 *rec;
    double *out;
    double lo[3], d[3], inv_d[3];
    int n[3], nb[3], img_shift, n_img;
    double box[3];
    ShapeTab tab;
    const uint32_t *seg_off;     // work items over the brick lists (work_items.cuh); ntiles = number of bricks
    int ntiles;
    int etop;                    // the float32 weights are relative to 2^etop (the top of the current band)
};

// One CTA per work item of a brick (a whole brick list, or an interleaved share of a long one), four autonomous warps (no CTA barrier): warp w owns the 4x4x8 column (x,y quadrant) of the brick and
// walks the brick's list on its own, 32 entries at a time: every lane stages one entry (float64 -> brick-relative float32),
// tests it against the warp's column, hits are compacted into the warp's shared-memory slots with a ballot (entries whose
// column lies wholly in the outer annulus q >= 1 of the cubic spline go to a second, cheaper loop), then every lane
// evaluates the hits for its 4 voxels (contiguous in z).  For batches with enough hits the staging lane also writes the
// entry's squared in-plane distances to the 16 (x, y) voxel columns and its squared z-distances to the 8 levels (in units of
// h), as the 2-D kernel does with its rows and columns: an evaluating lane then fetches one in-plane value and four level
// values (LDS.32 + LDS.128) and the squared radius of a voxel is one FADD instead of 11 instructions per entry and lane.
constexpr int kBrickTabMinHits = 10;
struct __align__(16) BrickSlot {
    float4 axy[4];       // squared in-plane distance to voxel column (x = i, y = j) at [i].{x,y,z,w}[j]   -- or the classic view:
                         // axy[0] = {ux*sx, uy*sy, uz*sz, c}, axy[1] = {sx, sy, sz, -}
    float4 cz[2];        // squared z-distance to levels 0..3, 4..7
    float4 w;            // {c, -, -, -}
};
static_assert(sizeof(BrickSlot) == 112, "slot layout");

template <int SHAPE>
__global__ void __launch_bounds__(kAcc3Threads) brick_accum_kernel(Acc3 a)
{
    __shared__ BrickSlot sB[4][32];
    TileWork w;
    if (!resolve_work(a, w)) return;
    const int brick = w.tile;
    const uint32_t beg = __shfl_sync(0xffffffffu, w.beg, 0), total = __shfl_sync(0xffffffffu, w.cnt, 0);   // uniform loop control
    const uint32_t w_first = __shfl_sync(0xffffffffu, w.first, 0), w_step = __shfl_sync(0xffffffffu, w.step, 0);
    if (total == 0) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int bz = brick % a.nb[2], by = (brick / a.nb[2]) % a.nb[1], bx = brick / (a.nb[2] * a.nb[1]);
    const int X0 = bx * BRICK, Y0 = by * BRICK, Z0 = bz * BRICK;
    const int xl = 4 * (warp >> 1) + (lane >> 3);
    const int yl = 4 * (warp & 1) + ((lane >> 1) & 3);
    const int zl = 4 * (lane & 1);
    const float xf = (float)xl, yf = (float)yl;
    const float zf0 = (float)zl, zf1 = (float)(zl + 1), zf2 = (float)(zl + 2), zf3 = (float)(zl + 3);
    const float lox = 4.f * (float)(warp >> 1), loy = 4.f * (float)(warp & 1);
    const float d0 = (float)a.d[0], d1 = (float)a.d[1], d2 = (float)a.d[2];
    BrickSlot *const slots = sB[warp];
    float acc[4] = { 0.f, 0.f, 0.f, 0.f };
    double acc64[4] = { 0.0, 0.0, 0.0, 0.0 };
    int since_fold = 0;

    for (uint32_t base = w_first; base < total; base += w_step) {
        const uint32_t j = base + lane;
        bool hit = false, outer = false;
        float4 P = make_float4(0.f, 0.f, 0.f, 0.f), S = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < total) {
            const uint64_t e = a.sorted[beg + j];
            const uint32_t idx = (uint32_t)e, m = ((uint32_t)(e >> 32)) & ((1u << a.img_shift) - 1u);
            const Rec3 r = a.rec[idx];
            const float fx = (float)((r.x + image_shift3(a.n_img, a.box, (int)m, 0) - a.lo[0]) * a.inv_d[0] - (double)X0);
            const float fy = (float)((r.y + image_shift3(a.n_img, a.box, (int)m, 1) - a.lo[1]) * a.inv_d[1] - (double)Y0);
            const float fz = (float)((r.z + image_shift3(a.n_img, a.box, (int)m, 2) - a.lo[2]) * a.inv_d[2] - (double)Z0);
            const float sx = d0 * r.inv_h, sy = d1 * r.inv_h, sz = d2 * r.inv_h;
            const float ddx = fmaxf(fmaxf(lox - fx, fx - (lox + 3.f)), 0.f) * sx;
            const float ddy = fmaxf(fmaxf(loy - fy, fy - (loy + 3.f)), 0.f) * sy;
            const float ddz = fmaxf(fmaxf(-fz, fz - 7.f), 0.f) * sz;
            const float qmin2 = ddx * ddx + ddy * ddy + ddz * ddz;
            hit = qmin2 < 4.0001f;
            outer = hit && SHAPE == SHAPE_CUBIC && qmin2 >= 1.0f;
            P = make_float4(fx * sx, fy * sy, fz * sz, SHAPE == SHAPE_CUBIC ? 2.0f * r.c : r.c);   // cubic: loops return f/2
            S = make_float4(sx, sy, sz, 0.f);
        }
        const unsigned ball_f = __ballot_sync(0xffffffffu, hit && !outer);
        const unsigned ball_o = __ballot_sync(0xffffffffu, outer);
        const int nf = __popc(ball_f), no = __popc(ball_o);
        if (nf + no == 0) continue;
        const unsigned lt = (1u << lane) - 1u;
        const int dst = outer ? 31 - __popc(ball_o & lt) : __popc(ball_f & lt);
        if (nf + no >= kBrickTabMinHits) {
            if (hit) {
                BrickSlot *d = slots + dst;
                float ax2[4], by2[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float tx = fmaf(-(lox + (float)i), S.x, P.x), ty = fmaf(-(loy + (float)i), S.y, P.y);
                    ax2[i] = tx * tx; by2[i] = ty * ty;
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) d->axy[i] = make_float4(ax2[i] + by2[0], ax2[i] + by2[1], ax2[i] + by2[2], ax2[i] + by2[3]);
                float cz[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { const float t = fmaf(-(float)i, S.z, P.z); cz[i] = t * t; }
                d->cz[0] = make_float4(cz[0], cz[1], cz[2], cz[3]);
                d->cz[1] = make_float4(cz[4], cz[5], cz[6], cz[7]);
                d->w = make_float4(P.w, 0.f, 0.f, 0.f);
            }
            __syncwarp();
            const int col = lane >> 1;                           // (x, y) voxel column of this lane inside the warp's 4 x 4: x = col >> 2, y = col & 3
            for (int e = 0; e < nf; ++e) {
                const float axy = reinterpret_cast<const float *>(slots[e].axy)[col];
                const float4 c = slots[e].cz[lane & 1];
                const float cc = slots[e].w.x;
                acc[0] = fmaf(cc, shape_half_full<SHAPE>(axy + c.x, a.tab), acc[0]);
                acc[1] = fmaf(cc, shape_half_full<SHAPE>(axy + c.y, a.tab), acc[1]);
                acc[2] = fmaf(cc, shape_half_full<SHAPE>(axy + c.z, a.tab), acc[2]);
                acc[3] = fmaf(cc, shape_half_full<SHAPE>(axy + c.w, a.tab), acc[3]);
            }
            if (SHAPE == SHAPE_CUBIC) {
                for (int e = 32 - no; e < 32; ++e) {
                    const float axy = reinterpret_cast<const float *>(slots[e].axy)[col];
                    const float4 c = slots[e].cz[lane & 1];
                    const float cc = slots[e].w.x;
                    const float a0 = __saturatef(fmaf(fast_sqrt(axy + c.x), -0.5f, 1.0f)), a1 = __saturatef(fmaf(fast_sqrt(axy + c.y), -0.5f, 1.0f));
                    const float a2 = __saturatef(fmaf(fast_sqrt(axy + c.z), -0.5f, 1.0f)), a3 = __saturatef(fmaf(fast_sqrt(axy + c.w), -0.5f, 1.0f));
                    acc[0] = fmaf(cc, a0 * a0 * a0, acc[0]);
                    acc[1] = fmaf(cc, a1 * a1 * a1, acc[1]);
                    acc[2] = fmaf(cc, a2 * a2 * a2, acc[2]);
                    acc[3] = fmaf(cc, a3 * a3 * a3, acc[3]);
                }
            }
        } else {
            if (hit) {
                slots[dst].axy[0] = P;
                slots[dst].axy[1] = S;
            }
            __syncwarp();
            for (int e = 0; e < nf; ++e) {
                const float4 s = slots[e].axy[1];
                const float4 q = slots[e].axy[0];
                const float ax = fmaf(-xf, s.x, q.x), by2 = fmaf(-yf, s.y, q.y);
                const float axy = fmaf(by2, by2, ax * ax);
                const float c0 = fmaf(-zf0, s.z, q.z), c1 = fmaf(-zf1, s.z, q.z), c2 = fmaf(-zf2, s.z, q.z), c3 = fmaf(-zf3, s.z, q.z);
                acc[0] = fmaf(q.w, shape_half_full<SHAPE>(fmaf(c0, c0, axy), a.tab), acc[0]);
                acc[1] = fmaf(q.w, shape_half_full<SHAPE>(fmaf(c1, c1, axy), a.tab), acc[1]);
                acc[2] = fmaf(q.w, shape_half_full<SHAPE>(fmaf(c2, c2, axy), a.tab), acc[2]);
                acc[3] = fmaf(q.w, shape_half_full<SHAPE>(fmaf(c3, c3, axy), a.tab), acc[3]);
            }
            if (SHAPE == SHAPE_CUBIC) {
                for (int e = 32 - no; e < 32; ++e) {
                    const float4 s = slots[e].axy[1];
                    const float4 q = slots[e].axy[0];
                    const float cc = q.w;
                    const float ax = fmaf(-xf, s.x, q.x), by2 = fmaf(-yf, s.y, q.y);
                    const float axy = fmaf(by2, by2, ax * ax);
                    const float c0 = fmaf(-zf0, s.z, q.z), c1 = fmaf(-zf1, s.z, q.z), c2 = fmaf(-zf2, s.z, q.z), c3 = fmaf(-zf3, s.z, q.z);
                    float a0 = __saturatef(fmaf(fast_sqrt(fmaf(c0, c0, axy)), -0.5f, 1.0f));
                    float a1 = __saturatef(fmaf(fast_sqrt(fmaf(c1, c1, axy)), -0.5f, 1.0f));
                    float a2 = __saturatef(fmaf(fast_sqrt(fmaf(c2, c2, axy)), -0.5f, 1.0f));
                    float a3 = __saturatef(fmaf(fast_sqrt(fmaf(c3, c3, axy)), -0.5f, 1.0f));
                    acc[0] = fmaf(cc, a0 * a0 * a0, acc[0]);
                    acc[1] = fmaf(cc, a1 * a1 * a1, acc[1]);
                    acc[2] = fmaf(cc, a2 * a2 * a2, acc[2]);
                    acc[3] = fmaf(cc, a3 * a3 * a3, acc[3]);
                }
            }
        }
        __syncwarp();
        since_fold += nf + no;
        if (since_fold >= 96) {
            since_fold = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) { acc64[k] += (double)acc[k]; acc[k] = 0.f; }
        }
    }
    const int xi = X0 + xl, yi = Y0 + yl;
    if (xi < a.n[0] && yi < a.n[1]) {
        // the sums are in units of 2^E: two exact power-of-two factors (one could overflow at the ends of the exponent range)
        const int e = min(max(a.etop, -2040), 2040), e1 = e / 2, e2 = e - e1;
        const double sc1 = __longlong_as_double((long long)(e1 + 1023) << 52), sc2 = __longlong_as_double((long long)(e2 + 1023) << 52);
        double *row = a.out + ((size_t)xi * a.n[1] + yi) * a.n[2];
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (Z0 + zl + k < a.n[2]) {
                const double v = (acc64[k] + (double)acc[k]) * sc1 * sc2;
                if (w.atomic_out) atomicAdd(row + Z0 + zl + k, v); else row[Z0 + zl + k] += v;
            }
    }
}

__global__ void bbox_cls3_kernel(P3 p, int32_t *__restrict__ bbox, uint8_t *__restrict__ cls)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const double x0[3] = { p.pos[3 * i], p.pos[3 * i + 1], p.pos[3 * i + 2] };
    const double h = p.h[i], R2 = radius2(h);
    for (int m = 0; m < p.n_img; ++m) {
        const double q[3] = { AST_DADD(x0[0], image_shift3(p.n_img, p.box, m, 0)), AST_DADD(x0[1], image_shift3(p.n_img, p.box, m, 1)), AST_DADD(x0[2], image_shift3(p.n_img, p.box, m, 2)) };
        Bin3 b = classify3<BRICK>(p.ax, q, h, R2, p.small_max_vox, p.huge_min_bricks);
        const int64_t j = (int64_t)m * p.n + i;
        if (bbox)
            for (int c = 0; c < 3; ++c) { bbox[6 * j + 2 * c] = b.lo[c]; bbox[6 * j + 2 * c + 1] = b.hi[c]; }
        if (cls) cls[j] = (uint8_t)b.cls;
    }
}

constexpr int64_t kDefaultSmallMaxVox = 27;
constexpr int64_t kDefaultHugeMinBricks = 512;

struct Layout3 {
    int64_t nb, nbricks, pair_cap, huge_cap;
    uint64_t *block_pairs, *block_huge;
    Rec3 *rec;
    uint32_t *pcount;
    uint64_t *pmask;
    uint64_t *pairs_a, *pairs_b, *huge;
    uint32_t *tbeg, *tend, *seg_off, *seg_tmp;
    uint64_t *hoff, *hoff_tmp;
    int *wexp;
    void *sort_ws;
    PresortBuffers pre;          // only with AST_FLAG_ORDER_AUTO / _ALWAYS
    size_t bytes;
};

static int validate3(const ast_grid3d_params *p)
{
    AST_REQUIRE(p != nullptr, "params is null");
    AST_REQUIRE(p->n >= 0 && p->n < (int64_t)0xffffffffll, "n out of range");
    AST_REQUIRE(p->nx > 0 && p->ny > 0 && p->nz > 0, "grid size must be positive");
    const int64_t nbr = (int64_t)((p->nx + BRICK - 1) / BRICK) * ((p->ny + BRICK - 1) / BRICK) * ((p->nz + BRICK - 1) / BRICK);
    AST_REQUIRE(nbr < (1ll << 26), "grid too large (more than 2^26 bricks)");
    AST_REQUIRE(kernel_valid(p->kernel_id), "unknown kernel id %d", p->kernel_id);
    if (p->kernel_id == AST_KERNEL_TABLE)
        AST_REQUIRE(p->kernel_table != nullptr && p->kernel_table_n >= 2 && (p->kernel_dim == 2 || p->kernel_dim == 3),
                    "AST_KERNEL_TABLE needs kernel_table (device), kernel_table_n >= 2 and kernel_dim 2 or 3");
    for (int c = 0; c < 3; ++c) AST_REQUIRE(p->hi[c] > p->lo[c], "empty or inverted grid bounds");
    if (p->flags & AST_FLAG_PERIODIC)
        for (int c = 0; c < 3; ++c) AST_REQUIRE(p->box[c] > 0, "periodic gridding needs box[0..2] > 0");
    AST_REQUIRE(p->pair_capacity >= 0 && p->pair_capacity < (1ll << 32), "pair_capacity out of range");
    AST_REQUIRE(p->huge_capacity >= 0 && p->huge_capacity < (1ll << 32), "huge_capacity out of range");
    return AST_OK;
}

static Layout3 layout3(const ast_grid3d_params *p, void *ws)
{
    Layout3 L;
    L.nb = (p->n + kBin3Threads - 1) / kBin3Threads;
    if (L.nb < 1) L.nb = 1;
    L.nbricks = (int64_t)((p->nx + BRICK - 1) / BRICK) * ((p->ny + BRICK - 1) / BRICK) * ((p->nz + BRICK - 1) / BRICK);
    L.pair_cap = p->pair_capacity > 0 ? p->pair_capacity : 1;
    L.huge_cap = p->huge_capacity > 0 ? p->huge_capacity : 1;
    Carver c(ws);
    L.block_pairs = c.take<uint64_t>(L.nb + 1);
    L.block_huge = c.take<uint64_t>(L.nb + 1);
    L.rec = c.take<Rec3>(p->n > 0 ? p->n : 1);
    L.pcount = c.take<uint32_t>(p->n > 0 ? p->n : 1);
    L.pmask = c.take<uint64_t>(p->n > 0 ? p->n : 1);
    L.pairs_a = c.take<uint64_t>(L.pair_cap);
    L.pairs_b = c.take<uint64_t>(L.pair_cap);
    L.huge = c.take<uint64_t>(L.huge_cap);
    L.tbeg = c.take<uint32_t>(L.nbricks);
    L.tend = c.take<uint32_t>(L.nbricks);
    L.seg_off = c.take<uint32_t>(L.nbricks + 1);
    L.seg_tmp = (uint32_t *)c.take<char>(scan_workspace_bytes<uint32_t>(L.nbricks + 1));
    L.wexp = c.take<int>(2);
    L.hoff = c.take<uint64_t>(L.huge_cap + 1);
    L.hoff_tmp = (uint64_t *)c.take<char>(scan_workspace_bytes<uint64_t>(L.huge_cap + 1));
    L.sort_ws = c.take<char>(sort_workspace_bytes(L.pair_cap));
    memset(&L.pre, 0, sizeof L.pre);
    if (p->flags & (AST_FLAG_ORDER_AUTO | AST_FLAG_ORDER_ALWAYS)) {
        const size_t n = (size_t)(p->n > 0 ? p->n : 1);
        L.pre.counts = c.take<unsigned long long>(2);
        L.pre.ka = c.take<uint64_t>(n);
        L.pre.kb = c.take<uint64_t>(n);
        L.pre.sort_ws = c.take<char>(sort_workspace_bytes((int64_t)n));
        L.pre.spos = c.take<double>(3 * n);
        L.pre.sh = c.take<double>(n);
        L.pre.sprop[0] = c.take<double>(n);
        L.pre.sprop[1] = nullptr;
    }
    L.bytes = c.bytes();
    return L;
}

static P3 make_p3(const ast_grid3d_params *p, const double *pos, const double *h, const double *prop, double *out)
{
    P3 a;
    a.pos = pos; a.h = h; a.prop = prop; a.out = out;
    a.n = p->n;
    a.kernel_id = p->kernel_id;
    a.shape = kernel_shape(p->kernel_id);
    a.norm_c = p->kernel_id == AST_KERNEL_TABLE ? 1.0 : kernel_norm(p->kernel_id, 1.0);
    a.norm_dim = p->kernel_id == AST_KERNEL_TABLE ? p->kernel_dim : ((p->kernel_id == 0 || p->kernel_id == 2) ? 3 : 2);
    a.tab.tab = (const float2 *)p->kernel_table;
    a.tab.n = p->kernel_table_n;
    a.tab.scale = 0.5f * (float)p->kernel_table_n;
    const int n3[3] = { p->nx, p->ny, p->nz };
    for (int c = 0; c < 3; ++c) {
        a.ax[c] = make_axis(p->lo[c], p->hi[c], n3[c]);
        a.nb[c] = (n3[c] + BRICK - 1) / BRICK;
    }
    const bool per = (p->flags & AST_FLAG_PERIODIC) != 0;
    a.n_img = per ? 27 : 1;
    a.img_shift = per ? 5 : 0;
    for (int c = 0; c < 3; ++c) a.box[c] = per ? p->box[c] : 0.0;
    a.small_max_vox = p->small_max_vox >= 0 ? p->small_max_vox : kDefaultSmallMaxVox;
    a.huge_min_bricks = p->huge_min_bricks >= 0 ? p->huge_min_bricks : kDefaultHugeMinBricks;
    a.wexp = nullptr;
    return a;
}

}  // namespace ast

using namespace ast;

extern "C" int ast_grid3d_workspace_bytes(const ast_grid3d_params *p, size_t *bytes)
{
    int rc = validate3(p);
    if (rc) return rc;
    AST_REQUIRE(bytes != nullptr, "bytes is null");
    *bytes = layout3(p, nullptr).bytes;
    return AST_OK;
}

extern "C" int ast_grid3d(const ast_grid3d_params *p, const double *pos, const double *h, const double *prop, double *out,
                          void *workspace, size_t workspace_bytes, void *stream, ast_project2d_stats *stats)
{
    int rc = validate3(p);
    if (rc) return rc;
    AST_REQUIRE(out != nullptr, "out is null");
    AST_REQUIRE(p->n == 0 || (pos && h && prop), "null input pointer");
    Layout3 L = layout3(p, workspace);
    if (workspace == nullptr || workspace_bytes < L.bytes) {
        set_error("workspace too small: need %zu bytes, have %zu", L.bytes, workspace_bytes);
        return AST_EWORKSPACE;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const bool timing = (p->flags & AST_FLAG_TIMING) != 0;
    StageTimer tm(timing, s), tk(timing, s);
    ast_project2d_stats st;
    memset(&st, 0, sizeof st);
    tm.begin(7);
    tk.begin(6);
    // optional spatial pre-ordering (presort.cuh): key = brick of the particle's own position
    if ((p->flags & (AST_FLAG_ORDER_AUTO | AST_FLAG_ORDER_ALWAYS)) && p->n > 0) {
        OrderGrid og;
        memset(&og, 0, sizeof og);
        og.dims = 3;
        const int n3[3] = { p->nx, p->ny, p->nz };
        for (int k = 0; k < 3; ++k) {
            og.col[k] = k;
            og.lo[k] = p->lo[k];
            og.inv_cell[k] = 1.0 / ((p->hi[k] - p->lo[k]) / n3[k] * BRICK);
            og.n[k] = (n3[k] + BRICK - 1) / BRICK;
        }
        int done = 0, nl = 0;
        const double *props1[1] = { prop };
        AST_CUDA_TRY(presort_particles((p->flags & AST_FLAG_ORDER_ALWAYS) ? 2 : 1, og, pos, h, props1, 1, p->n, L.pre, s, &done, &nl));
        st.n_launches += nl;
        st.reordered = done;
        if (done) { pos = L.pre.spos; h = L.pre.sh; prop = L.pre.sprop[0]; }
    }
    P3 a = make_p3(p, pos, h, prop, out);
    a.pcount = L.pcount; a.pmask = L.pmask; a.wexp = L.wexp;
    const size_t nvox = (size_t)p->nx * p->ny * p->nz;
    if (!(p->flags & AST_FLAG_ACCUMULATE)) AST_CUDA_TRY(cudaMemsetAsync(out, 0, sizeof(double) * nvox, s));
    AST_CUDA_TRY(cudaMemsetAsync(L.block_pairs, 0, sizeof(uint64_t) * (L.nb + 1), s));
    AST_CUDA_TRY(cudaMemsetAsync(L.block_huge, 0, sizeof(uint64_t) * (L.nb + 1), s));
    AST_CUDA_TRY(cudaMemsetAsync(L.wexp, 0, 2 * sizeof(int), s));
    tk.end();
    uint64_t totals[2] = { 0, 0 };
    int wexp[2] = { 0, 0 };
    if (p->n > 0) {
        tk.begin(0);
        {
            int dev = 0, sm = 148;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev);
            const int64_t want = (p->n + 255) / 256;
            wexp3_kernel<<<(unsigned)(want < (int64_t)sm * 8 ? want : (int64_t)sm * 8), 256, 0, s>>>(a, L.wexp);
        }
        if (a.shape == SHAPE_CUBIC) bin3_kernel<SHAPE_CUBIC, true><<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, L.rec, L.block_pairs, L.block_huge);
        else if (a.shape == SHAPE_WENDLAND) bin3_kernel<SHAPE_WENDLAND, true><<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, L.rec, L.block_pairs, L.block_huge);
        else bin3_kernel<SHAPE_TABLE, true><<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, L.rec, L.block_pairs, L.block_huge);
        tk.end();
        tk.begin(1);
        scan_exclusive_kernel<uint64_t><<<1, kScanThreads, 0, s>>>(L.block_pairs, L.nb + 1, nullptr);
        scan_exclusive_kernel<uint64_t><<<1, kScanThreads, 0, s>>>(L.block_huge, L.nb + 1, nullptr);
        tk.end();
        st.n_launches += 4;
        AST_CUDA_TRY(cudaGetLastError());
        AST_CUDA_TRY(cudaMemcpyAsync(&totals[0], L.block_pairs + L.nb, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaMemcpyAsync(&totals[1], L.block_huge + L.nb, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaMemcpyAsync(wexp, L.wexp, sizeof wexp, cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaStreamSynchronize(s));
    }
    const uint64_t T = totals[0], H = totals[1];
    st.n_pairs = (int64_t)T;
    st.n_huge = (int64_t)H;
    if (T + H > 0 && p->pair_capacity <= 0) {
        set_error("pair_capacity is 0 but %llu pairs and %llu large-h particles need the brick path", (unsigned long long)T,
                  (unsigned long long)H);
        if (stats) *stats = st;
        return AST_EWORKSPACE;
    }
    if (T + H > 0) {
        // pair_capacity and huge_capacity are WINDOWS: the combined pair order -- tiled pairs, then the member bricks of the
        // current window of the large-h list -- is walked through the pair window in rounds, so no capacity can fail after the
        // binning kernel has deposited the few-voxel particles
        const uint64_t cap = (uint64_t)L.pair_cap, hcap = (uint64_t)L.huge_cap;
        const int key_bits = ceil_log2_u64((uint64_t)L.nbricks);     // the image bits below the brick key are NOT sorted on
        Acc3 c;
        c.tbeg = L.tbeg; c.tend = L.tend; c.huge = L.huge; c.rec = L.rec; c.out = out;
        for (int k = 0; k < 3; ++k) {
            c.lo[k] = a.ax[k].vmin; c.d[k] = a.ax[k].d; c.inv_d[k] = a.ax[k].inv_d; c.n[k] = a.ax[k].n; c.nb[k] = a.nb[k];
        }
        c.img_shift = a.img_shift;
        c.n_img = a.n_img;
        c.tab = a.tab;
        c.n_huge = 0u;
        const int n_bands = n_bands3(wexp[0], wexp[1]);
        int rec_band = 0;                                           // the band whose weights the records hold (bin3_kernel: 0)
        for (int k = 0; k < 3; ++k) c.box[k] = a.box[k];
        static const int sm_count = [] { int dev = 0, n = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); return n; }();
        int64_t round_no = 0;
        const uint64_t n_hwin = H ? (H + hcap - 1) / hcap : 1;
        for (uint64_t hw = 0; hw < n_hwin; ++hw) {
            uint64_t HP = 0;
            uint32_t n_hent = 0;
            if (H) {                    // the large-h window: list entries [h0, h1) -> member-brick counts -> offsets
                const uint64_t h0 = hw * hcap, h1 = (h0 + hcap < H) ? h0 + hcap : H;
                n_hent = (uint32_t)(h1 - h0);
                tk.begin(2);
                emit3_kernel<<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, L.block_pairs, L.block_huge, 0, 0, L.pairs_a, L.huge, h0, h1);
                AST_CUDA_TRY(cudaMemsetAsync(L.hoff + n_hent, 0, sizeof(uint64_t), s));
                huge_bricks_kernel<false><<<(n_hent + 7) / 8, 256, 0, s>>>(a, L.huge, n_hent, L.hoff, 0, 0, 0, nullptr);
                int nlh = 0;
                AST_CUDA_TRY(scan_exclusive<uint64_t>(L.hoff, (int64_t)n_hent + 1, L.hoff_tmp, nullptr, s, &nlh));
                st.n_launches += 2 + nlh;
                tk.end();
                AST_CUDA_TRY(cudaMemcpyAsync(&HP, L.hoff + n_hent, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
                AST_CUDA_TRY(cudaStreamSynchronize(s));
                st.n_pairs += (int64_t)HP;
            }
            const uint64_t base = hw == 0 ? T : 0, total = base + HP;
            if (total == 0) continue;
            const uint64_t rounds = (total + cap - 1) / cap;
            uint64_t per_round = rounds > 1 ? (((total + rounds - 1) / rounds + 8191ull) & ~8191ull) : cap;
            if (per_round > cap) per_round = cap;
            for (uint64_t r = 0; r * per_round < total; ++r, ++round_no) {
                const uint64_t w0 = r * per_round, w1 = (w0 + per_round < total) ? w0 + per_round : total;
                const int64_t nw = (int64_t)(w1 - w0);
                tk.begin(2);
                if (hw == 0 && w0 < T)
                    emit3_kernel<<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, L.block_pairs, L.block_huge, w0, w1 < T ? w1 : T, L.pairs_a, L.huge, 0, 0);
                if (HP > 0 && w1 > base)
                    huge_bricks_kernel<true><<<(n_hent + 7) / 8, 256, 0, s>>>(a, L.huge, n_hent, L.hoff, base, w0, w1, L.pairs_a);
                tk.end();
                int in_b = 0, nl = 0;
                tk.begin(3);
                AST_CUDA_TRY(radix_sort_u64(L.pairs_a, L.pairs_b, nw, 32 + a.img_shift, key_bits, L.sort_ws, s, &in_b, &nl));
                tk.end();
                tk.begin(4);
                AST_CUDA_TRY(cudaMemsetAsync(L.tbeg, 0, sizeof(uint32_t) * L.nbricks, s));
                AST_CUDA_TRY(cudaMemsetAsync(L.tend, 0, sizeof(uint32_t) * L.nbricks, s));
                c.sorted = in_b ? L.pairs_b : L.pairs_a;
                brick_range_kernel<<<(unsigned)((nw + 255) / 256), 256, 0, s>>>(c.sorted, nw, a.img_shift, L.tbeg, L.tend);
                tk.end();
                // work items: long brick lists (cluster cores) are shared by several CTAs, see work_items.cuh
                const uint32_t seg_target = segment_target(nw, (int64_t)sm_count * 8);
                c.seg_off = L.seg_off; c.ntiles = (int)L.nbricks;
                tile_segments_kernel<<<(unsigned)((L.nbricks + 1 + 255) / 256), 256, 0, s>>>(L.tbeg, L.tend, 0u, seg_target, (int)L.nbricks, L.seg_off);
                int nls = 0;
                AST_CUDA_TRY(scan_exclusive<uint32_t>(L.seg_off, L.nbricks + 1, L.seg_tmp, nullptr, s, &nls));
                const int64_t max_items = L.nbricks + nw / (int64_t)seg_target;
                tk.begin(5);
                for (int j = 0; j < n_bands; ++j) {
                    const Band3 b = band3(wexp[0], wexp[1], j);
                    if (j != rec_band) {
                        rec3_weights_kernel<<<(unsigned)((p->n + 255) / 256), 256, 0, s>>>(a, L.rec, b);
                        rec_band = j;
                        st.n_launches += 1;
                    }
                    c.etop = b.top;
                    if (a.shape == SHAPE_CUBIC) brick_accum_kernel<SHAPE_CUBIC><<<(unsigned)max_items, kAcc3Threads, 0, s>>>(c);
                    else if (a.shape == SHAPE_WENDLAND) brick_accum_kernel<SHAPE_WENDLAND><<<(unsigned)max_items, kAcc3Threads, 0, s>>>(c);
                    else brick_accum_kernel<SHAPE_TABLE><<<(unsigned)max_items, kAcc3Threads, 0, s>>>(c);
                }
                tk.end();
                st.n_launches += 5 + n_bands + nl + nls;
                AST_CUDA_TRY(cudaGetLastError());
            }
        }
        st.n_rounds = round_no;
    }
    tm.end();
    if (timing) {
        float total_ms[8];
        tk.collect(st.stage_ms, 8);
        tm.collect(total_ms, 8);
        st.stage_ms[7] = total_ms[7];
    }
    if (stats) *stats = st;
    return AST_OK;
}

extern "C" int ast_bin3d(const ast_grid3d_params *p, const double *pos, const double *h, int32_t *bbox, uint8_t *cls,
                         uint64_t *pairs_sorted, uint64_t *huge, int64_t *counts, void *workspace, size_t workspace_bytes,
                         void *stream)
{
    int rc = validate3(p);
    if (rc) return rc;
    AST_REQUIRE(p->n == 0 || (pos && h), "null input pointer");
    Layout3 L = layout3(p, workspace);
    if (workspace == nullptr || workspace_bytes < L.bytes) {
        set_error("workspace too small: need %zu bytes, have %zu", L.bytes, workspace_bytes);
        return AST_EWORKSPACE;
    }
    cudaStream_t s = (cudaStream_t)stream;
    P3 a = make_p3(p, pos, h, nullptr, nullptr);
    a.pcount = L.pcount; a.pmask = L.pmask;
    uint64_t totals[2] = { 0, 0 };
    AST_CUDA_TRY(cudaMemsetAsync(L.block_pairs, 0, sizeof(uint64_t) * (L.nb + 1), s));
    AST_CUDA_TRY(cudaMemsetAsync(L.block_huge, 0, sizeof(uint64_t) * (L.nb + 1), s));
    if (p->n > 0) {
        if (bbox || cls) bbox_cls3_kernel<<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, bbox, cls);
        AST_KERNEL_CHECK(s, "bbox_cls3_kernel");
        bin3_kernel<SHAPE_CUBIC, false><<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, L.rec, L.block_pairs, L.block_huge);
        AST_KERNEL_CHECK(s, "bin3_kernel");
        scan_exclusive_kernel<uint64_t><<<1, kScanThreads, 0, s>>>(L.block_pairs, L.nb + 1, nullptr);
        scan_exclusive_kernel<uint64_t><<<1, kScanThreads, 0, s>>>(L.block_huge, L.nb + 1, nullptr);
        AST_KERNEL_CHECK(s, "scan_exclusive_kernel");
        AST_CUDA_TRY(cudaMemcpyAsync(&totals[0], L.block_pairs + L.nb, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaMemcpyAsync(&totals[1], L.block_huge + L.nb, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaStreamSynchronize(s));
    }
    const uint64_t T = totals[0], H = totals[1];
    uint64_t HP = 0;
    if (H > (uint64_t)p->huge_capacity || H > (uint64_t)L.huge_cap) {
        if (counts) { counts[0] = (int64_t)T; counts[1] = (int64_t)H; }
        set_error("capacity too small: need %llu huge entries", (unsigned long long)H);
        return AST_EWORKSPACE;
    }
    if (H > 0) {
        const uint32_t nh = (uint32_t)H;
        emit3_kernel<<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, L.block_pairs, L.block_huge, 0, 0, L.pairs_a, L.huge, 0, H);
        AST_CUDA_TRY(cudaMemsetAsync(L.hoff + nh, 0, sizeof(uint64_t), s));
        huge_bricks_kernel<false><<<(nh + 7) / 8, 256, 0, s>>>(a, L.huge, nh, L.hoff, 0, 0, 0, nullptr);
        AST_CUDA_TRY(scan_exclusive<uint64_t>(L.hoff, (int64_t)nh + 1, L.hoff_tmp, nullptr, s));
        AST_CUDA_TRY(cudaMemcpyAsync(&HP, L.hoff + nh, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaStreamSynchronize(s));
    }
    const uint64_t total = T + HP;
    if (counts) { counts[0] = (int64_t)total; counts[1] = (int64_t)H; }
    if (total > (uint64_t)p->pair_capacity) {
        set_error("capacity too small: need %llu pairs and %llu huge entries", (unsigned long long)total, (unsigned long long)H);
        return AST_EWORKSPACE;
    }
    if (total + H > 0) {
        if (T > 0) emit3_kernel<<<(unsigned)L.nb, kBin3Threads, 0, s>>>(a, L.block_pairs, L.block_huge, 0, T, L.pairs_a, L.huge, 0, 0);
        if (HP > 0) huge_bricks_kernel<true><<<((uint32_t)H + 7) / 8, 256, 0, s>>>(a, L.huge, (uint32_t)H, L.hoff, T, 0, total, L.pairs_a);
        AST_CUDA_TRY(cudaGetLastError());
        if (huge && H) AST_CUDA_TRY(cudaMemcpyAsync(huge, L.huge, sizeof(uint64_t) * H, cudaMemcpyDeviceToDevice, s));
        if (pairs_sorted && total) {
            int in_b = 0;
            const int key_bits = ceil_log2_u64((uint64_t)L.nbricks);
            AST_CUDA_TRY(radix_sort_u64(L.pairs_a, L.pairs_b, (int64_t)total, 32 + a.img_shift, key_bits, L.sort_ws, s, &in_b));
            AST_CUDA_TRY(cudaMemcpyAsync(pairs_sorted, in_b ? L.pairs_b : L.pairs_a, sizeof(uint64_t) * total,
                                         cudaMemcpyDeviceToDevice, s));
        }
    }
    AST_CUDA_TRY(cudaStreamSynchronize(s));
    return AST_OK;
}
