// project2d.cu -- 2-D line-of-sight projection of SPH particles onto a pixel map, sm_100a.
//
// Replaces create_image -> process_chunk -> calculate_pixel_value -> kernel_func of the reference
// (tools/projections/_projector.py:75-120,13-73; _pixel_calculations.pyx:9-36; _kernels.pyx:9-20).
// The reference gathers: for every pixel it scans every candidate particle.  Here the work is turned
// round (scatter by particle, gather by screen tile):
//
//   K1 bin_tma_kernel    persistent CTAs, inputs staged through shared memory by the TMA engine (cp.async.bulk + mbarrier);
//      (+ bin_kernel)    one thread per particle: float64 bbox (ast_geom.h), class, pair count and image mask; particles
//                        whose bbox is a few pixels are deposited right here with float64 atomics (the HBM-bound
//                        regime: inputs are read exactly once); the others get a 32-byte record.
//   scan                 exclusive scan of the per-block pair counts.
//   K3 emit_kernel       writes (tile key << 32 | particle) pairs in emit order (one enumeration: counts come from K1).
//   radix sort           stable, by tile key (scan_sort.cuh).
//   K5 pair_record_kernel  first/last pair of every tile, and per sorted pair the tile-relative float32 coordinates and
//                        weights the accumulate kernel needs (computed once, stored in list order).
//   K5b tile_segments    work items: long tile lists are shared by several CTAs with interleaved batches (work_items.cuh).
//   K6 rowcol_accum_kernel  one CTA per work item of a 32x32-pixel tile, 8 autonomous warps each owning an 8x16 sub-tile,
//                        2x2 pixels per thread in registers; every warp stages 32 list entries at a time through its own
//                        shared-memory slots, culls them against its sub-tile, stores the hits' squared row / column
//                        distances and evaluates them (one MUFU.SQRT per pixel); float32 partial sums are folded into
//                        float64 accumulators; the tile is written once.
//   large-h particles    (more than huge_min_tiles tiles: enumerating them inside one thread of K1 / K3 would stall its warp)
//                        go on a list; huge_tiles_kernel gives every entry a WARP that enumerates its tiles 32 at a time and
//                        appends (tile, particle) pairs behind the tiled ones, so the same sort / pair records / accumulate
//                        handle them and no tile ever walks particles that miss it.
#include <string.h>

#include "ast_geom.h"
#include "ast_math.h"
#include "block_utils.cuh"
#include "common.cuh"
#include "presort.cuh"
#include "scan_sort.cuh"
#include "work_items.cuh"

namespace ast {

constexpr int TILE = AST_TILE;
constexpr int kBinThreads = 256;

struct __align__(32) Rec {
    double pa, pb;             // in-plane position, float64 (tile-relative float32 is derived at staging time)
    float inv_h;               // 1/h, computed in float64 and narrowed once per particle
    float c[AST_MAX_PROPS];    // mantissa of prop * norm(h) in [0.5, 1) (or 0 / inf / NaN), see split_weight
    int16_t e[AST_MAX_PROPS];  // its binary exponent
};
static_assert(sizeof(Rec) == 32, "record is one 32-byte sector");

// The tile kernels work on float32 weights, the reference on float64 in any unit system (a luminosity in erg/s times
// 1/(pi h^3) with h in Mpc is ~1e48; Msun masses with lengths in cm ~1e-59: both outside float32), and one call may mix
// weights hundreds of binary orders apart (an ion column density: ion fractions of 1e-40 next to 1).  A weight is therefore
// stored as a float32 mantissa and its own binary exponent; K1 also takes the largest and the smallest exponent of every
// weight field over the particles that have records.  The pair weights are staged in exponent BANDS of kWeightBand binary
// orders: band j of field k stages mantissa * 2^(e - T_j) for T_j - kWeightBand < e <= T_j (T_0 = the largest exponent,
// T_j = T_0 - j kWeightBand) and 0 otherwise, the tile sums are formed in those units and multiplied by 2^T_j in float64
// when they are added to the map.  A staged weight is then at least 2^-kWeightBand, so even times a shape factor near the
// support edge it stays a normal float.  Nearly every call spans fewer orders than one band: it stages and accumulates
// once, as it always did; each further band repeats the staging and the accumulate kernel over the same sorted pairs.
// Powers of two only: no rounding is added anywhere.
constexpr int kZeroExp = -32768;
constexpr int kExpBias = 1 << 20;       // stored exponents are exponent + kExpBias (maximum) and kExpBias - exponent (minimum),
                                        // both > 0, so a zeroed control block means "none"
constexpr int kWeightBand = 100;
constexpr int kExpWords = (AST_MAX_PROPS * (int)sizeof(int) + 7) / 8;    // 64-bit words of one exponent array in the control block
__device__ __forceinline__ void split_weight(double c, float &m, int &e)
{
    if (c == 0.0) { m = 0.f; e = kZeroExp; return; }
    if (!(fabs(c) < INFINITY)) { m = (float)c; e = 0; return; }            // inf / NaN propagate as they do in the reference
    int ex;
    m = (float)frexp(c, &ex);
    e = ex;
}

struct P2 {
    const double *pos, *h;
    const double *prop[AST_MAX_PROPS];
    double *out;
    int64_t n;
    int a_col, b_col, n_prop, kernel_id, shape, norm_dim;
    double norm_c;                      // norm(h) = norm_c / h^norm_dim
    ShapeTab tab;                       // AST_KERNEL_TABLE only
    Axis1 ax, ay;
    double nxd1, nyd1;                  // (double)nx + 1, (double)ny + 1 (int -> double conversions cost XU cycles per particle)
    int ntx, nty, n_img, img_shift;     // sort key = tile_key << img_shift | image
    double box_a, box_b;                // periodic image m = 3*(ia+1) + (ib+1), shift = (ia*box_a, ib*box_b)
    int64_t small_max_px, huge_min_tiles;
    size_t map_stride;
    // written by K1 for the blocks that have pairs or large-h entries, read by K3 (which then enumerates tiles only once):
    uint32_t *pcount;                   // pairs of particle i
    uint32_t *pmask;                    // bit m: image m is tiled, bit 16 + m: image m is on the large-h list; bit 15 (single image
                                        // only): the member tiles of the image are in ptmask / ptorg, K3 need not recompute them
    uint64_t *ptmask, *ptorg;           // member tiles as a bit mask over the tile bbox (bit = (tx - tx0) * rows + (ty - ty0), at most
                                        // 64 tiles) and tx0 | ty0 << 24 | rows << 48
    int *wexp;                          // [AST_MAX_PROPS] maximum weight exponent of the call + kExpBias (atomicMax by K1; 0 = no
                                        // weight seen), see split_weight
    int *wmin;                          // [AST_MAX_PROPS] kExpBias - minimum weight exponent of the call (atomicMax by K1)
    unsigned long long *totals;         // [2] pairs and large-h entries of the call (atomicAdd by the K1 blocks that have any)
};


// periodic image shifts (0 for a single image); arithmetic instead of a parameter-space table, see grid3d.cu
__host__ __device__ __forceinline__ double image_shift_a(int n_img, double box_a, int m) { return n_img == 1 ? 0.0 : (double)(m / 3 - 1) * box_a; }
__host__ __device__ __forceinline__ double image_shift_b(int n_img, double box_b, int m) { return n_img == 1 ? 0.0 : (double)(m % 3 - 1) * box_b; }

// 1/x to ~1e-15 relative: float32 reciprocal seed + one Newton step in float64 (an IEEE float64 division costs ~40
// instructions on the device; weights only need 1e-7)
__device__ __forceinline__ double fast_rcp64(double x)
{
    const double r = (double)__frcp_rn((float)x);
    return r * (2.0 - x * r);
}

// norm(h) = norm_c * inv_h^2 (2-D normalisations) or norm_c * inv_h^3 (3-D), norm_c from kernel_norm(kid, 1)
__device__ __forceinline__ double norm_from_inv_h(const P2 &p, double inv_h)
{
    const double t = p.norm_c * inv_h * inv_h;
    return p.norm_dim == 3 ? t * inv_h : t;
}

// direct deposit of a small-footprint particle image: exact float64 mask, float32 shape, float64 atomics
template <int SHAPE, int NP>
__device__ __forceinline__ void deposit_small(const P2 &p, const Box2 &bb, double pa, double pb, double R2, float inv_h2,
                                              const double *coef)
{
    for (int xi = bb.x0; xi <= bb.x1; ++xi) {
        const double dx2 = dist2(p.ax, pa, xi);
        double *row = p.out + (size_t)xi * (size_t)p.ay.n;
        for (int yi = bb.y0; yi <= bb.y1; ++yi) {
            const double r2 = AST_DADD(dx2, dist2(p.ay, pb, yi));
            if (r2 < R2) {
                const double f = (double)shape_eval<SHAPE>(fast_sqrt((float)r2 * inv_h2), p.tab);
#pragma unroll
                for (int k = 0; k < NP; ++k) atomicAdd(row + k * p.map_stride + yi, coef[k] * f);
            }
        }
    }
}

// Sub-pixel fast path of the direct deposit: when the support diameter 4h is below two pixels on both axes
// (2h*inv_d <= 1 - 1e-9) at most the two samples at/after the particle can satisfy the 1-D condition on each axis, so
// the canonical bbox is at most 2x2 (class "direct" whenever small_max_px >= 4) and the four candidates are tested with
// the exact float64 mask directly -- no bbox search.  This is the HBM-bound regime of the path.
template <int SHAPE, int NP>
__device__ __forceinline__ void deposit_subpixel(const P2 &p, double pa, double pb, double R2, double inv_h2, const double *coef)
{
    const double tx = AST_DMUL(AST_DSUB(pa, p.ax.vmin), p.ax.inv_d), ty = AST_DMUL(AST_DSUB(pb, p.ay.vmin), p.ay.inv_d);
    if (!(tx > -2.0 && tx < p.nxd1 && ty > -2.0 && ty < p.nyd1)) return;   // also NaN / inf
    // floor() already is the sample index as a double: X(i) = vmin + i*d needs no int -> double conversion
    const double fx = floor(tx), fy = floor(ty);
    const int i0 = (int)fx, j0 = (int)fy;
    double dx2[2], dy2[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double tx_k = AST_DSUB(pa, AST_DADD(p.ax.vmin, AST_DMUL(fx + (double)k, p.ax.d)));
        const double ty_k = AST_DSUB(pb, AST_DADD(p.ay.vmin, AST_DMUL(fy + (double)k, p.ay.d)));
        dx2[k] = (i0 + k >= 0 && i0 + k < p.ax.n) ? AST_DMUL(tx_k, tx_k) : INFINITY;
        dy2[k] = (j0 + k >= 0 && j0 + k < p.ay.n) ? AST_DMUL(ty_k, ty_k) : INFINITY;
    }
    // exact float64 mask for the four candidates first, then ONE deposit loop over the hits of this lane: with four separate
    // predicated deposit blocks every block ran for the few lanes that hit that particular candidate (ncu: 22.8 of 32 lanes
    // active over the kernel); here pass n serves the n-th hit of every lane that has one.  Conversions run on the XU pipe
    // (a quarter of the FP32 rate; ncu: XU 41 % busy in this kernel), so q^2 is narrowed to float32 per HIT, not per candidate.
    double r2[4];
    unsigned hit = 0u;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        r2[c] = AST_DADD(dx2[c >> 1], dy2[c & 1]);
        hit |= (r2[c] < R2) ? (1u << c) : 0u;
    }
    while (hit) {
        const int c = __ffs((int)hit) - 1;
        hit &= hit - 1u;
        const double rr = (c & 2) ? ((c & 1) ? r2[3] : r2[2]) : ((c & 1) ? r2[1] : r2[0]);
        const double f = (double)shape_eval<SHAPE>(fast_sqrt((float)(rr * inv_h2)), p.tab);
        double *o = p.out + (size_t)(i0 + (c >> 1)) * (size_t)p.ay.n + (size_t)(j0 + (c & 1));
#pragma unroll
        for (int k = 0; k < NP; ++k) atomicAdd(o + k * p.map_stride, coef[k] * f);
    }
}

// is the support of a particle below one pixel on both axes (sub-pixel fast path)?  One definition for K0 and K1.
__device__ __forceinline__ bool is_subpixel(const P2 &p, double h2)
{
    return p.small_max_px >= 4 && h2 * p.ax.inv_d <= 1.0 - 1e-9 && h2 * p.ay.inv_d <= 1.0 - 1e-9;
}

// per-particle body of K1: classification, pair / large-h counts, direct deposit, record
// SKIP_SUB: the sub-pixel particles of this block were already deposited by subpixel_tma_kernel (K0)
template <int SHAPE, bool DEPOSIT, int NP, bool PER, bool SKIP_SUB = false>
__device__ __forceinline__ void bin_particle(const P2 &p, int64_t i, double pa0, double pb0, double h, double *coef /* [NP] props */,
                                             Rec *__restrict__ rec, uint32_t &npairs, uint32_t &nhuge, uint32_t &mask)
{
    const double R2 = radius2(h);
    const double h2 = AST_DMUL(2.0, h);
    if (!(h > 0.0 && h2 < INFINITY)) return;
    const bool subpixel = is_subpixel(p, h2);
    if (SKIP_SUB && subpixel) return;
    float inv_h2 = 0.f, inv_hf = 0.f;
    double inv_h2d = 0.0;
    if (DEPOSIT) {
        const double inv_h = fast_rcp64(h);
        const double nrm = norm_from_inv_h(p, inv_h);
#pragma unroll
        for (int k = 0; k < NP; ++k) coef[k] *= nrm;
        inv_hf = (float)inv_h;
        inv_h2d = inv_h * inv_h;
        inv_h2 = (float)inv_h2d;
    }
    const int n_img = PER ? p.n_img : 1;                       // compile-time 1 without periodic images
    if (subpixel) {
        if (DEPOSIT)
            for (int m = 0; m < n_img; ++m)
                deposit_subpixel<SHAPE, NP>(p, AST_DADD(pa0, image_shift_a(n_img, p.box_a, m)),
                                            AST_DADD(pb0, image_shift_b(n_img, p.box_b, m)), R2, inv_h2d, coef);
        return;
    }
    bool need_rec = false;
    // images m = 3 ia + ib in ascending order; an x shift that cannot reach the map prunes its three images at once
    const int nt = n_img == 1 ? 1 : 3;
    for (int ia = 0; ia < nt; ++ia) {
        const double pa = AST_DADD(pa0, n_img == 1 ? 0.0 : (double)(ia - 1) * p.box_a);
        if (!may_touch(p.ax, pa, h2)) continue;                                   // image cannot reach the map
        for (int ib = 0; ib < nt; ++ib) {
            const double pb = AST_DADD(pb0, n_img == 1 ? 0.0 : (double)(ib - 1) * p.box_b);
            if (!may_touch(p.ay, pb, h2)) continue;
            const int m = 3 * ia + ib;
            Bin2 b = classify2<TILE>(p.ax, p.ay, pa, pb, h, R2, p.small_max_px, p.huge_min_tiles);
            if (b.cls == CLS_SMALL) {
                if (DEPOSIT) deposit_small<SHAPE, NP>(p, b.bb, pa, pb, R2, inv_h2, coef);
            } else if (b.cls == CLS_TILED) {
                const int rows = b.ty1 - b.ty0 + 1;
                if (!PER && DEPOSIT && (b.tx1 - b.tx0 + 1) * rows <= 64) {
                    // single image with a small tile bbox: remember WHICH tiles are members, so that K3 writes the pairs from
                    // 16 bytes instead of redoing the float64 geometry from the position and h (8.0 -> 6.6 ms at config 3)
                    uint64_t tm = 0;
                    npairs += (uint32_t)for_each_tile2_xy<TILE>(p.ax, p.ay, pa, pb, R2, b, [&](int tx, int ty) {
                        tm |= 1ull << ((tx - b.tx0) * rows + (ty - b.ty0));
                    });
                    p.ptmask[i] = tm;
                    p.ptorg[i] = (uint64_t)(uint32_t)b.tx0 | ((uint64_t)(uint32_t)b.ty0 << 24) | ((uint64_t)rows << 48);
                    mask |= 0x8000u;
                } else {
                    npairs += (uint32_t)for_each_tile2<TILE>(p.ax, p.ay, pa, pb, R2, b, p.nty, [](uint32_t) {});
                }
                mask |= 1u << m;
                need_rec = true;
            } else if (b.cls == CLS_HUGE) {
                ++nhuge;
                mask |= 1u << (16 + m);
                need_rec = true;
            }
        }
    }
    if (need_rec && DEPOSIT) {
        Rec r;
        r.pa = pa0; r.pb = pb0; r.inv_h = inv_hf;
#pragma unroll
        for (int k = 0; k < AST_MAX_PROPS; ++k) {
            int e = kZeroExp;
            r.c[k] = 0.f;
            if (k < NP) split_weight(coef[k < NP ? k : 0], r.c[k], e);
            r.e[k] = (int16_t)e;
            // running maximum and minimum of the call: a plain (possibly stale) read settles them for all but the first few
            // warps, the atomic only runs when this particle would move one
            if (k < NP && e != kZeroExp) {
                if (e + kExpBias > __ldcg(p.wexp + k)) atomicMax(p.wexp + k, e + kExpBias);
                if (kExpBias - e > __ldcg(p.wmin + k)) atomicMax(p.wmin + k, kExpBias - e);
            }
        }
        rec[i] = r;
    }
}

// K1.  DEPOSIT=false is the index-only variant used by ast_bin2d (NP is then irrelevant).  One particle per thread,
// plain global loads; block b of the launch handles particle block b + block_offset.
template <int SHAPE, bool DEPOSIT, int NP, bool PER>
__global__ void __launch_bounds__(kBinThreads) bin_kernel(P2 p, Rec *__restrict__ rec, uint64_t *__restrict__ block_pairs,
                                                          uint64_t *__restrict__ block_huge, int64_t block_offset)
{
    __shared__ uint64_t red[34];
    const int64_t blk = (int64_t)blockIdx.x + block_offset;
    const int64_t i = blk * kBinThreads + threadIdx.x;
    uint32_t npairs = 0, nhuge = 0, mask = 0;
    if (i < p.n) {
        // every load of this particle is issued before anything depends on one of them
        const double pa0 = p.pos[3 * i + p.a_col], pb0 = p.pos[3 * i + p.b_col], h = p.h[i];
        double coef[NP];
        if (DEPOSIT) {
#pragma unroll
            for (int k = 0; k < NP; ++k) coef[k] = p.prop[k][i];
        }
        bin_particle<SHAPE, DEPOSIT, NP, PER>(p, i, pa0, pb0, h, coef, rec, npairs, nhuge, mask);
    }
    // one 64-bit reduction for both counts (pairs of a thread < 2^31 by validate2, large-h entries <= 9)
    const uint64_t packed = block_sum_u64(((uint64_t)nhuge << 44) | (uint64_t)npairs, red);
    if (packed != 0ull && i < p.n) { p.pcount[i] = npairs; p.pmask[i] = mask; }     // K3 only visits blocks with entries
    if (threadIdx.x == 0) {
        block_pairs[blk] = packed & ((1ull << 44) - 1ull);
        block_huge[blk] = packed >> 44;
        if (packed != 0ull && p.totals) {
            atomicAdd(p.totals, (unsigned long long)(packed & ((1ull << 44) - 1ull)));
            if (packed >> 44) atomicAdd(p.totals + 1, (unsigned long long)(packed >> 44));
        }
    }
}

// ---- TMA-staged K1 -------------------------------------------------------------------------------------------------
// Persistent CTAs stream the particle arrays through shared memory with 1-D bulk copies (cp.async.bulk, the TMA engine)
// signalled on mbarriers, two stages deep: while the CTA works on particle block b the copies of block b + gridDim are
// already in flight, so HBM latency is hidden independently of occupancy.  Only full blocks of 256 particles go through
// here (16-byte alignment of every copy); the tail block uses bin_kernel.
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

template <int NP>
struct __align__(128) BinStage {
    double pos[3 * kBinThreads];
    double h[kBinThreads];
    double prop[NP][kBinThreads];
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// K0 (round 2): the sub-pixel pass.  Same persistent TMA pipeline as K1, but the only thing it does is the sub-pixel fast path:
// a particle whose support is below one pixel is deposited here (exact float64 mask on its 2x2 candidates), anything else only
// marks its block as "heavy" for K1.  The point is occupancy: this path needs 40 registers, the general classification
// 64-80, and the HBM-bound regime of the whole library (every particle sub-pixel) is latency-limited -- ncu on K1 there:
// issue 72 %, 2.0 eligible warps per scheduler, "wait" 2.1 and barrier 1.3 stalls per issue at 4 CTAs per SM.  With SPH-realistic
// supports K0 streams the inputs once for nothing: 0.9 ms of a 278 ms step at config 3.
template <int SHAPE, int NP, bool PER>
__global__ void __launch_bounds__(kBinThreads, 6) subpixel_tma_kernel(P2 p, uint64_t *__restrict__ block_pairs,
                                                                      uint64_t *__restrict__ block_huge, uint8_t *__restrict__ block_heavy,
                                                                      unsigned long long *__restrict__ heavy_count, int64_t n_full_blocks)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    BinStage<NP> *st = reinterpret_cast<BinStage<NP> *>(smem_raw);
    __shared__ __align__(8) uint64_t bar[2];
    const int tid = threadIdx.x;
    constexpr uint32_t kBytes = (uint32_t)sizeof(BinStage<NP>);
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int64_t blk, int s) {
        mbar_expect_tx(&bar[s], kBytes);
        const int64_t i0 = blk * kBinThreads;
        tma_load_1d(st[s].pos, p.pos + 3 * i0, 3 * kBinThreads * 8, &bar[s]);
        tma_load_1d(st[s].h, p.h + i0, kBinThreads * 8, &bar[s]);
#pragma unroll
        for (int k = 0; k < NP; ++k) tma_load_1d(st[s].prop[k], p.prop[k] + i0, kBinThreads * 8, &bar[s]);
    };
    int64_t blk = blockIdx.x;
    if (tid == 0 && blk < n_full_blocks) issue(blk, 0);
    uint32_t phase_bits = 0u;
    unsigned cta_heavy = 0u;
    const int n_img = PER ? p.n_img : 1;
    for (int it = 0; blk < n_full_blocks; blk += gridDim.x, ++it) {
        const int s = it & 1;
        const int64_t next = blk + gridDim.x;
        if (tid == 0 && next < n_full_blocks) issue(next, s ^ 1);     // stage s^1 was released by the barrier below
        mbar_wait(&bar[s], (phase_bits >> s) & 1u);
        phase_bits ^= 1u << s;
        const double pa0 = st[s].pos[3 * tid + p.a_col], pb0 = st[s].pos[3 * tid + p.b_col], h = st[s].h[tid];
        double coef[NP];
#pragma unroll
        for (int k = 0; k < NP; ++k) coef[k] = st[s].prop[k][tid];
        const double h2 = AST_DMUL(2.0, h);
        bool heavy = false;
        if (h > 0.0 && h2 < INFINITY) {
            if (is_subpixel(p, h2)) {
                const double inv_h = fast_rcp64(h), nrm = norm_from_inv_h(p, inv_h), R2 = radius2(h);
#pragma unroll
                for (int k = 0; k < NP; ++k) coef[k] *= nrm;
                for (int m = 0; m < n_img; ++m)
                    deposit_subpixel<SHAPE, NP>(p, AST_DADD(pa0, image_shift_a(n_img, p.box_a, m)),
                                                AST_DADD(pb0, image_shift_b(n_img, p.box_b, m)), R2, inv_h * inv_h, coef);
            } else {
                heavy = true;
            }
        }
        const int any_heavy = __syncthreads_or(heavy);            // also releases stage s for the next bulk copy
        if (tid == 0) {
            block_heavy[blk] = any_heavy ? 1 : 0;
            if (any_heavy) ++cta_heavy;
            else { block_pairs[blk] = 0; block_huge[blk] = 0; }  // K1 skips the block: its scan entries are zero
        }
    }
    if (tid == 0 && cta_heavy) atomicAdd(heavy_count, (unsigned long long)cta_heavy);
}

// NSTAGE stages of 256 particles per CTA: NSTAGE - 1 bulk copies are in flight while one stage is worked on.  With K0 in
// front (SKIP_SUB) the CTA only visits the blocks K0 marked heavy: thread 0 looks up the next marked block of its stride and
// publishes its index with the stage (or -1 at the end, arriving on the barrier itself).
template <int SHAPE, int NP, bool PER, int NSTAGE, int MINB, bool SKIP_SUB>
__global__ void __launch_bounds__(kBinThreads, MINB) bin_tma_kernel(P2 p, Rec *__restrict__ rec, uint64_t *__restrict__ block_pairs,
                                                                    uint64_t *__restrict__ block_huge, int64_t n_full_blocks,
                                                                    const uint8_t *__restrict__ block_heavy,
                                                                    const unsigned long long *__restrict__ heavy_count)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    BinStage<NP> *st = reinterpret_cast<BinStage<NP> *>(smem_raw);
    __shared__ __align__(8) uint64_t bar[NSTAGE];
    __shared__ int64_t sblk[NSTAGE];
    __shared__ uint64_t red[34];
    if (SKIP_SUB && *heavy_count == 0ull) return;                   // nothing for K1: every particle was sub-pixel (or invalid)
    const int tid = threadIdx.x;
    constexpr uint32_t kBytes = (uint32_t)sizeof(BinStage<NP>);
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < NSTAGE; ++k) mbar_init(&bar[k], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    int64_t scan = blockIdx.x;                                     // thread 0: next candidate block of this CTA's stride
    auto fill = [&](int s) {          // one elected thread: next block to visit -> stage s (bulk copies), or the end marker
        while (SKIP_SUB && scan < n_full_blocks && !block_heavy[scan]) scan += gridDim.x;
        const int64_t blk = scan < n_full_blocks ? scan : -1;
        scan += gridDim.x;
        sblk[s] = blk;
        if (blk < 0) { mbar_arrive(&bar[s]); return; }
        mbar_expect_tx(&bar[s], kBytes);
        const int64_t i0 = blk * kBinThreads;
        tma_load_1d(st[s].pos, p.pos + 3 * i0, 3 * kBinThreads * 8, &bar[s]);
        tma_load_1d(st[s].h, p.h + i0, kBinThreads * 8, &bar[s]);
#pragma unroll
        for (int k = 0; k < NP; ++k) tma_load_1d(st[s].prop[k], p.prop[k] + i0, kBinThreads * 8, &bar[s]);
    };
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < NSTAGE - 1; ++k) fill(k);
    }
    uint32_t phase_bits = 0u;                                   // bit s = parity to wait for on stage s (kept in a register)
    uint64_t cta_pairs = 0, cta_huge = 0;                       // thread 0: totals of the blocks this CTA handled
    int s = 0;
    for (;;) {
        // the stage worked on in the previous iteration was released by the barrier at its end: refill it
        if (tid == 0) fill(s == 0 ? NSTAGE - 1 : s - 1);
        mbar_wait(&bar[s], (phase_bits >> s) & 1u);
        phase_bits ^= 1u << s;
        const int64_t blk = sblk[s];
        if (blk < 0) break;                                     // uniform: no block left for this CTA
        const int64_t i = blk * kBinThreads + tid;
        const double pa0 = st[s].pos[3 * tid + p.a_col], pb0 = st[s].pos[3 * tid + p.b_col], h = st[s].h[tid];
        double coef[NP];
#pragma unroll
        for (int k = 0; k < NP; ++k) coef[k] = st[s].prop[k][tid];
        uint32_t npairs = 0, nhuge = 0, mask = 0;
        bin_particle<SHAPE, true, NP, PER, SKIP_SUB>(p, i, pa0, pb0, h, coef, rec, npairs, nhuge, mask);
        // one barrier-with-vote tells whether any thread has pairs / large-h entries at all (in the direct-deposit regime none
        // has): only then pay for the full block reduction.  The barrier also releases stage s for the next bulk copy.
        uint64_t packed = ((uint64_t)nhuge << 44) | (uint64_t)npairs;
        if (__syncthreads_or(packed != 0ull)) {
            p.pcount[i] = npairs;
            p.pmask[i] = mask;
            packed = block_sum_u64(packed, red);
        }
        if (tid == 0) {
            block_pairs[blk] = packed & ((1ull << 44) - 1ull);
            block_huge[blk] = packed >> 44;
            cta_pairs += packed & ((1ull << 44) - 1ull);
            cta_huge += packed >> 44;
        }
        s = s + 1 == NSTAGE ? 0 : s + 1;
    }
    if (tid == 0) {                                   // one atomic per persistent CTA and count, none in the direct-deposit regime
        if (cta_pairs) atomicAdd(p.totals, (unsigned long long)cta_pairs);
        if (cta_huge) atomicAdd(p.totals + 1, (unsigned long long)cta_huge);
    }
}

// K3: pairs with global emit index in [w0, w1) are written to pairs[g - w0]; large-h entries with list index in [h0, h1)
// to huge[gh - h0] (either window may be empty).
__global__ void __launch_bounds__(kBinThreads) emit_kernel(P2 p, const uint64_t *__restrict__ pairs_excl,
                                                           const uint64_t *__restrict__ huge_excl, uint64_t w0, uint64_t w1,
                                                           uint64_t *__restrict__ pairs, uint64_t *__restrict__ huge,
                                                           uint64_t h0, uint64_t h1)
{
    constexpr int kStage = 512;                             // pairs staged per warp and round
    __shared__ uint32_t sm[34];
    __shared__ uint64_t sbuf[kBinThreads / 32][kStage];
    const uint64_t pbase = pairs_excl[blockIdx.x], pnext = pairs_excl[blockIdx.x + 1];
    const uint64_t hbase = huge_excl[blockIdx.x], hnext = huge_excl[blockIdx.x + 1];
    const bool any_pairs = pnext > pbase && pnext > w0 && pbase < w1;
    const bool any_huge = hnext > hbase && hnext > h0 && hbase < h1;
    if (!any_pairs && !any_huge) return;                    // uniform for the block
    const int64_t i = (int64_t)blockIdx.x * kBinThreads + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // counts and image masks come from K1 (it wrote them for every block that has entries): one enumeration here, not two
    uint32_t npairs = 0, nhuge = 0, mask = 0;
    if (i < p.n) {
        npairs = p.pcount[i];
        mask = p.pmask[i];
        nhuge = (uint32_t)__popc(mask >> 16);
    }
    uint32_t tot;
    uint64_t g = pbase + block_excl_scan_u32(npairs, sm, &tot);
    uint64_t gh = hbase + block_excl_scan_u32(nhuge, sm, &tot);
    if (!any_pairs) mask &= 0xffff0000u;                    // only the large-h entries are wanted
    if (!any_huge) mask &= 0x0000ffffu;
    // Single-image particles whose member tiles K1 stored (the bulk): no geometry here, just the set bits of the mask in emit
    // order (tx, then ty ascending).  A thread's pairs are consecutive in the output, neighbouring threads' ranges adjoin: the
    // warp's pairs form ONE contiguous range.  Written straight from the threads that is an 8-byte store to 32 different
    // sectors per instruction; staged through the warp's shared-memory window the range goes out in full sectors
    // (6.6 -> 5.9 ms at config 3).
    const bool staged = (mask & 0x8000u) != 0u;
    if (__any_sync(0xffffffffu, staged)) {
        const uint64_t warp_base = __shfl_sync(0xffffffffu, g, 0);
        const uint32_t warp_total = (uint32_t)(__shfl_sync(0xffffffffu, g + npairs, 31) - warp_base);
        const uint32_t rel = (uint32_t)(g - warp_base);
        uint64_t tm = 0, org = 0;
        if (staged) { tm = p.ptmask[i]; org = p.ptorg[i]; }
        const int tx0 = (int)(org & 0xffffffu), ty0 = (int)((org >> 24) & 0xffffffu), rows = staged ? (int)(org >> 48) : 1;
        uint64_t *buf = sbuf[warp];
        for (uint32_t c0 = 0; c0 < warp_total; c0 += kStage) {
            for (int o = lane; o < kStage; o += 32) buf[o] = ~0ull;                 // slots of threads that write their own pairs
            __syncwarp();
            if (staged && rel < c0 + kStage && rel + npairs > c0) {
                uint64_t t = tm;
                uint32_t pos = rel;
                while (t) {
                    const int bit = __ffsll((long long)t) - 1;
                    t &= t - 1ull;
                    if (pos >= c0 && pos < c0 + kStage) {
                        const int dx = bit / rows, dy = bit - dx * rows;
                        buf[pos - c0] = ((uint64_t)(uint32_t)((tx0 + dx) * p.nty + ty0 + dy) << 32) | (uint64_t)(uint32_t)i;
                    }
                    ++pos;
                }
            }
            __syncwarp();
            const uint32_t nc = warp_total - c0 < (uint32_t)kStage ? warp_total - c0 : (uint32_t)kStage;
            for (uint32_t o = lane; o < nc; o += 32) {
                const uint64_t v = buf[o], gp = warp_base + c0 + o;
                if (v != ~0ull && gp >= w0 && gp < w1) pairs[gp - w0] = v;
            }
            __syncwarp();
        }
    }
    if (i >= p.n || staged || mask == 0u) return;
    const double pa0 = p.pos[3 * i + p.a_col], pb0 = p.pos[3 * i + p.b_col], h = p.h[i], R2 = radius2(h);
    for (int m = 0; m < p.n_img; ++m) {
        if (!((mask >> m) & 0x10001u)) continue;                           // image m has neither pairs nor a large-h entry
        if ((mask >> (16 + m)) & 1u) {                                     // classes come from K1's masks: no re-classification
            if (gh >= h0 && gh < h1) huge[gh - h0] = ((uint64_t)m << 32) | (uint64_t)(uint32_t)i;
            ++gh;
            continue;
        }
        const double pa = AST_DADD(pa0, image_shift_a(p.n_img, p.box_a, m)), pb = AST_DADD(pb0, image_shift_b(p.n_img, p.box_b, m));
        Bin2 b = classify2<TILE>(p.ax, p.ay, pa, pb, h, R2, p.small_max_px, p.huge_min_tiles);
        for_each_tile2<TILE>(p.ax, p.ay, pa, pb, R2, b, p.nty, [&](uint32_t key) {
            if (g >= w0 && g < w1)
                pairs[g - w0] = ((uint64_t)((key << p.img_shift) | (uint32_t)m) << 32) | (uint64_t)(uint32_t)i;
            ++g;
        });
    }
}

// Large-h split: one WARP per entry of the large-h list.  The tile bbox of the entry is enumerated 32 tiles at a time in emit
// order (tx ascending, then ty ascending) with the same membership test as for_each_tile2 (at least one pixel of tile /\ bbox
// inside the support).  WRITE = false: hoff[e] = number of member tiles.  WRITE = true: hoff holds the exclusive scan of those
// counts; pair number g = base + hoff[e] + rank goes to pairs[g - w0] when it falls into the window [w0, w1).  The pairs have
// the format of the tiled ones, so everything downstream (sort, pair records, accumulate) is shared.
template <bool WRITE>
__global__ void __launch_bounds__(256) huge_tiles_kernel(P2 p, const uint64_t *__restrict__ huge, uint32_t n_entries,
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
        if (gend <= w0 || g >= w1) return;                  // no pair of this entry falls into the window
    }
    const uint64_t ent = huge[e];
    const int64_t i = (int64_t)(uint32_t)ent;
    const int m = (int)(ent >> 32);
    const double h = p.h[i], R2 = radius2(h);
    const double pa = AST_DADD(p.pos[3 * i + p.a_col], image_shift_a(p.n_img, p.box_a, m));
    const double pb = AST_DADD(p.pos[3 * i + p.b_col], image_shift_b(p.n_img, p.box_b, m));
    const Bin2 b = classify2<TILE>(p.ax, p.ay, pa, pb, h, R2, p.small_max_px, p.huge_min_tiles);
    const int nrow = b.ty1 - b.ty0 + 1;
    const int64_t nt = (int64_t)(b.tx1 - b.tx0 + 1) * (int64_t)nrow;      // <= 0 only if the entry were not CLS_HUGE
    uint32_t cnt = 0;
    const unsigned lt = (1u << lane) - 1u;
    for (int64_t t0 = 0; t0 < nt; t0 += 32) {
        const int64_t t = t0 + lane;
        bool in = false;
        uint32_t key = 0;
        if (t < nt) {
            const int tx = b.tx0 + (int)(t / nrow), ty = b.ty0 + (int)(t % nrow);
            const int xa = tx * TILE > b.bb.x0 ? tx * TILE : b.bb.x0, xb = tx * TILE + TILE - 1 < b.bb.x1 ? tx * TILE + TILE - 1 : b.bb.x1;
            const int ya = ty * TILE > b.bb.y0 ? ty * TILE : b.bb.y0, yb = ty * TILE + TILE - 1 < b.bb.y1 ? ty * TILE + TILE - 1 : b.bb.y1;
            in = AST_DADD(min_dist2(p.ax, pa, xa, xb), min_dist2(p.ay, pb, ya, yb)) < R2;
            key = (uint32_t)(tx * p.nty + ty);
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

// K6
struct Acc {
    const uint64_t *sorted;
    const uint32_t *tbeg, *tend;
    const Rec *rec;
    double *out;
    double x_min, y_min, dx, dy, inv_dx, inv_dy;
    int nx, ny, ntx, nty, img_shift, n_img;
    double box_a, box_b;
    ShapeTab tab;
    size_t map_stride;
    const float4 *pp;             // per sorted pair: {fx, fy, sx, sy} tile-relative float32 (pair_record_kernel)
    const float2 *pc;             // per sorted pair: weights (x 2 for the cubic spline, whose loops return f/2)
    const uint32_t *seg_off;      // [ntiles + 1] exclusive scan of the segments per tile; seg_off[ntiles] = number of work items
    uint32_t seg_target;          // target list entries per segment
    uint32_t n_huge;              // always 0 here (work_items.cuh is shared with the 3-D grid, which still walks a global list)
    int ntiles;
    int etop[AST_MAX_PROPS];      // exponent band of the staged weights (see split_weight): exponents etop - kWeightBand < e <=
    int ebot[AST_MAX_PROPS];      // etop (ebot <= e <= etop, ebot = kZeroExp in the lowest band) are staged relative to 2^etop
};

// pair weight of band [ebot, etop] relative to 2^etop, 0 outside it
__device__ __forceinline__ float stage_weight(float c, int e, int etop, int ebot)
{
    return (e >= ebot && e <= etop) ? ldexpf(c, max(e - etop, -300)) : 0.f;
}

// K5: first / one-past-last sorted pair of every tile (arrays pre-zeroed), and every sorted pair is turned into the two things the accumulate kernel
// needs -- tile-relative float32 coordinates {fx, fy, sx, sy} and the weights -- ONCE, here.  The accumulate kernel used to do
// this for every pair in each of its 8 warps (sorted pair -> dependent 32-byte record gather -> float64 arithmetic): 10 % of
// its instructions and 19 % of its stall samples (ncu source view, profiles/r01_v4_summary.md).  Same expressions, same values.
template <int SHAPE, int NP>
__global__ void __launch_bounds__(256) pair_record_kernel(Acc a, int64_t n, uint32_t *__restrict__ tbeg, uint32_t *__restrict__ tend,
                                                          float4 *__restrict__ pp, float2 *__restrict__ pc)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t e = a.sorted[i];
    const uint32_t key = (uint32_t)(e >> 32), t = key >> a.img_shift, m = key & ((1u << a.img_shift) - 1u);
    if (i == 0 || ((uint32_t)(a.sorted[i - 1] >> 32) >> a.img_shift) != t) tbeg[t] = (uint32_t)i;
    if (i == n - 1 || ((uint32_t)(a.sorted[i + 1] >> 32) >> a.img_shift) != t) tend[t] = (uint32_t)(i + 1);
    const Rec r = a.rec[(uint32_t)e];
    const int tx = (int)t / a.nty, ty = (int)t - tx * a.nty;
    const double ox = (double)(tx * TILE), oy = (double)(ty * TILE);
    const float fx = (float)((r.pa + image_shift_a(a.n_img, a.box_a, (int)m) - a.x_min) * a.inv_dx - ox);
    const float fy = (float)((r.pb + image_shift_b(a.n_img, a.box_b, (int)m) - a.y_min) * a.inv_dy - oy);
    const float cscale = SHAPE == SHAPE_CUBIC ? 2.0f : 1.0f;
    pp[i] = make_float4(fx, fy, (float)a.dx * r.inv_h, (float)a.dy * r.inv_h);
    // weights of the current band relative to its top 2^etop_k: mantissa * 2^(e - etop_k), at most 1 in magnitude
    const float w0 = stage_weight(r.c[0], r.e[0], a.etop[0], a.ebot[0]);
    const float w1 = NP > 1 ? stage_weight(r.c[1], r.e[1], a.etop[1], a.ebot[1]) : 0.f;
    pc[i] = make_float2(cscale * w0, cscale * w1);
}

// K6: one CTA per work item of a 32x32 tile; every warp walks the list on its own for its own 8x16 sub-tile (no CTA
// barrier anywhere), 2x2 pixels per thread.  Per 32 list entries each lane loads one staged pair record, tests it against the
// warp's sub-tile, the hits are ballot-compacted into the warp's shared-memory slots, then all lanes evaluate them.  For
// batches with enough hits the lane that staged an entry also computes the entry's squared x-distances to the 8 pixel
// columns and squared y-distances to the 16 pixel rows of the sub-tile (in units of h) and stores them with the
// weights: the evaluating lanes then fetch their two column and two row values (LDS.64 + LDS.128) instead of
// recomputing them 32 lanes wide, and the per-pixel work is FADD, MUFU.SQRT, shape, NP FFMA.  The cubic spline is
// evaluated as f/2 = min(1/2 + s(3q/8 - 3/4), sat(1 - q/2)^3), s = q^2 (the first argument is the inner branch
// 1 - 3/2 q^2 + 3/4 q^3 of _kernels.pyx:17, the second the outer branch 1/4 (2-q)^3 of :19; inner - outer = -(1-q)^3/2
// changes sign exactly at q = 1, so the minimum selects the right branch and is 0 beyond q = 2), with the weights
// doubled at staging time.  Sparse batches (fewer than kRowColMinHits hits) take the classic per-lane coordinates.
// The quad is evaluated as two pixel pairs, one per column, with the packed float32 forms of ast_math.h (bit-identical to
// the scalar ones): per pixel of the full list the SASS is 1/2 FADD2, MUFU.SQRT, FFMA.SAT, 1 FFMA2 and 1 FMUL2 of shape,
// FMNMX and NP/2 FFMA2, i.e. 6 instructions for NP = 1 (7 with the slot loads and the loop control), 3 in the inner-only
// and 4 in the outer-annulus list.  This saves issue slots, not FMA-pipe time: a packed instruction holds the FMA pipe for
// two cycles, so a full-list pixel still costs ~7 FMA-pipe cycles next to the 8 XU cycles of its warp-wide MUFU.SQRT.
constexpr int kRowColMinHits = 8;
struct __align__(16) RowColSlot {
    float4 ax[2];        // squared x-distance (in h) to the 8 pixel columns of the sub-tile
    float4 byc[8];       // {squared y-distance to rows 2j, 2j+1, c0, c1}
};
static_assert(sizeof(RowColSlot) == 160, "slot layout");

template <int SHAPE, int NP>
__global__ void __launch_bounds__(256, 3) rowcol_accum_kernel(Acc a)
{
    constexpr int NW = 8, WY = 2, SX = 8, SY = 16, PX = 2, PY = 2, LY = SY / PY, NPIX = PX * PY;
    __shared__ RowColSlot sS[NW][32];

    TileWork w;
    if (!resolve_work(a, w)) return;
    const int tile = w.tile;
    // the work item is the same for every thread of the CTA; saying so (broadcast from lane 0) lets the compiler keep the loop
    // control in uniform registers and drop the divergence checks around the warp collectives below
    const uint32_t beg = __shfl_sync(0xffffffffu, w.beg, 0), total = __shfl_sync(0xffffffffu, w.cnt, 0);
    const uint32_t w_first = __shfl_sync(0xffffffffu, w.first, 0), w_step = __shfl_sync(0xffffffffu, w.step, 0);
    if (total == 0) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tile / a.nty, ty = tile - tx * a.nty;
    const int X0 = tx * TILE, Y0 = ty * TILE;
    const int sub_x = SX * (warp / WY), sub_y = SY * (warp % WY);
    const int xl = sub_x + PX * (lane / LY), yl = sub_y + PY * (lane % LY);
    const float xf[PX] = { (float)xl, (float)(xl + 1) }, yf[PY] = { (float)yl, (float)(yl + 1) };
    const float lox = (float)sub_x, hix = (float)(sub_x + SX - 1), loy = (float)sub_y, hiy = (float)(sub_y + SY - 1);
    RowColSlot *const slots = sS[warp];
    // classic view of the same storage: {ux*sx, uy*sy, sx, sy} in ax[0], {c0, c1} in the first half of ax[1]

    // float32 sums per pixel pair: acc[k][ix] = {pixel (xl + ix, yl), pixel (xl + ix, yl + 1)}, the two rows of one column,
    // whose row values sit side by side in byc and whose column value is a broadcast operand of FADD2
    float2 acc[NP][PX];
    double acc64[NP][NPIX];
#pragma unroll
    for (int k = 0; k < NP; ++k) {
#pragma unroll
        for (int ix = 0; ix < PX; ++ix) acc[k][ix] = f2(0.f);
#pragma unroll
        for (int j = 0; j < NPIX; ++j) acc64[k][j] = 0.0;
    }
    // one staged entry of a dense batch: the lane's two column values, its two row values and the weights
    auto eval_slot = [&](int e, auto shape2) {
        const float2 ax2 = reinterpret_cast<const float2 *>(slots[e].ax)[lane >> 3];
        const float4 bc = slots[e].byc[lane & 7];
        const float2 by = make_float2(bc.x, bc.y);
        const float2 f0 = shape2(__fadd2_rn(by, f2(ax2.x))), f1 = shape2(__fadd2_rn(by, f2(ax2.y)));
        acc[0][0] = __ffma2_rn(f2(bc.z), f0, acc[0][0]); acc[0][1] = __ffma2_rn(f2(bc.z), f1, acc[0][1]);
        if (NP > 1) { acc[NP - 1][0] = __ffma2_rn(f2(bc.w), f0, acc[NP - 1][0]); acc[NP - 1][1] = __ffma2_rn(f2(bc.w), f1, acc[NP - 1][1]); }
    };
    const auto full2 = [&](float2 s) { return shape_half_full2<SHAPE>(s, a.tab); };

    int since_fold = 0;
    for (uint32_t base = w_first; base < total; base += w_step) {
        const uint32_t j = base + lane;
        bool hit = false, outer = false, inner = false;
        float4 P = make_float4(0.f, 0.f, 0.f, 0.f);
        float2 C = make_float2(0.f, 0.f);
        if (j < total) {
            const float4 q = a.pp[beg + j];                      // staged once per pair by pair_record_kernel (coalesced)
            C = a.pc[beg + j];
            const float fx = q.x, fy = q.y, sx = q.z, sy = q.w;
            const float ddx = fmaxf(fmaxf(lox - fx, fx - hix), 0.f) * sx;
            const float ddy = fmaxf(fmaxf(loy - fy, fy - hiy), 0.f) * sy;
            const float qmin2 = ddx * ddx + ddy * ddy;
            hit = qmin2 < 4.0001f;
            outer = hit && SHAPE == SHAPE_CUBIC && qmin2 >= 1.0f;
            if (SHAPE == SHAPE_CUBIC) {
                // farthest pixel of the sub-tile: if even that one has q < 1 every pixel takes the inner branch alone
                const float fdx = fmaxf(fx - lox, hix - fx) * sx, fdy = fmaxf(fy - loy, hiy - fy) * sy;
                inner = hit && (fdx * fdx + fdy * fdy < 0.9999f);
            }
            P = make_float4(fx * sx, fy * sy, sx, sy);
        }
        // slots: mixed hits from the front, then inner-only hits, outer-annulus hits from the back
        const unsigned ball_f = __ballot_sync(0xffffffffu, hit && !outer && !inner);
        const unsigned ball_o = __ballot_sync(0xffffffffu, outer);
        const unsigned ball_i = SHAPE == SHAPE_CUBIC ? __ballot_sync(0xffffffffu, inner) : 0u;
        const int nf = __popc(ball_f), no = __popc(ball_o), ni = __popc(ball_i), nh = nf + no + ni;
        if (nh == 0) continue;
        const unsigned lt = (1u << lane) - 1u;
        const int dst = outer ? 31 - __popc(ball_o & lt) : (inner ? nf + __popc(ball_i & lt) : __popc(ball_f & lt));
        if (nh >= kRowColMinHits) {
            if (hit) {
                RowColSlot *d = slots + dst;
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { const float t = fmaf(-(lox + (float)i), P.z, P.x); v[i] = t * t; }
                d->ax[0] = make_float4(v[0], v[1], v[2], v[3]);
                d->ax[1] = make_float4(v[4], v[5], v[6], v[7]);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float t0 = fmaf(-(loy + (float)(2 * i)), P.w, P.y), t1 = fmaf(-(loy + (float)(2 * i + 1)), P.w, P.y);
                    d->byc[i] = make_float4(t0 * t0, t1 * t1, C.x, C.y);
                }
            }
            __syncwarp();
            // unrolled by 4: one entry per iteration spends ~7 of its ~33 instructions on the loop control and the slot address
#pragma unroll 4
            for (int e = 0; e < nf; ++e) eval_slot(e, full2);
            if (SHAPE == SHAPE_CUBIC) {
                // every pixel has q < 1: f/2 = 1/2 + s (3q/8 - 3/4)
#pragma unroll 4
                for (int e = nf; e < nf + ni; ++e) eval_slot(e, [](float2 s) { return shape_half_inner2(s); });
#pragma unroll 4
                for (int e = 32 - no; e < 32; ++e) eval_slot(e, [](float2 s) { return shape_half_outer2(s); });
            }
        } else {
            if (hit) {
                slots[dst].ax[0] = P;
                *reinterpret_cast<float2 *>(&slots[dst].ax[1]) = C;
            }
            __syncwarp();
            // sparse batch: full and outer-annulus hits alike through the general shape
            for (int e = 0; e < nh; ++e) {
                const int sl = e < nf + ni ? e : 32 - nh + e;
                const float4 q = slots[sl].ax[0];
                const float2 c = *reinterpret_cast<const float2 *>(&slots[sl].ax[1]);
                float ax2[PX], by2[PY];
#pragma unroll
                for (int i = 0; i < PX; ++i) { const float t = fmaf(-xf[i], q.z, q.x); ax2[i] = t * t; }
#pragma unroll
                for (int i = 0; i < PY; ++i) { const float t = fmaf(-yf[i], q.w, q.y); by2[i] = t * t; }
                // scalar on purpose: ax2 + by2 of two products in registers is contracted to an FFMA here, which a packed
                // FADD2 would not reproduce bit for bit
#pragma unroll
                for (int ix = 0; ix < PX; ++ix) {
                    const float f0 = shape_half_full<SHAPE>(ax2[ix] + by2[0], a.tab), f1 = shape_half_full<SHAPE>(ax2[ix] + by2[1], a.tab);
                    acc[0][ix].x = fmaf(c.x, f0, acc[0][ix].x); acc[0][ix].y = fmaf(c.x, f1, acc[0][ix].y);
                    if (NP > 1) { acc[NP - 1][ix].x = fmaf(c.y, f0, acc[NP - 1][ix].x); acc[NP - 1][ix].y = fmaf(c.y, f1, acc[NP - 1][ix].y); }
                }
            }
        }
        __syncwarp();
        since_fold += nh;
        if (since_fold >= 96) {
            since_fold = 0;
#pragma unroll
            for (int k = 0; k < NP; ++k)
#pragma unroll
                for (int ix = 0; ix < PX; ++ix) {
                    acc64[k][ix * PY] += (double)acc[k][ix].x;
                    acc64[k][ix * PY + 1] += (double)acc[k][ix].y;
                    acc[k][ix] = f2(0.f);
                }
        }
    }
    // the sums are in units of 2^etop_k: two exact power-of-two factors (etop_k spans -1073 .. 1024, one factor could overflow)
    double sc1[NP], sc2[NP];
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const int e = min(max(a.etop[k], -2040), 2040), e1 = e / 2, e2 = e - e1;
        sc1[k] = __longlong_as_double((long long)(e1 + 1023) << 52);
        sc2[k] = __longlong_as_double((long long)(e2 + 1023) << 52);
    }
#pragma unroll
    for (int ix = 0; ix < PX; ++ix) {
        const int xi = X0 + xl + ix;
        if (xi >= a.nx) continue;
#pragma unroll
        for (int iy = 0; iy < PY; ++iy) {
            const int yi = Y0 + yl + iy;
            if (yi >= a.ny) continue;
#pragma unroll
            for (int k = 0; k < NP; ++k) {
                double *o = a.out + k * a.map_stride + (size_t)xi * a.ny + yi;
                const double v = (acc64[k][ix * PY + iy] + (double)(iy ? acc[k][ix].y : acc[k][ix].x)) * sc1[k] * sc2[k];
                if (w.atomic_out) atomicAdd(o, v); else *o += v;
            }
        }
    }
}

// exact contributor count (reference mask) per pixel, for parity tests
__global__ void contrib_count_kernel(P2 p, int32_t *__restrict__ count)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const double pa0 = p.pos[3 * i + p.a_col], pb0 = p.pos[3 * i + p.b_col], h = p.h[i];
    const double R2 = radius2(h);
    for (int m = 0; m < p.n_img; ++m) {
        const double pa = AST_DADD(pa0, image_shift_a(p.n_img, p.box_a, m)), pb = AST_DADD(pb0, image_shift_b(p.n_img, p.box_b, m));
        int x0, x1, y0, y1;
        if (!range1(p.ax, pa, h, R2, x0, x1) || !range1(p.ay, pb, h, R2, y0, y1)) continue;
        for (int xi = x0; xi <= x1; ++xi) {
            const double dx2 = dist2(p.ax, pa, xi);
            for (int yi = y0; yi <= y1; ++yi)
                if (AST_DADD(dx2, dist2(p.ay, pb, yi)) < R2) atomicAdd(count + (size_t)xi * p.ay.n + yi, 1);
        }
    }
}

// bbox + class per particle image, for parity tests
__global__ void bbox_cls_kernel(P2 p, int32_t *__restrict__ bbox, uint8_t *__restrict__ cls)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const double pa0 = p.pos[3 * i + p.a_col], pb0 = p.pos[3 * i + p.b_col], h = p.h[i];
    const double R2 = radius2(h);
    for (int m = 0; m < p.n_img; ++m) {
        const double pa = AST_DADD(pa0, image_shift_a(p.n_img, p.box_a, m)), pb = AST_DADD(pb0, image_shift_b(p.n_img, p.box_b, m));
        Bin2 b = classify2<TILE>(p.ax, p.ay, pa, pb, h, R2, p.small_max_px, p.huge_min_tiles);
        const int64_t j = (int64_t)m * p.n + i;
        if (bbox) {
            bbox[4 * j] = b.bb.x0; bbox[4 * j + 1] = b.bb.x1; bbox[4 * j + 2] = b.bb.y0; bbox[4 * j + 3] = b.bb.y1;
        }
        if (cls) cls[j] = (uint8_t)b.cls;
    }
}

__global__ void kernel_eval_kernel(int kid, const double *__restrict__ r, const double *__restrict__ h, double *__restrict__ out,
                                   int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = kernel_f64(kid, r[i], h[i]);
}

// ------------------------------------------------------------------------------------------------ host side
constexpr int64_t kDefaultSmallMaxPx = 36;      // measured (benchmarks/small_max_probe.py): 36 beats 16 by 21 % at 2.2-pixel supports, 64 loses 22 % at 4.5
constexpr int64_t kDefaultHugeMinTiles = 256;

// Workspace.  One pair window of pair_capacity elements; more pairs are walked through it in rounds.
struct RoundSet {
    float4 *pp;                 // win staged pair records
    float2 *pc;                 // win staged pair weights (lives in the ping-pong buffer the sort leaves free)
    uint32_t *tbeg, *tend, *seg_off, *seg_tmp;
};
struct Layout2 {
    int64_t nb;                 // bin blocks
    int64_t ntiles;
    int64_t win, huge_cap;
    uint64_t *block_pairs, *block_huge;   // nb + 1 each
    uint64_t *scan_tmp;
    Rec *rec;
    uint64_t *pairs_a, *pairs_b, *huge, *hoff, *hoff_tmp;
    uint32_t *pcount, *pmask;
    uint64_t *ptmask, *ptorg;
    unsigned long long *ctrl;   // control block: totals[2], heavy block count, then the biased maximum and minimum weight exponents
                                // (int[AST_MAX_PROPS] each, kExpWords words each); zeroed per call
    int *wexp, *wmin;
    uint8_t *block_heavy;       // nb flags written by K0: the block holds particles K1 has to classify
    PresortBuffers pre;         // only with AST_FLAG_ORDER_AUTO / _ALWAYS
    RoundSet set;
    void *sort_ws;
    size_t bytes;
};

static int validate2(const ast_project2d_params *p)
{
    AST_REQUIRE(p != nullptr, "params is null");
    AST_REQUIRE(p->n >= 0 && p->n < (int64_t)0xffffffffll, "n = %lld out of range [0, 2^32-1)", (long long)p->n);
    AST_REQUIRE(p->axis >= 0 && p->axis <= 2, "axis = %d is not 0, 1 or 2", p->axis);
    AST_REQUIRE(p->nx > 0 && p->ny > 0, "image_size (%d, %d) must be positive", p->nx, p->ny);
    AST_REQUIRE((int64_t)((p->nx + TILE - 1) / TILE) * ((p->ny + TILE - 1) / TILE) < (1ll << 27), "image too large");
    AST_REQUIRE(kernel_valid(p->kernel_id), "unknown kernel id %d", p->kernel_id);
    if (p->kernel_id == AST_KERNEL_TABLE)
        AST_REQUIRE(p->kernel_table != nullptr && p->kernel_table_n >= 2 && (p->kernel_dim == 2 || p->kernel_dim == 3),
                    "AST_KERNEL_TABLE needs kernel_table (device), kernel_table_n >= 2 and kernel_dim 2 or 3");
    AST_REQUIRE(p->n_prop >= 1 && p->n_prop <= AST_MAX_PROPS, "n_prop = %d not in [1, %d]", p->n_prop, AST_MAX_PROPS);
    AST_REQUIRE(p->x_max > p->x_min && p->y_max > p->y_min, "empty or inverted map bounds");
    if (p->flags & AST_FLAG_PERIODIC) AST_REQUIRE(p->box_a > 0 && p->box_b > 0, "periodic projection needs box_a, box_b > 0");
    AST_REQUIRE(p->pair_capacity >= 0 && p->pair_capacity < (1ll << 32), "pair_capacity out of range");
    AST_REQUIRE(p->huge_capacity >= 0 && p->huge_capacity < (1ll << 31), "huge_capacity out of range");
    return AST_OK;
}

static Layout2 layout2(const ast_project2d_params *p, void *ws)
{
    Layout2 L;
    L.nb = (p->n + kBinThreads - 1) / kBinThreads;
    if (L.nb < 1) L.nb = 1;
    L.ntiles = (int64_t)((p->nx + TILE - 1) / TILE) * ((p->ny + TILE - 1) / TILE);
    L.win = p->pair_capacity > 0 ? p->pair_capacity : 1;
    L.huge_cap = p->huge_capacity > 0 ? p->huge_capacity : 1;
    Carver c(ws);
    L.block_pairs = c.take<uint64_t>(L.nb + 1);
    L.block_huge = c.take<uint64_t>(L.nb + 1);
    L.scan_tmp = c.take<uint64_t>(2 * scan_num_blocks(L.nb + 1) + 2);
    L.rec = c.take<Rec>(p->n > 0 ? p->n : 1);
    L.pcount = c.take<uint32_t>(p->n > 0 ? p->n : 1);
    L.pmask = c.take<uint32_t>(p->n > 0 ? p->n : 1);
    L.ptmask = c.take<uint64_t>(p->n > 0 ? p->n : 1);
    L.ptorg = c.take<uint64_t>(p->n > 0 ? p->n : 1);
    L.ctrl = c.take<unsigned long long>(3 + 2 * kExpWords);
    L.wexp = reinterpret_cast<int *>(L.ctrl ? L.ctrl + 3 : nullptr);
    L.wmin = reinterpret_cast<int *>(L.ctrl ? L.ctrl + 3 + kExpWords : nullptr);
    L.block_heavy = c.take<uint8_t>(L.nb + 1);
    L.pairs_a = c.take<uint64_t>(L.win);
    L.pairs_b = c.take<uint64_t>(L.win);
    L.huge = c.take<uint64_t>(L.huge_cap);
    L.hoff = c.take<uint64_t>(L.huge_cap + 1);
    L.hoff_tmp = (uint64_t *)c.take<char>(scan_workspace_bytes<uint64_t>(L.huge_cap + 1));
    L.set.pp = c.take<float4>(L.win);
    L.set.pc = nullptr;                                   // chosen per round: the sort's free ping-pong buffer
    L.set.tbeg = c.take<uint32_t>(L.ntiles);
    L.set.tend = c.take<uint32_t>(L.ntiles);
    L.set.seg_off = c.take<uint32_t>(L.ntiles + 1);
    L.set.seg_tmp = c.take<uint32_t>(scan_num_blocks(L.ntiles + 1) + 2);
    L.sort_ws = c.take<char>(sort_workspace_bytes(L.win));
    memset(&L.pre, 0, sizeof L.pre);
    if (p->flags & (AST_FLAG_ORDER_AUTO | AST_FLAG_ORDER_ALWAYS)) {
        const size_t n = (size_t)(p->n > 0 ? p->n : 1);
        L.pre.counts = c.take<unsigned long long>(2);
        L.pre.ka = c.take<uint64_t>(n);
        L.pre.kb = c.take<uint64_t>(n);
        L.pre.sort_ws = c.take<char>(sort_workspace_bytes((int64_t)n));
        L.pre.spos = c.take<double>(3 * n);
        L.pre.sh = c.take<double>(n);
        for (int k = 0; k < AST_MAX_PROPS; ++k) L.pre.sprop[k] = k < p->n_prop ? c.take<double>(n) : nullptr;
    }
    L.bytes = c.bytes();
    return L;
}

static P2 make_p2(const ast_project2d_params *p, const double *pos, const double *h, const double *const *prop, double *out)
{
    P2 a;
    a.pos = pos; a.h = h; a.out = out;
    for (int k = 0; k < AST_MAX_PROPS; ++k) a.prop[k] = (prop && k < p->n_prop) ? prop[k] : nullptr;
    a.n = p->n;
    plane_columns(p->axis, a.a_col, a.b_col);
    a.n_prop = p->n_prop;
    a.kernel_id = p->kernel_id;
    a.shape = kernel_shape(p->kernel_id);
    a.norm_c = p->kernel_id == AST_KERNEL_TABLE ? 1.0 : kernel_norm(p->kernel_id, 1.0);
    a.norm_dim = p->kernel_id == AST_KERNEL_TABLE ? p->kernel_dim : ((p->kernel_id == 0 || p->kernel_id == 2) ? 3 : 2);
    a.tab.tab = (const float2 *)p->kernel_table;
    a.tab.n = p->kernel_table_n;
    a.tab.scale = 0.5f * (float)p->kernel_table_n;
    a.ax = make_axis(p->x_min, p->x_max, p->nx);
    a.ay = make_axis(p->y_min, p->y_max, p->ny);
    a.nxd1 = (double)p->nx + 1.0; a.nyd1 = (double)p->ny + 1.0;
    a.ntx = (p->nx + TILE - 1) / TILE;
    a.nty = (p->ny + TILE - 1) / TILE;
    const bool per = (p->flags & AST_FLAG_PERIODIC) != 0;
    a.n_img = per ? 9 : 1;
    a.img_shift = per ? 4 : 0;
    a.box_a = per ? p->box_a : 0.0;
    a.box_b = per ? p->box_b : 0.0;
    a.small_max_px = p->small_max_px >= 0 ? p->small_max_px : kDefaultSmallMaxPx;
    a.huge_min_tiles = p->huge_min_tiles >= 0 ? p->huge_min_tiles : kDefaultHugeMinTiles;
    a.map_stride = (size_t)p->nx * (size_t)p->ny;
    a.pcount = nullptr; a.pmask = nullptr; a.wexp = nullptr; a.wmin = nullptr; a.totals = nullptr; a.ptmask = nullptr; a.ptorg = nullptr;
    return a;
}

template <int SHAPE>
static void launch_accum(int np, const Acc &a, int64_t n_items, cudaStream_t s)
{
    if (np == 1) rowcol_accum_kernel<SHAPE, 1><<<(unsigned)n_items, 256, 0, s>>>(a);
    else rowcol_accum_kernel<SHAPE, 2><<<(unsigned)n_items, 256, 0, s>>>(a);
}

}  // namespace ast

using namespace ast;

extern "C" int ast_project2d_workspace_bytes(const ast_project2d_params *p, size_t *bytes)
{
    int rc = validate2(p);
    if (rc) return rc;
    AST_REQUIRE(bytes != nullptr, "bytes is null");
    *bytes = layout2(p, nullptr).bytes;
    return AST_OK;
}

namespace {

// everything one call needs on the host
struct Run2 {
    const ast_project2d_params *p;
    P2 a;
    Layout2 L;
    Acc c;
    cudaStream_t s;
    float2 *pc;                    // staged weights of the current round
    const uint64_t *sorted;        // sorted pairs of the current round
    int n_bands;                   // exponent bands of the call (1 unless the weights of one field span more than kWeightBand)
    int emax[AST_MAX_PROPS], nbk[AST_MAX_PROPS];   // largest weight exponent and number of bands per field
    ast_project2d_stats st;
    StageTimer *tk;
    int sm_count;
};

// band j of every field into R.c (see split_weight); a field with fewer bands stages zeros from its last band on
static void set_band(Run2 &R, int j)
{
    for (int k = 0; k < AST_MAX_PROPS; ++k) {
        const int top = R.emax[k] - j * kWeightBand;
        R.c.etop[k] = j < R.nbk[k] ? top : R.emax[k];
        R.c.ebot[k] = j < R.nbk[k] ? (j + 1 == R.nbk[k] ? kZeroExp : top - kWeightBand + 1) : R.emax[k] + 1;
    }
}

// K5 over the sorted pairs of the current round: tile ranges, coordinates and the weights of the band in R.c
static void launch_pair_records(Run2 &R, int64_t nw)
{
    const RoundSet &S = R.L.set;
    Acc c = R.c;
    c.sorted = R.sorted;
    const unsigned nbk = (unsigned)((nw + 255) / 256);
    cudaStream_t q = R.s;
#define AST_LAUNCH_PR(SH) do { if (R.p->n_prop == 1) pair_record_kernel<SH, 1><<<nbk, 256, 0, q>>>(c, nw, S.tbeg, S.tend, S.pp, R.pc); \
                               else pair_record_kernel<SH, 2><<<nbk, 256, 0, q>>>(c, nw, S.tbeg, S.tend, S.pp, R.pc); } while (0)
    if (R.a.shape == SHAPE_CUBIC) AST_LAUNCH_PR(SHAPE_CUBIC);
    else if (R.a.shape == SHAPE_WENDLAND) AST_LAUNCH_PR(SHAPE_WENDLAND);
    else AST_LAUNCH_PR(SHAPE_TABLE);
#undef AST_LAUNCH_PR
    R.st.n_launches += 1;
}

// index work of one round: pairs [w0, w1) of the combined emit order -- tiled pairs [0, T), then the pairs of the current
// large-h window [base, base + HP): emit, stable sort by tile key, pair records, tile ranges, work items.
static int prep_round(Run2 &R, uint64_t w0, uint64_t w1, uint64_t T, uint64_t base, uint64_t HP, uint32_t n_hent, uint32_t *seg_target)
{
    const Layout2 &L = R.L;
    const RoundSet &S = L.set;
    cudaStream_t q = R.s;
    const int64_t nw = (int64_t)(w1 - w0);
    R.tk->begin(2);
    if (w0 < T) {
        emit_kernel<<<(unsigned)L.nb, kBinThreads, 0, q>>>(R.a, L.block_pairs, L.block_huge, w0, w1 < T ? w1 : T, L.pairs_a, L.huge, 0, 0);
        R.st.n_launches += 1;
    }
    if (HP > 0 && w1 > base) {
        huge_tiles_kernel<true><<<(n_hent + 7) / 8, 256, 0, q>>>(R.a, L.huge, n_hent, L.hoff, base, w0, w1, L.pairs_a);
        R.st.n_launches += 1;
    }
    R.tk->end();
    int in_b = 0, nl = 0;
    const int key_bits = ceil_log2_u64((uint64_t)L.ntiles);     // the image bits below the tile key are NOT sorted on
    R.tk->begin(3);
    AST_CUDA_TRY(radix_sort_u64(L.pairs_a, L.pairs_b, nw, 32 + R.a.img_shift, key_bits, L.sort_ws, q, &in_b, &nl));
    R.tk->end();
    R.st.n_launches += nl;
    R.tk->begin(4);
    AST_CUDA_TRY(cudaMemsetAsync(S.tbeg, 0, sizeof(uint32_t) * L.ntiles, q));
    AST_CUDA_TRY(cudaMemsetAsync(S.tend, 0, sizeof(uint32_t) * L.ntiles, q));
    R.sorted = in_b ? L.pairs_b : L.pairs_a;
    R.pc = reinterpret_cast<float2 *>(in_b ? L.pairs_a : L.pairs_b);      // 8 bytes per pair, like the pairs
    launch_pair_records(R, nw);
    *seg_target = segment_target(nw, (int64_t)R.sm_count * 4);
    tile_segments_kernel<<<(unsigned)((L.ntiles + 1 + 255) / 256), 256, 0, q>>>(S.tbeg, S.tend, 0u, *seg_target, (int)L.ntiles, S.seg_off);
    nl = 0;
    AST_CUDA_TRY(scan_exclusive<uint32_t>(S.seg_off, L.ntiles + 1, S.seg_tmp, nullptr, q, &nl));
    R.st.n_launches += 1 + nl;
    R.tk->end();
    AST_CUDA_TRY(cudaGetLastError());
    return AST_OK;
}

static int accumulate_round(Run2 &R, int64_t nw, uint32_t seg_target)
{
    const Layout2 &L = R.L;
    const RoundSet &S = L.set;
    Acc c = R.c;
    c.sorted = nullptr;
    c.tbeg = S.tbeg; c.tend = S.tend; c.pp = S.pp; c.pc = R.pc; c.seg_off = S.seg_off; c.seg_target = seg_target;
    const int64_t max_items = L.ntiles + nw / (int64_t)seg_target;      // sum_t max(1, ceil(cnt_t / target)) <= this
    R.tk->begin(5);
    if (R.a.shape == SHAPE_CUBIC) launch_accum<SHAPE_CUBIC>(R.p->n_prop, c, max_items, R.s);
    else if (R.a.shape == SHAPE_WENDLAND) launch_accum<SHAPE_WENDLAND>(R.p->n_prop, c, max_items, R.s);
    else launch_accum<SHAPE_TABLE>(R.p->n_prop, c, max_items, R.s);
    R.tk->end();
    R.st.n_launches += 1;
    AST_CUDA_TRY(cudaGetLastError());
    return AST_OK;
}

}  // namespace

extern "C" int ast_project2d(const ast_project2d_params *p, const double *pos, const double *h, const double *const *prop,
                             double *out, void *workspace, size_t workspace_bytes, void *stream, ast_project2d_stats *stats)
{
    int rc = validate2(p);
    if (rc) return rc;
    AST_REQUIRE(out != nullptr, "out is null");
    AST_REQUIRE(p->n == 0 || (pos && h && prop), "null input pointer");
    for (int k = 0; k < p->n_prop && p->n > 0; ++k) AST_REQUIRE(prop[k] != nullptr, "prop[%d] is null", k);
    Run2 R;
    R.p = p;
    R.L = layout2(p, workspace);
    const Layout2 &L = R.L;
    if (workspace == nullptr || workspace_bytes < L.bytes) {
        set_error("workspace too small: need %zu bytes, have %zu", L.bytes, workspace_bytes);
        return AST_EWORKSPACE;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const bool timing = (p->flags & AST_FLAG_TIMING) != 0;
    StageTimer tm(timing, s);
    StageTimer tk(timing, s);
    R.tk = &tk;
    R.s = s;
    memset(&R.st, 0, sizeof R.st);
    ast_project2d_stats &st = R.st;
    tm.begin(7);
    // optional spatial pre-ordering (presort.cuh): key = tile of the particle's own position (timed with the memsets, stage 6)
    const double *sorted_prop[AST_MAX_PROPS] = { nullptr, nullptr };
    tk.begin(6);
    if ((p->flags & (AST_FLAG_ORDER_AUTO | AST_FLAG_ORDER_ALWAYS)) && p->n > 0) {
        OrderGrid og;
        memset(&og, 0, sizeof og);
        og.dims = 2;
        plane_columns(p->axis, og.col[0], og.col[1]);
        const int nt[2] = { (p->nx + TILE - 1) / TILE, (p->ny + TILE - 1) / TILE };
        const double lo2[2] = { p->x_min, p->y_min }, d2[2] = { (p->x_max - p->x_min) / p->nx, (p->y_max - p->y_min) / p->ny };
        for (int k = 0; k < 2; ++k) { og.lo[k] = lo2[k]; og.inv_cell[k] = 1.0 / (d2[k] * TILE); og.n[k] = nt[k]; }
        og.n[2] = 1;
        int done = 0, nl = 0;
        AST_CUDA_TRY(presort_particles((p->flags & AST_FLAG_ORDER_ALWAYS) ? 2 : 1, og, pos, h, prop, p->n_prop, p->n, L.pre, s, &done, &nl));
        st.n_launches += nl;
        st.reordered = done;
        if (done) {
            pos = L.pre.spos; h = L.pre.sh;
            for (int k = 0; k < p->n_prop; ++k) sorted_prop[k] = L.pre.sprop[k];
            prop = sorted_prop;
        }
    }
    R.a = make_p2(p, pos, h, prop, out);
    P2 &a = R.a;
    a.pcount = L.pcount; a.pmask = L.pmask; a.wexp = L.wexp; a.wmin = L.wmin; a.totals = L.ctrl; a.ptmask = L.ptmask; a.ptorg = L.ptorg;
    { int dev = 0; R.sm_count = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&R.sm_count, cudaDevAttrMultiProcessorCount, dev); }

    if (!(p->flags & AST_FLAG_ACCUMULATE)) AST_CUDA_TRY(cudaMemsetAsync(out, 0, sizeof(double) * a.map_stride * p->n_prop, s));
    AST_CUDA_TRY(cudaMemsetAsync(L.ctrl, 0, sizeof(unsigned long long) * (3 + 2 * kExpWords), s));     // totals, heavy count, exponents
    tk.end();
    uint64_t totals[2] = { 0, 0 };
    unsigned long long ctl[3 + 2 * kExpWords];
    memset(ctl, 0, sizeof ctl);
    if (p->n > 0) {
        tk.begin(0);
        {
            // full blocks through the TMA-staged persistent kernel when every bulk copy is 16-byte aligned, the tail
            // block (and everything, when AST_BIN_TMA=0 or a pointer is misaligned) through the plain kernel
            bool aligned = ((uintptr_t)pos % 16 == 0) && ((uintptr_t)h % 16 == 0);
            for (int k = 0; k < p->n_prop; ++k) aligned = aligned && ((uintptr_t)prop[k] % 16 == 0);
            static const bool use_tma = env_flag("AST_BIN_TMA", true);
            const int64_t n_full = (aligned && use_tma) ? p->n / kBinThreads : 0;
            if (n_full > 0) {
                // persistent grid: one wave of resident CTAs (multiple of the SM count)
                // K0 (sub-pixel pass, 40 registers, 6 CTAs per SM) deposits every particle whose support is below one pixel and
                // marks the other blocks; K1 (general classification, 80 registers) then visits the marked blocks only and
                // returns at once when there is none.  AST_BIN_K0=0 runs K1 alone over all blocks.
                static const bool use_k0 = env_flag("AST_BIN_K0", true);
#define AST_LAUNCH_K(KERN, SMEM, ...)                                                                                   \
    do {                                                                                                                \
        auto kern = KERN;                                                                                               \
        const size_t smem = (SMEM);                                                                                     \
        if (smem > 40 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
        int per_sm = 1;                                                                                                 \
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kBinThreads, smem);                                \
        int64_t grid = (int64_t)R.sm_count * (per_sm > 0 ? per_sm : 1);     /* persistent: one wave of resident CTAs */  \
        if (grid > n_full) grid = n_full;                                                                               \
        kern<<<(unsigned)grid, kBinThreads, smem, s>>>(__VA_ARGS__);                                                    \
    } while (0)
    // measured on K1 alone (512^3 particles with sub-pixel supports; stages x CTAs per SM): 2 x 3
    // (80 registers) 1.581 ms, 4 x 3: 1.587, 2 x 4 (64 registers, no spills): 1.469, 4 x 4: 1.488, 2 x 5 (48 registers,
    // spills): 1.608, 2 x 6: 2.000 -- occupancy, not pipeline depth, hides the latency; hence K0.  With SPH-realistic supports
    // the 80-register build of K1 is the faster one (7.18 against 7.69 ms at config 3).
#define AST_LAUNCH_TMA(SH, NPV, PERV)                                                                                   \
    do {                                                                                                                \
        if (use_k0) {                                                                                                   \
            AST_LAUNCH_K((subpixel_tma_kernel<SH, NPV, PERV>), 2 * sizeof(BinStage<NPV>), a, L.block_pairs, L.block_huge, \
                         L.block_heavy, L.ctrl + 2, n_full);                                                            \
            AST_LAUNCH_K((bin_tma_kernel<SH, NPV, PERV, 2, 3, true>), 2 * sizeof(BinStage<NPV>), a, L.rec, L.block_pairs, \
                         L.block_huge, n_full, L.block_heavy, L.ctrl + 2);                                              \
            st.n_launches += 1;                                                                                         \
        } else {                                                                                                        \
            AST_LAUNCH_K((bin_tma_kernel<SH, NPV, PERV, 2, 4, false>), 2 * sizeof(BinStage<NPV>), a, L.rec, L.block_pairs, \
                         L.block_huge, n_full, nullptr, nullptr);                                                       \
        }                                                                                                               \
    } while (0)
                {
                    const bool per = a.n_img > 1;
#define AST_D2(SH) do { if (p->n_prop == 1) { if (per) AST_LAUNCH_TMA(SH, 1, true); else AST_LAUNCH_TMA(SH, 1, false); } \
                        else { if (per) AST_LAUNCH_TMA(SH, 2, true); else AST_LAUNCH_TMA(SH, 2, false); } } while (0)
                    if (a.shape == SHAPE_CUBIC) AST_D2(SHAPE_CUBIC);
                    else if (a.shape == SHAPE_WENDLAND) AST_D2(SHAPE_WENDLAND);
                    else AST_D2(SHAPE_TABLE);
#undef AST_D2
                }
#undef AST_LAUNCH_TMA
#undef AST_LAUNCH_K
                st.n_launches += 1;
            }
            const int64_t n_rest = L.nb - n_full;
            if (n_rest > 0) {
#define AST_LAUNCH_BIN(SH, NPV, PERV) bin_kernel<SH, true, NPV, PERV><<<(unsigned)n_rest, kBinThreads, 0, s>>>(a, L.rec, L.block_pairs, L.block_huge, n_full)
                {
                    const bool per = a.n_img > 1;
#define AST_D2(SH) do { if (p->n_prop == 1) { if (per) AST_LAUNCH_BIN(SH, 1, true); else AST_LAUNCH_BIN(SH, 1, false); } \
                        else { if (per) AST_LAUNCH_BIN(SH, 2, true); else AST_LAUNCH_BIN(SH, 2, false); } } while (0)
                    if (a.shape == SHAPE_CUBIC) AST_D2(SHAPE_CUBIC);
                    else if (a.shape == SHAPE_WENDLAND) AST_D2(SHAPE_WENDLAND);
                    else AST_D2(SHAPE_TABLE);
#undef AST_D2
                }
#undef AST_LAUNCH_BIN
                st.n_launches += 1;
            }
        }
        tk.end();
        AST_CUDA_TRY(cudaGetLastError());
        // the K1 blocks that have pairs or large-h entries added them to the control block: when nothing needs the tile path
        // (the HBM-bound regime: every particle was deposited by K1) the call ends here, without the scan.  The weight
        // exponents come with the same copy: they decide the bands.
        AST_CUDA_TRY(cudaMemcpyAsync(ctl, L.ctrl, sizeof ctl, cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaStreamSynchronize(s));
        totals[0] = ctl[0]; totals[1] = ctl[1];
        if (totals[0] + totals[1] > 0) {
            tk.begin(1);
            // entries 0..nb-1 were written by the binning kernels; the sentinel entry nb becomes the total
            AST_CUDA_TRY(cudaMemsetAsync(L.block_pairs + L.nb, 0, sizeof(uint64_t), s));
            AST_CUDA_TRY(cudaMemsetAsync(L.block_huge + L.nb, 0, sizeof(uint64_t), s));
            int nl = 0;
            AST_CUDA_TRY(scan2_exclusive<uint64_t>(L.block_pairs, L.block_huge, L.nb + 1, L.scan_tmp, s, &nl));
            st.n_launches += nl;
            tk.end();
        }
    }
    const uint64_t T = totals[0], H = totals[1];
    st.n_pairs = (int64_t)T;
    st.n_huge = (int64_t)H;
    if (T + H > 0 && p->pair_capacity <= 0) {
        // nothing was deposited by the tile path yet, but the direct deposits of K1 are in `out`: the header documents it
        set_error("pair_capacity is 0 but %llu pairs and %llu large-h particles need the tile path", (unsigned long long)T,
                  (unsigned long long)H);
        if (stats) *stats = st;
        return AST_EWORKSPACE;
    }
    if (T + H > 0) {
        Acc &c = R.c;
        memset(&c, 0, sizeof c);
        c.rec = L.rec; c.out = out;
        c.x_min = a.ax.vmin; c.y_min = a.ay.vmin; c.dx = a.ax.d; c.dy = a.ay.d; c.inv_dx = a.ax.inv_d; c.inv_dy = a.ay.inv_d;
        c.nx = p->nx; c.ny = p->ny; c.ntx = a.ntx; c.nty = a.nty; c.img_shift = a.img_shift;
        c.n_img = a.n_img; c.box_a = a.box_a; c.box_b = a.box_b; c.tab = a.tab;
        c.map_stride = a.map_stride; c.ntiles = (int)L.ntiles; c.n_huge = 0u;
        int wexp[AST_MAX_PROPS], wmin[AST_MAX_PROPS];
        memcpy(wexp, ctl + 3, sizeof wexp);
        memcpy(wmin, ctl + 3 + kExpWords, sizeof wmin);
        R.n_bands = 1;
        for (int k = 0; k < AST_MAX_PROPS; ++k) {
            const bool any = k < p->n_prop && wexp[k] > 0;        // 0: no non-zero weight in this field
            R.emax[k] = wexp[k] - kExpBias;
            R.nbk[k] = any ? (R.emax[k] - (kExpBias - wmin[k])) / kWeightBand + 1 : 1;
            if (R.nbk[k] > R.n_bands) R.n_bands = R.nbk[k];
        }
        set_band(R, 0);

        int rc2 = AST_OK;
        int64_t round_no = 0;
        const uint64_t hcap = (uint64_t)L.huge_cap;
        const uint64_t n_hwin = H ? (H + hcap - 1) / hcap : 1;
        for (uint64_t hw = 0; hw < n_hwin && rc2 == AST_OK; ++hw) {
            // ---- the large-h window: list entries [h0, h1) -> member-tile counts -> offsets (all on the caller's stream)
            uint64_t HP = 0;
            uint32_t n_hent = 0;
            if (H) {
                const uint64_t h0 = hw * hcap, h1 = (h0 + hcap < H) ? h0 + hcap : H;
                n_hent = (uint32_t)(h1 - h0);
                tk.begin(2);
                emit_kernel<<<(unsigned)L.nb, kBinThreads, 0, s>>>(a, L.block_pairs, L.block_huge, 0, 0, L.pairs_a, L.huge, h0, h1);
                AST_CUDA_TRY(cudaMemsetAsync(L.hoff + n_hent, 0, sizeof(uint64_t), s));
                huge_tiles_kernel<false><<<(n_hent + 7) / 8, 256, 0, s>>>(a, L.huge, n_hent, L.hoff, 0, 0, 0, nullptr);
                int nl = 0;
                AST_CUDA_TRY(scan_exclusive<uint64_t>(L.hoff, (int64_t)n_hent + 1, L.hoff_tmp, nullptr, s, &nl));
                st.n_launches += 2 + nl;
                tk.end();
                AST_CUDA_TRY(cudaMemcpyAsync(&HP, L.hoff + n_hent, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
                AST_CUDA_TRY(cudaStreamSynchronize(s));
                st.n_pairs += (int64_t)HP;
            }
            const uint64_t base = hw == 0 ? T : 0, total = base + HP;
            if (total == 0) continue;
            // rounds over the combined pair order
            const uint64_t win = (uint64_t)L.win;
            const uint64_t rounds = (total + win - 1) / win;
            uint64_t per_round = rounds > 1 ? (((total + rounds - 1) / rounds + 8191ull) & ~8191ull) : win;   // even rounds
            if (per_round > win) per_round = win;
            for (uint64_t r = 0; r * per_round < total && rc2 == AST_OK; ++r, ++round_no) {
                const uint64_t w0 = r * per_round, w1 = (w0 + per_round < total) ? w0 + per_round : total;
                uint32_t seg_target = 1024;
                if (R.n_bands > 1) set_band(R, 0);
                rc2 = prep_round(R, w0, w1, hw == 0 ? T : 0, base, HP, n_hent, &seg_target);
                if (rc2) break;
                rc2 = accumulate_round(R, (int64_t)(w1 - w0), seg_target);
                for (int j = 1; j < R.n_bands && rc2 == AST_OK; ++j) {       // the further bands over the same sorted pairs
                    set_band(R, j);
                    launch_pair_records(R, (int64_t)(w1 - w0));
                    rc2 = accumulate_round(R, (int64_t)(w1 - w0), seg_target);
                }
            }
        }
        st.n_rounds = round_no;
        if (rc2) { if (stats) *stats = st; return rc2; }
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

extern "C" int ast_bin2d(const ast_project2d_params *p, const double *pos, const double *h, int32_t *bbox, uint8_t *cls,
                         uint64_t *pairs_emit, uint64_t *pairs_sorted, uint64_t *huge, int64_t *counts, void *workspace,
                         size_t workspace_bytes, void *stream)
{
    int rc = validate2(p);
    if (rc) return rc;
    AST_REQUIRE(p->n == 0 || (pos && h), "null input pointer");
    Layout2 L = layout2(p, workspace);
    if (workspace == nullptr || workspace_bytes < L.bytes) {
        set_error("workspace too small: need %zu bytes, have %zu", L.bytes, workspace_bytes);
        return AST_EWORKSPACE;
    }
    cudaStream_t s = (cudaStream_t)stream;
    P2 a = make_p2(p, pos, h, nullptr, nullptr);
    a.pcount = L.pcount; a.pmask = L.pmask; a.wexp = L.wexp; a.totals = nullptr; a.ptmask = L.ptmask; a.ptorg = L.ptorg;
    uint64_t *pa = L.pairs_a, *pb = L.pairs_b;
    const int64_t cap = L.win;
    uint64_t totals[2] = { 0, 0 };
    uint64_t HP = 0;
    AST_CUDA_TRY(cudaMemsetAsync(L.block_pairs, 0, sizeof(uint64_t) * (L.nb + 1), s));
    AST_CUDA_TRY(cudaMemsetAsync(L.block_huge, 0, sizeof(uint64_t) * (L.nb + 1), s));
    if (p->n > 0) {
        if (bbox || cls) bbox_cls_kernel<<<(unsigned)L.nb, kBinThreads, 0, s>>>(a, bbox, cls);
        bin_kernel<SHAPE_CUBIC, false, 1, true><<<(unsigned)L.nb, kBinThreads, 0, s>>>(a, L.rec, L.block_pairs, L.block_huge, 0);
        scan_exclusive_kernel<uint64_t><<<1, kScanThreads, 0, s>>>(L.block_pairs, L.nb + 1, nullptr);
        scan_exclusive_kernel<uint64_t><<<1, kScanThreads, 0, s>>>(L.block_huge, L.nb + 1, nullptr);
        AST_CUDA_TRY(cudaGetLastError());
        AST_CUDA_TRY(cudaMemcpyAsync(&totals[0], L.block_pairs + L.nb, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaMemcpyAsync(&totals[1], L.block_huge + L.nb, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaStreamSynchronize(s));
    }
    const uint64_t T = totals[0], H = totals[1];
    if (H > (uint64_t)L.huge_cap) {
        if (counts) { counts[0] = (int64_t)T; counts[1] = (int64_t)H; }
        set_error("capacity too small: need %llu huge entries", (unsigned long long)H);
        return AST_EWORKSPACE;
    }
    if (H > 0) {
        const uint32_t nh = (uint32_t)H;
        emit_kernel<<<(unsigned)L.nb, kBinThreads, 0, s>>>(a, L.block_pairs, L.block_huge, 0, 0, pa, L.huge, 0, H);
        AST_CUDA_TRY(cudaMemsetAsync(L.hoff + nh, 0, sizeof(uint64_t), s));
        huge_tiles_kernel<false><<<(nh + 7) / 8, 256, 0, s>>>(a, L.huge, nh, L.hoff, 0, 0, 0, nullptr);
        AST_CUDA_TRY(scan_exclusive<uint64_t>(L.hoff, (int64_t)nh + 1, L.hoff_tmp, nullptr, s));
        AST_CUDA_TRY(cudaMemcpyAsync(&HP, L.hoff + nh, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        AST_CUDA_TRY(cudaStreamSynchronize(s));
    }
    const uint64_t total = T + HP;
    if (counts) { counts[0] = (int64_t)total; counts[1] = (int64_t)H; }
    if (total > (uint64_t)p->pair_capacity || total > (uint64_t)cap) {
        set_error("capacity too small: need %llu pairs and %llu huge entries", (unsigned long long)total, (unsigned long long)H);
        return AST_EWORKSPACE;
    }
    if (total + H > 0) {
        if (T > 0) emit_kernel<<<(unsigned)L.nb, kBinThreads, 0, s>>>(a, L.block_pairs, L.block_huge, 0, T, pa, L.huge, 0, 0);
        if (HP > 0) huge_tiles_kernel<true><<<((uint32_t)H + 7) / 8, 256, 0, s>>>(a, L.huge, (uint32_t)H, L.hoff, T, 0, total, pa);
        AST_CUDA_TRY(cudaGetLastError());
        if (pairs_emit && total)
            AST_CUDA_TRY(cudaMemcpyAsync(pairs_emit, pa, sizeof(uint64_t) * total, cudaMemcpyDeviceToDevice, s));
        if (huge && H) AST_CUDA_TRY(cudaMemcpyAsync(huge, L.huge, sizeof(uint64_t) * H, cudaMemcpyDeviceToDevice, s));
        if (pairs_sorted && total) {
            int in_b = 0;
            const int key_bits = ceil_log2_u64((uint64_t)L.ntiles);
            AST_CUDA_TRY(radix_sort_u64(pa, pb, (int64_t)total, 32 + a.img_shift, key_bits, L.sort_ws, s, &in_b));
            AST_CUDA_TRY(cudaMemcpyAsync(pairs_sorted, in_b ? pb : pa, sizeof(uint64_t) * total, cudaMemcpyDeviceToDevice, s));
        }
    }
    AST_CUDA_TRY(cudaStreamSynchronize(s));
    return AST_OK;
}

extern "C" int ast_contrib_count2d(const ast_project2d_params *p, const double *pos, const double *h, int32_t *count, void *stream)
{
    int rc = validate2(p);
    if (rc) return rc;
    AST_REQUIRE(count != nullptr && (p->n == 0 || (pos && h)), "null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    P2 a = make_p2(p, pos, h, nullptr, nullptr);
    AST_CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int32_t) * a.map_stride, s));
    if (p->n > 0) contrib_count_kernel<<<(unsigned)((p->n + 127) / 128), 128, 0, s>>>(a, count);
    AST_CUDA_TRY(cudaGetLastError());
    return AST_OK;
}

extern "C" int ast_kernel_eval(int kernel_id, const double *r, const double *h, double *out, int64_t n, void *stream)
{
    AST_REQUIRE(kernel_valid(kernel_id) && kernel_id != AST_KERNEL_TABLE, "unknown kernel id %d", kernel_id);
    AST_REQUIRE(n >= 0 && (n == 0 || (r && h && out)), "null pointer or negative n");
    if (n > 0) kernel_eval_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(kernel_id, r, h, out, n);
    AST_CUDA_TRY(cudaGetLastError());
    return AST_OK;
}

extern "C" int ast_sort_workspace_bytes(int64_t n, size_t *bytes)
{
    AST_REQUIRE(bytes != nullptr && n >= 0, "bad argument");
    *bytes = sort_workspace_bytes(n);
    return AST_OK;
}

extern "C" int ast_radix_sort_u64(uint64_t *keys, uint64_t *tmp, int64_t n, int bit_lo, int n_bits, void *workspace,
                                  size_t workspace_bytes, void *stream, int *result_in_tmp)
{
    AST_REQUIRE(n >= 0 && n < (1ll << 32), "n out of range");
    AST_REQUIRE(bit_lo >= 0 && n_bits >= 0 && bit_lo + n_bits <= 64, "bad bit range");
    AST_REQUIRE(result_in_tmp != nullptr, "result_in_tmp is null");
    if (workspace_bytes < sort_workspace_bytes(n) || (n > 0 && (!keys || !tmp || !workspace))) {
        set_error("sort workspace too small or null buffers");
        return AST_EWORKSPACE;
    }
    AST_CUDA_TRY(radix_sort_u64(keys, tmp, n, bit_lo, n_bits, workspace, (cudaStream_t)stream, result_in_tmp));
    return AST_OK;
}
