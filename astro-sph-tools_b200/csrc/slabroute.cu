// slabroute.cu -- packing kernel of the multi-GPU exchanges along x-slabs: the k-NN exchange (SURVEY 8(e): slabs along x +
// ghost zones) and the 3-D gridding exchange (each rank owns an x-slab of the grid).  One kernel, two destination policies.
//
// Every rank holds an arbitrary set of particles (the reference's per-rank read, io/EAGLE/_SnapshotEAGLE.py:120-130) and has
// to send each of them to the rank that OWNS its slab and, as a ghost, to every rank whose slab lies within the ghost width
// w of it.  The torch version of this step walks the particle array once per destination rank (remainder, where, two
// nonzero, a cat and a gather: ~10 passes of n_local per rank of the job); here it is two passes in all:
//   count  one ballot per (kind, destination) and warp -> per-block counts, table [kind][destination][block]
//   scan   one exclusive scan over the flattened table = first send row of every (kind, destination, block)
//   write  the same ballots again -> rank inside the warp / block -> send row; the particle's position goes straight into
//          the send buffer and its index into src_index (the way h finds back home)
// Send buffer layout: [owned -> rank 0 | owned -> rank 1 | ... | ghosts -> rank 0 | ghosts -> rank 1 | ...], inside each piece
// ascending particle index (blocks, warps and lanes are walked in order), which is also what the torch version produces.
// Two all-to-all calls (owned, then ghosts) then leave the receiver with [owned from all | ghosts from all] without a reorder.
// Gridding has one kind: a particle goes to every rank whose planes its support reaches (GridRoute), rows (x, y, z, h, prop).
#include "ast_geom.h"
#include "common.cuh"
#include "scan_sort.cuh"

namespace ast {

constexpr int kRouteMaxWorld = 32;

// A destination policy R provides
//   kKinds                    pieces of the send buffer per destination rank (kind-major: [kind 0 -> 0 | kind 0 -> 1 | ...])
//   n, world                  local particles, ranks
//   dests(i, m)               m[k] bit g: particle i goes to rank g as kind k (the count and the write pass call the same code)
//   put(send, idx, row, i)    write particle i as send row `row`
struct KnnRoute {
    static constexpr int kKinds = 2;                 // 0 = owned, 1 = ghost
    const double *pos;            // (n, 3)
    const int64_t *owner;         // (n) owning rank of every particle (from the global histogram plan)
    int64_t n;
    int world, periodic, covers_all;
    double length, w;
    double b_lo[kRouteMaxWorld], b_hi[kRouteMaxWorld];

    // bit g of the result: the particle goes to rank g as a ghost
    __device__ __forceinline__ uint32_t ghosts(double x, int own) const
    {
        uint32_t m = 0;
        for (int g = 0; g < world; ++g) {
            if (g == own) continue;
            double d;
            if (periodic) {
                double t = fmod(x - b_lo[g], length);
                if (t < 0.0) t += length;
                const double seg = b_hi[g] - b_lo[g];
                d = t <= seg ? 0.0 : fmin(t - seg, length - t);
            } else {
                d = fmax(fmax(b_lo[g] - x, x - b_hi[g]), 0.0);
            }
            if (d <= w || covers_all) m |= 1u << g;
        }
        return m;
    }
    __device__ __forceinline__ void dests(int64_t i, uint32_t *m) const
    {
        int own = (int)owner[i];
        if (own < 0 || own >= world) own = -1;                         // (never from _slab_plan; such a particle would be dropped)
        m[0] = own >= 0 ? 1u << own : 0u;
        m[1] = ghosts(pos[3 * i], own);
    }
    __device__ __forceinline__ void put(double *send, int64_t *src_index, int64_t row, int64_t i) const
    {
        send[3 * row] = pos[3 * i]; send[3 * row + 1] = pos[3 * i + 1]; send[3 * row + 2] = pos[3 * i + 2];
        src_index[row] = i;
    }
};

// Rank g owns planes [e[g], e[g+1]) of the whole grid.  The ranges are range1 on the whole grid's axes and the image shifts
// are bin3_kernel's, so a particle reaches a rank exactly when ast_grid3d with that rank's x window would deposit it.
struct GridRoute {
    static constexpr int kKinds = 1;
    const double *pos, *h, *prop;
    int64_t n;
    int world, periodic;
    Axis1 ax[3];
    double box[3];
    int e[kRouteMaxWorld + 1];

    __device__ __forceinline__ void dests(int64_t i, uint32_t *m) const
    {
        m[0] = 0u;
        const double hh = h[i], R2 = radius2(hh);
        const int nt = periodic ? 3 : 1;
        int lo, up;
        for (int c = 1; c < 3; ++c) {                                    // some image must reach the grid along y and along z
            bool any = false;
            for (int t = 0; t < nt && !any; ++t)
                any = range1(ax[c], AST_DADD(pos[3 * i + c], periodic ? (double)(t - 1) * box[c] : 0.0), hh, R2, lo, up);
            if (!any) return;
        }
        for (int t = 0; t < nt; ++t) {
            if (!range1(ax[0], AST_DADD(pos[3 * i], periodic ? (double)(t - 1) * box[0] : 0.0), hh, R2, lo, up)) continue;
            for (int g = 0; g < world; ++g)
                if (e[g] < e[g + 1] && e[g] <= up && lo < e[g + 1]) m[0] |= 1u << g;
        }
    }
    __device__ __forceinline__ void put(double *send, int64_t *, int64_t row, int64_t i) const
    {
        double *r = send + 5 * row;
        r[0] = pos[3 * i]; r[1] = pos[3 * i + 1]; r[2] = pos[3 * i + 2]; r[3] = h[i]; r[4] = prop[i];
    }
};

// table[(kind * world + g) * nblocks + block].  WRITE: a row at or beyond send_rows (the rows the caller allocated from the
// counted total) is not written; it sets *overflow instead.
template <class R, bool WRITE>
__global__ void __launch_bounds__(256) slab_route_kernel(R a, uint64_t *__restrict__ table, int64_t nblocks, double *__restrict__ send,
                                                         int64_t *__restrict__ src_index, int64_t send_rows, int *__restrict__ overflow)
{
    __shared__ uint32_t wcount[2 * kRouteMaxWorld][8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t i = (int64_t)blockIdx.x * 256 + tid;
    uint32_t m[R::kKinds];
    for (int k = 0; k < R::kKinds; ++k) m[k] = 0u;
    if (i < a.n) a.dests(i, m);
    for (int k = 0; k < R::kKinds; ++k)
        for (int g = 0; g < a.world; ++g) {
            const unsigned b = __ballot_sync(0xffffffffu, (m[k] >> g) & 1u);
            if (lane == 0) wcount[k * a.world + g][warp] = __popc(b);
        }
    __syncthreads();
    if (!WRITE) {
        if (tid < R::kKinds * a.world) {
            uint32_t s = 0;
            for (int w = 0; w < 8; ++w) s += wcount[tid][w];
            table[(int64_t)tid * nblocks + blockIdx.x] = s;
        }
        return;
    }
    // (all lanes stay to the end: the ballots below are full-warp)
    const unsigned lt = (1u << lane) - 1u;
    for (int k = 0; k < R::kKinds; ++k)
        for (int g = 0; g < a.world; ++g) {
            const bool in = (m[k] >> g) & 1u;
            const unsigned b = __ballot_sync(0xffffffffu, in);
            if (!in) continue;
            const int piece = k * a.world + g;
            uint32_t before = 0;
            for (int w = 0; w < warp; ++w) before += wcount[piece][w];
            const int64_t row = (int64_t)table[(int64_t)piece * nblocks + blockIdx.x] + before + __popc(b & lt);
            if (row < send_rows) a.put(send, src_index, row, i);
            else *overflow = 1;
        }
}

// counts[p] = table entry of the first block of the NEXT piece - first block of this piece
__global__ void slab_route_counts_kernel(const uint64_t *__restrict__ table, const uint64_t *__restrict__ total, int64_t nblocks, int pieces,
                                         int64_t *__restrict__ counts)
{
    const int p = threadIdx.x;
    if (p >= pieces) return;
    const uint64_t b = table[(int64_t)p * nblocks], e = p + 1 < pieces ? table[(int64_t)(p + 1) * nblocks] : *total;
    counts[p] = (int64_t)(e - b);
}

static int64_t route_blocks(int64_t n) { return n > 0 ? (n + 255) / 256 : 1; }

static size_t route_workspace(int pieces, int64_t n)
{
    const int64_t entries = (int64_t)pieces * route_blocks(n);
    Carver c(nullptr);
    c.take<uint64_t>(entries + 1);
    c.take<char>(scan_workspace_bytes<uint64_t>(entries + 1));
    return c.bytes();
}

// count pass + scan: counts[0 .. kKinds*world) and, in the workspace, the scanned block table (first send row of every
// piece and block) that the write pass reads
template <class R>
static int route_count(const R &a, int64_t *counts, void *workspace, size_t workspace_bytes, cudaStream_t s)
{
    const int pieces = R::kKinds * a.world;
    const size_t need = route_workspace(pieces, a.n);
    if (!workspace || workspace_bytes < need) { set_error("workspace too small: need %zu bytes, have %zu", need, workspace_bytes); return AST_EWORKSPACE; }
    const int64_t nb = route_blocks(a.n), entries = (int64_t)pieces * nb;
    Carver c(workspace);
    uint64_t *table = c.take<uint64_t>(entries + 1);
    uint64_t *tmp = (uint64_t *)c.take<char>(scan_workspace_bytes<uint64_t>(entries + 1));
    AST_CUDA_TRY(cudaMemsetAsync(table, 0, sizeof(uint64_t) * (entries + 1), s));
    if (a.n > 0) slab_route_kernel<R, false><<<(unsigned)nb, 256, 0, s>>>(a, table, nb, nullptr, nullptr, 0, nullptr);
    AST_KERNEL_CHECK(s, "slab_route_kernel<count>");
    AST_CUDA_TRY(scan_exclusive<uint64_t>(table, entries, tmp, table + entries, s));      // total behind the table
    slab_route_counts_kernel<<<1, 64, 0, s>>>(table, table + entries, nb, pieces, counts);
    AST_KERNEL_CHECK(s, "slab_route_counts_kernel");
    return AST_OK;
}

template <class R>
static int route_write(const R &a, double *send, int64_t *src_index, int64_t send_rows, int *overflow, void *workspace,
                       size_t workspace_bytes, cudaStream_t s)
{
    const size_t need = route_workspace(R::kKinds * a.world, a.n);
    if (!workspace || workspace_bytes < need) { set_error("workspace too small: need %zu bytes, have %zu", need, workspace_bytes); return AST_EWORKSPACE; }
    const int64_t nb = route_blocks(a.n);
    Carver c(workspace);
    uint64_t *table = c.take<uint64_t>((int64_t)R::kKinds * a.world * nb + 1);      // scanned by route_count on the same workspace
    slab_route_kernel<R, true><<<(unsigned)nb, 256, 0, s>>>(a, table, nb, send, src_index, send_rows, overflow);
    AST_KERNEL_CHECK(s, "slab_route_kernel<write>");
    return AST_OK;
}

}  // namespace ast

using namespace ast;

// ---- k-NN exchange
static int route_validate(const ast_slab_route_params *p)
{
    AST_REQUIRE(p != nullptr, "params is null");
    AST_REQUIRE(p->n >= 0, "n < 0");
    AST_REQUIRE(p->world >= 1 && p->world <= kRouteMaxWorld, "world = %d not in [1, %d]", p->world, kRouteMaxWorld);
    AST_REQUIRE(p->w >= 0.0, "ghost width < 0");
    AST_REQUIRE(!p->periodic || p->length > 0.0, "periodic routing needs length > 0");
    return AST_OK;
}

static KnnRoute knn_route(const ast_slab_route_params *p, const double *pos, const int64_t *owner)
{
    KnnRoute a;
    memset(&a, 0, sizeof a);
    a.pos = pos; a.owner = owner; a.n = p->n; a.world = p->world; a.periodic = p->periodic; a.covers_all = p->covers_all;
    a.length = p->length; a.w = p->w;
    for (int g = 0; g < p->world; ++g) { a.b_lo[g] = p->bounds[g]; a.b_hi[g] = p->bounds[g + 1]; }
    return a;
}

extern "C" int ast_slab_route_workspace_bytes(const ast_slab_route_params *p, size_t *bytes)
{
    int rc = route_validate(p);
    if (rc) return rc;
    AST_REQUIRE(bytes != nullptr, "bytes is null");
    *bytes = route_workspace(KnnRoute::kKinds * p->world, p->n);
    return AST_OK;
}

extern "C" int ast_slab_route_count(const ast_slab_route_params *p, const double *pos, const int64_t *owner, int64_t *counts,
                                    void *workspace, size_t workspace_bytes, void *stream)
{
    int rc = route_validate(p);
    if (rc) return rc;
    AST_REQUIRE(counts != nullptr && (p->n == 0 || (pos && owner)), "null pointer");
    return route_count(knn_route(p, pos, owner), counts, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int ast_slab_route_write(const ast_slab_route_params *p, const double *pos, const int64_t *owner, double *send,
                                    int64_t *src_index, void *workspace, size_t workspace_bytes, void *stream)
{
    int rc = route_validate(p);
    if (rc) return rc;
    if (p->n == 0) return AST_OK;
    AST_REQUIRE(pos && owner && send && src_index, "null pointer");
    // (this ABI has no row count: the caller allocates the counted total, so no row bound is passed)
    return route_write(knn_route(p, pos, owner), send, src_index, INT64_MAX, nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- 3-D gridding on x-slabs
static int grid_route_validate(const ast_grid_route_params *p)
{
    AST_REQUIRE(p != nullptr, "params is null");
    AST_REQUIRE(p->n >= 0, "n < 0");
    AST_REQUIRE(p->world >= 1 && p->world <= kRouteMaxWorld, "world = %d not in [1, %d]", p->world, kRouteMaxWorld);
    AST_REQUIRE(p->nx > 0 && p->ny > 0 && p->nz > 0, "grid size must be positive");
    for (int c = 0; c < 3; ++c) AST_REQUIRE(p->hi[c] > p->lo[c], "empty or inverted grid bounds");
    if (p->periodic)
        for (int c = 0; c < 3; ++c) AST_REQUIRE(p->box[c] > 0, "periodic routing needs box[0..2] > 0");
    AST_REQUIRE(p->edges[0] >= 0 && p->edges[p->world] <= p->nx, "plane edges must lie in [0, nx = %d]", p->nx);
    for (int g = 0; g < p->world; ++g) AST_REQUIRE(p->edges[g] <= p->edges[g + 1], "plane edges must not decrease");
    return AST_OK;
}

static GridRoute grid_route(const ast_grid_route_params *p, const double *pos, const double *h, const double *prop)
{
    GridRoute a;
    memset(&a, 0, sizeof a);
    a.pos = pos; a.h = h; a.prop = prop; a.n = p->n; a.world = p->world; a.periodic = p->periodic ? 1 : 0;
    const int n3[3] = { p->nx, p->ny, p->nz };
    for (int c = 0; c < 3; ++c) {
        a.ax[c] = make_axis(p->lo[c], p->hi[c], n3[c]);
        a.box[c] = p->periodic ? p->box[c] : 0.0;
    }
    for (int g = 0; g <= p->world; ++g) a.e[g] = p->edges[g];
    return a;
}

extern "C" int ast_grid_route_workspace_bytes(const ast_grid_route_params *p, size_t *bytes)
{
    int rc = grid_route_validate(p);
    if (rc) return rc;
    AST_REQUIRE(bytes != nullptr, "bytes is null");
    *bytes = route_workspace(GridRoute::kKinds * p->world, p->n);
    return AST_OK;
}

extern "C" int ast_grid_route_count(const ast_grid_route_params *p, const double *pos, const double *h, int64_t *counts,
                                    void *workspace, size_t workspace_bytes, void *stream)
{
    int rc = grid_route_validate(p);
    if (rc) return rc;
    AST_REQUIRE(counts != nullptr && (p->n == 0 || (pos && h)), "null pointer");
    return route_count(grid_route(p, pos, h, nullptr), counts, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int ast_grid_route_write(const ast_grid_route_params *p, const double *pos, const double *h, const double *prop,
                                    double *send, int64_t send_rows, int32_t *overflow, void *workspace, size_t workspace_bytes,
                                    void *stream)
{
    int rc = grid_route_validate(p);
    if (rc) return rc;
    AST_REQUIRE(overflow != nullptr, "overflow is null");
    AST_REQUIRE(send_rows >= 0 && (send_rows == 0 || send != nullptr), "send is null");
    AST_REQUIRE(p->n == 0 || (pos && h && prop), "null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    AST_CUDA_TRY(cudaMemsetAsync(overflow, 0, sizeof(int32_t), s));
    if (p->n == 0) return AST_OK;
    return route_write(grid_route(p, pos, h, prop), send, nullptr, send_rows, overflow, workspace, workspace_bytes, s);
}
