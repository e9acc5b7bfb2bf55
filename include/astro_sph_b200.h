/*
 * astro_sph_b200.h -- C ABI of the B200-native SPH deposition / smoothing-length library
 * (libastsph_b200.so, built from astro-sph-tools_b200/csrc by nvcc for sm_100a).
 *
 * This is the drop-in boundary for the hot path of QuasarX1/astro-sph-tools.  Each entry point names the
 * reference interface it replaces (paths relative to /root/reference/src/astro_sph_tools/).  In the
 * reference the FFI boundary is Python -> Cython, crossed once PER PIXEL
 * (tools/projections/_pixel_calculations.pyx:9-10 calculate_pixel_value, called from
 * tools/projections/_projector.py:53-71); here it is crossed once PER MAP.
 *
 * Conventions
 *   - every function returns an ast_status (0 = ok); ast_last_error() gives the message of the last
 *     failure on the calling thread;
 *   - all data pointers are DEVICE pointers unless the parameter is documented "host";
 *   - the library never allocates or frees device memory: inputs, outputs and workspace are caller-owned
 *     (the Python host layer hands torch-owned buffers in by raw pointer);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it except where a function
 *     is documented to synchronise;
 *   - positions are (N,3) row-major float64 exactly as the reference readers hand them out
 *     (io/data_structures/_SnapshotBase.py:708-725), h and the per-particle weights are (N,) float64
 *     (:599-616, :618-637); maps are float64 row-major out[xi*ny + yi] like the reference's img[xi, yi]
 *     (tools/projections/_projector.py:88,117).
 */
#ifndef ASTRO_SPH_B200_H
#define ASTRO_SPH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AST_ABI_VERSION 1
#define AST_MAX_PROPS 2          /* weight fields deposited in one pass (mass and mass*T for config 2) */
#define AST_TILE 32              /* screen tile edge in pixels (tile key = tx * ceil(ny/32) + ty) */
#define AST_BRICK 8              /* voxel brick edge for the 3-D grid (brick key = (bx*nby + by)*nbz + bz) */

typedef enum ast_status {
    AST_OK = 0,
    AST_EINVAL = 1,              /* bad argument (shape, axis, kernel id, null pointer) */
    AST_EWORKSPACE = 2,          /* workspace or a capacity is too small; see ast_last_error() */
    AST_ECUDA = 3,               /* a CUDA runtime call or kernel launch failed */
    AST_EUNSUPPORTED = 4
} ast_status;

/* SPH kernels W(r,h); all have support r < 2h, the reference's hard mask (_pixel_calculations.pyx:31). */
typedef enum ast_kernel {
    AST_KERNEL_CUBIC_SPLINE_3D = 0,   /* the reference's `quartic_spline_kernel` (tools/projections/_kernels.pyx:9-20):
                                         M4 cubic spline, 1/(pi h^3) normalisation */
    AST_KERNEL_WENDLAND_C2_2D = 1,    /* 7/(pi H^2) (1-u)^4 (1+4u), u = r/H, H = 2h  (surface density) */
    AST_KERNEL_WENDLAND_C2_3D = 2,    /* 21/(2 pi H^3) (1-u)^4 (1+4u) */
    AST_KERNEL_CUBIC_SPLINE_2D = 3,   /* M4 cubic spline with 10/(7 pi h^2) */
    AST_KERNEL_TABLE = 4              /* W(r,h) = f(r/h) / h^kernel_dim with f tabulated by the caller on q in [0,2]: this is
                                         how an arbitrary `kernel_func` callable of the reference (_projector.py:86) is served */
} ast_kernel;

enum {
    AST_FLAG_PERIODIC = 1,       /* deposit the 9 (2-D) / 27 (3-D) periodic images, shifts ia*box_a etc. */
    AST_FLAG_ACCUMULATE = 2,     /* add to `out` instead of zeroing it first */
    AST_FLAG_TIMING = 4,         /* record CUDA events around every stage and return stage_ms (synchronises) */
    AST_FLAG_ORDER_AUTO = 8,     /* look at a sample of consecutive particles; if they are far apart in space (an incoherent input
                                    order) sort the particles by the tile / brick of their own position first and run on the copy
                                    (one more stream synchronisation, workspace grows by ~64 bytes per particle) */
    AST_FLAG_ORDER_ALWAYS = 16   /* pre-order without looking */
};

/* ---- 2-D line-of-sight projection ------------------------------------------------------------------
 * Replaces create_image / process_chunk / calculate_pixel_value
 * (tools/projections/_projector.py:75-120, :13-73, _pixel_calculations.pyx:9-36):
 *   out[p][xi][yi] = sum_i prop_p[i] * W(sqrt(r2), h_i)  over  r2 = (pa - X)^2 + (pb - Y)^2 < (2 h_i)^2
 *   X = x_min + xi*(x_max-x_min)/nx, Y = y_min + yi*(y_max-y_min)/ny   (pixel LOWER corner)
 *   (pa, pb) = position columns (1,2) / (0,2) / (0,1) for axis 0 / 1 / 2. */
typedef struct ast_project2d_params {
    int64_t n;                   /* particles */
    int32_t axis;                /* 0 = X, 1 = Y, 2 = Z  (CoordinateAxes, _CoordinateAxes.py:7-9) */
    int32_t nx, ny;              /* image_size */
    int32_t kernel_id;           /* ast_kernel */
    int32_t n_prop;              /* 1..AST_MAX_PROPS weight arrays -> that many maps */
    int32_t flags;
    double x_min, x_max, y_min, y_max;
    double box_a, box_b;         /* periodic lengths along the two in-plane axes (AST_FLAG_PERIODIC) */
    int64_t small_max_px;        /* bbox area (pixels) up to which a particle is deposited directly; <0 = default */
    int64_t huge_min_tiles;      /* tile-bbox count above which a particle image goes on the large-h list and is split across its
                                    tiles by a warp of its own (huge_tiles_kernel); <0 = default */
    int64_t pair_capacity;       /* WINDOW of (tile, particle) pairs the workspace holds; more pairs take more rounds */
    int64_t huge_capacity;       /* WINDOW of large-h list entries; a longer list is walked window by window */
    const float *kernel_table;   /* AST_KERNEL_TABLE: DEVICE array of 2*kernel_table_n floats, entry j = {f(q_j), f(q_j+1)-f(q_j)},
                                    q_j = 2j/kernel_table_n; linear interpolation, 0 for q >= 2 */
    int32_t kernel_table_n;      /* number of intervals */
    int32_t kernel_dim;          /* 2 or 3: the power of h in the normalisation */
} ast_project2d_params;

typedef struct ast_project2d_stats {
    int64_t n_pairs;             /* (tile, particle-image) pairs emitted, those of the large-h list included */
    int64_t n_huge;              /* particle-images on the large-h list */
    int64_t n_rounds;            /* passes over the pair window (1 unless pair_capacity < n_pairs or huge_capacity < n_huge) */
    int64_t n_launches;          /* kernels launched by this call */
    float stage_ms[8];           /* AST_FLAG_TIMING: 0 bin+direct deposit, 1 scan, 2 emit, 3 sort, 4 tile ranges / pair records,
                                    5 tile accumulate, 6 pre-ordering + memset, 7 total */
    int32_t reordered;           /* 1: the particles were pre-ordered (AST_FLAG_ORDER_AUTO found the input incoherent, or _ALWAYS) */
    int32_t reserved;
} ast_project2d_stats;

int ast_project2d_workspace_bytes(const ast_project2d_params *p, size_t *bytes /* host */);

/* prop: HOST array of n_prop DEVICE pointers.  out: n_prop*nx*ny doubles.  stats: host, nullable.
 * Synchronises the stream once after the binning kernel (a 16-byte read of the pair / large-h totals; when both are zero
 * the call ends there) and once more per large-h window.  pair_capacity and huge_capacity are windows: no value > 0 can
 * make the call fail, and nothing is deposited twice.  The one AST_EWORKSPACE that can be returned AFTER `out` has been
 * written to (the direct deposits of the binning kernel) is pair_capacity <= 0 with particles that need the tile path.
 * Weights are float64 and keep float64 range, also when one call mixes weights far apart (the tile path stores mantissa +
 * exponent and sums in exponent bands of 100 binary orders, each in units of its largest power of two, scaled back in
 * float64). */
int ast_project2d(const ast_project2d_params *p, const double *pos, const double *h,
                  const double *const *prop, double *out, void *workspace, size_t workspace_bytes,
                  void *stream, ast_project2d_stats *stats);

/* ---- index work, exposed for the bit-exact parity tests (no reference symbol: the reference is a gather;
 * the definitions follow _pixel_calculations.pyx:11-14,30-31, see DESIGN.md "Index work") ------------
 * bbox: n_img*N*4 int32 (x0,x1,y0,y1 inclusive; empty = 0,-1,0,-1), row j = m*N + i.
 * cls:  n_img*N uint8 (0 empty, 1 direct, 2 tiled, 3 global list).
 * pairs_emit / pairs_sorted: pair_capacity uint64 each, element = (sort_key << 32) | particle,
 *   sort_key = tile_key * (periodic ? 16 : 1) + image; the tiled pairs in emit order (particle, image, tx, ty ascending)
 *   are followed by the pairs of the large-h entries (entry by entry in list order, tiles tx-then-ty ascending).
 *   huge: huge_capacity uint64 = (image << 32) | particle.
 * counts (host): [0] pairs (large-h pairs included), [1] large-h entries.  Any output pointer may be null.  Synchronises.
 * Here the capacities ARE limits (AST_EWORKSPACE when the caller's arrays are too small); no map is touched. */
int ast_bin2d(const ast_project2d_params *p, const double *pos, const double *h,
              int32_t *bbox, uint8_t *cls, uint64_t *pairs_emit, uint64_t *pairs_sorted, uint64_t *huge,
              int64_t *counts, void *workspace, size_t workspace_bytes, void *stream);

/* exact contributor count per pixel: the reference mask r2 < (2h)^2 in float64 (int32 map nx*ny) */
int ast_contrib_count2d(const ast_project2d_params *p, const double *pos, const double *h, int32_t *count,
                        void *stream);

/* ---- SPH kernel evaluation, replaces quartic_spline_kernel(double[:] r, double[:] h)
 * (tools/projections/_kernels.pyx:9-20) for any ast_kernel, float64 ------------------------------- */
int ast_kernel_eval(int kernel_id, const double *r, const double *h, double *out, int64_t n, void *stream);

/* ---- device radix sort of 64-bit elements by bits [bit_lo, bit_lo+n_bits), stable.  keys and tmp hold n
 * elements; *result_in_tmp (host) tells which buffer has the result.  Exposed for tests. */
int ast_sort_workspace_bytes(int64_t n, size_t *bytes);
int ast_radix_sort_u64(uint64_t *keys, uint64_t *tmp, int64_t n, int bit_lo, int n_bits, void *workspace,
                       size_t workspace_bytes, void *stream, int *result_in_tmp);

/* ---- 3-D voxel gridding (EXTENSION named by BASELINE.json; no reference function; same rules as 2-D:
 * voxel lower-corner sample, r2 = (dx^2+dy^2)+dz^2 < (2h)^2) -------------------------------------- */
typedef struct ast_grid3d_params {
    int64_t n;
    int32_t nx, ny, nz;
    int32_t kernel_id;
    int32_t flags;
    int32_t reserved;
    double lo[3], hi[3];
    double box[3];
    int64_t small_max_vox;       /* bbox volume up to which a particle is deposited directly; <0 = default */
    int64_t huge_min_bricks;     /* brick-bbox count above which a particle image goes on the large-h list and is split across its
                                    bricks by a warp of its own (huge_bricks_kernel); <0 = default */
    int64_t pair_capacity;       /* WINDOW of (brick, particle) pairs, as in ast_project2d_params */
    int64_t huge_capacity;       /* WINDOW of large-h list entries */
    const float *kernel_table;   /* as in ast_project2d_params */
    int32_t kernel_table_n;
    int32_t kernel_dim;
    /* x window: compute planes [x_begin, x_end) of the nx-plane grid only; out holds (x_end - x_begin)*ny*nz doubles,
     * plane x_begin first.  0, 0 = the whole grid.  Every voxel corner is the whole grid's (lo[0] + (x_begin + i)*d, d =
     * (hi[0] - lo[0])/nx), so a window's voxels have the same contributors, bit for bit, as in the whole-grid call; bricks
     * and bboxes are numbered from x_begin.  AST_EINVAL unless 0 <= x_begin < x_end <= nx (or both 0).  Appended at the
     * end of the struct: every earlier field keeps its offset, so the ABI version is unchanged. */
    int32_t x_begin, x_end;
} ast_grid3d_params;

int ast_grid3d_workspace_bytes(const ast_grid3d_params *p, size_t *bytes);
int ast_grid3d(const ast_grid3d_params *p, const double *pos, const double *h, const double *prop,
               double *out, void *workspace, size_t workspace_bytes, void *stream, ast_project2d_stats *stats);

/* 3-D index work for the bit-exact parity tests: bbox n_img*N*6 int32 (x0,x1,y0,y1,z0,z1), cls n_img*N uint8,
 * pairs_sorted pair_capacity uint64 = (sort_key << 32) | particle with sort_key = brick_key * (periodic ? 32 : 1) + image,
 * brick_key = (bx*nby + by)*nbz + bz, sorted (stably) by brick_key only; the tiled pairs are followed by the member bricks
 * of the large-h entries (list order; bx, by, bz ascending); huge = (image << 32) | particle; counts (host) = {pairs (large-h
 * pairs included), large-h entries}.  Here the capacities are limits.  Synchronises.  With an x window the bboxes are the
 * whole grid's clipped to the window and shifted by -x_begin (empty when the x range misses the window), and classes,
 * pairs and the large-h list follow from those bboxes and the window's bricks. */
int ast_bin3d(const ast_grid3d_params *p, const double *pos, const double *h, int32_t *bbox, uint8_t *cls,
              uint64_t *pairs_sorted, uint64_t *huge, int64_t *counts, void *workspace, size_t workspace_bytes,
              void *stream);

/* ---- smoothing lengths by k nearest neighbours, replaces the KDTree branch of
 * SnapshotSWIFT.get_smoothing_lengths (io/SWIFT/_SnapshotSWIFT.py:62-83):
 *   h_out[i] = K-th smallest sqrt((dx*dx+dy*dy)+dz*dz) over all particles j, i itself included;
 *   box > 0: each delta is first wrapped by -+box when |delta| > box/2 (scipy boxsize semantics) and
 *   positions must satisfy 0 <= x < box.  idx_out (nullable): N*k int32 neighbour indices, ascending
 *   (distance, index).  dist_out (nullable): N*k float64.  Positions must lie in [lo, hi] per axis (open
 *   box) -- the cell grid is built over that extent. */
/* flags: by default the h-only call (idx_out == dist_out == NULL) runs the selection kernel (csrc/knn_select.cuh: CTA per block
 * of cells, float32 histogram + exact float64 band) and hands the queries it cannot verify to the lock-step kernel, in which
 * the 32 queries of a warp walk their ring traversals together; calls that want neighbour lists take the lock-step kernel.
 * AST_KNN_NO_SELECT: lock-step kernel alone.  AST_KNN_DIVERGING: the first query kernel (every thread walks its traversal on
 * its own).  All give the same bits (tuning / tests).  AST_KNN_FULL_BUILD: with a query subset, build the cell list from ALL
 * particles instead of those within reach of the queries. */
enum { AST_KNN_DIVERGING = 1, AST_KNN_FULL_BUILD = 4, AST_KNN_NO_SELECT = 8 };
typedef struct ast_knn_params {
    int64_t n;
    int32_t k;
    int32_t flags;
    double box;                  /* > 0: periodic cube [0, box)^3 ; <= 0: open */
    double lo[3], hi[3];         /* extent of the positions (open box); ignored when periodic */
    double cell_target;          /* mean particles per cell; <= 0 = default (1.75) */
    int64_t q_begin, q_count;    /* queries = particles [q_begin, q_begin + q_count); q_count <= 0 = all.  Multi-GPU:
                                    every rank holds all positions and answers its own slice of the queries.
                                    h_out / idx_out / dist_out hold q_count rows, row = particle - q_begin. */
} ast_knn_params;

int ast_knn_workspace_bytes(const ast_knn_params *p, size_t *bytes);
int ast_knn_h(const ast_knn_params *p, const double *pos, double *h_out, int32_t *idx_out, double *dist_out,
              void *workspace, size_t workspace_bytes, void *stream);

/* k nearest DATA points (p->n of them, cell list built over them; p->lo/hi = their extent, or p->box) of each of n_query
 * separate QUERY points: replaces KDTree(centres, boxsize=L).query(particles[, k]) of the nearest-halo script
 * (_scripts/find_nearest_haloes.py:207-215).  dist_out / idx_out: n_query*k, ascending (distance, index); either may be
 * null.  Same arithmetic as ast_knn_h (bit-equal to scipy).  Workspace: ast_knn_workspace_bytes(p). */
int ast_knn_query(const ast_knn_params *p, const double *data_pos, const double *query_pos, int64_t n_query,
                  double *dist_out, int32_t *idx_out, void *workspace, size_t workspace_bytes, void *stream);

/* ---- particle-ID matching (SURVEY 8(f) N4), replaces the sort / intersect1d / searchsorted arithmetic of the reference's
 * ArrayReorder family (tools/_ArrayReorder.py:744-768, :988-1038; used at io/EAGLE/_CatalogueSUBFIND.py:292-295):
 * source_index_of_target[j] = index i of the source ID equal to target_ids[j] (smallest i if the source repeats an ID),
 * or -1 (no match, or filtered out).  Filters (nullable): uint8 masks, 0 = the element does not take part.
 * INT64_MIN is reserved.  All pointers are device pointers. */
int ast_match_ids_workspace_bytes(int64_t n_source, size_t *bytes);
int ast_match_ids(const int64_t *source_ids, int64_t n_source, const uint8_t *source_filter, const int64_t *target_ids,
                  int64_t n_target, const uint8_t *target_filter, int64_t *source_index_of_target, void *workspace,
                  size_t workspace_bytes, void *stream);
/* out[j] = src[index[j]] for rows of row_bytes bytes where index[j] >= 0 (other rows untouched): applies a matching */
int ast_gather_rows(const void *src, int64_t row_bytes, const int64_t *index, int64_t n_out, void *out, void *stream);

/* ---- N-D linear table interpolation and fused per-particle weights (SURVEY 8(f) N3), replaces
 * IonisationTableBase.__call__ / evaluate_at_redshift (data_structures/_IonisationTable.py:44-58: scipy
 * RegularGridInterpolator, method "linear", bounds_error=False, fill_value=-inf; HM01 tables loaded at
 * io/ionisation_tables/_HM01.py:73-97).  Bit-equal to scipy in float64.  Coordinates come as one device pointer and element
 * stride per dimension, so an (N,ndim) row-major gas_state (x_cols[d] = gas_state + d, stride ndim) and separate
 * per-particle arrays (stride 1) are both served without a copy; dimension `fixed_dim` (>= 0) takes `fixed_value` for every
 * point (evaluate_at_redshift).  out[i] = value, or 10^value with AST_TABLE_POW10, times base[i] when base is not null
 * (element mass x ion fraction = the weight array of an ion column-density map; outside the table 10^-inf = 0). */
#define AST_TABLE_MAX_DIM 4
enum { AST_TABLE_POW10 = 1 };
typedef struct ast_table_params {
    int32_t ndim;                              /* 1..AST_TABLE_MAX_DIM */
    int32_t shape[AST_TABLE_MAX_DIM];          /* grid points per dimension, each >= 2 */
    const double *axes[AST_TABLE_MAX_DIM];     /* device: ascending grid coordinates of each dimension */
    const double *table;                       /* device: values, C order (dimension 0 slowest) */
    double fill_value;                         /* result outside the grid (the reference uses -inf) */
    int32_t fixed_dim;                         /* -1, or the dimension held at fixed_value */
    int32_t flags;                             /* AST_TABLE_POW10 */
    double fixed_value;
} ast_table_params;
int ast_table_interp(const ast_table_params *t, const double *const *x_cols /* host array of ndim device pointers */,
                     const int64_t *x_strides /* host, in elements */, int64_t n, const double *base /* nullable */,
                     double *out, void *stream);

/* ---- multi-GPU k-NN exchange (SURVEY 8(e): slabs along x + ghost zones): packing of the send buffer.  Rank g owns
 * x in [bounds[g], bounds[g+1]); `owner[i]` is the owning rank of local particle i (decided on the bins of a global histogram so
 * that every rank derives the same owner); a particle also goes, as a ghost, to every other rank whose slab lies within `w`
 * of it (distance along the circle of circumference `length` from bounds[0] when `periodic`; every rank when `covers_all`).
 * ast_slab_route_count fills counts[0..world) = owned rows per destination and counts[world..2 world) = ghost rows per
 * destination (device, int64) and leaves the scanned block table in the workspace; ast_slab_route_write (same params, same
 * workspace, after the count) writes the send buffer  [owned -> 0 | owned -> 1 | ... | ghosts -> 0 | ghosts -> 1 | ...]
 * (rows of 3 doubles, ascending particle index inside each piece) and src_index[row] = local particle index.
 * The per-rank particle split is the reference's io/EAGLE/_SnapshotEAGLE.py:120-130; the search itself is ast_knn_h. */
#define AST_ROUTE_MAX_WORLD 32
typedef struct ast_slab_route_params {
    int64_t n;
    int32_t world, periodic, covers_all, reserved;
    double length, w;
    double bounds[AST_ROUTE_MAX_WORLD + 1];
} ast_slab_route_params;
int ast_slab_route_workspace_bytes(const ast_slab_route_params *p, size_t *bytes);
int ast_slab_route_count(const ast_slab_route_params *p, const double *pos, const int64_t *owner, int64_t *counts,
                         void *workspace, size_t workspace_bytes, void *stream);
int ast_slab_route_write(const ast_slab_route_params *p, const double *pos, const int64_t *owner, double *send,
                         int64_t *src_index, void *workspace, size_t workspace_bytes, void *stream);

/* ---- multi-GPU 3-D gridding: routing of particles to x-slabs of the grid.  Rank g owns planes [e[g], e[g+1]) of the
 * whole grid (lo, hi, nx, ny, nz; box when periodic); particle i goes to rank g iff some periodic image of it (the particle
 * itself when not periodic) has a non-empty contributor range on the whole grid's x axis that meets [e[g], e[g+1]), and
 * some image has a non-empty range on y and on z: exactly the particles that ast_grid3d with that x window would deposit
 * (same ranges, same float64 arithmetic).  ast_grid_route_count fills counts[0..world) (device, int64) and leaves the
 * scanned block table in the workspace; ast_grid_route_write (same params, same workspace, after the count) writes rows
 * (x, y, z, h, prop) of 5 doubles, [-> rank 0 | -> rank 1 | ...], ascending particle index inside each piece.  send_rows
 * is the number of rows `send` holds (the counted total): a row beyond it is not written and sets *overflow (device int32,
 * zeroed by the call) to 1. */
typedef struct ast_grid_route_params {
    int64_t n;
    int32_t world, periodic;
    int32_t nx, ny, nz, reserved;
    double lo[3], hi[3], box[3];
    int32_t edges[AST_ROUTE_MAX_WORLD + 1];   /* plane edges e[0..world], non-decreasing, e[0] >= 0, e[world] <= nx */
} ast_grid_route_params;
int ast_grid_route_workspace_bytes(const ast_grid_route_params *p, size_t *bytes);
int ast_grid_route_count(const ast_grid_route_params *p, const double *pos, const double *h, int64_t *counts,
                         void *workspace, size_t workspace_bytes, void *stream);
int ast_grid_route_write(const ast_grid_route_params *p, const double *pos, const double *h, const double *prop,
                         double *send, int64_t send_rows, int32_t *overflow, void *workspace, size_t workspace_bytes,
                         void *stream);

/* ---- misc ---- */
const char *ast_last_error(void);
int ast_abi_version(void);
int ast_tile_size(void);
int ast_device_sm_count(int *sm_count /* host */);

#ifdef __cplusplus
}
#endif
#endif /* ASTRO_SPH_B200_H */
