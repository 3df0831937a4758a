/*
 * liboctreelib_b200 -- C ABI of the B200-native octreelib grid pipeline.
 *
 * The reference (prime-slam/octreelib) is pure Python and has no FFI of its own; its "operator
 * interface" for this path is the Python class surface.  Every entry point below is what a
 * binding of that surface needs, and names the reference code it replaces (paths relative to the
 * reference repository root).  The Python host in `octreelib_b200/` binds these with ctypes; a
 * reference maintainer would add the same stubs (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; every function returns an ol_status (0 = OK); ol_last_error() gives the
 *     message of the last failure on the calling thread.
 *   - one forest handle = one CUDA device + one stream + one caller thread.
 *   - device memory comes from the caller's allocator callbacks (the Python binding passes
 *     torch's caching allocator); with NULL callbacks the library uses cudaMallocAsync.
 *   - `*_host` pointers are host memory, `*_dev` pointers are device memory on the forest's device.
 *   - poses are identified by a dense "pose index" = order of insertion (0, 1, 2, ...); the host
 *     keeps the user's pose-number <-> index map.
 */
#ifndef OCTREELIB_B200_H
#define OCTREELIB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OL_ABI_VERSION 2
#define OL_MAX_DEPTH 21 /* 3 * 21 = 63 Morton bits */

typedef enum ol_status {
    OL_OK = 0,
    OL_ERR_INVALID = 1,     /* bad argument                         -> ValueError */
    OL_ERR_CUDA = 2,        /* CUDA runtime failure                 -> RuntimeError */
    OL_ERR_ALLOC = 3,       /* allocator callback failed            -> MemoryError */
    OL_ERR_RANGE = 4,       /* cell coordinates do not fit the key  -> ValueError */
    OL_ERR_OUT_OF_NODE = 5, /* octree/octree.py:98 IndexError       -> IndexError */
    OL_ERR_DEPTH_CAP = 6,   /* reference would recurse deeper       -> RecursionError */
    OL_ERR_NONFINITE = 7,   /* NaN / inf input                      -> ValueError */
    OL_ERR_STATE = 8,       /* call not valid in the current state  -> RuntimeError */
    OL_ERR_POSE = 9,        /* unknown pose index                   -> KeyError */
    OL_ERR_INTERNAL = 10,   /* self-check failed (RANSAC verify)    -> AssertionError */
    OL_ERR_CAPACITY = 11,   /* exchange receive buffer too small    -> the host binding grows it and retries */
    OL_ERR_UNSUPPORTED = 12 /* result the grid cannot represent     -> NotImplementedError */
} ol_status;

typedef void *(*ol_alloc_fn)(void *user, size_t bytes);
typedef void (*ol_free_fn)(void *user, void *ptr);

typedef struct ol_forest ol_forest; /* opaque: a Grid (many cells) or one OctreeManager cell */

typedef struct ol_forest_config {
    double voxel_edge_length; /* GridConfig.voxel_edge_length, grid/grid_base.py:70 */
    double corner[3];         /* GridConfig.corner, grid/grid_base.py:71; single_cell: corner_min */
    int32_t single_cell;      /* 1 = one fixed cell (OctreeManager / Octree used directly,
                                 octree_manager/octree_manager.py:21-34): no cell hashing */
    int32_t max_depth;        /* octree depth cap, 1..OL_MAX_DEPTH (reference: unbounded) */
    int32_t device;           /* CUDA device ordinal */
    int32_t reserved;
    void *stream;             /* cudaStream_t all work is enqueued on */
    ol_alloc_fn alloc;        /* device allocator callbacks (may be NULL) */
    ol_free_fn free;
    void *alloc_user;
} ol_forest_config;

typedef struct ol_forest_stats {
    int64_t n_points_inserted; /* all points ever inserted */
    int64_t n_points_alive;    /* after filter / RANSAC masks */
    int64_t n_poses;
    int64_t n_cells;
    int64_t n_cell_poses;  /* (cell, pose) pairs that own an octree (-1 from ol_forest_stats_light while not built) */
    int64_t n_leaves;      /* leaves of the shared per-cell tree shape, empty ones included */
    int64_t n_internal;    /* internal (split) nodes */
    int64_t n_blocks;      /* non-empty (pose, leaf) pairs = RANSAC blocks */
    int64_t max_block_size;
    int64_t max_depth_reached;
    int64_t key_bits;      /* significant bits of the packed cell key */
    int64_t device_bytes_peak;
    int64_t sample_oob_seen; /* 1 if a RANSAC sample index int32(R*n + start) ever fell outside its block (it is clamped
                                into the block; the reference, ransac/cuda_ransac.py:104-107, would read a neighbouring
                                block's point there).  bench.py asserts 0. */
} ol_forest_stats;

/* ---- library ------------------------------------------------------------------------------ */
int ol_abi_version(void);
const char *ol_last_error(void);

/* ---- forest lifetime ------------------------------------------------------------------------ */
/* Grid.__init__ (grid/grid.py:49-56) / OctreeManager.__init__ (octree_manager.py:21-34) */
int ol_forest_create(const ol_forest_config *config, ol_forest **out);
int ol_forest_destroy(ol_forest *f);

/* ---- Grid.insert_points, grid/grid.py:58-109 ------------------------------------------------
 * Appends one pose's cloud ([n][3] float64, host or device memory).  Returns the new pose index.
 * The re-insert ValueError (grid.py:65-66) is raised by the host, which owns pose numbers.
 * Pageable host sources are consumed before the call returns; a PAGE-LOCKED host source and a DEVICE source are read
 * asynchronously on the forest's stream and must stay unchanged until that work has run (any call that returns results
 * has waited for it; memory recycled in stream order on the same stream - torch's caching allocator - is safe). */
int ol_forest_insert(ol_forest *f, const double *xyz, int64_t n, int32_t src_on_device, int32_t *out_pose_index);

/* The same for `count` DEVICE-resident clouds at once (a host array of device pointers and their point counts): every
 * cloud becomes one new pose, in order; *out_first_pose_index = index of the first.  One exact growth of the point
 * array and one copy kernel instead of a driver call per pose - the Python host defers `insert_points` of CUDA tensors
 * into such a batch and flushes it before the next grid operation. */
int ol_forest_insert_batch(ol_forest *f, const double *const *xyz_dev_ptrs_host, const int64_t *sizes_host, int32_t count,
                           int32_t *out_first_pose_index);

/* Multi-GPU form: the cloud is a concatenation of `n_segments` runs, run s holding
 * `seg_sizes[s]` points of pose index `seg_pose[s]` whose first point has index `seg_first[s]`
 * inside that pose's original cloud (what an all-to-all delivers: one run per (source rank, pose)).
 * Pose indices may repeat and need not be dense; `n_poses_total` fixes the pose count. */
int ol_forest_insert_segments(ol_forest *f, const double *xyz, int64_t n, int32_t src_on_device,
                              const int64_t *seg_sizes, const int32_t *seg_pose, const int64_t *seg_first,
                              int32_t n_segments, int32_t n_poses_total);

/* ---- Grid.subdivide, grid/grid.py:244-258 -> OctreeManager.subdivide, octree_manager.py:36-66 --
 * Level-synchronous split of every cell: a node splits iff (#points of the listed poses inside it)
 * > max_points (criterion `len(points) > max_points`, octree/octree.py:26).  n_poses == 0 means
 * "all poses of the cell" (octree_manager.py:46-47).  The shape is imposed on every pose. */
int ol_forest_subdivide(ol_forest *f, int64_t max_points, const int32_t *pose_indices, int32_t n_poses);

/* Same, but the per-node decision comes from a count -> {0,1} table (an arbitrary count-only
 * criterion list folded by the host); counts >= table_len use split_beyond. */
int ol_forest_subdivide_table(ol_forest *f, const uint8_t *split_table_host, int64_t table_len, int32_t split_beyond,
                              const int32_t *pose_indices, int32_t n_poses);

/* Size thresholds (BASELINE north_star: "splitting by point-count and size thresholds").  The reference's criteria see
 * only the points (octree/octree.py:26), so a node-size limit is a property of the criterion OBJECT
 * (octreelib_b200/criteria.py: MaxPoints(n, max_depth=, min_edge=), MaxDepth, MinEdge); the host folds a criterion list
 * into a rule that is piecewise constant in the octree level: entry e applies to the levels
 * [first_level[e], first_level[e + 1]) (first_level[0] == 0, ascending; the last entry applies to every deeper level).
 * Threshold form: level_max_points[e] (a node splits iff count > it; 1 << 62 = never); table form (split_tables_host !=
 * NULL): split_tables_host[e][count] with split_beyond[e] for counts >= table_len. */
int ol_forest_subdivide_levels(ol_forest *f, const int32_t *first_level, int32_t n_entries, const int64_t *level_max_points,
                               const uint8_t *split_tables_host, int64_t table_len, const int32_t *split_beyond,
                               const int32_t *pose_indices, int32_t n_poses);

/* Geometric criteria (octreelib_b200/criteria.py: MaxExtent, MaxThickness, Planar).  A term looks at the points a node
 * holds (the listed poses' points for a subdivision with pose indices), all in float64:
 *   extent    = max over the axes of (max coordinate - min coordinate), 0 for an empty node;
 *   thickness = sqrt(max(smallest eigenvalue of the population covariance, 0)), the RMS distance of the points from
 *               their least-squares plane; 0 for fewer than 3 points.
 * A term holds iff the node has at least min_points points and  stat > value (OL_GEOM_GT) / stat <= value (OL_GEOM_LE).
 * The reference evaluates such criteria per node in Python (octree/octree.py:26, :111). */
#define OL_GEOM_EXTENT 0
#define OL_GEOM_THICKNESS 1
#define OL_GEOM_GT 0
#define OL_GEOM_LE 1
#define OL_GEOM_MAX_TERMS 8 /* terms per rule entry */
typedef struct ol_geom_term {
    int32_t stat;       /* OL_GEOM_EXTENT / OL_GEOM_THICKNESS */
    int32_t op;         /* OL_GEOM_GT / OL_GEOM_LE */
    int64_t min_points; /* >= 0 */
    double value;       /* >= 0 */
} ol_geom_term;

/* Grid.subdivide with criteria that look at coordinates (octree/octree.py:20-32 with e.g. "split while not planar"):
 * the arguments of ol_forest_subdivide_levels plus, per entry e, n_terms[e] terms (at most OL_GEOM_MAX_TERMS) stored
 * back to back in `terms` (entry 0 first).  A node of a level of entry e splits iff the count rule says so OR one of
 * the entry's terms holds.  Counts as a subdivide call (the leaf order across calls, ol_forest_export_leaves). */
int ol_forest_subdivide_geometric(ol_forest *f, const int32_t *first_level, int32_t n_entries, const int64_t *level_max_points,
                                  const uint8_t *split_tables_host, int64_t table_len, const int32_t *split_beyond,
                                  const ol_geom_term *terms, const int32_t *n_terms, const int32_t *pose_indices,
                                  int32_t n_poses);

/* ---- Grid.filter, grid/grid.py:260-267 -> octree/octree.py:102-112 --------------------------
 * A (pose, leaf) block of n points survives iff keep_table[min(n, table_len-1)] != 0; the tree
 * shape is unchanged.  n_poses == 0: all poses. */
int ol_forest_filter(ol_forest *f, const uint8_t *keep_table_host, int64_t table_len, const int32_t *pose_indices,
                     int32_t n_poses);
/* Same, with geometric terms (octree/octree.py:111, e.g. "keep planar leaves"): a block of a listed pose survives iff
 * the keep table says so AND all n_terms terms (at most OL_GEOM_MAX_TERMS) hold on its points. */
int ol_forest_filter_geometric(ol_forest *f, const uint8_t *keep_table_host, int64_t table_len, const ol_geom_term *terms,
                               int32_t n_terms, const int32_t *pose_indices, int32_t n_poses);

/* ---- Grid.map_leaf_points_cuda_ransac, grid/grid.py:124-215 ---------------------------------
 * table_host: [H][K] float64 uniform [0,1) hypothesis table (ransac/cuda_ransac.py:39-41).
 * pose_rank[p]: position of pose index p in the reference's batch order (= its pose number when
 * numbers are 0..P-1, grid.py:149-157).  With apply != 0 the inlier masks are applied
 * (grid.py:203-215); otherwise they are only stored for export.
 * pose_start (NULL for a forest that holds the whole grid): multi-GPU, slab partition - pose_start[p] = index, inside
 * its batch of the reference's layout (cuda_ransac.py:65-67), of the first point of pose index p that THIS forest holds
 * = (points of the batch's earlier poses on all ranks) + (points of pose p on the lower ranks); poses_per_batch is then
 * only informative.  The host derives it from one all-gather of ol_forest_pose_point_counts. */
int ol_forest_ransac(ol_forest *f, const double *table_host, int32_t H, int32_t K, double threshold,
                     const int32_t *pose_rank, int32_t poses_per_batch, int32_t apply, uint32_t flags,
                     const int64_t *pose_start);
/* out_host[p] = points currently stored for pose index p ([n_poses] int64) */
int ol_forest_pose_point_counts(ol_forest *f, int64_t *out_host);
/* applies the mask of the last ol_forest_ransac(apply = 0) call (grid.py:203-215) */
int ol_forest_apply_mask(ol_forest *f);

/* OctreeManager.apply_mask / Octree.apply_mask (octree_manager.py:173-180, octree/octree.py:265-274):
 * mask_host[n] covers the points of pose `pose_index` in the order of ol_forest_export_points(order 0);
 * points with mask 0 are removed. */
int ol_forest_apply_pose_mask(ol_forest *f, const int32_t *pose_rank, int32_t pose_index, const uint8_t *mask_host,
                              int64_t n);

/* ---- declarative leaf maps: Grid.map_leaf_points, grid.py:111-122 -> octree.py:114-123 ------------
 * (octreelib_b200/leaf_maps.py: Centroid, Shrink, FirstPoints).  Every non-empty (pose, leaf) block of the listed poses
 * (n_poses == 0: all poses) is mapped on the device, in float64, bit for bit like numpy on the block's points in
 * ol_forest_export_points(order 0) order:
 *   OL_MAP_CENTROID  the block becomes its mean, cloud.mean(axis=0) (sequential row sum / n);      param ignored
 *   OL_MAP_SHRINK    every point p becomes c + param * (p - c), c the block's mean, no FMA;         param finite
 *   OL_MAP_FIRST     the block keeps its first min(param, n) points (K7 compaction only);           param >= 0
 * A result that is a subsequence of the block's own rows (a centroid equal to one of its points, a shrink that changes
 * no point) keeps those rows, as the host path does with a callable.  Any other result replaces the block: its points
 * are removed, the new rows are appended to the pose (one segment per pose, continuing the pose's point indices) and the
 * grid is rebuilt with the same shape (scheme replay).  A new row outside the leaf it was computed from
 * (lo <= p < lo + edge per axis, non-finite fails) returns OL_ERR_UNSUPPORTED before anything changes; an appended row
 * that lands in another leaf after the rebuild returns OL_ERR_STATE.  rows_appended_host (NULL or [number of poses]
 * int64) receives the rows appended to every pose index. */
#define OL_MAP_CENTROID 0
#define OL_MAP_SHRINK 1
#define OL_MAP_FIRST 2
int ol_forest_map_leaves(ol_forest *f, int32_t op, double param, const int32_t *pose_indices, int32_t n_poses,
                         int64_t *rows_appended_host);

/* Octree.subdivide_as / OctreeNode.subdivide_as (octree/octree.py:34-53, 222-227): copy the subdivision scheme of one
 * octree onto another.  ol_forest_export_shape lists the split nodes of a forest (cell coordinates q[n][3], depth, Morton
 * path from the cell root: 3 bits per level); with NULL arrays only *out_n is written.  ol_forest_impose_shape makes
 * exactly the listed nodes the split nodes of the target (rebuilt from its cell roots the next time the shape is
 * needed): nodes the target lacks are split, nodes the list lacks are collapsed, points are re-routed; n = 0 collapses
 * every cell to one leaf.  Depth limit: 9 levels.  (The reference forgets to put a collapsed node back into its leaf
 * list, octree.py:48-53; this library keeps it, like the CPU oracle.) */
int ol_forest_export_shape(ol_forest *f, int64_t *q, uint32_t *depth, uint64_t *path, int64_t *out_n);
int ol_forest_impose_shape(ol_forest *f, const int64_t *q, const uint32_t *depth, const uint64_t *path, int64_t n);

/* ---- Grid.locate_points (no counterpart in the reference, whose only way is insert_points of a new pose) ----------
 * The leaf every query point would be routed into by inserting it as a new pose under the current scheme (grid.py:72-76
 * for the cell, octree.py:73-97 level by level for the path), without inserting it: nothing changes.  -1 where a
 * coordinate is not finite, the cell does not exist (cell coordinates outside the packed key range included), or the
 * point leaves its node above the leaf (insertion would raise IndexError, octree.py:98).
 * xyz[n][3] float64; on_device != 0: xyz and out are device pointers and the call is stream-ordered, else host
 * pointers and the call synchronises.  leaf_to_row (device, int32[L], may be NULL) maps a leaf-table index to the value
 * written (-1 stays -1); NULL writes the leaf-table index (ol_forest_export_leaves order). */
int ol_forest_locate(ol_forest *f, const double *xyz, int64_t n, int32_t on_device, const int32_t *leaf_to_row,
                     int64_t *out);

/* ---- measurement support (bench.py): per-stage CUDA-event timers on the forest's stream -------
 * ol_forest_profile(f, 1) clears and enables the timers; ol_forest_profile_read synchronises, writes
 * one line "stage_name launches total_ms" per stage into buf and clears the records.
 * ol_launch_count: kernels launched by this library in this process so far. */
int ol_forest_profile(ol_forest *f, int32_t enable);
int ol_forest_profile_read(ol_forest *f, char *buf, int64_t buf_len, int64_t *out_len);
uint64_t ol_launch_count(void);
/* Device blocks obtained through the allocator callbacks are kept in a process-wide cache when a forest (or a transient
 * call context) releases them, keyed by (callbacks, user pointer, stream), and are handed to the next forest on the same
 * stream - a pipeline step builds a fresh forest and would otherwise re-enter the host allocator ~30 times.  The cache
 * is bounded (environment OL_CACHE_BYTES, default a quarter of the device memory) and emptied on allocation failure.
 * ol_release_cached_memory returns every cached block through the free callback it came from (bytes released): call it
 * before tearing an allocator down.  The reference has no counterpart (numpy / numba manage their own memory). */
uint64_t ol_release_cached_memory(void);

/* ---- counters: Grid.n_leaves / n_points / n_nodes, grid/grid.py:343-362 ---------------------- */
int ol_forest_stats_get(ol_forest *f, ol_forest_stats *out);
/* same, but builds no derived table: n_blocks / max_block_size are -1 when the (pose, leaf) block table is stale
 * (after a filter / RANSAC mask); synchronises the stream, so it doubles as the step's completion point */
int ol_forest_stats_light(ol_forest *f, ol_forest_stats *out);
/* out[p] = {n_leaves, n_points, n_nodes} for pose index p, [n_poses][3] int64 */
int ol_forest_pose_counts(ol_forest *f, int64_t *out_host);

/* ---- exports (host buffers sized from ol_forest_stats_get; any pointer may be NULL) ----------
 * cells, lexicographic by signed (ix,iy,iz) (grid.py:79-81):
 *   q[C][3] integer cell coordinates, corner[C][3] float64 cell corner, first_pose[C] pose index
 *   that created the cell (dict order of grid.py:56), n_nodes[C] nodes of the cell's tree,
 *   leaf_begin[C+1] range of the cell's leaves in the leaf table below. */
int ol_forest_export_cells(ol_forest *f, int64_t *q, double *corner, int32_t *first_pose, int64_t *n_nodes,
                           int64_t *leaf_begin);
/* (cell, pose) pairs, sorted by (cell, pose index): which poses own an octree in which cell */
int ol_forest_export_cell_poses(ol_forest *f, int32_t *cell, int32_t *pose);
/* leaves in the reference's enumeration order (cells lexicographic, inside a cell the
 * `_cached_leaves` order of octree/octree_base.py:48-49 + octree/octree.py:183-191):
 *   corner[L][3], edge[L] (octree.py:181-187), cell[L], depth[L], parent_epoch[L] = number of the subdivide call that
 *   split the leaf's parent (0 for an unsplit cell root).
 * This is the order of a grid that was subdivided ONCE.  Every pose octree of the reference keeps its leaf list across
 * calls (octree_base.py:48-49, octree.py:183-191), so after a SECOND subdivide the order of pose p inside a cell is
 * (max(parent_epoch, number of calls made before p was inserted), order above): the block table below and everything
 * derived from it (point exports, RANSAC batch layout, apply_pose_mask) follow that order on the device; a caller that
 * enumerates EMPTY leaves too applies the same rule to this table. */
int ol_forest_export_leaves(ol_forest *f, double *corner, double *edge, int32_t *cell, int32_t *depth, int32_t *parent_epoch);
/* non-empty (pose, leaf) blocks in the order Grid.get_leaf_points / the RANSAC batches use
 * (pose rank, then the reference's leaf order for that pose):  pose[B], leaf[B] (index into the leaf table), size[B]. */
int ol_forest_export_blocks(ol_forest *f, const int32_t *pose_rank, int32_t *pose, int32_t *leaf, int32_t *size);
/* Point statistics of the same blocks, in the same order, for one pose (pose_index >= 0) or all (-1): what a plane-based
 * back end reads instead of reducing Grid.get_leaf_points(...)[i].get_points() (grid.py:217-232) leaf by leaf.  Per row:
 * pose[B], n[B], mean[B][3], cov[B][6] (population covariance xx, xy, xz, yy, yz, zz), extent[B][3] (max - min per axis).
 * *out_n = number of rows; with every array NULL only *out_n is written. */
int ol_forest_export_block_stats(ol_forest *f, const int32_t *pose_rank, int32_t pose_index, int32_t *pose, int64_t *n,
                                 double *mean, double *cov, double *extent, int64_t *out_n);
/* the block table as it was when ol_forest_ransac last ran (before the masks were applied), same
 * order, plus per block: plane[B][4] float32, best[B] (hypothesis index, -1 = skipped because the
 * block has fewer than K points, ransac/cuda_ransac.py:96-97), best_count[B] (its inlier count).
 * scored_only != 0 keeps only the fitted blocks (best >= 0).
 * *out_n = number of rows (pass NULL arrays first to size the buffers). */
int ol_forest_export_ransac(ol_forest *f, int32_t scored_only, int32_t *pose, int32_t *leaf, int32_t *size, float *plane,
                            int32_t *best, int32_t *best_count, int64_t *out_n);
/* points of one pose (pose_index >= 0) or of all poses (-1, pose-rank-major):
 *   order 0: block order of ol_forest_export_blocks, original input order inside a block
 *   order 1: cells lexicographic, depth-first leaf order inside a cell (octree.py:55-65)
 * xyz[n][3] float64, idx[n] index of the point in its pose's inserted cloud, cell[n] cell index,
 * mask[n] last RANSAC inlier mask (order 0 only, before it was applied). */
int ol_forest_export_points(ol_forest *f, const int32_t *pose_rank, int32_t pose_index, int32_t order, double *xyz,
                            int64_t *idx, int32_t *cell, uint8_t *mask, int64_t *out_n);

/* ---- CudaRansac.evaluate, ransac/cuda_ransac.py:43-81 (kernel-level boundary) ----------------
 * points_dev [n][3] float64, block_sizes_dev [B] int32 back to back, table_dev [H][K] float64;
 * outputs: mask_dev [n] uint8, plane_dev [B][4] float32, best_dev [B], best_count_dev [B]
 * (the three per-block outputs may be NULL).
 * flags: OL_RANSAC_NO_TMA      plain loads instead of TMA bulk staging
 *        OL_RANSAC_EXACT_ONLY  evaluate every hypothesis with the reference's float64 arithmetic (no FP32 pre-filter)
 *        OL_RANSAC_VERIFY      exact evaluation of everything + check that every count lies inside its pre-filter
 *                              interval (returns OL_ERR_INTERNAL if one does not)
 *        OL_RANSAC_STATS       accumulate pre-filter statistics (ol_ransac_stats_read)
 * All modes return identical results. */
#define OL_RANSAC_NO_TMA 1u
#define OL_RANSAC_EXACT_ONLY 2u
#define OL_RANSAC_VERIFY 4u
#define OL_RANSAC_STATS 8u
int ol_ransac_evaluate(void *stream, const double *points_dev, int64_t n, const int32_t *block_sizes_dev, int64_t B,
                       const double *table_dev, int32_t H, int32_t K, double threshold, uint8_t *mask_dev,
                       float *plane_dev, int32_t *best_dev, int32_t *best_count_dev, uint32_t flags,
                       ol_alloc_fn alloc, ol_free_fn free_fn, void *alloc_user);

/* what the RANSAC kernels executed since the last reset (OL_RANSAC_STATS / OL_RANSAC_VERIFY launches; device-wide
 * synchronisation): out[0] blocks, [1] hypotheses that went through the float32 pre-filter, [2] trivial intervals,
 * [3] exact evaluations of pre-filter candidates, [4] early exits, [5] interval violations (verify mode),
 * [6] exact float64 plane fits (util.py:28-84, ~152 flops each at K = 6), [7] exact float64 point-plane distance
 * evaluations (util.py:16-24, 6 flops each; the final mask pass included), [8] float32 distance evaluations of the
 * pre-filter (6 flops each) */
int ol_ransac_stats_read(uint64_t out[16], int32_t reset);

/* Measured arithmetic peaks of this GPU at its current clocks (dense FMA throughput, 2 flops per FMA, 8 independent chains
 * per thread): the roofline denominators of the RANSAC kernel, which is bound by the FP64 pipe (SURVEY.md 8(d): "the bench
 * must calibrate with an FMA microbenchmark at the observed clock").  Either pointer may be NULL.  Synchronises. */
int ol_measure_fma_peak(void *stream, double *out_fp64_tflops, double *out_fp32_tflops);

/* ---- multi-GPU routing (no counterpart in the single-process reference; SURVEY.md 8(e)) --------
 * A cell (all poses of it) is owned by ONE rank, a function of its cell coordinates:
 *   hash  (slab_bounds_host == NULL)  ol_host_cell_owner(ix, iy, iz, world)
 *   slab  (slab_bounds_host = world - 1 ascending cell-x boundaries)  owner = #{k : bound[k] <= ix}; order preserving, so
 *         the reference's lexicographic cell order (grid/grid.py:79-81) is the rank-major concatenation of the local ones
 *         and its batch-global block_start_indices (ransac/cuda_ransac.py:65-67) can be reproduced exactly across ranks
 *         (ol_forest_ransac: pose_start).  ol_slab_histogram gives every rank what it needs to pick the boundaries as
 *         count quantiles: out_dev = int64[2 + n_bins] {min ix, max ix, counts of n_bins equal-width bins over that
 *         range} of a 1-in-8 sample of the rank's points; enqueued on the stream, not synchronised.
 * ol_partition_by_owner reorders a rank's local cloud xyz_dev ([n][3] float64, a concatenation of
 * n_segments runs = poses) into out_xyz_dev grouped by owner rank, stable inside (owner, run), and
 * returns counts[owner][run] (host, int64) - the send layout of one all-to-all, the exchange of the multi-GPU grid where
 * ol_exchange_run cannot run (a backend other than NCCL, or no peer-mapped memory).  Synchronises. */
uint32_t ol_host_cell_owner(int64_t qx, int64_t qy, int64_t qz, uint32_t world);
int ol_slab_histogram(void *stream, const double *xyz_dev, int64_t n, double edge, double corner_x, int32_t n_bins,
                      int64_t *out_dev);
int ol_partition_by_owner(void *stream, const double *xyz_dev, int64_t n, const int64_t *seg_sizes_host, int32_t n_segments,
                          double edge, const double corner[3], int32_t world, const int64_t *slab_bounds_host,
                          double *out_xyz_dev, int64_t *out_counts_host, ol_alloc_fn alloc, ol_free_fn free_fn,
                          void *alloc_user);

/* ---- fused exchange over peer-mapped memory (csrc/exchange.cu) ----------------------------------------------------------
 * The production path of the multi-GPU grid when the ranks of a node can map each other's memory: owner rule, counting,
 * routing and the hand-over to the receiving forest in one call, with every inter-rank dependency resolved on the device
 * (flags in peer-mapped control blocks; no library collective, ONE host wait).  The host binding provides the memory:
 *   ctrl_ptrs_host[r]              control block of rank r mapped into THIS process, ol_exchange_ctrl_bytes(world, n_poses)
 *                                  bytes each, zero-filled once before the first exchange (all ranks, then a barrier);
 *   data_ptrs_host[b * world + r]  receive buffer b of rank r (rows_cap x 3 float64), n_buffers >= 1 of them so that a
 *                                  forest can keep using buffer b while the next exchange fills buffer b + 1.
 * ol_exchange_run is collective (every rank calls it with the same slabs / buffer): it routes the rank's local clouds
 * (clouds_dev_ptrs_host[k] = [sizes_host[k]][3] float64 on the device, pose numbers poses_host[k] ascending) and makes the
 * EMPTY forest f adopt receive buffer `buffer` as its point array: (source rank, pose) runs in the order the reference would
 * have seen the points of a pose when the ranks hold increasing index ranges of it.  The buffer must stay untouched until f is
 * destroyed or ol_forest_disown_points(f) copied the points out.  info_out[4] = rows sent to other ranks, rows received,
 * rows kept, largest receive total of any rank; bounds_out[world - 1] = the slab boundaries chosen (slabs != 0; count
 * quantiles of the leading cell coordinate, identical on every rank); pose_sizes_out[world][n_poses] (uint32) = rows of every
 * pose held by every rank afterwards (what the batch-global block starts of ol_forest_ransac's pose_start need).
 * Returns OL_ERR_CAPACITY (on every rank alike) when a rank would receive more than rows_cap rows: nothing was routed;
 * create a larger exchange and call again. */
typedef struct ol_exchange ol_exchange;
int64_t ol_exchange_ctrl_bytes(int32_t world, int32_t n_poses);
int ol_exchange_create(int32_t world, int32_t rank, int32_t n_poses, int64_t rows_cap, int32_t n_buffers,
                       void *const *ctrl_ptrs_host, void *const *data_ptrs_host, int32_t device, ol_exchange **out);
int ol_exchange_destroy(ol_exchange *x);
int ol_exchange_run(ol_exchange *x, ol_forest *f, const double *const *clouds_dev_ptrs_host, const int64_t *sizes_host,
                    const int32_t *poses_host, int32_t count, int32_t slabs, int32_t buffer, int64_t *info_out,
                    int64_t *bounds_out, uint32_t *pose_sizes_out);
/* copies an adopted point array into memory of the forest's own (no-op otherwise); synchronises */
int ol_forest_disown_points(ol_forest *f);

/* ---- primitives, exported so that tests can check them in isolation -------------------------- */
/* stable LSD radix sort of (key, value) pairs on bits [begin_bit, end_bit); result in keys_dev/vals_dev */
int ol_sort_pairs_u64(void *stream, uint64_t *keys_dev, uint32_t *vals_dev, int64_t n, int32_t begin_bit,
                      int32_t end_bit, ol_alloc_fn alloc, ol_free_fn free_fn, void *alloc_user);
int ol_sort_pairs_u32(void *stream, uint32_t *keys_dev, uint32_t *vals_dev, int64_t n, int32_t begin_bit,
                      int32_t end_bit, ol_alloc_fn alloc, ol_free_fn free_fn, void *alloc_user);
/* test hook: 1 = use the three-kernel LSD sort instead of onesweep (both must give identical results) */
int ol_debug_force_legacy_sort(int32_t on);
/* exclusive prefix sum, in place allowed; total written to *total_host if non-NULL (synchronises) */
int ol_exclusive_scan_u32(void *stream, const uint32_t *in_dev, uint32_t *out_dev, int64_t n, uint64_t *total_host,
                          ol_alloc_fn alloc, ol_free_fn free_fn, void *alloc_user);
/* host restatement of numpy's float64 floor_divide (grid.py:72-76), for CPU-side tests */
double ol_host_floor_divide(double a, double b);
/* cell coordinate + Morton code of one point exactly as the device computes them (CPU-side tests) */
int ol_host_point_key(double edge, const double corner[3], int32_t single_cell, int32_t depth, const double p[3],
                      int64_t q[3], uint64_t *morton, int32_t *bad_level);

#ifdef __cplusplus
}
#endif
#endif /* OCTREELIB_B200_H */
