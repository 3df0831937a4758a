// Declarative leaf maps of Grid.map_leaf_points (grid.py:111-122 -> octree.py:114-123) on the device: Centroid, Shrink and
// FirstPoints (octreelib_b200/leaf_maps.py).  Forest::map_leaves (forest_host2.inl) drives the passes below.
//
// The results must equal numpy's bit for bit.  For a C-contiguous (n, 3) float64 cloud, `cloud.mean(axis=0)` is the
// sequential sum of the rows in order, starting from +0.0, followed by one division by float64(n) (numpy does not sum
// pairwise along axis 0; tests/test_cpu_leaf_maps.py pins this).  A block's points sit at consecutive positions in the
// order export_points(order 0) hands them to the host function, so one thread per block reproduces the sum; the order
// is fixed, no tree reduction.  Shrink is c + factor * (p - c): three rounded operations per coordinate, no FMA
// (explicit __d*_rn intrinsics, and the library is built with -fmad=false anyway).
//
// The host path turns a result that is a subsequence of the block's own rows into a keep-mask instead of replacing the
// block (ForestHost._as_selection): a centroid that is bit-equal (==) to a row of its block keeps the first such row, and
// a shrink that leaves every row unchanged keeps the block as it is.  The passes reproduce that, and only blocks that
// are really replaced are checked against their leaf (lo <= p < lo + edge, per coordinate; a NaN fails).
#pragma once
#include "forest.cuh"

namespace ol {

constexpr uint32_t LEAF_MAP_NO_MATCH = 0xffffffffu;
constexpr int LEAF_MEAN_UNROLL = 8;

__device__ __forceinline__ bool leaf_map_mapped(const uint8_t* __restrict__ listed, const int32_t* __restrict__ blk_pose, uint32_t b) {
    return !listed || listed[blk_pose[b]];
}

// lo <= v < lo + edge on every axis, with the leaf geometry of K5 (depth-0 leaves: the cell corner, or the forest's
// corner for a single cell, and the voxel edge - exactly what the host path compares against)
__device__ __forceinline__ bool leaf_map_inside(const double v[3], const double* __restrict__ leaf_corner,
                                                const double* __restrict__ leaf_edge, uint32_t li) {
    const double e = leaf_edge[li];
    bool in = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double lo = leaf_corner[(size_t)li * 3 + a];
        in = in && v[a] >= lo && v[a] < __dadd_rn(lo, e);
    }
    return in;
}

__device__ __forceinline__ void leaf_shrink_row(const double p[3], const double c[3], double f, double out[3]) {
#pragma unroll
    for (int a = 0; a < 3; ++a) out[a] = __dadd_rn(c[a], __dmul_rn(f, __dsub_rn(p[a], c[a])));
}

// one thread per (listed) block: sequential float64 sum of the block's rows, then one division.  The loads of
// LEAF_MEAN_UNROLL rows are issued before their dependent adds.  check != 0 (Centroid): the mean itself is the
// replacement row and is checked against the leaf here.
__global__ void __launch_bounds__(256) leaf_mean_kernel(uint32_t nb, const uint32_t* __restrict__ blk_start,
                                                        const int32_t* __restrict__ blk_pose, const uint8_t* __restrict__ listed,
                                                        const uint32_t* __restrict__ perm, const double* __restrict__ xyz,
                                                        const uint32_t* __restrict__ blk_leaf, const uint32_t* __restrict__ cache_rank,
                                                        const double* __restrict__ leaf_corner, const double* __restrict__ leaf_edge,
                                                        int check, double* __restrict__ mean, uint8_t* __restrict__ oob) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb || !leaf_map_mapped(listed, blk_pose, b)) return;
    const uint32_t s = blk_start[b], e = blk_start[b + 1];
    double sx = 0.0, sy = 0.0, sz = 0.0;
    uint32_t i = s;
    for (; i + LEAF_MEAN_UNROLL <= e; i += LEAF_MEAN_UNROLL) {
        uint32_t r[LEAF_MEAN_UNROLL];
        double v[LEAF_MEAN_UNROLL][3];
#pragma unroll
        for (int k = 0; k < LEAF_MEAN_UNROLL; ++k) r[k] = perm[i + k];
#pragma unroll
        for (int k = 0; k < LEAF_MEAN_UNROLL; ++k) {
            v[k][0] = xyz[(size_t)r[k] * 3 + 0];
            v[k][1] = xyz[(size_t)r[k] * 3 + 1];
            v[k][2] = xyz[(size_t)r[k] * 3 + 2];
        }
#pragma unroll
        for (int k = 0; k < LEAF_MEAN_UNROLL; ++k) {
            sx = __dadd_rn(sx, v[k][0]);
            sy = __dadd_rn(sy, v[k][1]);
            sz = __dadd_rn(sz, v[k][2]);
        }
    }
    for (; i < e; ++i) {
        const size_t r = perm[i];
        sx = __dadd_rn(sx, xyz[r * 3 + 0]);
        sy = __dadd_rn(sy, xyz[r * 3 + 1]);
        sz = __dadd_rn(sz, xyz[r * 3 + 2]);
    }
    const double n = (double)(e - s);
    const double m[3] = {__ddiv_rn(sx, n), __ddiv_rn(sy, n), __ddiv_rn(sz, n)};
    mean[(size_t)b * 3 + 0] = m[0];
    mean[(size_t)b * 3 + 1] = m[1];
    mean[(size_t)b * 3 + 2] = m[2];
    if (check && !leaf_map_inside(m, leaf_corner, leaf_edge, cache_rank[blk_leaf[b]])) oob[b] = 1;
}

// one thread per position of a listed block, once the means are known.
//   Centroid: the first position whose row == the mean (atomicMin) - the block is then a selection of that row.
//   Shrink:   changed[b] = some row differs from its original; oob[b] = some row is outside the leaf.
// (changed / oob are only ever set to 1: the plain byte stores of several threads agree)
__global__ void __launch_bounds__(256) leaf_point_pass_kernel(uint32_t n, int op, double factor, const uint32_t* __restrict__ blk_of_pos,
                                                              const int32_t* __restrict__ blk_pose, const uint8_t* __restrict__ listed,
                                                              const uint32_t* __restrict__ perm, const double* __restrict__ xyz,
                                                              const double* __restrict__ mean, const uint32_t* __restrict__ blk_leaf,
                                                              const uint32_t* __restrict__ cache_rank,
                                                              const double* __restrict__ leaf_corner,
                                                              const double* __restrict__ leaf_edge, uint32_t* __restrict__ match,
                                                              uint8_t* __restrict__ changed, uint8_t* __restrict__ oob) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t b = blk_of_pos[i];
    if (!leaf_map_mapped(listed, blk_pose, b)) return;
    const size_t r = perm[i];
    const double p[3] = {xyz[r * 3 + 0], xyz[r * 3 + 1], xyz[r * 3 + 2]};
    const double c[3] = {mean[(size_t)b * 3 + 0], mean[(size_t)b * 3 + 1], mean[(size_t)b * 3 + 2]};
    if (op == OL_MAP_CENTROID) {
        if (p[0] == c[0] && p[1] == c[1] && p[2] == c[2]) atomicMin(&match[b], i);
        return;
    }
    double o[3];
    leaf_shrink_row(p, c, factor, o);
    if (!(o[0] == p[0] && o[1] == p[1] && o[2] == p[2])) changed[b] = 1;
    if (!leaf_map_inside(o, leaf_corner, leaf_edge, cache_rank[blk_leaf[b]])) oob[b] = 1;
}

// per block in reference order: rows it appends (0 for a selection or an unlisted block) and whether it appends at all;
// a replaced block with a row outside its leaf raises DEVERR_LEAF_MAP
__global__ void leaf_map_count_kernel(uint32_t nb, int op, const uint32_t* __restrict__ ref_order, const uint32_t* __restrict__ blk_start,
                                      const int32_t* __restrict__ blk_pose, const uint8_t* __restrict__ listed,
                                      const uint32_t* __restrict__ match, const uint8_t* __restrict__ changed,
                                      const uint8_t* __restrict__ oob, uint32_t* __restrict__ rows_ref,
                                      uint32_t* __restrict__ replaced_ref, uint32_t* __restrict__ err) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nb) return;
    const uint32_t b = ref_order[j];
    uint32_t rows = 0;
    if (leaf_map_mapped(listed, blk_pose, b)) {
        if (op == OL_MAP_CENTROID)
            rows = match[b] == LEAF_MAP_NO_MATCH ? 1u : 0u;
        else
            rows = changed[b] ? blk_start[b + 1] - blk_start[b] : 0u;
    }
    rows_ref[j] = rows;
    replaced_ref[j] = rows ? 1u : 0u;
    if (rows && oob[b]) atomicOr(err, (uint32_t)DEVERR_LEAF_MAP);
}

// first / one-past-last reference position of every pose's blocks (the reference order is pose-index major)
__global__ void pose_span_kernel(uint32_t nb, const uint32_t* __restrict__ ref_order, const int32_t* __restrict__ blk_pose,
                                 uint32_t* __restrict__ pose_lo, uint32_t* __restrict__ pose_hi) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nb) return;
    const int32_t p = blk_pose[ref_order[j]];
    if (j == 0 || blk_pose[ref_order[j - 1]] != p) pose_lo[p] = j;
    if (j + 1 == nb || blk_pose[ref_order[j + 1]] != p) pose_hi[p] = j + 1;
}

__global__ void pose_rows_kernel(int n_poses, uint32_t nb, const uint32_t* __restrict__ pose_lo, const uint32_t* __restrict__ pose_hi,
                                 const uint32_t* __restrict__ row_off, const unsigned long long* __restrict__ total,
                                 unsigned long long* __restrict__ pose_rows) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_poses) return;
    const uint32_t lo = pose_lo[p], hi = pose_hi[p];
    const unsigned long long end = hi < nb ? (unsigned long long)row_off[hi] : *total;
    pose_rows[p] = hi > lo ? end - row_off[lo] : 0ull;
}

// per replaced block: the identity of its leaf (cell coordinates, depth, Morton path) for the post-rebuild check, and the
// Centroid row
__global__ void leaf_map_emit_block_kernel(uint32_t nb, int op, const uint32_t* __restrict__ ref_order, const uint32_t* __restrict__ rows_ref,
                                           const uint32_t* __restrict__ row_off, const uint32_t* __restrict__ ord,
                                           const uint32_t* __restrict__ blk_leaf, const uint32_t* __restrict__ lcell,
                                           const uint8_t* __restrict__ ldepth, const uint64_t* __restrict__ lpath,
                                           const uint64_t* __restrict__ cell_key, KeyParams kp, const double* __restrict__ mean,
                                           long long* __restrict__ src_q, uint32_t* __restrict__ src_depth,
                                           uint64_t* __restrict__ src_path, double* __restrict__ out, uint32_t* __restrict__ row_src) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nb || !rows_ref[j]) return;
    const uint32_t b = ref_order[j], o = ord[j], k = blk_leaf[b];
    long long q[3] = {0, 0, 0};
    if (!kp.single_cell) unpack_cell(kp, cell_key[lcell[k]], q);
    src_q[(size_t)o * 3 + 0] = q[0];
    src_q[(size_t)o * 3 + 1] = q[1];
    src_q[(size_t)o * 3 + 2] = q[2];
    src_depth[o] = ldepth[k];
    src_path[o] = lpath[k];
    if (op == OL_MAP_CENTROID) {
        const uint32_t d = row_off[j];
        out[(size_t)d * 3 + 0] = mean[(size_t)b * 3 + 0];
        out[(size_t)d * 3 + 1] = mean[(size_t)b * 3 + 1];
        out[(size_t)d * 3 + 2] = mean[(size_t)b * 3 + 2];
        row_src[d] = o;
    }
}

// Shrink rows of the replaced blocks, in the block's point order (the row recomputed exactly as in leaf_point_pass_kernel)
__global__ void __launch_bounds__(256) leaf_shrink_emit_kernel(uint32_t n, double factor, const uint32_t* __restrict__ blk_of_pos,
                                                               const uint32_t* __restrict__ blk_start, const uint32_t* __restrict__ refpos,
                                                               const uint32_t* __restrict__ rows_ref, const uint32_t* __restrict__ row_off,
                                                               const uint32_t* __restrict__ ord, const uint32_t* __restrict__ perm,
                                                               const double* __restrict__ xyz, const double* __restrict__ mean,
                                                               double* __restrict__ out, uint32_t* __restrict__ row_src) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t b = blk_of_pos[i], j = refpos[b];
    if (!rows_ref[j]) return;
    const size_t r = perm[i];
    const double p[3] = {xyz[r * 3 + 0], xyz[r * 3 + 1], xyz[r * 3 + 2]};
    const double c[3] = {mean[(size_t)b * 3 + 0], mean[(size_t)b * 3 + 1], mean[(size_t)b * 3 + 2]};
    double o[3];
    leaf_shrink_row(p, c, factor, o);
    const uint32_t d = row_off[j] + (i - blk_start[b]);
    out[(size_t)d * 3 + 0] = o[0];
    out[(size_t)d * 3 + 1] = o[1];
    out[(size_t)d * 3 + 2] = o[2];
    row_src[d] = ord[j];
}

// keep flag of every position (K7 input): unlisted blocks keep everything; FirstPoints keeps the first k positions of a
// block, Centroid the matching row of a selection block, Shrink the unchanged blocks
__global__ void leaf_map_keep_kernel(uint32_t n, int op, uint32_t first_k, const uint32_t* __restrict__ blk_of_pos,
                                     const uint32_t* __restrict__ blk_start, const int32_t* __restrict__ blk_pose,
                                     const uint8_t* __restrict__ listed, const uint32_t* __restrict__ match,
                                     const uint8_t* __restrict__ changed, uint8_t* __restrict__ keep) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t b = blk_of_pos[i];
    uint8_t k = 1;
    if (leaf_map_mapped(listed, blk_pose, b)) {
        if (op == OL_MAP_FIRST)
            k = i - blk_start[b] < first_k;
        else if (op == OL_MAP_CENTROID)
            k = match[b] == i;
        else
            k = !changed[b];
    }
    keep[i] = k;
}

// after the rebuild: every appended row (rank >= n0) must sit in the leaf its block came from, compared by cell
// coordinates, depth and Morton path (leaf and cell indices are renumbered by the rebuild)
__global__ void leaf_map_check_kernel(uint32_t n, uint32_t n0, const uint32_t* __restrict__ perm, const uint32_t* __restrict__ leaf_of,
                                      const uint32_t* __restrict__ lcell, const uint8_t* __restrict__ ldepth,
                                      const uint64_t* __restrict__ lpath, const uint64_t* __restrict__ cell_key, KeyParams kp,
                                      const uint32_t* __restrict__ row_src, const long long* __restrict__ src_q,
                                      const uint32_t* __restrict__ src_depth, const uint64_t* __restrict__ src_path,
                                      uint32_t* __restrict__ err) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t r = perm[i];
    if (r < n0) return;
    const uint32_t o = row_src[r - n0], k = leaf_of[i];
    long long q[3] = {0, 0, 0};
    if (!kp.single_cell) unpack_cell(kp, cell_key[lcell[k]], q);
    const bool same = q[0] == src_q[(size_t)o * 3 + 0] && q[1] == src_q[(size_t)o * 3 + 1] && q[2] == src_q[(size_t)o * 3 + 2] &&
                      (uint32_t)ldepth[k] == src_depth[o] && lpath[k] == src_path[o];
    if (!same) atomicOr(err, (uint32_t)DEVERR_LEAF_MOVED);
}

}  // namespace ol
