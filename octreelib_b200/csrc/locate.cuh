// Grid.locate_points on the device: the leaf every query point would be routed into by insert_points of a new pose,
// without inserting it.  Forest::locate (forest_host2.inl) makes the tables current and launches the kernel below.
//
// One thread per query, no new geometry: the cell coordinates and the in-cell Morton code come from the same
// pointkey.cuh calls as the key pass (keygen_kernel, pow2 reciprocal included), so a query lands exactly where an
// inserted point would.  Then
//   1. the cell: binary search of the sorted packed keys (cell_key), after a range check of every coordinate field (a
//      coordinate outside the packed range cannot belong to an existing cell and is never wrapped into another one);
//   2. the leaf: the cell's leaves are contiguous in depth-first order (the range of cell_leaf_begin) and, because every
//      split makes all eight children, tile the cell; their paths, padded to depth_reached levels, ascend.  The leaf is
//      the last one whose padded path is <= the query's code at depth_reached;
//   3. -1 when a coordinate is not finite, the cell does not exist, or the point leaves its node above the leaf
//      (bad_level < depth: insertion raises IndexError there, DEVERR_OUT_OF_NODE).
// The result is the leaf's index in the reference's enumeration (cache_rank), optionally mapped through leaf_to_row.
// Traffic: 24 B read + 8 B written per query; the key, leaf and rank tables are read through L2.
#pragma once
#include "forest.cuh"

namespace ol {

constexpr int LOCATE_THREADS = 256;

struct LocateTables {
    const uint64_t* cell_key;         // [C] ascending packed cell keys (without pose bits)
    const uint32_t* cell_leaf_begin;  // [C + 1] first leaf of every cell (same range in DFS and reference order)
    const uint64_t* lpath;            // [L] DFS order: Morton digits from the cell root, 3 bits per level
    const uint8_t* ldepth;            // [L]
    const uint32_t* cache_rank;       // [L] DFS leaf -> leaf-table index
    const int32_t* leaf_to_row;       // [L] leaf-table index -> value written (NULL: the index itself)
    uint32_t C;
    int depth;                        // depth_reached (<= OL_MAX_DEPTH: at most 63 code bits, shifts stay below 64)
    int field_bits[3];                // width of the x / y / z field of the packed cell key
};

__global__ void __launch_bounds__(LOCATE_THREADS) locate_kernel(const double* __restrict__ xyz, int64_t n, KeyParams kp,
                                                                LocateTables t, int64_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * LOCATE_THREADS + threadIdx.x;
    if (i >= n) return;
    const double p[3] = {xyz[i * 3 + 0], xyz[i * 3 + 1], xyz[i * 3 + 2]};
    int64_t res = -1;
    do {
        if (!(isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2])) || t.C == 0) break;
        long long q[3] = {0, 0, 0};
        uint32_t c = 0;
        if (!kp.single_cell) {
            uint64_t key = 0;
            bool in_range = true;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double qa = cell_coord_inv(p[a], kp.corner[a], kp.edge, kp.inv_edge);
                if (!(fabs(qa) < 4503599627370496.0)) {  // 2^52, like the key pass
                    in_range = false;
                    break;
                }
                q[a] = (long long)qa;
                const long long rel = q[a] - kp.qmin[a];  // |q|, |qmin| < 2^52: no overflow
                const int w = t.field_bits[a];
                if (rel < 0 || (w < 63 && (rel >> w) != 0)) {
                    in_range = false;
                    break;
                }
                const int s = kp.shift[a] - kp.pose_bits;
                if (s < 64) key |= (uint64_t)rel << s;
            }
            if (!in_range) break;
            uint32_t lo = 0, hi = t.C;  // first cell with cell_key >= key
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (t.cell_key[mid] < key)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            if (lo == t.C || t.cell_key[lo] != key) break;
            c = lo;
        }
        double c0[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) c0[a] = cell_corner_coord(q[a], kp.corner[a], kp.edge, kp.single_cell);
        int bad;
        const unsigned long long m = point_morton(p, c0, kp.edge, t.depth, &bad);
        // the cell's first leaf has the all-zero path, so the answer is inside [lo, hi)
        uint32_t lo = t.cell_leaf_begin[c], hi = t.cell_leaf_begin[c + 1];
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if ((t.lpath[mid] << (3 * (t.depth - (int)t.ldepth[mid]))) <= m)
                lo = mid;
            else
                hi = mid;
        }
        if (bad < (int)t.ldepth[lo]) break;
        const uint32_t j = t.cache_rank[lo];
        res = t.leaf_to_row ? (int64_t)t.leaf_to_row[j] : (int64_t)j;
    } while (false);
    out[i] = res;
}

}  // namespace ol
