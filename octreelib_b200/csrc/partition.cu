// Multi-GPU routing (SURVEY.md 8(e)): owner rank = a function of the grid-cell key, stable partition of a rank's local
// points by owner so that one exchange delivers every cell's points - of all poses - to a single GPU.  Two owner rules:
//   hash  owner = hash(ix, iy, iz) mod world
//   slab  owner = number of boundaries b_1 <= ... <= b_{world-1} that are <= ix: an ORDER-PRESERVING hash of the cell key
//         (the leading cell coordinate).  Cells are enumerated lexicographically by (ix, iy, iz) in the reference
//         (grid/grid.py:79-81, 217-232), so with slabs every cell of rank r precedes every cell of rank r + 1: the global
//         leaf order is the rank-major concatenation of the local ones, and the reference's batch-global
//         `block_start_indices` (ransac/cuda_ransac.py:65-67) of a block is the local one plus the pose's point count on
//         the lower ranks - exact with one small all-gather.  The boundaries are count quantiles of ix over all ranks
//         (ol_slab_histogram + one all-gather), chosen identically by every rank.
// ol_partition_by_owner is the staged exchange, the fallback where the fused one (exchange.cu) cannot run: a staging copy
// grouped by owner and the counts of one all-to-all.  The reference has no counterpart (single process); the cell
// coordinates are the ones of /root/reference/octreelib/grid/grid.py:72-76.
#include <climits>

#include "common.cuh"
#include "pointkey.cuh"
#include "primitives.cuh"

namespace ol {

namespace {

constexpr int ROUTE_MAX_WORLD = 64;
struct OwnerRule {
    int slabs;                            // 0 = hash of (ix, iy, iz), 1 = slab of ix
    long long bound[ROUTE_MAX_WORLD];     // slabs: world - 1 ascending boundaries
};

__global__ void owner_kernel(const double* __restrict__ xyz, uint32_t n, double edge, double c0, double c1, double c2,
                             uint32_t world, const __grid_constant__ OwnerRule rule, uint32_t* __restrict__ owner,
                             uint32_t* __restrict__ iota, uint32_t* __restrict__ err) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double qx = cell_coord(xyz[(size_t)i * 3 + 0], c0, edge);
    const double qy = cell_coord(xyz[(size_t)i * 3 + 1], c1, edge);
    const double qz = cell_coord(xyz[(size_t)i * 3 + 2], c2, edge);
    uint32_t o = 0;
    if (fabs(qx) < 4503599627370496.0 && fabs(qy) < 4503599627370496.0 && fabs(qz) < 4503599627370496.0) {
        if (rule.slabs) {
            const long long ix = (long long)qx;
            for (uint32_t k = 0; k + 1 < world; ++k) o += rule.bound[k] <= ix ? 1u : 0u;
        } else {
            o = cell_owner((long long)qx, (long long)qy, (long long)qz, world);
        }
    } else
        atomicOr(err, (uint32_t)(isfinite(qx + qy + qz) ? DEVERR_CELL_RANGE : DEVERR_NONFINITE));
    owner[i] = o;
    iota[i] = i;
}

__global__ void route_gather_kernel(uint32_t n, const double* __restrict__ xyz, const uint32_t* __restrict__ perm,
                                    double* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t r = perm[i];
    out[(size_t)i * 3 + 0] = xyz[r * 3 + 0];
    out[(size_t)i * 3 + 1] = xyz[r * 3 + 1];
    out[(size_t)i * 3 + 2] = xyz[r * 3 + 2];
}

// (owner, segment) runs are contiguous after the stable sort: record where each run starts / ends
__global__ void route_counts_kernel(uint32_t n, const uint32_t* __restrict__ owner_sorted, const uint32_t* __restrict__ perm,
                                    const uint32_t* __restrict__ seg_start, int n_seg, unsigned long long* __restrict__ run_begin,
                                    unsigned long long* __restrict__ run_end) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    auto seg_of = [&](uint32_t r) {
        int lo = 0, hi = n_seg;
        while (hi - lo > 1) {
            int mid = (lo + hi) >> 1;
            if (seg_start[mid] <= r)
                lo = mid;
            else
                hi = mid;
        }
        return lo;
    };
    const uint32_t o = owner_sorted[i];
    const int s = seg_of(perm[i]);
    const size_t slot = (size_t)o * n_seg + s;
    const bool head = (i == 0) || owner_sorted[i - 1] != o || seg_of(perm[i - 1]) != s;
    const bool tail = (i == n - 1) || owner_sorted[i + 1] != o || seg_of(perm[i + 1]) != s;
    if (head) run_begin[slot] = i;
    if (tail) run_end[slot] = (unsigned long long)i + 1;
}

// ---- slab boundaries: range and histogram of the leading cell coordinate ---------------------------------------------
// Both kernels look at every SLAB_SAMPLE-th point only: the boundaries balance the load, they need not be exact quantiles
// (ownership itself is decided per point from the boundaries), and a LiDAR sweep keeps thousands of consecutive points in
// the same column of cells - counted one by one they would all hit the same shared-memory counter.
constexpr uint32_t SLAB_SAMPLE = 8;

__global__ void __launch_bounds__(256) slab_range_kernel(const double* __restrict__ xyz, uint32_t n, double edge, double c0,
                                                         long long* __restrict__ out /*[0] min ix, [1] max ix*/) {
    long long lo = LLONG_MAX, hi = LLONG_MIN;
    const uint32_t m = (n + SLAB_SAMPLE - 1) / SLAB_SAMPLE;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < m; k += gridDim.x * blockDim.x) {
        const double q = cell_coord(xyz[(size_t)k * SLAB_SAMPLE * 3], c0, edge);
        if (fabs(q) < 4503599627370496.0) {
            const long long ix = (long long)q;
            lo = ix < lo ? ix : lo;
            hi = ix > hi ? ix : hi;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
        lo = l2 < lo ? l2 : lo;
        hi = h2 > hi ? h2 : hi;
    }
    if ((threadIdx.x & 31) == 0) {
        if (lo != LLONG_MAX) atomicMin(&out[0], lo);
        if (hi != LLONG_MIN) atomicMax(&out[1], hi);
    }
}

// counts[k] = sampled points whose ix falls into bin k = (ix - min ix) / width, width = ceil((max - min + 1) / n_bins)
__global__ void __launch_bounds__(256) slab_hist_kernel(const double* __restrict__ xyz, uint32_t n, double edge, double c0,
                                                        int n_bins, long long* __restrict__ out /*[2 + n_bins]*/) {
    extern __shared__ unsigned int s_h[];
    for (int k = threadIdx.x; k < n_bins; k += blockDim.x) s_h[k] = 0u;
    __syncthreads();
    const long long lo = out[0], hi = out[1];
    const long long width = hi >= lo ? ((hi - lo + 1) + n_bins - 1) / n_bins : 1;
    const uint32_t m = (n + SLAB_SAMPLE - 1) / SLAB_SAMPLE;
    const uint32_t m_pad = (m + 31u) & ~31u;  // whole warps take part in the match
    const int lane = threadIdx.x & 31;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < m_pad; k += gridDim.x * blockDim.x) {
        int bin = -1;
        if (k < m) {
            const double q = cell_coord(xyz[(size_t)k * SLAB_SAMPLE * 3], c0, edge);
            if (fabs(q) < 4503599627370496.0) bin = (int)(((long long)q - lo) / width);
        }
        const uint32_t peers = __match_any_sync(0xffffffffu, bin);  // one shared-memory atomic per distinct bin and warp
        if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&s_h[bin], (unsigned int)__popc(peers));
    }
    __syncthreads();
    for (int k = threadIdx.x; k < n_bins; k += blockDim.x)
        if (s_h[k]) atomicAdd(reinterpret_cast<unsigned long long*>(&out[2 + k]), (unsigned long long)s_h[k]);
}

}  // namespace
}  // namespace ol

extern "C" {

// out_dev: int64[2 + n_bins] = {min ix, max ix, counts of n_bins equal-width bins over [min ix, max ix]} of this rank's points
// (min > max when the rank holds no point).  Enqueued on `stream`; no synchronisation.
int ol_slab_histogram(void* stream, const double* xyz_dev, int64_t n, double edge, double corner_x, int32_t n_bins,
                      int64_t* out_dev) {
    using namespace ol;
    try {
        OL_REQUIRE(n >= 0 && n < (1ll << 31) && n_bins >= 1 && n_bins <= 8192 && edge > 0, OL_ERR_INVALID, "bad histogram arguments");
        cudaStream_t st = (cudaStream_t)stream;
        OL_CUDA(cudaMemsetAsync(out_dev, 0, sizeof(int64_t) * (size_t)(2 + n_bins), st));
        const long long init[2] = {LLONG_MAX, LLONG_MIN};
        OL_CUDA(cudaMemcpyAsync(out_dev, init, sizeof(init), cudaMemcpyHostToDevice, st));
        if (n == 0) return OL_OK;
        const unsigned g = (unsigned)std::min<int64_t>((n / SLAB_SAMPLE + 256) / 256, 148 * 8);
        slab_range_kernel<<<g, 256, 0, st>>>(xyz_dev, (uint32_t)n, edge, corner_x, reinterpret_cast<long long*>(out_dev));
        OL_CHECK_LAUNCH();
        slab_hist_kernel<<<g, 256, sizeof(unsigned int) * (size_t)n_bins, st>>>(xyz_dev, (uint32_t)n, edge, corner_x, n_bins,
                                                                             reinterpret_cast<long long*>(out_dev));
        OL_CHECK_LAUNCH();
    } catch (const ol::Error& e) {
        ol::set_last_error(e.code, e.msg);
        return e.code;
    }
    return OL_OK;
}


uint32_t ol_host_cell_owner(int64_t qx, int64_t qy, int64_t qz, uint32_t world) { return ol::cell_owner(qx, qy, qz, world); }

// Owner per point, stable sort by owner, gather into that order; counts[owner][run] are read back (one synchronisation).
int ol_partition_by_owner(void* stream, const double* xyz_dev, int64_t n, const int64_t* seg_sizes_host, int32_t n_segments,
                          double edge, const double corner[3], int32_t world, const int64_t* slab_bounds_host, double* out_xyz_dev,
                          int64_t* out_counts_host, ol_alloc_fn alloc, ol_free_fn free_fn, void* alloc_user) {
    using namespace ol;
    try {
        Ctx c;
        c.stream = (cudaStream_t)stream;
        c.alloc_fn = alloc;
        c.free_fn = free_fn;
        c.alloc_user = alloc_user;
        c.pool_enabled = true;
        OL_REQUIRE(n >= 0 && n < (1ll << 31) && n_segments >= 1 && world >= 1 && world <= ROUTE_MAX_WORLD && edge > 0, OL_ERR_INVALID,
                   "bad partition arguments");
        OwnerRule rule{};
        if (slab_bounds_host) {
            rule.slabs = 1;
            for (int k = 0; k + 1 < world; ++k) {
                OL_REQUIRE(k == 0 || slab_bounds_host[k] >= slab_bounds_host[k - 1], OL_ERR_INVALID, "slab boundaries must ascend");
                rule.bound[k] = slab_bounds_host[k];
            }
        }
        for (int64_t k = 0; k < (int64_t)world * n_segments; ++k) out_counts_host[k] = 0;
        if (n == 0) return OL_OK;
        const uint32_t m = (uint32_t)n;
        std::vector<uint32_t> seg_start((size_t)n_segments + 1, 0);
        for (int s = 0; s < n_segments; ++s) seg_start[s + 1] = seg_start[s] + (uint32_t)seg_sizes_host[s];
        OL_REQUIRE(seg_start[n_segments] == m, OL_ERR_INVALID, "segment sizes do not add up to n");
        DevBuf<uint32_t> err(c, 1), k0(c, m), k1(c, m), v0(c, m), v1(c, m), d_seg(c, seg_start.size());
        DevBuf<unsigned long long> rb(c, (size_t)world * n_segments), re(c, (size_t)world * n_segments);
        err.zero();
        rb.zero();
        re.zero();
        h2d(c, d_seg.get(), seg_start.data(), seg_start.size());
        const unsigned g = (m + 255) / 256;
        owner_kernel<<<g, 256, 0, c.stream>>>(xyz_dev, m, edge, corner[0], corner[1], corner[2], (uint32_t)world, rule, k0.get(),
                                              v0.get(), err.get());
        OL_CHECK_LAUNCH();
        int w = radix_sort_pairs<uint32_t>(c, k0.get(), k1.get(), v0.get(), v1.get(), m, 0, bit_length_u64((uint64_t)world - 1));
        const uint32_t* ks = w ? k1.get() : k0.get();
        const uint32_t* vs = w ? v1.get() : v0.get();
        route_gather_kernel<<<g, 256, 0, c.stream>>>(m, xyz_dev, vs, out_xyz_dev);
        OL_CHECK_LAUNCH();
        route_counts_kernel<<<g, 256, 0, c.stream>>>(m, ks, vs, d_seg.get(), n_segments, rb.get(), re.get());
        OL_CHECK_LAUNCH();
        std::vector<unsigned long long> hb((size_t)world * n_segments), he((size_t)world * n_segments);
        uint32_t herr = 0;
        d2h(c, hb.data(), rb.get(), hb.size());
        d2h(c, he.data(), re.get(), he.size());
        d2h(c, &herr, err.get(), 1);
        c.sync();
        OL_REQUIRE(!(herr & DEVERR_NONFINITE), OL_ERR_NONFINITE, "point cloud contains NaN or infinite coordinates");
        OL_REQUIRE(!(herr & DEVERR_CELL_RANGE), OL_ERR_RANGE, "cell coordinates out of the representable range");
        for (size_t k = 0; k < hb.size(); ++k) out_counts_host[k] = (int64_t)(he[k] - hb[k]);
    } catch (const ol::Error& e) {
        ol::set_last_error(e.code, e.msg);
        return e.code;
    }
    return OL_OK;
}

}  // extern "C"
