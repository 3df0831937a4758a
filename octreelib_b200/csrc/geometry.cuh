// Point statistics of segments of the current point order, for the geometric criteria (criteria.py: MaxExtent,
// MaxThickness, Planar) and Grid.leaf_statistics.  A segment is a leaf of one level of K4 (split_levels) or a
// (pose, leaf) block (filter, export).  Per segment: count, per-axis min / max, and - COV - mean and population
// covariance, all in float64.
//
// Deterministic reduction (no atomics): the segment is cut into chunks of GEOM_CHUNK positions; ONE warp reduces a chunk
// (lane l takes the positions l, l + 32, ... in order, then a fixed xor butterfly), and ONE thread per segment merges the
// chunk partials in chunk order.  The order of every floating-point operation is a function of the segment alone.
// The sums are taken relative to the segment's PIVOT, the point at its first position: a point of the node, so that
// |p - pivot| <= extent whatever the offset of the map (a leaf 1e5 m from the origin keeps its precision).
//
// Error bound used by the tests (tests/test_gpu_geometric_criteria.py restates it).  u = 2^-53, n = points of the segment,
// E = its largest per-axis extent, M = its largest |coordinate|, C = the exact population covariance of the points.
//   device:  |d - fl(d)| <= u|d| with |d| <= E; each of the six sums of n products has error <= (n + 2) u n E^2 (any
//            summation order), so an entry of ss/n is off by <= (n + 3) u E^2, the mean offset md = s/n by <= (n + 2) u E,
//            md_a md_b by <= 2 (n + 3) u E^2: every entry of the covariance is off by <= 3 (n + 4) u E^2, the 2-norm of
//            the error matrix by <= 9 (n + 4) u E^2.  Jacobi rotations (sym3_min_eigenvalue) are backward stable:
//            <= 8 u ||C||_F <= 24 u E^2 more.  |lambda_dev - lambda_min(C)| <= 9 (n + 8) u E^2.
//   numpy:   two-pass covariance on the raw coordinates: the mean is off by <= d0 = (n + 2) u (M + E), so every entry is
//            off by <= 2 (E + d0) d0 + (n + 3) u (E + d0)^2; eigvalsh (LAPACK) adds <= 24 u (E + d0)^2 (taken as the
//            same constant as Jacobi).
//   dl = 9 (n + 8) u E^2 + 3 [2 (E + d0) d0 + (n + 3) u (E + d0)^2] + 24 u (E + d0)^2 bounds |lambda_dev - lambda_numpy|;
//   sqrt(max(., 0)) then gives  |thickness_dev - thickness_numpy| <= min(sqrt(dl), dl / thickness_numpy)
//   (|sqrt a - sqrt b| <= |a - b| / (sqrt a + sqrt b)).  Extent is exact: min / max are exact and the subtraction is one
//   IEEE operation, as in numpy.
#pragma once

namespace ol {

constexpr uint32_t GEOM_CHUNK = 1024;  // positions per warp task (32 per lane)

// moments of a run of positions; s / ss relative to the segment's pivot
struct GeomPartial {
    double mn[3], mx[3];
    double s[3];
    double ss[6];  // xx xy xz yy yz zz
    uint32_t n, pad;
};

struct GeomStats {
    long long n;
    double ext[3], mean[3], cov[6];
    double extent, thickness;
};

// what the split decision of a level reads per leaf
struct GeomLeaf {
    double extent, thickness;
    long long n;
};

__device__ __forceinline__ void geom_empty(GeomPartial& m) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        m.mn[a] = __longlong_as_double(0x7ff0000000000000ll);   // +inf
        m.mx[a] = __longlong_as_double((long long)0xfff0000000000000ull);  // -inf
        m.s[a] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) m.ss[i] = 0.0;
    m.n = 0;
    m.pad = 0;
}

template <bool COV>
__device__ __forceinline__ void geom_merge(GeomPartial& m, const GeomPartial& o) {
    m.n += o.n;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        m.mn[a] = fmin(m.mn[a], o.mn[a]);
        m.mx[a] = fmax(m.mx[a], o.mx[a]);
        if (COV) m.s[a] += o.s[a];
    }
    if (COV) {
#pragma unroll
        for (int i = 0; i < 6; ++i) m.ss[i] += o.ss[i];
    }
}

// smallest eigenvalue of the symmetric 3x3 matrix c = (xx, xy, xz, yy, yz, zz): cyclic Jacobi rotations until the
// off-diagonal part is below round-off (quadratic convergence: 3-5 sweeps; 16 at most)
__device__ inline double sym3_min_eigenvalue(const double c[6]) {
    double a[3][3] = {{c[0], c[1], c[2]}, {c[1], c[3], c[4]}, {c[2], c[4], c[5]}};
#pragma unroll 1
    for (int sweep = 0; sweep < 16; ++sweep) {
        if (a[0][1] == 0.0 && a[0][2] == 0.0 && a[1][2] == 0.0) break;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int p = r == 2 ? 1 : 0, q = r == 0 ? 1 : 2;
            const double apq = a[p][q];
            if (apq == 0.0) continue;
            if (fabs(apq) <= 1e-17 * (fabs(a[p][p]) + fabs(a[q][q]))) {  // below round-off of the diagonal
                a[p][q] = a[q][p] = 0.0;
                continue;
            }
            const double theta = (a[q][q] - a[p][p]) / (2.0 * apq);
            const double t = fabs(theta) > 1e150 ? 0.5 / theta : copysign(1.0, theta) / (fabs(theta) + sqrt(theta * theta + 1.0));
            const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
            a[p][p] -= t * apq;
            a[q][q] += t * apq;
            a[p][q] = a[q][p] = 0.0;
            const int o = 3 - p - q;
            const double aop = a[o][p], aoq = a[o][q];
            a[o][p] = a[p][o] = cs * aop - sn * aoq;
            a[o][q] = a[q][o] = sn * aop + cs * aoq;
        }
    }
    return fmin(a[0][0], fmin(a[1][1], a[2][2]));
}

template <bool COV>
__device__ __forceinline__ GeomStats geom_finish(const GeomPartial& m, const double pv[3]) {
    GeomStats g;
    g.n = m.n;
    g.extent = 0.0;
    g.thickness = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        g.ext[a] = m.n ? m.mx[a] - m.mn[a] : 0.0;
        g.extent = fmax(g.extent, g.ext[a]);
        g.mean[a] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) g.cov[i] = 0.0;
    if (COV && m.n) {
        const double n = (double)m.n;
        double md[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            md[a] = m.s[a] / n;
            g.mean[a] = pv[a] + md[a];
        }
        g.cov[0] = m.ss[0] / n - md[0] * md[0];
        g.cov[1] = m.ss[1] / n - md[0] * md[1];
        g.cov[2] = m.ss[2] / n - md[0] * md[2];
        g.cov[3] = m.ss[3] / n - md[1] * md[1];
        g.cov[4] = m.ss[4] / n - md[1] * md[2];
        g.cov[5] = m.ss[5] / n - md[2] * md[2];
        if (m.n >= 3) g.thickness = sqrt(fmax(sym3_min_eigenvalue(g.cov), 0.0));
    }
    return g;
}

__device__ __forceinline__ bool geom_term_holds(const ol_geom_term& t, long long n, double extent, double thickness) {
    if (n < t.min_points) return false;
    const double s = t.stat == OL_GEOM_EXTENT ? extent : thickness;
    return t.op == OL_GEOM_GT ? s > t.value : s <= t.value;
}

// positions whose point belongs to a listed pose (listed == nullptr: every position)
struct PoseFilter {
    const uint32_t* seg_start;
    const int32_t* seg_pose;
    int n_seg;
    const uint8_t* listed;
    __device__ __forceinline__ bool operator()(uint32_t r) const {
        return !listed || listed[seg_pose[seg_of_rank(seg_start, n_seg, r)]] != 0;
    }
};

// the leaves of one level (leaves of other depths are empty segments)
struct LevelSegs {
    const uint32_t* lstart;
    const uint8_t* ldepth;
    int level;
    __device__ __forceinline__ void range(uint32_t k, uint32_t& b, uint32_t& e) const {
        b = lstart[k];
        e = (int)ldepth[k] == level ? lstart[k + 1] : b;
    }
};

// (pose, leaf) blocks
struct BlockSegs {
    const uint32_t* start;
    __device__ __forceinline__ void range(uint32_t k, uint32_t& b, uint32_t& e) const {
        b = start[k];
        e = start[k + 1];
    }
};

__device__ __forceinline__ uint32_t geom_chunks(uint32_t len) { return len / GEOM_CHUNK + (len % GEOM_CHUNK != 0u); }

template <class Seg>
__global__ void geom_chunk_count_kernel(uint32_t n_seg, Seg seg, uint32_t* __restrict__ cnt) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_seg) return;
    uint32_t b, e;
    seg.range(k, b, e);
    cnt[k] = geom_chunks(e - b);
}

// one warp per chunk (grid-stride over the chunks); off = exclusive scan of the chunk counts, *n_chunks its total
template <bool COV, class Seg>
__global__ void __launch_bounds__(256) geom_chunk_kernel(uint32_t n_seg, Seg seg, const uint32_t* __restrict__ off,
                                                         const unsigned long long* __restrict__ n_chunks,
                                                         const uint32_t* __restrict__ perm, const double* __restrict__ P,
                                                         PoseFilter member, GeomPartial* __restrict__ part) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t total = (uint32_t)*n_chunks;
    const uint32_t stride = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < total; c += stride) {
        uint32_t lo = 0, hi = n_seg;  // segment of chunk c: the last k with off[k] <= c
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (off[mid] <= c)
                lo = mid;
            else
                hi = mid;
        }
        uint32_t b, e;
        seg.range(lo, b, e);
        const uint32_t p0 = b + (c - off[lo]) * GEOM_CHUNK;
        const uint32_t p1 = min(e, p0 + GEOM_CHUNK);
        const uint32_t rp = perm[b];
        const double pv0 = P[(size_t)rp * 3 + 0], pv1 = P[(size_t)rp * 3 + 1], pv2 = P[(size_t)rp * 3 + 2];
        GeomPartial m;
        geom_empty(m);
        for (uint32_t i = p0 + lane; i < p1; i += 32u) {
            const uint32_t r = perm[i];
            if (!member(r)) continue;
            const double x = P[(size_t)r * 3 + 0], y = P[(size_t)r * 3 + 1], z = P[(size_t)r * 3 + 2];
            m.n += 1;
            m.mn[0] = fmin(m.mn[0], x);
            m.mn[1] = fmin(m.mn[1], y);
            m.mn[2] = fmin(m.mn[2], z);
            m.mx[0] = fmax(m.mx[0], x);
            m.mx[1] = fmax(m.mx[1], y);
            m.mx[2] = fmax(m.mx[2], z);
            if (COV) {
                const double dx = x - pv0, dy = y - pv1, dz = z - pv2;
                m.s[0] += dx;
                m.s[1] += dy;
                m.s[2] += dz;
                m.ss[0] += dx * dx;
                m.ss[1] += dx * dy;
                m.ss[2] += dx * dz;
                m.ss[3] += dy * dy;
                m.ss[4] += dy * dz;
                m.ss[5] += dz * dz;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            GeomPartial t = m;
            t.n = __shfl_xor_sync(0xffffffffu, m.n, o);
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                t.mn[a] = __shfl_xor_sync(0xffffffffu, m.mn[a], o);
                t.mx[a] = __shfl_xor_sync(0xffffffffu, m.mx[a], o);
                if (COV) t.s[a] = __shfl_xor_sync(0xffffffffu, m.s[a], o);
            }
            if (COV) {
#pragma unroll
                for (int i = 0; i < 6; ++i) t.ss[i] = __shfl_xor_sync(0xffffffffu, m.ss[i], o);
            }
            geom_merge<COV>(m, t);  // x + y on one lane, y + x on its partner: the same value on both
        }
        if (lane == 0) part[c] = m;
    }
}

// one thread per segment: the chunk partials in chunk order, then the statistics
template <bool COV, class Seg, class Emit>
__global__ void geom_merge_kernel(uint32_t n_seg, Seg seg, const uint32_t* __restrict__ off, const uint32_t* __restrict__ perm,
                                  const double* __restrict__ P, const GeomPartial* __restrict__ part, Emit emit) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_seg) return;
    uint32_t b, e;
    seg.range(k, b, e);
    GeomPartial m;
    geom_empty(m);
    double pv[3] = {0.0, 0.0, 0.0};
    if (e > b) {
        const uint32_t nc = geom_chunks(e - b), c0 = off[k];
        for (uint32_t j = 0; j < nc; ++j) geom_merge<COV>(m, part[c0 + j]);
        const uint32_t rp = perm[b];
        pv[0] = P[(size_t)rp * 3 + 0];
        pv[1] = P[(size_t)rp * 3 + 1];
        pv[2] = P[(size_t)rp * 3 + 2];
    }
    emit(k, geom_finish<COV>(m, pv));
}

// K4: what DecideIn<., ., true> reads
struct GeomLevelEmit {
    GeomLeaf* geo;
    __device__ __forceinline__ void operator()(uint32_t k, const GeomStats& g) const { geo[k] = GeomLeaf{g.extent, g.thickness, g.n}; }
};

// filter: a block of a listed pose loses its keep flag unless every term holds
struct GeomFilterEmit {
    const int32_t* blk_pose;
    const uint8_t* listed;
    const ol_geom_term* terms;
    int n_terms;
    uint8_t* keep;
    __device__ __forceinline__ void operator()(uint32_t k, const GeomStats& g) const {
        if (listed && !listed[blk_pose[k]]) return;
        bool all = true;
        for (int t = 0; t < n_terms; ++t) all = all && geom_term_holds(terms[t], g.n, g.extent, g.thickness);
        if (!all) keep[k] = 0;
    }
};

// export: the statistics themselves
struct GeomStatsEmit {
    long long* n;
    double* mean;
    double* cov;
    double* ext;
    __device__ __forceinline__ void operator()(uint32_t k, const GeomStats& g) const {
        n[k] = g.n;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            mean[(size_t)k * 3 + a] = g.mean[a];
            ext[(size_t)k * 3 + a] = g.ext[a];
        }
#pragma unroll
        for (int i = 0; i < 6; ++i) cov[(size_t)k * 6 + i] = g.cov[i];
    }
};

}  // namespace ol
