// Fused multi-GPU exchange: owner computation, counting, routing over NVLink and the hand-over to the receiving forest,
// with every inter-rank dependency resolved ON THE DEVICE.
//
// Why: the grid shards by cell (every cell is independent in the reference: grid/grid.py:255-258, 266-267), so one exchange
// moves every point to the rank that owns its cell and everything afterwards is local.  On 8 GPUs a rank's share of the
// 100 M-point map is processed in ~2.5 ms of kernels; an exchange built from library collectives with host round trips
// (histogram all-gather + read-back, count all-gather + read-back, two barriers, a staging copy and an insert copy) cost
// more than 1.5 ms of that.  Here:
//   * ranks talk through CONTROL BLOCKS in peer-mapped memory: a rank writes its payload locally, then raises a flag in
//     every peer's block (st.release.sys); consumers spin on their own flags (ld.acquire.sys) and read the peers' payloads
//     over NVLink.  No NCCL call, no host round trip; three flag rounds per exchange.
//   * slab boundaries (order-preserving owner rule, partition.cu) are computed on the device, by every rank identically,
//     from integer arithmetic on the ranks' histograms (bisection on the combined cumulative count).
//   * ONE counting pass (owner byte per point, per-tile / per-(owner, pose) counts, bounding box, NaN check) and ONE
//     scatter pass that stages a tile in shared memory grouped by owner and stores contiguous runs straight into the
//     owners' receive buffers (256-byte warp stores; order inside (source rank, pose) is the input order).
//   * the receiving forest adopts the receive buffer as its point array (no insert copy, no bounding-box pass, no bounding
//     box read-back: the cell-coordinate range of what can arrive is known from the ranks' boxes and the slab bounds).
//   * the host waits for ONE event (after the count round) to learn the (source, pose) runs it receives; the scatter and the
//     final flag round run on the GPU meanwhile.
// The reference has no counterpart (single process); cell coordinates as in grid/grid.py:72-76.
#include <climits>

#include "exchange.cuh"
#include "forest.cuh"
#include "pointkey.cuh"
#include "primitives.cuh"

namespace ol {

namespace {

constexpr unsigned long long XCHG_TIMEOUT_NS = 20ull * 1000ull * 1000ull * 1000ull;
constexpr uint32_t XERR_TIMEOUT = 1u << 30;

struct XTile {
    const double* src;   // first point of the tile
    uint32_t n;          // points in the tile (<= XCHG_TILE)
    uint32_t first_row;  // index of the tile's first point in the rank's concatenated local cloud
    int32_t pose;
    int32_t pad;
};

// one local cloud; the tile table is expanded from these on the device (xchg_tiles_kernel): the host uploads ~100 rows
// instead of building and staging thousands of tile descriptors per step
struct XCloud {
    const double* src;
    uint32_t n;           // points
    uint32_t first_row;   // index of the cloud's first point in the rank's concatenated local cloud
    uint32_t first_tile;  // index of the cloud's first tile
    int32_t pose;
};

struct XParams {
    double edge, c0, c1, c2;
    double inv_edge;  // 1 / edge for power-of-two edges (exact), else 0: common.cuh, npy_floor_divide_inv
    int world, rank, n_poses, slabs;
    long long rows_cap;
    unsigned long long epoch;
};

struct XPeers {
    unsigned char* ctrl[XCHG_MAX_WORLD];
    double* data[XCHG_MAX_WORLD];
};

// scratch layout
struct XScratch {
    static constexpr size_t BOUNDS = 0;                       // int64 [64]
    static constexpr size_t BASE = 512;                       // int64 [64]
    static constexpr size_t TOT = 1024;                       // uint32 [64][64]
    static constexpr size_t MISC = TOT + 4 * 64 * 64;         // uint32: 0 ticket, 1 overflow, 2 err
    static constexpr size_t BBOX = MISC + 16;                 // int64 [6] union of the ranks' boxes
    static constexpr size_t PREFIX = BBOX + 48;               // uint64 [world][XCHG_BINS + 1]
    __host__ __device__ static size_t pose_size(int world) { return PREFIX + 8 * (size_t)world * (XCHG_BINS + 1); }  // uint32 [world][n_poses]
    static size_t bytes(int world, int n_poses) { return pose_size(world) + 4 * (size_t)world * (size_t)n_poses; }
};

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ void signal_peer(unsigned char* peer_ctrl, int stage, int me, unsigned long long epoch) {
    unsigned long long* p = reinterpret_cast<unsigned long long*>(peer_ctrl + XchgCtrl::FLAG) + (size_t)stage * XCHG_MAX_WORLD + me;
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(epoch) : "memory");
}

// returns false on timeout
__device__ __forceinline__ bool wait_flag(const unsigned char* my_ctrl, int stage, int src, unsigned long long epoch) {
    const unsigned long long* p = reinterpret_cast<const unsigned long long*>(my_ctrl + XchgCtrl::FLAG) + (size_t)stage * XCHG_MAX_WORLD + src;
    const unsigned long long t0 = globaltimer_ns();
    for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
        if (v >= epoch) return true;
        if (globaltimer_ns() - t0 > XCHG_TIMEOUT_NS) return false;
        __nanosleep(200);
    }
}

// ---- reset of this rank's payloads and scratch -------------------------------------------------------------------------
__global__ void xchg_init_kernel(unsigned char* my_ctrl, unsigned char* scratch, int world, int n_poses) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t* hist = reinterpret_cast<uint32_t*>(my_ctrl + XchgCtrl::HIST);
    uint32_t* cube = reinterpret_cast<uint32_t*>(my_ctrl + XchgCtrl::CUBE);
    uint32_t* psz = reinterpret_cast<uint32_t*>(scratch + XScratch::pose_size(world));
    const size_t wp = (size_t)world * n_poses;
    if (i < XCHG_BINS) hist[i] = 0u;
    if (i < wp) {
        cube[i] = 0u;
        psz[i] = 0u;
    }
    if (i < 64 * 64) reinterpret_cast<uint32_t*>(scratch + XScratch::TOT)[i] = 0u;
    if (i < 4) reinterpret_cast<uint32_t*>(scratch + XScratch::MISC)[i] = 0u;
    if (i < 6) {
        const long long v = i < 3 ? LLONG_MAX : LLONG_MIN;
        reinterpret_cast<long long*>(my_ctrl + XchgCtrl::BBOX)[i] = v;
        reinterpret_cast<long long*>(scratch + XScratch::BBOX)[i] = v;
    }
    if (i == 0) {
        reinterpret_cast<long long*>(my_ctrl + XchgCtrl::RANGE)[0] = LLONG_MAX;
        reinterpret_cast<long long*>(my_ctrl + XchgCtrl::RANGE)[1] = LLONG_MIN;
        *reinterpret_cast<uint32_t*>(my_ctrl + XchgCtrl::ERR) = 0u;
    }
}

// ---- stage A (slabs only): sampled range and histogram of the leading cell coordinate ------------------------------------
constexpr uint32_t XCHG_SAMPLE = 8;  // every 8th point: the boundaries balance the load, ownership is decided per point

__global__ void __launch_bounds__(256) xchg_range_kernel(const XTile* __restrict__ tiles, uint32_t n_tiles, XParams p,
                                                         unsigned char* my_ctrl) {
    long long lo = LLONG_MAX, hi = LLONG_MIN;
    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const XTile T = tiles[t];
        const uint32_t k = threadIdx.x * XCHG_SAMPLE;
        if (k < T.n) {
            const double q = cell_coord_inv(T.src[(size_t)k * 3], p.c0, p.edge, p.inv_edge);
            if (fabs(q) < 4503599627370496.0) {
                const long long ix = (long long)q;
                lo = ix < lo ? ix : lo;
                hi = ix > hi ? ix : hi;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
        lo = l2 < lo ? l2 : lo;
        hi = h2 > hi ? h2 : hi;
    }
    if ((threadIdx.x & 31) == 0) {
        long long* r = reinterpret_cast<long long*>(my_ctrl + XchgCtrl::RANGE);
        if (lo != LLONG_MAX) atomicMin(&r[0], lo);
        if (hi != LLONG_MIN) atomicMax(&r[1], hi);
    }
}

__global__ void __launch_bounds__(256) xchg_hist_kernel(const XTile* __restrict__ tiles, uint32_t n_tiles, XParams p,
                                                        unsigned char* my_ctrl) {
    __shared__ unsigned int s_h[XCHG_BINS];
    for (int k = threadIdx.x; k < XCHG_BINS; k += blockDim.x) s_h[k] = 0u;
    __syncthreads();
    const long long* r = reinterpret_cast<const long long*>(my_ctrl + XchgCtrl::RANGE);
    const long long lo = r[0], hi = r[1];
    const long long width = hi >= lo ? ((hi - lo + 1) + XCHG_BINS - 1) / XCHG_BINS : 1;
    const int lane = threadIdx.x & 31;
    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const XTile T = tiles[t];
        const uint32_t k = threadIdx.x * XCHG_SAMPLE;
        int bin = -1;
        if (k < T.n) {
            const double q = cell_coord_inv(T.src[(size_t)k * 3], p.c0, p.edge, p.inv_edge);
            if (fabs(q) < 4503599627370496.0) bin = (int)(((long long)q - lo) / width);
        }
        const uint32_t peers = __match_any_sync(0xffffffffu, bin);  // one shared-memory atomic per distinct bin and warp
        if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&s_h[bin], (unsigned int)__popc(peers));
    }
    __syncthreads();
    uint32_t* out = reinterpret_cast<uint32_t*>(my_ctrl + XchgCtrl::HIST);
    for (int k = threadIdx.x; k < XCHG_BINS; k += blockDim.x)
        if (s_h[k]) atomicAdd(&out[k], s_h[k]);
}

// sampled points of one rank with cell x < `x` (piecewise linear inside a bin; integer / double arithmetic that every rank
// evaluates identically)
__device__ inline unsigned long long rank_cdf(long long lo, long long hi, const unsigned long long* prefix, long long x) {
    if (lo > hi || x <= lo) return 0ull;
    if (x > hi) return prefix[XCHG_BINS];
    const long long width = ((hi - lo + 1) + XCHG_BINS - 1) / XCHG_BINS;
    const long long k = (x - lo) / width, rem = (x - lo) - k * width;
    const unsigned long long cnt = prefix[k + 1] - prefix[k];
    return prefix[k] + (unsigned long long)((double)cnt * ((double)rem / (double)width));
}

// flag round A + slab boundaries: one CTA, one warp per rank for the prefix sums, one thread per boundary for the bisection
__global__ void __launch_bounds__(1024) xchg_sync_a_kernel(XParams p, const __grid_constant__ XPeers peers, unsigned char* scratch,
                                                           unsigned char* host) {
    __shared__ long long s_lo[XCHG_MAX_WORLD], s_hi[XCHG_MAX_WORLD];
    __shared__ int s_timeout;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned char* my_ctrl = peers.ctrl[p.rank];
    if (tid == 0) s_timeout = 0;
    __syncthreads();
    if (tid < p.world) signal_peer(peers.ctrl[tid], 0, p.rank, p.epoch);
    if (tid < p.world && !wait_flag(my_ctrl, 0, tid, p.epoch)) s_timeout = 1;
    __syncthreads();
    if (s_timeout) {
        if (tid == 0) {
            atomicOr(reinterpret_cast<uint32_t*>(scratch + XScratch::MISC) + 2, XERR_TIMEOUT);
            reinterpret_cast<volatile long long*>(host + XchgHost::HDR)[8] = 1;
        }
        return;
    }
    unsigned long long* prefix = reinterpret_cast<unsigned long long*>(scratch + XScratch::PREFIX);
    for (int r = warp; r < p.world; r += 32) {
        const unsigned char* c = peers.ctrl[r];
        if (lane == 0) {
            s_lo[r] = reinterpret_cast<const long long*>(c + XchgCtrl::RANGE)[0];
            s_hi[r] = reinterpret_cast<const long long*>(c + XchgCtrl::RANGE)[1];
        }
        const uint32_t* h = reinterpret_cast<const uint32_t*>(c + XchgCtrl::HIST);
        unsigned long long run = 0;
        unsigned long long* pr = prefix + (size_t)r * (XCHG_BINS + 1);
        for (int b0 = 0; b0 < XCHG_BINS; b0 += 32) {
            const unsigned long long v = h[b0 + lane];
            unsigned long long inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long up = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += up;
            }
            pr[b0 + lane] = run + inc - v;
            run += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (lane == 0) pr[XCHG_BINS] = run;
    }
    __syncthreads();
    long long* bounds = reinterpret_cast<long long*>(scratch + XScratch::BOUNDS);
    if (tid < p.world - 1) {
        long long glo = LLONG_MAX, ghi = LLONG_MIN;
        unsigned long long total = 0;
        for (int r = 0; r < p.world; ++r) {
            if (s_lo[r] <= s_hi[r]) {
                glo = s_lo[r] < glo ? s_lo[r] : glo;
                ghi = s_hi[r] > ghi ? s_hi[r] : ghi;
                total += prefix[(size_t)r * (XCHG_BINS + 1) + XCHG_BINS];
            }
        }
        long long b = 0;
        if (glo <= ghi) {
            // target count of boundary tid + 1 of world: total (tid + 1) / world, kept in 64 bits (total < 2^31)
            const unsigned long long target = total * (unsigned long long)(tid + 1) / (unsigned long long)p.world;
            long long a = glo, z = ghi + 1;  // smallest x in [glo, ghi + 1] whose combined count reaches the target
            while (a < z) {
                const long long mid = a + (z - a) / 2;
                unsigned long long f = 0;
                for (int r = 0; r < p.world; ++r) f += rank_cdf(s_lo[r], s_hi[r], prefix + (size_t)r * (XCHG_BINS + 1), mid);
                if (f >= target)
                    z = mid;
                else
                    a = mid + 1;
            }
            b = a;
        }
        bounds[tid] = b;
        reinterpret_cast<volatile long long*>(host + XchgHost::BOUNDS)[tid] = b;
    }
}

// tile t -> its cloud (bisection over the clouds' first tiles) -> descriptor
__global__ void xchg_tiles_kernel(const XCloud* __restrict__ clouds, int n_clouds, uint32_t n_tiles, XTile* __restrict__ tiles) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    int lo = 0, hi = n_clouds;  // last cloud with first_tile <= t (clouds without points own no tile and are skipped by the search)
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (clouds[mid].first_tile <= t)
            lo = mid;
        else
            hi = mid;
    }
    const XCloud c = clouds[lo];
    const uint32_t off = (t - c.first_tile) * (uint32_t)XCHG_TILE;
    XTile T;
    T.src = c.src + (size_t)off * 3;
    T.n = min((uint32_t)XCHG_TILE, c.n - off);
    T.first_row = c.first_row + off;
    T.pose = c.pose;
    T.pad = 0;
    tiles[t] = T;
}

// ---- counting pass ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) xchg_count_kernel(const XTile* __restrict__ tiles, uint32_t n_tiles, XParams p,
                                                         const long long* __restrict__ bounds, uint8_t* __restrict__ owner_out,
                                                         uint32_t* __restrict__ tile_cnt, unsigned char* my_ctrl) {
    __shared__ uint32_t s_cnt[XCHG_MAX_WORLD];
    __shared__ long long s_bound[XCHG_MAX_WORLD];
    __shared__ long long s_bb[6];
    __shared__ uint32_t s_err;
    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t tile = blockIdx.x;
    const XTile T = tiles[tile];
    if (tid < XCHG_MAX_WORLD) {
        s_cnt[tid] = 0u;
        s_bound[tid] = (p.slabs && tid < p.world - 1) ? bounds[tid] : LLONG_MAX;
    }
    if (tid < 6) s_bb[tid] = tid < 3 ? LLONG_MAX : LLONG_MIN;
    if (tid == 0) s_err = 0u;
    __syncthreads();
    double mn0 = INFINITY, mn1 = INFINITY, mn2 = INFINITY, mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY;
    uint32_t err = 0u;
    // the tile in groups of four rows: the twelve loads of a group are issued together, then the arithmetic and the
    // warp-synchronous counting (inside one loop every row waited for its own loads)
    constexpr int XG = 4;
    static_assert((XCHG_TILE / 256) % XG == 0, "tile rows must come in groups of XG");
    for (int r0 = 0; r0 < XCHG_TILE / 256; r0 += XG) {
    double px[XG], py[XG], pz[XG];
#pragma unroll
    for (int g = 0; g < XG; ++g) {
        const uint32_t idx = (uint32_t)(r0 + g) * 256u + (uint32_t)tid;
        const bool in = idx < T.n;
        px[g] = in ? T.src[(size_t)idx * 3] : 0.0;
        py[g] = in ? T.src[(size_t)idx * 3 + 1] : 0.0;
        pz[g] = in ? T.src[(size_t)idx * 3 + 2] : 0.0;
    }
#pragma unroll
    for (int g = 0; g < XG; ++g) {
        const int r = r0 + g;
        const uint32_t idx = (uint32_t)r * 256u + (uint32_t)tid;
        uint32_t o = 0xffffffffu;
        if (idx < T.n) {
            const double x = px[g], y = py[g], z = pz[g];
            o = 0u;
            if (!isfinite(x + y + z)) {
                err |= DEVERR_NONFINITE;
            } else {
                mn0 = fmin(mn0, x), mx0 = fmax(mx0, x);
                mn1 = fmin(mn1, y), mx1 = fmax(mx1, y);
                mn2 = fmin(mn2, z), mx2 = fmax(mx2, z);
                const double qx = cell_coord_inv(x, p.c0, p.edge, p.inv_edge);
                if (p.slabs) {
                    if (fabs(qx) < 4503599627370496.0) {
                        const long long ix = (long long)qx;
                        for (int k = 0; k + 1 < p.world; ++k) o += s_bound[k] <= ix ? 1u : 0u;
                    } else
                        err |= DEVERR_CELL_RANGE;
                } else {
                    const double qy = cell_coord_inv(y, p.c1, p.edge, p.inv_edge), qz = cell_coord_inv(z, p.c2, p.edge, p.inv_edge);
                    if (fabs(qx) < 4503599627370496.0 && fabs(qy) < 4503599627370496.0 && fabs(qz) < 4503599627370496.0)
                        o = cell_owner((long long)qx, (long long)qy, (long long)qz, (uint32_t)p.world);
                    else
                        err |= DEVERR_CELL_RANGE;
                }
            }
            owner_out[(size_t)T.first_row + idx] = (uint8_t)o;
        }
        const uint32_t peers = __match_any_sync(0xffffffffu, o);
        if (o != 0xffffffffu && lane == __ffs(peers) - 1) atomicAdd(&s_cnt[o], (uint32_t)__popc(peers));
    }
    }  // groups of rows
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn0 = fmin(mn0, __shfl_xor_sync(0xffffffffu, mn0, o)), mx0 = fmax(mx0, __shfl_xor_sync(0xffffffffu, mx0, o));
        mn1 = fmin(mn1, __shfl_xor_sync(0xffffffffu, mn1, o)), mx1 = fmax(mx1, __shfl_xor_sync(0xffffffffu, mx1, o));
        mn2 = fmin(mn2, __shfl_xor_sync(0xffffffffu, mn2, o)), mx2 = fmax(mx2, __shfl_xor_sync(0xffffffffu, mx2, o));
        err |= __shfl_xor_sync(0xffffffffu, err, o);
    }
    if (lane == 0) {
        if (mn0 <= mx0) {
            atomicMin(&s_bb[0], double_to_ordered(mn0)), atomicMax(&s_bb[3], double_to_ordered(mx0));
            atomicMin(&s_bb[1], double_to_ordered(mn1)), atomicMax(&s_bb[4], double_to_ordered(mx1));
            atomicMin(&s_bb[2], double_to_ordered(mn2)), atomicMax(&s_bb[5], double_to_ordered(mx2));
        }
        if (err) atomicOr(&s_err, err);
    }
    __syncthreads();
    uint32_t* cube = reinterpret_cast<uint32_t*>(my_ctrl + XchgCtrl::CUBE);
    if (tid < p.world) {
        const uint32_t c = s_cnt[tid];
        tile_cnt[(size_t)tid * n_tiles + tile] = c;
        if (c) atomicAdd(&cube[(size_t)tid * p.n_poses + T.pose], c);
    }
    if (tid < 3 && s_bb[tid] != LLONG_MAX) atomicMin(reinterpret_cast<long long*>(my_ctrl + XchgCtrl::BBOX) + tid, s_bb[tid]);
    if (tid >= 3 && tid < 6 && s_bb[tid] != LLONG_MIN) atomicMax(reinterpret_cast<long long*>(my_ctrl + XchgCtrl::BBOX) + tid, s_bb[tid]);
    if (tid == 0 && s_err) atomicOr(reinterpret_cast<uint32_t*>(my_ctrl + XchgCtrl::ERR), s_err);
}

// ---- flag round B + routing plan: CTA s handles source rank s; the last CTA to finish derives the bases and the summary ----
__global__ void __launch_bounds__(256) xchg_sync_b_kernel(XParams p, const __grid_constant__ XPeers peers, unsigned char* scratch,
                                                          unsigned char* host) {
    __shared__ uint32_t s_red[8];
    __shared__ int s_flag;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = blockIdx.x;
    unsigned char* my_ctrl = peers.ctrl[p.rank];
    uint32_t* misc = reinterpret_cast<uint32_t*>(scratch + XScratch::MISC);
    if (tid == 0) {
        signal_peer(peers.ctrl[s], 1, p.rank, p.epoch);
        s_flag = wait_flag(my_ctrl, 1, s, p.epoch) ? 1 : 0;
        if (!s_flag) atomicOr(&misc[2], XERR_TIMEOUT);
    }
    __syncthreads();
    const bool ok = s_flag != 0;
    const unsigned char* c = peers.ctrl[s];
    const uint32_t* cube = reinterpret_cast<const uint32_t*>(c + XchgCtrl::CUBE);
    uint32_t* tot = reinterpret_cast<uint32_t*>(scratch + XScratch::TOT);
    uint32_t* psz = reinterpret_cast<uint32_t*>(scratch + XScratch::pose_size(p.world));
    volatile uint32_t* h_recv = reinterpret_cast<volatile uint32_t*>(host + XchgHost::COUNTS);
    if (ok) {
        for (int d = 0; d < p.world; ++d) {
            uint32_t sum = 0;
            for (int q = tid; q < p.n_poses; q += 256) {
                const uint32_t v = cube[(size_t)d * p.n_poses + q];
                sum += v;
                if (v) atomicAdd(&psz[(size_t)d * p.n_poses + q], v);
                if (d == p.rank) h_recv[(size_t)s * p.n_poses + q] = v;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            if (lane == 0) s_red[warp] = sum;
            __syncthreads();
            if (tid == 0) {
                uint32_t t = 0;
                for (int w = 0; w < 8; ++w) t += s_red[w];
                tot[s * XCHG_MAX_WORLD + d] = t;
            }
            __syncthreads();
        }
        if (tid < 3) atomicMin(reinterpret_cast<long long*>(scratch + XScratch::BBOX) + tid, reinterpret_cast<const long long*>(c + XchgCtrl::BBOX)[tid]);
        if (tid >= 3 && tid < 6) atomicMax(reinterpret_cast<long long*>(scratch + XScratch::BBOX) + tid, reinterpret_cast<const long long*>(c + XchgCtrl::BBOX)[tid]);
        if (tid == 6) atomicOr(&misc[2], *reinterpret_cast<const uint32_t*>(c + XchgCtrl::ERR));
    }
    // last CTA: bases, overflow check, cell-coordinate range, summary for the host
    __threadfence();
    __syncthreads();
    if (tid == 0) s_flag = (atomicAdd(&misc[0], 1u) == (uint32_t)p.world - 1u) ? 1 : 0;
    __syncthreads();
    if (!s_flag) return;
    __threadfence();
    volatile long long* hdr = reinterpret_cast<volatile long long*>(host + XchgHost::HDR);
    long long* base = reinterpret_cast<long long*>(scratch + XScratch::BASE);
    const volatile uint32_t* vtot = tot;
    __shared__ long long s_max;
    if (tid == 0) s_max = 0;
    __syncthreads();
    if (tid < p.world) {
        long long b = 0, all = 0;
        for (int r = 0; r < p.world; ++r) {
            const long long v = (long long)vtot[r * XCHG_MAX_WORLD + tid];
            if (r < p.rank) b += v;
            all += v;
        }
        base[tid] = b;
        atomicMax(&s_max, all);
        if (tid == p.rank) hdr[9] = all;
    }
    __syncthreads();
    if (tid == 0) {
        const long long mx = s_max;
        hdr[1] = mx;
        if (mx > p.rows_cap) misc[1] = 1u;
        uint32_t err = *reinterpret_cast<volatile uint32_t*>(&misc[2]);
        const volatile long long* bb = reinterpret_cast<const volatile long long*>(scratch + XScratch::BBOX);
        const long long* bounds = reinterpret_cast<const long long*>(scratch + XScratch::BOUNDS);
        const double corner[3] = {p.c0, p.c1, p.c2};
        for (int a = 0; a < 3; ++a) {
            long long qlo = 0, qhi = 0;
            if (bb[a] <= bb[3 + a]) {
                const double lo = cell_coord(ordered_to_double(bb[a]), corner[a], p.edge);
                const double hi = cell_coord(ordered_to_double(bb[3 + a]), corner[a], p.edge);
                if (fabs(lo) < 4503599627370496.0 && fabs(hi) < 4503599627370496.0) {
                    qlo = (long long)lo;
                    qhi = (long long)hi;
                } else
                    err |= DEVERR_CELL_RANGE;
            }
            if (a == 0 && p.slabs) {  // only cells of this rank's slab can arrive
                if (p.rank > 0 && bounds[p.rank - 1] > qlo) qlo = bounds[p.rank - 1];
                if (p.rank < p.world - 1 && bounds[p.rank] - 1 < qhi) qhi = bounds[p.rank] - 1;
                if (qhi < qlo) qhi = qlo;
            }
            hdr[2 + a] = qlo;
            hdr[5 + a] = qhi;
        }
        hdr[0] = (long long)err;
        if (err & XERR_TIMEOUT) hdr[8] = 1;
    }
    volatile uint32_t* h_psz = h_recv + (size_t)p.world * p.n_poses;
    const volatile uint32_t* vpsz = psz;
    for (size_t i = tid; i < (size_t)p.world * p.n_poses; i += 256) h_psz[i] = vpsz[i];
    __threadfence_system();
}

// ---- scatter pass ---------------------------------------------------------------------------------------------------------
// dynamic shared memory: double pts[XCHG_TILE * 3] | uint32 wcnt[64 groups][world] | uint16 pos[XCHG_TILE] | per-owner tables
__global__ void __launch_bounds__(256) xchg_scatter_kernel(const XTile* __restrict__ tiles, uint32_t n_tiles, XParams p,
                                                           const uint8_t* __restrict__ owner, const uint32_t* __restrict__ tile_off,
                                                           const unsigned char* __restrict__ scratch,
                                                           const __grid_constant__ XPeers peers) {
    extern __shared__ __align__(16) unsigned char smem[];
    if (reinterpret_cast<const uint32_t*>(scratch + XScratch::MISC)[1]) return;  // a receive buffer would overflow: nothing is written
    const int W = p.world;
    double* s_pts = reinterpret_cast<double*>(smem);
    uint32_t* s_wcnt = reinterpret_cast<uint32_t*>(smem + (size_t)XCHG_TILE * 24);
    uint16_t* s_pos = reinterpret_cast<uint16_t*>(s_wcnt + 64 * W);
    uint32_t* s_first = reinterpret_cast<uint32_t*>(s_pos + XCHG_TILE);     // [W + 1] first staged row of every owner
    long long* s_row0 = reinterpret_cast<long long*>(s_first + XCHG_MAX_WORLD + 2);  // [W] destination row of that first row
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tile = blockIdx.x;
    const XTile T = tiles[tile];
    for (int i = tid; i < 64 * W; i += 256) s_wcnt[i] = 0u;
    __syncthreads();
    uint32_t own[XCHG_TILE / 256], rnk[XCHG_TILE / 256];
#pragma unroll
    for (int r = 0; r < XCHG_TILE / 256; ++r) {  // every owner byte of the thread first, then the warp-synchronous ranking
        const uint32_t idx = (uint32_t)r * 256u + (uint32_t)tid;
        own[r] = idx < T.n ? (uint32_t)owner[(size_t)T.first_row + idx] : 0xffffffffu;
    }
#pragma unroll
    for (int r = 0; r < XCHG_TILE / 256; ++r) {
        const uint32_t o = own[r];
        const uint32_t m = __match_any_sync(0xffffffffu, o);
        rnk[r] = (uint32_t)__popc(m & ((1u << lane) - 1u));
        if (o != 0xffffffffu && lane == __ffs(m) - 1) s_wcnt[(r * 8 + warp) * W + (int)o] = (uint32_t)__popc(m);
    }
    __syncthreads();
    if (tid < W) {  // exclusive scan over the 64 (round, warp) groups, per owner
        uint32_t run = 0;
        for (int g = 0; g < 64; ++g) {
            const uint32_t c = s_wcnt[g * W + tid];
            s_wcnt[g * W + tid] = run;
            run += c;
        }
        s_first[tid + 1] = run;  // counts for now
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t run = 0;
        s_first[0] = 0;
        for (int o = 0; o < W; ++o) {
            const uint32_t c = s_first[o + 1];
            s_first[o + 1] = run + c;
            run += c;
        }
    }
    __syncthreads();
    if (tid < W) {
        const long long* base = reinterpret_cast<const long long*>(scratch + XScratch::BASE);
        s_row0[tid] = base[tid] + (long long)(tile_off[(size_t)tid * n_tiles + tile] - tile_off[(size_t)tid * n_tiles]);
    }
#pragma unroll
    for (int r = 0; r < XCHG_TILE / 256; ++r) {
        const uint32_t idx = (uint32_t)r * 256u + (uint32_t)tid;
        if (own[r] != 0xffffffffu) s_pos[idx] = (uint16_t)(s_first[own[r]] + s_wcnt[(r * 8 + warp) * W + (int)own[r]] + rnk[r]);
    }
    __syncthreads();
    const uint32_t nd = T.n * 3u;
    for (uint32_t f = tid; f < nd; f += 256) {  // coalesced read of the tile, grouped by owner in shared memory
        const uint32_t row = f / 3u, cc = f - row * 3u;
        s_pts[(uint32_t)s_pos[row] * 3u + cc] = T.src[f];
    }
    __syncthreads();
    for (uint32_t f = tid; f < nd; f += 256) {  // contiguous runs straight into the owners' receive buffers
        const uint32_t row = f / 3u, cc = f - row * 3u;
        int o = 0;
        while (o + 1 < W && s_first[o + 1] <= row) ++o;
        peers.data[o][(size_t)(s_row0[o] + (long long)(row - s_first[o])) * 3 + cc] = s_pts[f];
    }
}

// flag round C: every rank's rows have landed in this rank's receive buffer
__global__ void xchg_sync_c_kernel(XParams p, const __grid_constant__ XPeers peers, unsigned char* scratch, unsigned char* host) {
    const int tid = threadIdx.x;
    if (tid < p.world) {
        signal_peer(peers.ctrl[tid], 2, p.rank, p.epoch);
        if (!wait_flag(peers.ctrl[p.rank], 2, tid, p.epoch)) {
            atomicOr(reinterpret_cast<uint32_t*>(scratch + XScratch::MISC) + 2, XERR_TIMEOUT);
            reinterpret_cast<volatile long long*>(host + XchgHost::HDR)[8] = 1;
        }
    }
}

}  // namespace

Exchange::Exchange(int world_, int rank_, int n_poses_, int64_t rows_cap_, int nbuf_, void* const* ctrl_ptrs, void* const* data_ptrs,
                   int device_)
    : world(world_), rank(rank_), n_poses(n_poses_), nbuf(nbuf_), device(device_), rows_cap(rows_cap_) {
    OL_REQUIRE(world >= 1 && world <= XCHG_MAX_WORLD && rank >= 0 && rank < world && n_poses >= 1 && nbuf >= 1 && rows_cap >= 0,
               OL_ERR_INVALID, "bad exchange arguments");
    OL_CUDA(cudaSetDevice(device));
    for (int r = 0; r < world; ++r) ctrl.push_back(static_cast<unsigned char*>(ctrl_ptrs[r]));
    for (int k = 0; k < nbuf * world; ++k) data.push_back(static_cast<double*>(data_ptrs[k]));
    OL_CUDA(cudaMallocHost(reinterpret_cast<void**>(&host), XchgHost::bytes(world, n_poses)));
    memset(host, 0, XchgHost::bytes(world, n_poses));
    scratch_bytes = XScratch::bytes(world, n_poses);
    OL_CUDA(cudaMalloc(reinterpret_cast<void**>(&scratch), scratch_bytes));
    OL_CUDA(cudaMemset(scratch, 0, scratch_bytes));
    OL_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    OL_CUDA(cudaFuncSetAttribute(xchg_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
}

Exchange::~Exchange() {
    if (ev) cudaEventDestroy(ev);
    if (scratch) cudaFree(scratch);
    if (host) cudaFreeHost(host);
}

void Exchange::run(Forest& f, const double* const* clouds, const int64_t* sizes, const int32_t* poses, int count, int slabs, int buf,
                   int64_t* info, int64_t* bounds_out, uint32_t* pose_sizes_out) {
    OL_REQUIRE(f.N == 0 && f.n_poses == 0, OL_ERR_STATE, "the exchange fills an empty forest");
    OL_REQUIRE(buf >= 0 && buf < nbuf && count >= 0, OL_ERR_INVALID, "bad exchange arguments");
    Ctx& c = f.ctx;
    cudaStream_t st = c.stream;
    // tile table of the local clouds (poses ascending, so that a (source rank, pose) run is contiguous at the receiver)
    std::vector<XCloud> cloud_rows;
    cloud_rows.reserve((size_t)count);
    size_t n_local = 0, n_tiles_sz = 0;
    int last_pose = -1;
    for (int k = 0; k < count; ++k) {
        OL_REQUIRE(sizes[k] >= 0 && poses[k] >= 0 && poses[k] < n_poses, OL_ERR_POSE, "pose number out of range");
        OL_REQUIRE(poses[k] >= last_pose, OL_ERR_INVALID, "clouds must be ordered by pose number");
        last_pose = poses[k];
        if (sizes[k] > 0) cloud_rows.push_back(XCloud{clouds[k], (uint32_t)sizes[k], (uint32_t)n_local, (uint32_t)n_tiles_sz, poses[k]});
        n_tiles_sz += (size_t)((sizes[k] + XCHG_TILE - 1) / XCHG_TILE);
        n_local += (size_t)sizes[k];
        OL_REQUIRE(n_local < (1ull << 31), OL_ERR_INVALID, "more than 2^31 - 1 points per rank are not supported");
    }
    const uint32_t n_tiles = (uint32_t)n_tiles_sz;
    ++epoch;
    XParams p{};
    p.edge = f.cfg.voxel_edge_length;
    p.inv_edge = pow2_reciprocal(p.edge);
    p.c0 = f.cfg.corner[0], p.c1 = f.cfg.corner[1], p.c2 = f.cfg.corner[2];
    p.world = world, p.rank = rank, p.n_poses = n_poses, p.slabs = slabs ? 1 : 0;
    p.rows_cap = rows_cap;
    p.epoch = epoch;
    XPeers peers{};
    for (int r = 0; r < world; ++r) {
        peers.ctrl[r] = ctrl[r];
        peers.data[r] = data[(size_t)buf * world + r];
    }
    unsigned char* my_ctrl = ctrl[rank];
    DevBuf<XTile> d_tiles(c, std::max<size_t>(n_tiles, 1));
    DevBuf<uint8_t> d_owner(c, std::max<size_t>(n_local, 1));
    DevBuf<uint32_t> tile_cnt(c, (size_t)world * std::max<uint32_t>(n_tiles, 1));
    DevBuf<XCloud> d_clouds(c, std::max<size_t>(cloud_rows.size(), 1));
    h2d(c, d_clouds.get(), cloud_rows.data(), cloud_rows.size());
    if (n_tiles) {
        xchg_tiles_kernel<<<(n_tiles + 255) / 256, 256, 0, st>>>(d_clouds.get(), (int)cloud_rows.size(), n_tiles, d_tiles.get());
        OL_CHECK_LAUNCH();
    }
    volatile long long* hdr = reinterpret_cast<volatile long long*>(host + XchgHost::HDR);
    hdr[8] = 0;
    {
        ProfScope ps(c, "exchange_plan", (double)n_local);
        const size_t init_n = std::max<size_t>((size_t)world * n_poses, 64 * 64);
        xchg_init_kernel<<<(unsigned)((init_n + 255) / 256), 256, 0, st>>>(my_ctrl, scratch, world, n_poses);
        OL_CHECK_LAUNCH();
        if (slabs && world > 1) {
            if (n_tiles) {
                const unsigned g = std::min<unsigned>(n_tiles, (unsigned)c.num_sms * 8);
                xchg_range_kernel<<<g, 256, 0, st>>>(d_tiles.get(), n_tiles, p, my_ctrl);
                OL_CHECK_LAUNCH();
                xchg_hist_kernel<<<g, 256, 0, st>>>(d_tiles.get(), n_tiles, p, my_ctrl);
                OL_CHECK_LAUNCH();
            }
            xchg_sync_a_kernel<<<1, 1024, 0, st>>>(p, peers, scratch, host);
            OL_CHECK_LAUNCH();
        }
        if (n_tiles) {
            xchg_count_kernel<<<n_tiles, 256, 0, st>>>(d_tiles.get(), n_tiles, p, reinterpret_cast<const long long*>(scratch + XScratch::BOUNDS),
                                                      d_owner.get(), tile_cnt.get(), my_ctrl);
            OL_CHECK_LAUNCH();
            exclusive_scan_u32(c, tile_cnt.get(), tile_cnt.get(), (size_t)world * n_tiles, nullptr);
        }
        xchg_sync_b_kernel<<<world, 256, 0, st>>>(p, peers, scratch, host);
        OL_CHECK_LAUNCH();
    }
    OL_CUDA(cudaEventRecord(ev, st));
    {
        ProfScope ps(c, "exchange_route", (double)n_local);
        if (n_tiles) {
            const size_t smem = (size_t)XCHG_TILE * 24 + 4 * 64 * (size_t)world + 2 * XCHG_TILE + 4 * (XCHG_MAX_WORLD + 2) + 8 * XCHG_MAX_WORLD + 16;
            xchg_scatter_kernel<<<n_tiles, 256, smem, st>>>(d_tiles.get(), n_tiles, p, d_owner.get(), tile_cnt.get(), scratch, peers);
            OL_CHECK_LAUNCH();
        }
        xchg_sync_c_kernel<<<1, XCHG_MAX_WORLD, 0, st>>>(p, peers, scratch, host);
        OL_CHECK_LAUNCH();
    }
    // the ONE host wait of the exchange: the routing plan (the scatter and flag round C run meanwhile)
    OL_CUDA(cudaEventSynchronize(ev));
    const long long err = hdr[0], max_recv = hdr[1], received = hdr[9];
    OL_REQUIRE(!hdr[8] && !(err & XERR_TIMEOUT), OL_ERR_STATE, "multi-GPU exchange timed out waiting for a peer rank");
    OL_REQUIRE(!(err & DEVERR_NONFINITE), OL_ERR_NONFINITE, "point cloud contains NaN or infinite coordinates");
    OL_REQUIRE(!(err & DEVERR_CELL_RANGE), OL_ERR_RANGE, "cell coordinates out of the representable range");
    const uint32_t* h_recv = reinterpret_cast<const uint32_t*>(host + XchgHost::COUNTS);
    const uint32_t* h_psz = h_recv + (size_t)world * n_poses;
    if (info) {
        long long kept = 0;
        for (int q = 0; q < n_poses; ++q) kept += h_recv[(size_t)rank * n_poses + q];
        info[0] = (int64_t)n_local - kept;
        info[1] = received;
        info[2] = kept;
        info[3] = max_recv;
    }
    if (bounds_out)
        for (int k = 0; k + 1 < world; ++k) bounds_out[k] = slabs ? reinterpret_cast<const long long*>(host + XchgHost::BOUNDS)[k] : 0;
    if (pose_sizes_out) memcpy(pose_sizes_out, h_psz, 4 * (size_t)world * n_poses);
    if (max_recv > rows_cap) {
        c.sync();  // the skipped scatter and round C have drained; the caller grows the buffers (every rank saw the same totals)
        throw Error{OL_ERR_CAPACITY, "receive buffer too small: " + std::to_string(max_recv) + " rows needed"};
    }
    // (source rank, pose) runs of what arrives, in buffer order
    std::vector<int64_t> seg_sizes, seg_first;
    std::vector<int32_t> seg_pose;
    std::vector<long long> before((size_t)n_poses, 0);
    for (int s = 0; s < world; ++s)
        for (int q = 0; q < n_poses; ++q) {
            const uint32_t v = h_recv[(size_t)s * n_poses + q];
            if (!v) continue;
            seg_sizes.push_back(v);
            seg_pose.push_back(q);
            seg_first.push_back(before[q]);
            before[q] += v;
        }
    const long long qlo[3] = {hdr[2], hdr[3], hdr[4]}, qhi[3] = {hdr[5], hdr[6], hdr[7]};
    f.adopt_points(data[(size_t)buf * world + rank], (size_t)received, seg_sizes.data(), seg_pose.data(), seg_first.data(),
                   (int)seg_sizes.size(), n_poses, qlo, qhi);
    // Keys, sort and cell table are enqueued right behind the scatter (the cell-coordinate range came with the plan, so
    // nothing has to be read back first): the GPU keeps working while the host language returns from this call and
    // prepares the next one; the number of cells is picked up from the mailbox by that next call.
    f.build_enqueue();
}

}  // namespace ol
