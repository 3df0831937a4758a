// Device-wide primitives used by the forest pipeline: exclusive scan (u32), stable LSD radix sort of (key, u32 value)
// pairs (onesweep.cuh below 2^30 pairs, the three-kernel sort in this file above), run segmentation (one pass).
// All work is enqueued on Ctx::stream; temporaries come from Ctx::alloc.
#pragma once
#include "common.cuh"
#include "onesweep.cuh"

#include <type_traits>

namespace ol {

// =============================================================================================
// exclusive scan (uint32 / packed uint64), ONE kernel per call
//   n <= SCAN_SMALL_MAX : a single CTA walks the input in chunks (launch-latency bound inputs: tile counts, tables)
//   otherwise           : single-pass chained scan with decoupled look-back over 256 x ITEMS element tiles
//                         (tile order by an atomic ticket, two 64-bit status words per tile: aggregate / inclusive
//                         prefix, top bit = valid, so the word itself carries the data and no fence is needed).
// Traffic: element read once, written once.  All partial sums are carried in 64 bits; the outputs wrap to T.
// The uint64 form scans two packed 32-bit counters at once (hi | lo, no carry between them as long as the low
// total stays below 2^32) - used where two scans over the same index space would otherwise be needed.
// =============================================================================================
constexpr int SCAN_THREADS = 256;
constexpr size_t SCAN_SMALL_MAX = 16384;
constexpr unsigned long long SCAN_VALID = 1ull << 63;

__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) >= o) v += t;
    }
    return v;
}
__device__ __forceinline__ unsigned long long warp_inclusive_scan64(unsigned long long v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned long long t = __shfl_up_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) >= o) v += t;
    }
    return v;
}

// exclusive scan of one value per thread across a 256-thread block; returns block total via *total
__device__ __forceinline__ uint32_t block_exclusive_scan_256(uint32_t v, uint32_t* smem_warp /*[8]*/, uint32_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = warp_inclusive_scan(v);
    if (lane == 31) smem_warp[warp] = inc;
    __syncthreads();
    uint32_t wsum = (lane < 8) ? smem_warp[lane] : 0;
    uint32_t winc = warp_inclusive_scan(wsum);
    uint32_t wbase = __shfl_sync(0xffffffffu, winc - wsum, warp);
    uint32_t tot = __shfl_sync(0xffffffffu, winc, 7);
    __syncthreads();
    if (total) *total = tot;
    return wbase + inc - v;
}

// the same in 64 bits for any block size that is a multiple of 32 (<= 1024 threads)
__device__ __forceinline__ unsigned long long block_exclusive_scan64(unsigned long long v, unsigned long long* smem_warp /*[32]*/,
                                                                    unsigned long long* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    unsigned long long inc = warp_inclusive_scan64(v);
    if (lane == 31) smem_warp[warp] = inc;
    __syncthreads();
    unsigned long long wsum = (lane < nwarps) ? smem_warp[lane] : 0ull;
    unsigned long long winc = warp_inclusive_scan64(wsum);
    unsigned long long wbase = __shfl_sync(0xffffffffu, winc - wsum, warp);
    unsigned long long tot = __shfl_sync(0xffffffffu, winc, nwarps - 1);
    __syncthreads();
    if (total) *total = tot;
    return wbase + inc - v;
}

__device__ __forceinline__ unsigned long long scan_ld_status(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void scan_st_status(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// both status words of a tile (aggregate, inclusive prefix) in ONE 16-byte load: every word validates itself (top bit), so
// it does not matter whether the pair is read atomically - and a look-back round costs one trip to L2 instead of two
__device__ __forceinline__ void scan_ld_status2(const unsigned long long* p, unsigned long long& agg, unsigned long long& inc) {
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(agg), "=l"(inc) : "l"(p) : "memory");
}
// Chained-scan building block: the calling CTA owns tile `tile` (tiles are taken in ticket order) with aggregate
// `aggregate`; returns the sum of the aggregates of all earlier tiles (valid in every thread after the internal
// barriers) and publishes this tile's inclusive prefix.  status = [2 * tiles] words, zero-initialised:
// status[2 t] = aggregate of tile t, status[2 t + 1] = inclusive prefix through tile t, both | SCAN_VALID.
__device__ __forceinline__ unsigned long long lookback_exclusive_prefix(unsigned long long* __restrict__ status, uint32_t tile,
                                                                        unsigned long long aggregate,
                                                                        unsigned long long* s_prefix /*shared, 1 word (unused)*/) {
    // The WHOLE CTA looks back, blockDim.x predecessors per round.  All tiles of a launch become resident at about the
    // same time (a B200 holds more than a thousand 256-thread CTAs), so the nearest predecessor that already knows its
    // inclusive prefix is typically hundreds of tiles away: with one warp per round (32 tiles, one trip to L2 each) the
    // look-back alone took 15-25 us per scan; with 256 tiles per round it is a handful of rounds.
    (void)s_prefix;
    __shared__ unsigned long long s_sum[32];
    __shared__ uint32_t s_stop[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (int)(blockDim.x >> 5);
    if (threadIdx.x == 0) scan_st_status(status + 2 * (size_t)tile + (tile == 0 ? 1 : 0), SCAN_VALID | aggregate);
    unsigned long long prefix = 0;
    if (tile > 0) {
        long long look = (long long)tile - 1;
        while (true) {
            const long long idx = look - (long long)threadIdx.x;
            unsigned long long val = 0;
            bool stop = idx < 0;  // before the first tile: an inclusive prefix of 0
            if (idx >= 0) {
                while (true) {
                    unsigned long long agg, inc;
                    scan_ld_status2(status + 2 * (size_t)idx, agg, inc);
                    if (inc & SCAN_VALID) {
                        val = inc & ~SCAN_VALID;
                        stop = true;
                        break;
                    }
                    if (agg & SCAN_VALID) {
                        val = agg & ~SCAN_VALID;
                        break;
                    }
                }
            }
            const uint32_t stopmask = __ballot_sync(0xffffffffu, stop);
            const int first = stopmask ? (__ffs(stopmask) - 1) : 32;
            unsigned long long v = (lane <= first) ? val : 0ull;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) {
                s_sum[warp] = v;
                s_stop[warp] = stopmask ? 1u : 0u;
            }
            __syncthreads();
            bool done = false;
            for (int w = 0; w < nwarps; ++w) {  // warps in look-back order: nearest predecessors first
                prefix += s_sum[w];
                if (s_stop[w]) {
                    done = true;
                    break;
                }
            }
            __syncthreads();  // the partial sums are overwritten by the next round
            if (done) break;
            look -= (long long)blockDim.x;
        }
        if (threadIdx.x == 0) scan_st_status(status + 2 * (size_t)tile + 1, SCAN_VALID | (prefix + aggregate));
    }
    return prefix;
}

// input / output functors of the scans: in(i) -> T, out(i, exclusive prefix, in(i)); the plain forms read / write arrays
template <typename T>
struct ScanPtrIn {
    const T* p;
    __device__ __forceinline__ T operator()(size_t i) const { return p[i]; }
};
template <typename T>
struct ScanPtrOut {
    T* p;
    __device__ __forceinline__ void operator()(size_t i, T ex, T) const { p[i] = ex; }
};

template <typename T, int ITEMS, typename InFn, typename OutFn>
__global__ void __launch_bounds__(SCAN_THREADS) scan_lookback_kernel(InFn in, OutFn out, size_t n, uint32_t num_tiles,
                                                                      unsigned long long* __restrict__ status,
                                                                      unsigned long long* __restrict__ total_out, const Mail mail) {
    constexpr int TILE = SCAN_THREADS * ITEMS;
    __shared__ T tile[TILE + TILE / 32];
    __shared__ unsigned long long sw[32];
    __shared__ unsigned long long s_prefix;
    __shared__ uint32_t s_tile;
    if (threadIdx.x == 0) s_tile = atomicAdd(reinterpret_cast<uint32_t*>(status + 2 * (size_t)num_tiles), 1u);
    __syncthreads();
    const uint32_t t = s_tile;
    const size_t base = (size_t)t * TILE;
    {
        // all inputs of the thread first, THEN the shared-memory stores: the loads behind in(i) are independent and must be
        // in flight together (a store between two of them makes the warp wait for each load in turn)
        T staged[ITEMS];
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            const size_t i = base + (size_t)(j * SCAN_THREADS + threadIdx.x);
            staged[j] = (i < n) ? in(i) : (T)0;
        }
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            const int li = j * SCAN_THREADS + threadIdx.x;
            tile[li + (li >> 5)] = staged[j];
        }
    }
    __syncthreads();
    T v[ITEMS];
    unsigned long long s = 0;
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const int li = threadIdx.x * ITEMS + j;
        v[j] = tile[li + (li >> 5)];
        s += (unsigned long long)v[j];
    }
    unsigned long long tot;
    unsigned long long ex = block_exclusive_scan64(s, sw, &tot);
    const unsigned long long prefix = lookback_exclusive_prefix(status, t, tot, &s_prefix);
    if (t == num_tiles - 1 && threadIdx.x == 0) {
        if (total_out) *total_out = prefix + tot;
        mail_post(mail, prefix + tot);
    }
    ex += prefix;
    // the tile buffer now carries the exclusive prefixes back to the coalesced arrangement; the values stay in a
    // second pass through it only when the output functor needs them (cheap: shared memory)
    T w[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const int li = j * SCAN_THREADS + threadIdx.x;
        w[j] = tile[li + (li >> 5)];  // in(i) of the element this thread will write
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const int li = threadIdx.x * ITEMS + j;
        tile[li + (li >> 5)] = (T)ex;
        ex += (unsigned long long)v[j];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const int li = j * SCAN_THREADS + threadIdx.x;
        const size_t i = base + li;
        if (i < n) out(i, tile[li + (li >> 5)], w[j]);
    }
}

// single CTA (1024 threads, 4 consecutive elements per thread and chunk): inputs of a few thousand elements
template <typename T, typename InFn, typename OutFn>
__global__ void __launch_bounds__(1024) scan_small_kernel(InFn in, OutFn out, size_t n, unsigned long long* __restrict__ total_out,
                                                          const Mail mail) {
    __shared__ unsigned long long sw[32];
    unsigned long long carry = 0;
    for (size_t base = 0; base < n; base += 4096) {
        const size_t i0 = base + (size_t)threadIdx.x * 4;
        T v[4];
        unsigned long long s = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[j] = (i0 + j < n) ? in(i0 + j) : (T)0;
            s += (unsigned long long)v[j];
        }
        unsigned long long tot;
        unsigned long long ex = carry + block_exclusive_scan64(s, sw, &tot);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (i0 + j < n) out(i0 + j, (T)ex, v[j]);
            ex += (unsigned long long)v[j];
        }
        carry += tot;
    }
    if (threadIdx.x == 0) {
        if (total_out) *total_out = carry;
        mail_post(mail, carry);
    }
}

// out(i, sum_{j<i} in(j), in(i)) for i in [0, n).  If d_total != nullptr the 64-bit grand total is written there
// (device memory).  No host synchronisation.  `name` = profiler stage.
template <typename T, typename InFn, typename OutFn>
inline void transform_scan(Ctx& c, InFn in, OutFn out, size_t n, unsigned long long* d_total, const char* name = "scan",
                           const Mail& mail = Mail{}) {
    // n == 0 still launches (one CTA that finds nothing to do): the total and the mail are written by the kernel
    ProfScope ps(c, name, (double)n);
    if (n <= SCAN_SMALL_MAX) {
        scan_small_kernel<T, InFn, OutFn><<<1, 1024, 0, c.stream>>>(in, out, n, d_total, mail);
        OL_CHECK_LAUNCH();
        return;
    }
    constexpr int ITEMS = sizeof(T) == 4 ? 16 : 8;
    const size_t tiles = (n + SCAN_THREADS * ITEMS - 1) / (SCAN_THREADS * ITEMS);
    DevBuf<unsigned long long> own;
    unsigned long long* status = c.status_words(2 * tiles + 1);  // + the ticket counter
    if (!status) {
        own.reset(c, 2 * tiles + 1);
        own.zero();
        status = own.get();
    }
    scan_lookback_kernel<T, ITEMS, InFn, OutFn><<<(unsigned)tiles, SCAN_THREADS, 0, c.stream>>>(in, out, n, (uint32_t)tiles, status,
                                                                                              d_total, mail);
    OL_CHECK_LAUNCH();
}
// array form: out[i] = sum_{j<i} in[j]; in == out allowed
template <typename T>
inline void exclusive_scan(Ctx& c, const T* in, T* out, size_t n, unsigned long long* d_total) {
    transform_scan<T>(c, ScanPtrIn<T>{in}, ScanPtrOut<T>{out}, n, d_total);
}
inline void exclusive_scan_u32(Ctx& c, const uint32_t* in, uint32_t* out, size_t n, unsigned long long* d_total) {
    exclusive_scan<uint32_t>(c, in, out, n, d_total);
}

// =============================================================================================
// stable LSD radix sort of (key, u32 value) pairs.
// One pass = digit histogram per 4096-key tile -> exclusive scan of the (digit-major) count
// matrix -> stable scatter with warp-level match ranking.
// =============================================================================================
constexpr int SORT_THREADS = 256;
constexpr int SORT_ITEMS = 16;
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;
constexpr int SORT_WARPS = SORT_THREADS / 32;

template <typename KeyT>
__global__ void __launch_bounds__(SORT_THREADS) radix_hist_kernel(const KeyT* __restrict__ keys,
                                                                   uint32_t* __restrict__ counts, uint32_t n,
                                                                   uint32_t num_tiles, int shift, uint32_t nbins) {
    __shared__ uint32_t hist[256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = threadIdx.x; b < 256; b += SORT_THREADS) hist[b] = 0;
    __syncthreads();
    const uint32_t mask = nbins - 1;
    const uint32_t wbase = blockIdx.x * SORT_TILE + warp * (32 * SORT_ITEMS);
#pragma unroll 4
    for (int j = 0; j < SORT_ITEMS; ++j) {
        uint32_t i = wbase + j * 32 + lane;
        bool valid = i < n;
        uint32_t d = valid ? (uint32_t)((keys[i] >> shift) & mask) : 0xffffffffu;
        uint32_t peers = __match_any_sync(0xffffffffu, d);
        if (valid && lane == (__ffs(peers) - 1)) atomicAdd(&hist[d], __popc(peers));
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < nbins; b += SORT_THREADS) counts[(size_t)b * num_tiles + blockIdx.x] = hist[b];
}

template <typename KeyT>
__global__ void __launch_bounds__(SORT_THREADS) radix_scatter_kernel(const KeyT* __restrict__ keys_in,
                                                                      const uint32_t* __restrict__ vals_in,
                                                                      KeyT* __restrict__ keys_out,
                                                                      uint32_t* __restrict__ vals_out,
                                                                      const uint32_t* __restrict__ offsets, uint32_t n,
                                                                      uint32_t num_tiles, int shift, uint32_t nbins) {
    __shared__ uint32_t whist[SORT_WARPS][256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = threadIdx.x; b < SORT_WARPS * 256; b += SORT_THREADS) (&whist[0][0])[b] = 0;
    __syncthreads();
    const uint32_t mask = nbins - 1;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t wbase = blockIdx.x * SORT_TILE + warp * (32 * SORT_ITEMS);
    KeyT k[SORT_ITEMS];
    uint32_t rnk[SORT_ITEMS];
#pragma unroll
    for (int j = 0; j < SORT_ITEMS; ++j) {
        uint32_t i = wbase + j * 32 + lane;
        bool valid = i < n;
        k[j] = valid ? keys_in[i] : (KeyT)0;
        uint32_t d = valid ? (uint32_t)((k[j] >> shift) & mask) : 0xffffffffu;
        uint32_t peers = __match_any_sync(0xffffffffu, d);
        int leader = __ffs(peers) - 1;
        uint32_t old = 0;
        if (valid && lane == leader) {
            old = whist[warp][d];
            whist[warp][d] = old + __popc(peers);
        }
        old = __shfl_sync(0xffffffffu, old, leader);
        rnk[j] = old + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();
    // per digit: exclusive prefix over the warps of this tile, on top of the tile's global offset
    for (uint32_t b = threadIdx.x; b < nbins; b += SORT_THREADS) {
        uint32_t run = offsets[(size_t)b * num_tiles + blockIdx.x];
#pragma unroll
        for (int w = 0; w < SORT_WARPS; ++w) {
            uint32_t t = whist[w][b];
            whist[w][b] = run;
            run += t;
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < SORT_ITEMS; ++j) {
        uint32_t i = wbase + j * 32 + lane;
        if (i < n) {
            uint32_t d = (uint32_t)((k[j] >> shift) & mask);
            uint32_t dst = whist[warp][d] + rnk[j];
            keys_out[dst] = k[j];
            vals_out[dst] = vals_in[i];
        }
    }
}

// Sorts (keys0, vals0) by bits [begin_bit, end_bit) using (keys1, vals1) as the alternate buffer.
// Returns 0 if the result is in buffer 0, 1 if it is in buffer 1.  Onesweep (onesweep.cuh) below 2^30
// pairs; the three-kernel LSD sort in this file above that (and when g_force_legacy_sort is set: tests).
extern bool g_force_legacy_sort;
template <typename KeyT>
inline int radix_sort_pairs(Ctx& c, KeyT* keys0, KeyT* keys1, uint32_t* vals0, uint32_t* vals1, size_t n, int begin_bit,
                            int end_bit, bool main_sort = false) {
    OL_REQUIRE(n < (1ull << 31), OL_ERR_INVALID, "radix_sort_pairs: n must be < 2^31");
    int bits = end_bit - begin_bit;
    if (n <= 1 || bits <= 0) return 0;
    if (n < (1ull << 30) && !g_force_legacy_sort) return onesweep_sort_pairs<KeyT>(c, keys0, keys1, vals0, vals1, n, begin_bit, end_bit, main_sort);
    int passes = (bits + 7) / 8;
    int per = (bits + passes - 1) / passes;
    uint32_t tiles = (uint32_t)((n + SORT_TILE - 1) / SORT_TILE);
    DevBuf<uint32_t> counts(c, (size_t)256 * tiles);
    int cur = 0;
    int bit = begin_bit;
    for (int p = 0; p < passes; ++p) {
        int nb = (end_bit - bit < per) ? (end_bit - bit) : per;
        uint32_t nbins = 1u << nb;
        KeyT* kin = cur ? keys1 : keys0;
        KeyT* kout = cur ? keys0 : keys1;
        uint32_t* vin = cur ? vals1 : vals0;
        uint32_t* vout = cur ? vals0 : vals1;
        {
            ProfScope ps(c, sizeof(KeyT) == 8 ? "radix_hist_u64" : "radix_hist_u32", (double)n);
            radix_hist_kernel<KeyT><<<tiles, SORT_THREADS, 0, c.stream>>>(kin, counts.get(), (uint32_t)n, tiles, bit, nbins);
            OL_CHECK_LAUNCH();
        }
        exclusive_scan_u32(c, counts.get(), counts.get(), (size_t)nbins * tiles, nullptr);
        {
            ProfScope ps(c, sizeof(KeyT) == 8 ? "radix_scatter_u64" : "radix_scatter_u32", (double)n);
            radix_scatter_kernel<KeyT><<<tiles, SORT_THREADS, 0, c.stream>>>(kin, vin, kout, vout, counts.get(), (uint32_t)n,
                                                                               tiles, bit, nbins);
            OL_CHECK_LAUNCH();
        }
        cur ^= 1;
        bit += nb;
    }
    return cur;
}

// =============================================================================================
// run segmentation: maximal runs of equal key(i) over i in [0, n)  (K3 cells, (cell, pose) pairs, (pose, leaf) blocks)
//   runs_fused_kernel  head flags per 2048-element tile, chained scan of the tile head counts (decoupled look-back), ranks
//                      the heads with ballots, writes run_of_pos[i] and calls emit(run, i, key) for every head
// Traffic: the key inputs are read ONCE and run_of_pos is written once; no flag / scan arrays of length n.
// KeyFn:  __device__ uint64_t operator()(uint32_t i) const;      EmitFn: __device__ void operator()(uint32_t run, uint32_t i, uint64_t key) const
// =============================================================================================
constexpr int RUNS_THREADS = 256;
constexpr int RUNS_ITEMS = 8;
constexpr int RUNS_TILE = RUNS_THREADS * RUNS_ITEMS;

// A key functor may come in two stages: `load(i)` (the element's own coalesced loads) and `finish(loaded)` (what
// depends on them, e.g. a table search).  The kernels then issue the loads of all RUNS_ITEMS elements of a thread
// before the first search: with one stage, a search between two elements kept one DRAM load per thread in flight.
template <typename KeyFn, typename = void>
struct RunKey {
    static __device__ __forceinline__ uint64_t load(const KeyFn& k, uint32_t i) { return k(i); }
    static __device__ __forceinline__ uint64_t finish(const KeyFn&, uint64_t v) { return v; }
};
template <typename KeyFn>
struct RunKey<KeyFn, std::void_t<decltype(&KeyFn::finish)>> {
    static __device__ __forceinline__ uint64_t load(const KeyFn& k, uint32_t i) { return k.load(i); }
    static __device__ __forceinline__ uint64_t finish(const KeyFn& k, uint64_t v) { return k.finish(v); }
};

template <typename KeyFn>
__device__ __forceinline__ void runs_warp_flags(const KeyFn& key, uint32_t wbase, uint32_t n, int lane, uint32_t masks[RUNS_ITEMS],
                                                uint64_t keys[RUNS_ITEMS]) {
    // the warp walks RUNS_ITEMS x 32 consecutive elements; element (j, lane) = wbase + 32 j + lane
    uint64_t carry = 0;  // key of the element just before the current group of 32 (valid in every lane)
    bool have_carry = false;
    if (wbase > 0 && wbase < n) {
        carry = key(wbase - 1);
        have_carry = true;
    }
    // every key of the lane first (independent loads, all in flight together), then the shuffles
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j) {
        const uint32_t i = wbase + 32 * j + lane;
        keys[j] = i < n ? RunKey<KeyFn>::load(key, i) : 0ull;
    }
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j)
        if (wbase + 32 * j + lane < n) keys[j] = RunKey<KeyFn>::finish(key, keys[j]);
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j) {
        const uint32_t i = wbase + 32 * j + lane;
        const bool valid = i < n;
        const uint64_t k = keys[j];
        uint64_t prev = __shfl_up_sync(0xffffffffu, k, 1);
        bool has_prev = true;
        if (lane == 0) {
            prev = carry;
            has_prev = have_carry;
        }
        const bool head = valid && (!has_prev || prev != k);
        masks[j] = __ballot_sync(0xffffffffu, head);
        carry = __shfl_sync(0xffffffffu, k, 31);
        have_carry = true;
    }
}

// ONE pass: head flags per tile (ballots), chained scan of the tile head counts with decoupled look-back
// (lookback_exclusive_prefix above), emit.  The number of runs is only known when the kernel has finished, so the
// caller sizes the run tables by an upper bound (n, or what the key space allows) and reads *total_out afterwards.
template <typename KeyFn, typename EmitFn>
__global__ void __launch_bounds__(RUNS_THREADS) runs_fused_kernel(KeyFn key, EmitFn emit, uint32_t n, uint32_t num_tiles,
                                                                  unsigned long long* __restrict__ status,
                                                                  uint32_t* __restrict__ run_of_pos,
                                                                  unsigned long long* __restrict__ total_out,
                                                                  uint32_t* __restrict__ sentinel, const Mail mail) {
    __shared__ uint32_t s_w[RUNS_THREADS / 32];
    __shared__ unsigned long long s_prefix;
    __shared__ uint32_t s_tile;
    if (threadIdx.x == 0) s_tile = atomicAdd(reinterpret_cast<uint32_t*>(status + 2 * (size_t)num_tiles), 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t wbase = tile * RUNS_TILE + warp * (32 * RUNS_ITEMS);
    uint32_t masks[RUNS_ITEMS];
    uint64_t keys[RUNS_ITEMS];
    runs_warp_flags(key, wbase, n, lane, masks, keys);
    uint32_t cnt = 0;
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j) cnt += __popc(masks[j]);
    if (lane == 0) s_w[warp] = cnt;
    __syncthreads();
    uint32_t tile_total = 0, before = 0;
#pragma unroll
    for (int w = 0; w < RUNS_THREADS / 32; ++w) {
        if (w < warp) before += s_w[w];
        tile_total += s_w[w];
    }
    const unsigned long long prefix = lookback_exclusive_prefix(status, tile, (unsigned long long)tile_total, &s_prefix);
    if (tile == num_tiles - 1 && threadIdx.x == 0) {
        if (total_out) *total_out = prefix + tile_total;
        if (sentinel) sentinel[prefix + tile_total] = n;  // run_start[number of runs] = n closes the start table
        mail_post(mail, prefix + tile_total);
    }
    uint32_t run = (uint32_t)prefix + before;  // heads before this warp's first element
    const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j) {
        const uint32_t i = wbase + 32 * j + lane;
        const bool head = (masks[j] >> lane) & 1u;
        const uint32_t mine = run + __popc(masks[j] & lt) + (head ? 1u : 0u) - 1u;  // index of the run element i belongs to
        if (i < n) {
            if (run_of_pos) run_of_pos[i] = mine;
            if (head) emit(mine, i, keys[j]);
        }
        run += __popc(masks[j]);
    }
}

// TWO passes for large inputs (reduce-then-scan): the chained single-pass kernel above spends most of its time in the
// look-back (2048-element tiles, ~49 k of them for 100 M elements, hundreds in flight: 1.5 TB/s), whereas two streaming
// kernels with a small scan between them run at memory speed although the keys are evaluated again for the run heads:
//   runs_flags_kernel  head flags -> one bit word per 32 elements + the head count of every tile
//   (exclusive scan of the tile counts; its kernel posts the number of runs to the host)
//   runs_emit2_kernel  run index of every element from the bit words, emit for the heads
template <typename KeyFn>
__global__ void __launch_bounds__(RUNS_THREADS) runs_flags_kernel(KeyFn key, uint32_t n, uint32_t* __restrict__ flag_words,
                                                                  uint32_t* __restrict__ tile_cnt) {
    __shared__ uint32_t s_w[RUNS_THREADS / 32];
    const uint32_t tile = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t wbase = tile * RUNS_TILE + warp * (32 * RUNS_ITEMS);
    uint32_t masks[RUNS_ITEMS];
    uint64_t keys[RUNS_ITEMS];
    runs_warp_flags(key, wbase, n, lane, masks, keys);
    uint32_t cnt = 0;
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j) {
        cnt += __popc(masks[j]);
        if (lane == j && wbase + 32 * j < n) flag_words[(wbase >> 5) + j] = masks[j];
    }
    if (lane == 0) s_w[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < RUNS_THREADS / 32; ++w) t += s_w[w];
        tile_cnt[tile] = t;
    }
}

template <typename KeyFn, typename EmitFn>
__global__ void __launch_bounds__(RUNS_THREADS) runs_emit2_kernel(KeyFn key, EmitFn emit, uint32_t n, uint32_t num_tiles,
                                                                  const uint32_t* __restrict__ flag_words,
                                                                  const uint32_t* __restrict__ tile_off,
                                                                  const unsigned long long* __restrict__ d_total,
                                                                  uint32_t* __restrict__ run_of_pos, uint32_t* __restrict__ sentinel,
                                                                  uint32_t* __restrict__ word_off) {
    __shared__ uint32_t s_w[RUNS_THREADS / 32];
    const uint32_t tile = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t wbase = tile * RUNS_TILE + warp * (32 * RUNS_ITEMS);
    uint32_t masks[RUNS_ITEMS];
    uint32_t cnt = 0;
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j) {
        masks[j] = wbase + 32 * j < n ? flag_words[(wbase >> 5) + j] : 0u;
        cnt += __popc(masks[j]);
    }
    if (lane == 0) s_w[warp] = cnt;
    __syncthreads();
    uint32_t run = tile_off[tile];
#pragma unroll
    for (int w = 0; w < RUNS_THREADS / 32; ++w)
        if (w < warp) run += s_w[w];
    const uint32_t lt = (1u << lane) - 1u;
    uint64_t loaded[RUNS_ITEMS];  // the heads' key loads first, all in flight together (RunKey)
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j) {
        const uint32_t i = wbase + 32 * j + lane;
        loaded[j] = i < n && ((masks[j] >> lane) & 1u) ? RunKey<KeyFn>::load(key, i) : 0ull;
    }
#pragma unroll
    for (int j = 0; j < RUNS_ITEMS; ++j) {
        const uint32_t i = wbase + 32 * j + lane;
        const bool head = (masks[j] >> lane) & 1u;
        const uint32_t mine = run + __popc(masks[j] & lt) + (head ? 1u : 0u) - 1u;
        if (word_off && lane == j && wbase + 32 * j < n) word_off[(wbase >> 5) + j] = run;
        if (i < n) {
            if (run_of_pos) run_of_pos[i] = mine;
            if (head) emit(mine, i, RunKey<KeyFn>::finish(key, loaded[j]));
        }
        run += __popc(masks[j]);
    }
    if (tile == num_tiles - 1 && threadIdx.x == 0 && sentinel) sentinel[*d_total] = n;
}
constexpr size_t RUNS_TWO_PASS_MIN = (size_t)1 << 20;

// Segments [0, n) into maximal runs of equal key: calls emit(run, first position, key) per run, writes run_of_pos[i]
// (may be nullptr) and the number of runs to d_total (device, 64-bit).  Run tables must hold the caller's upper bound.
// `sentinel` (may be nullptr): a run-start table whose entry [number of runs] is set to n by the kernel itself, so that
// the host does not have to know the count to close the table.  `mail`: the count posted to the host (common.cuh).
// `words` / `word_off` (both or neither; (n + 31) / 32 entries each): the caller keeps the run index (common.cuh: RunIndex);
// the two-pass form then runs for every n.
template <typename KeyFn, typename EmitFn>
inline void segment_runs(Ctx& c, KeyFn key, EmitFn emit, size_t n, uint32_t* run_of_pos, unsigned long long* d_total,
                         uint32_t* sentinel = nullptr, const Mail& mail = Mail{}, uint32_t* words = nullptr,
                         uint32_t* word_off = nullptr) {
    OL_REQUIRE(n > 0, OL_ERR_INTERNAL, "segment_runs: empty input");
    const size_t tiles = (n + RUNS_TILE - 1) / RUNS_TILE;
    static const bool one_pass = getenv("OL_RUNS_ONE_PASS") != nullptr;  // debug / A-B: the chained kernel for every size
    if ((n >= RUNS_TWO_PASS_MIN && !one_pass) || words) {
        OL_REQUIRE(d_total != nullptr, OL_ERR_INTERNAL, "segment_runs: the two-pass form needs a device total");
        DevBuf<uint32_t> own_words, tile_cnt(c, tiles);
        if (!words) {
            own_words.reset(c, (n + 31) / 32);
            words = own_words.get();
        }
        runs_flags_kernel<KeyFn><<<(unsigned)tiles, RUNS_THREADS, 0, c.stream>>>(key, (uint32_t)n, words, tile_cnt.get());
        OL_CHECK_LAUNCH();
        transform_scan<uint32_t>(c, ScanPtrIn<uint32_t>{tile_cnt.get()}, ScanPtrOut<uint32_t>{tile_cnt.get()}, tiles, d_total, "scan", mail);
        runs_emit2_kernel<KeyFn, EmitFn><<<(unsigned)tiles, RUNS_THREADS, 0, c.stream>>>(key, emit, (uint32_t)n, (uint32_t)tiles,
                                                                                         words, tile_cnt.get(), d_total,
                                                                                         run_of_pos, sentinel, word_off);
        OL_CHECK_LAUNCH();
        return;
    }
    DevBuf<unsigned long long> own;
    unsigned long long* status = c.status_words(2 * tiles + 1);
    if (!status) {
        own.reset(c, 2 * tiles + 1);
        own.zero();
        status = own.get();
    }
    runs_fused_kernel<KeyFn, EmitFn><<<(unsigned)tiles, RUNS_THREADS, 0, c.stream>>>(key, emit, (uint32_t)n, (uint32_t)tiles, status,
                                                                                     run_of_pos, d_total, sentinel, mail);
    OL_CHECK_LAUNCH();
}

// =============================================================================================
// small elementwise helpers
// =============================================================================================
static __global__ void iota_kernel(uint32_t* out, uint32_t n, uint32_t first) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = first + i;
}

template <typename T>
__global__ void fill_kernel(T* out, size_t n, T v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = v;
}

template <typename T>
__global__ void gather_kernel(T* __restrict__ out, const T* __restrict__ in, const uint32_t* __restrict__ idx, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[idx[i]];
}

// highest set bit + 1 (0 for v == 0)
inline int bit_length_u64(uint64_t v) {
    int b = 0;
    while (v) {
        ++b;
        v >>= 1;
    }
    return b;
}

}  // namespace ol
