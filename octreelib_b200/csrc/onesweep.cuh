// Onesweep LSD radix sort of (key, u32 value) pairs (K2).
//
// Groups what the reference groups with `np.unique(axis=0)` + `argsort` + `np.split`
// (/root/reference/octreelib/grid/grid.py:79-90, octree/octree.py:78-89).  Stable, so the canonical
// (pose, input index) order inside a cell falls out of the sort.
//
//   os_hist_kernel   one read of the keys builds the digit histograms of ALL passes (shared-memory
//                    histograms, warp-level peer aggregation by ballots, one global atomic per bin and CTA)
//   os_scan_kernel   exclusive scan of every pass's <= 256 bins
//   os_pass_kernel   one launch per digit: tile histogram with ballot-based peer ranking, chained
//                    scan over tiles with decoupled look-back (single 32-bit status word per (tile, digit):
//                    2 flag bits + 30-bit count, so no fence is needed), keys and values reordered inside the
//                    tile through shared memory so that global stores are digit-run coalesced.
// Algorithmic traffic: 1 x sizeof(Key) for the histograms + per pass (sizeof(Key) + 4) read and written.
// Limits: n < 2^30 pairs per call (30-bit status payload); the caller falls back to the three-kernel sort above it.
#pragma once
#include "common.cuh"

namespace ol {

constexpr int OS_THREADS = 256;
constexpr int OS_ITEMS = 16;
constexpr int OS_TILE = OS_THREADS * OS_ITEMS;
constexpr int OS_WARPS = OS_THREADS / 32;
constexpr int OS_MAX_PASSES = 8;
constexpr int OS_LOOKBACK = 4;  // measured on the 100 M-pair pass: 1 -> 0.68 ms, 4 -> 0.617, 8 -> 0.627, 16 -> 0.653
constexpr uint32_t OS_FLAG_AGG = 1u << 30;
constexpr uint32_t OS_FLAG_INC = 2u << 30;
constexpr uint32_t OS_VAL_MASK = (1u << 30) - 1u;

// Lanes whose digit equals this lane's digit; invalid lanes only match each other.  MATCH.ANY is microcoded - its
// cost grows with the number of distinct values in the warp (~28 for random 8-bit digits: > 50 % of a pass on random
// keys).  A peer mask built from one ballot per digit bit is faster on random keys, but spatially coherent keys (LiDAR
// scan order) put few distinct digits in a warp, where MATCH.ANY is the cheaper instruction: measured 0.81 ms vs
// 1.2 ms per 100 M-pair pass on the bench workload.
__device__ __forceinline__ uint32_t os_match_digit(uint32_t d, bool valid) {
    return __match_any_sync(0xffffffffu, valid ? d : 0xffffffffu);
}

struct OsPlan {
    int passes;
    int bit[OS_MAX_PASSES];    // first bit of the pass's digit
    int nbits[OS_MAX_PASSES];  // digit width (<= 8)
};

inline OsPlan os_make_plan(int begin_bit, int end_bit) {
    OsPlan p{};
    const int bits = end_bit - begin_bit;
    p.passes = (bits + 7) / 8;
    const int per = (bits + p.passes - 1) / p.passes;
    int bit = begin_bit;
    for (int i = 0; i < p.passes; ++i) {
        p.bit[i] = bit;
        p.nbits[i] = (end_bit - bit < per) ? (end_bit - bit) : per;
        bit += p.nbits[i];
    }
    return p;
}

template <typename KeyT>
__global__ void __launch_bounds__(OS_THREADS) os_hist_kernel(const KeyT* __restrict__ keys, uint32_t n, OsPlan plan,
                                                             uint32_t* __restrict__ ghist /*[passes][256]*/) {
    // Every thread walks CONSECUTIVE keys (16 bytes per load) and counts runs of equal digits in registers: one shared
    // atomic per run instead of a MATCH.ANY + atomic per key and pass.  The pipeline's keys are spatially coherent (a LiDAR
    // scan sweeps through neighbouring cells), so a thread's four keys nearly always share their upper digits.
    __shared__ uint32_t h[OS_MAX_PASSES][256];
    for (int i = threadIdx.x; i < plan.passes * 256; i += OS_THREADS) (&h[0][0])[i] = 0;
    __syncthreads();
    constexpr int VEC = 16 / (int)sizeof(KeyT);  // keys per 16-byte load
    const uint32_t n_vec = (reinterpret_cast<uintptr_t>(keys) & 15u) ? 0u : n / VEC;  // unaligned input: key by key
    uint32_t run_d[OS_MAX_PASSES], run_c[OS_MAX_PASSES];
#pragma unroll
    for (int p = 0; p < OS_MAX_PASSES; ++p) run_d[p] = 0u, run_c[p] = 0u;
    auto add = [&](KeyT k) {
#pragma unroll
        for (int p = 0; p < OS_MAX_PASSES; ++p) {
            if (p >= plan.passes) break;
            const uint32_t d = (uint32_t)((k >> plan.bit[p]) & (KeyT)((1u << plan.nbits[p]) - 1u));
            if (d == run_d[p]) {
                ++run_c[p];
            } else {
                if (run_c[p]) atomicAdd(&h[p][run_d[p]], run_c[p]);
                run_d[p] = d;
                run_c[p] = 1u;
            }
        }
    };
    // four 16-byte loads in flight per thread, then their keys (a shared-memory atomic between two loads would make the
    // thread wait for each load in turn)
    constexpr int UNR = 4;
    const uint32_t stride = gridDim.x * OS_THREADS;
    for (uint32_t v0 = blockIdx.x * OS_THREADS + threadIdx.x; v0 < n_vec; v0 += stride * UNR) {
        if (sizeof(KeyT) == 4) {
            uint4 q[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const uint32_t v = v0 + (uint32_t)u * stride;
                q[u] = v < n_vec ? reinterpret_cast<const uint4*>(keys)[v] : make_uint4(0u, 0u, 0u, 0u);
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u)
                if (v0 + (uint32_t)u * stride < n_vec) add((KeyT)q[u].x), add((KeyT)q[u].y), add((KeyT)q[u].z), add((KeyT)q[u].w);
        } else {
            ulonglong2 q[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const uint32_t v = v0 + (uint32_t)u * stride;
                q[u] = v < n_vec ? reinterpret_cast<const ulonglong2*>(keys)[v] : make_ulonglong2(0ull, 0ull);
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u)
                if (v0 + (uint32_t)u * stride < n_vec) add((KeyT)q[u].x), add((KeyT)q[u].y);
        }
    }
    for (uint32_t i = n_vec * VEC + blockIdx.x * OS_THREADS + threadIdx.x; i < n; i += gridDim.x * OS_THREADS) add(keys[i]);  // the rest
#pragma unroll
    for (int p = 0; p < OS_MAX_PASSES; ++p) {
        if (p >= plan.passes) break;
        if (run_c[p]) atomicAdd(&h[p][run_d[p]], run_c[p]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < plan.passes * 256; i += OS_THREADS) {
        const uint32_t v = (&h[0][0])[i];
        if (v) atomicAdd(&ghist[i], v);
    }
}

// exclusive scan of each pass's 256 bins, in place (one CTA of 256 threads per pass)
static __global__ void __launch_bounds__(256) os_scan_kernel(uint32_t* __restrict__ ghist) {
    __shared__ uint32_t sw[8];
    uint32_t* h = ghist + (size_t)blockIdx.x * 256;
    const uint32_t v = h[threadIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) sw[warp] = inc;
    __syncthreads();
    uint32_t wbase = 0;
    for (int w = 0; w < warp; ++w) wbase += sw[w];
    h[threadIdx.x] = wbase + inc - v;
}

__device__ __forceinline__ uint32_t os_ld_status(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void os_st_status(uint32_t* p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

template <typename KeyT>
__global__ void __launch_bounds__(OS_THREADS, 3) os_pass_kernel(const KeyT* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                                                                KeyT* __restrict__ keys_out, uint32_t* __restrict__ vals_out,
                                                                const uint32_t* __restrict__ gbase /*[256] exclusive digit offsets*/,
                                                                uint32_t* __restrict__ status /*[tiles][256]*/,
                                                                uint32_t* __restrict__ tile_counter, uint32_t n, int shift, int nbits) {
    extern __shared__ __align__(16) unsigned char os_smem[];
    KeyT* s_keys = reinterpret_cast<KeyT*>(os_smem);                                // [OS_TILE]
    uint32_t* s_vals = reinterpret_cast<uint32_t*>(os_smem + sizeof(KeyT) * OS_TILE);  // [OS_TILE]
    uint32_t* s_whist = s_vals + OS_TILE;                                           // [OS_WARPS][256]
    uint32_t* s_delta = s_whist + OS_WARPS * 256;                                   // [256] global position - local position
    uint32_t* s_excl = s_delta + 256;                                               // [256] first local position of the digit
    uint32_t* s_vraw = s_excl + 256;                                                // [OS_TILE] values in input order (cp.async)
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp_scan[8];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_tile = atomicAdd(tile_counter, 1u);
    for (int i = threadIdx.x; i < OS_WARPS * 256; i += OS_THREADS) s_whist[i] = 0;
    __syncthreads();
    const uint32_t tile = s_tile;
    // The values are only needed for the tile reorder: start an asynchronous global -> shared copy of the tile's
    // values now (LDGSTS, no registers held) so that their latency hides behind ranking and the chained scan.
    {
        const uint32_t tbase = tile * OS_TILE;
        const uint32_t tcount = min((uint32_t)OS_TILE, n - tbase);
        if (tcount == (uint32_t)OS_TILE) {
            for (uint32_t e = threadIdx.x * 4; e < (uint32_t)OS_TILE; e += OS_THREADS * 4) {
                const uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_vraw + e);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(vals_in + tbase + e) : "memory");
            }
        } else {
            for (uint32_t e = threadIdx.x; e < tcount; e += OS_THREADS) {
                const uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_vraw + e);
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(vals_in + tbase + e) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    const uint32_t mask = (1u << nbits) - 1u;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t wbase = tile * OS_TILE + warp * (32 * OS_ITEMS);

    // ---- load, match, rank inside the warp (stable: item-major, then lane) ------------------------------------
    KeyT k[OS_ITEMS];
    uint16_t rnk[OS_ITEMS];
    uint32_t* wh = s_whist + warp * 256;
#pragma unroll
    for (int j = 0; j < OS_ITEMS; ++j) {
        const uint32_t i = wbase + j * 32 + lane;
        k[j] = (i < n) ? keys_in[i] : (KeyT)0;
    }
#pragma unroll
    for (int j = 0; j < OS_ITEMS; ++j) {
        const uint32_t i = wbase + j * 32 + lane;
        const bool valid = i < n;
        const uint32_t d = (uint32_t)(k[j] >> shift) & mask;
        const uint32_t peers = os_match_digit(d, valid);
        const int leader = __ffs(peers) - 1;
        uint32_t old = 0;
        if (valid && lane == leader) {
            old = wh[d];
            wh[d] = old + __popc(peers);
        }
        old = __shfl_sync(0xffffffffu, old, leader);
        rnk[j] = (uint16_t)(old + __popc(peers & lt));
        __syncwarp();
    }
    __syncthreads();

    // ---- per digit (thread d < 256): warp counts -> exclusive over warps, tile count, chained scan --------------
    const uint32_t d = threadIdx.x;
    const bool digit_thread = d < 256;
    uint32_t count = 0;
    uint32_t* my_status = status + (size_t)tile * 256 + (d & 255u);
    if (digit_thread) {
#pragma unroll
        for (int w = 0; w < OS_WARPS; ++w) {
            const uint32_t t = s_whist[w * 256 + d];
            s_whist[w * 256 + d] = count;
            count += t;
        }
        os_st_status(my_status, (tile == 0 ? OS_FLAG_INC : OS_FLAG_AGG) | count);
    }
    // local exclusive scan of the tile's digit counts (threads 0..255 = warps 0..7)
    uint32_t inc = count;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (digit_thread && lane == 31) s_warp_scan[warp] = inc;
    __syncthreads();
    uint32_t local_first = 0;
    if (digit_thread) {
        uint32_t wb = 0;
        for (int w = 0; w < warp; ++w) wb += s_warp_scan[w];
        local_first = wb + inc - count;
        s_excl[d] = local_first;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");  // this thread's share of the value copy has landed ...
    __syncthreads();                                      // ... and after the barrier everybody's has

    // ---- reorder inside the tile (shared memory): keys and values to their local sorted position.  This runs
    // BETWEEN publishing the tile's aggregate and the look-back, so the value loads and the shared-memory
    // scatter overlap with the predecessors finishing their own prefixes (shorter look-back walks).
#pragma unroll
    for (int j = 0; j < OS_ITEMS; ++j) {
        const uint32_t i = wbase + j * 32 + lane;
        if (i < n) {
            const uint32_t dg = (uint32_t)(k[j] >> shift) & mask;
            const uint32_t p = s_excl[dg] + wh[dg] + rnk[j];
            s_keys[p] = k[j];
            s_vals[p] = s_vraw[i - tile * OS_TILE];
        }
    }
    // ---- decoupled look-back: sum the aggregates of the preceding tiles until an inclusive prefix is found ----
    if (digit_thread) {
        uint32_t excl = 0;
        if (tile > 0) {
            // OS_LOOKBACK predecessors per round, their loads issued back to back: a walk that fetched one status word
            // per trip to L2 (~0.7 us each) could not keep up with the rate at which tiles start - several hundred tiles
            // are in flight, and most of them have only published their aggregate when a successor looks back
            const uint32_t* st = status + d;
            long long t = (long long)tile - 1;
            bool done = false;
            while (!done && t >= 0) {
                uint32_t sv[OS_LOOKBACK];
#pragma unroll
                for (int w = 0; w < OS_LOOKBACK; ++w)
                    sv[w] = (t - w >= 0) ? os_ld_status(st + (size_t)(t - w) * 256) : (OS_FLAG_INC | 0u);
#pragma unroll
                for (int w = 0; w < OS_LOOKBACK; ++w) {
                    if (!done) {
                        while ((sv[w] >> 30) == 0u) sv[w] = os_ld_status(st + (size_t)(t - w) * 256);
                        excl += sv[w] & OS_VAL_MASK;
                        if ((sv[w] >> 30) == 2u) done = true;
                    }
                }
                t -= OS_LOOKBACK;
            }
            os_st_status(my_status, OS_FLAG_INC | ((excl + count) & OS_VAL_MASK));
        }
        s_delta[d] = gbase[d] + excl - local_first;
    }
    __syncthreads();
    const uint32_t tile_n = min((uint32_t)OS_TILE, n - tile * OS_TILE);
#pragma unroll
    for (int j = 0; j < OS_ITEMS; ++j) {
        const uint32_t p = j * OS_THREADS + threadIdx.x;
        if (p < tile_n) {
            const KeyT key = s_keys[p];
            const uint32_t dst = s_delta[(uint32_t)(key >> shift) & mask] + p;
            keys_out[dst] = key;
            vals_out[dst] = s_vals[p];
        }
    }
}

template <typename KeyT>
inline size_t os_pass_smem() {
    return sizeof(KeyT) * OS_TILE + 4 * OS_TILE + 4 * (OS_WARPS * 256 + 256 + 256) + 4 * OS_TILE;
}

template <typename KeyT>
inline void os_launch_pass(Ctx& c, const KeyT* kin, const uint32_t* vin, KeyT* kout, uint32_t* vout, const uint32_t* gbase,
                           uint32_t* status, uint32_t* counter, uint32_t n, int shift, int nbits) {
    static bool attr_set = false;
    const size_t smem = os_pass_smem<KeyT>();
    if (!attr_set) {
        OL_CUDA(cudaFuncSetAttribute(os_pass_kernel<KeyT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    const uint32_t tiles = (n + OS_TILE - 1) / OS_TILE;
    os_pass_kernel<KeyT><<<tiles, OS_THREADS, smem, c.stream>>>(kin, vin, kout, vout, gbase, status, counter, n, shift, nbits);
    OL_CHECK_LAUNCH();
}

// Sorts (keys0, vals0) by bits [begin_bit, end_bit) using (keys1, vals1) as the alternate buffer.
// Returns 0 if the result is in buffer 0, 1 if it is in buffer 1.  Requires 1 < n < 2^30.
template <typename KeyT>
inline int onesweep_sort_pairs(Ctx& c, KeyT* keys0, KeyT* keys1, uint32_t* vals0, uint32_t* vals1, size_t n, int begin_bit,
                               int end_bit, bool main_sort = false) {
    const OsPlan plan = os_make_plan(begin_bit, end_bit);
    OL_REQUIRE(plan.passes <= OS_MAX_PASSES, OL_ERR_INVALID, "onesweep: too many digit passes");
    const uint32_t tiles = (uint32_t)((n + OS_TILE - 1) / OS_TILE);
    // [passes][256] histograms | [passes] tile counters | [tiles][256] status words (re-zeroed per pass)
    // (one status array PER PASS, all of them zeroed by one memset: a memset per pass was a 2 us operation plus a 2 us bubble)
    const size_t status_per_pass = (size_t)tiles * 256;
    DevBuf<uint32_t> ghist(c, (size_t)plan.passes * 256 + OS_MAX_PASSES), status(c, status_per_pass * (size_t)plan.passes);
    ghist.zero();
    status.zero();
    // the grid-wide sort of all points (Forest::build) is timed under its own names: bench.py's roofline object
    const char* hname = main_sort ? "sort_main_hist" : (sizeof(KeyT) == 8 ? "radix_hist_u64" : "radix_hist_u32");
    const char* sname = main_sort ? "sort_main_pass" : (sizeof(KeyT) == 8 ? "radix_scatter_u64" : "radix_scatter_u32");
    {
        ProfScope ps(c, hname, (double)n);
        const unsigned g = std::min<unsigned>(tiles, (unsigned)c.num_sms * 8);
        os_hist_kernel<KeyT><<<g, OS_THREADS, 0, c.stream>>>(keys0, (uint32_t)n, plan, ghist.get());
        OL_CHECK_LAUNCH();
        os_scan_kernel<<<plan.passes, 256, 0, c.stream>>>(ghist.get());
        OL_CHECK_LAUNCH();
    }
    int cur = 0;
    for (int p = 0; p < plan.passes; ++p) {
        KeyT* kin = cur ? keys1 : keys0;
        KeyT* kout = cur ? keys0 : keys1;
        uint32_t* vin = cur ? vals1 : vals0;
        uint32_t* vout = cur ? vals0 : vals1;
        uint32_t* status_p = status.get() + status_per_pass * (size_t)p;
        ProfScope ps(c, sname, (double)n);
        const uint32_t* gb = ghist.get() + (size_t)p * 256;
        uint32_t* ctr = ghist.get() + (size_t)plan.passes * 256 + p;
        os_launch_pass<KeyT>(c, kin, vin, kout, vout, gb, status_p, ctr, (uint32_t)n, plan.bit[p], plan.nbits[p]);
        cur ^= 1;
    }
    return cur;
}

}  // namespace ol
