// Common host/device helpers for liboctreelib_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <iterator>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/octreelib_b200.h"

namespace ol {

// ---------------------------------------------------------------------------------------------
// error handling: every C-ABI entry point returns an ol_status; details via ol_last_error().
// ---------------------------------------------------------------------------------------------
struct Error {
    int code;
    std::string msg;
};

void set_last_error(int code, const std::string& msg);

#define OL_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            throw ::ol::Error{OL_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)};    \
        }                                                                                          \
    } while (0)

// every kernel launch in the library is followed by OL_CHECK_LAUNCH(): it also counts launches.  With the environment
// variable OL_DEBUG_SYNC=1 every launch is followed by a device synchronisation, so that an asynchronous fault is reported
// at the launch that caused it (debug aid; never set in measurements).
extern unsigned long long g_launch_count;
extern int g_debug_sync;  // -1 = not read yet
inline bool debug_sync_enabled() {
    if (g_debug_sync < 0) {
        const char* e = getenv("OL_DEBUG_SYNC");
        g_debug_sync = (e && e[0] == '1') ? 1 : 0;
    }
    return g_debug_sync == 1;
}
#define OL_CHECK_LAUNCH()                                                                                              \
    do {                                                                                                               \
        ++::ol::g_launch_count;                                                                                        \
        OL_CUDA(cudaGetLastError());                                                                                   \
        if (::ol::debug_sync_enabled()) {                                                                              \
            cudaError_t _s = cudaDeviceSynchronize();                                                                  \
            if (_s != cudaSuccess)                                                                                     \
                throw ::ol::Error{OL_ERR_CUDA, std::string("kernel launched at ") + __FILE__ + ":" + std::to_string(__LINE__) + \
                                                   " failed: " + cudaGetErrorString(_s)};                              \
        }                                                                                                              \
    } while (0)

#define OL_REQUIRE(cond, code, text)                 \
    do {                                             \
        if (!(cond)) throw ::ol::Error{(code), (text)}; \
    } while (0)

// device-side error bits (accumulated with atomicOr into Ctx::d_err, read at sync points)
enum DevErr : uint32_t {
    DEVERR_NONFINITE = 1u,      // NaN / inf coordinate
    DEVERR_CELL_RANGE = 2u,     // cell coordinate outside the packed key range
    DEVERR_OUT_OF_NODE = 4u,    // point outside its node at a level that is being split (octree.py:98)
    DEVERR_DEPTH_CAP = 8u,      // a node still exceeds the criterion at the maximum depth
    DEVERR_SAMPLE_OOB = 16u,    // RANSAC sample index fell outside its block (clamped)
    DEVERR_FILTER_BOUND = 32u,  // RANSAC verify mode: an exact count left its pre-filter interval
    DEVERR_LEAF_MAP = 64u,      // a leaf map produced a row outside the leaf it was computed from (leaf_maps.cuh)
    DEVERR_LEAF_MOVED = 128u,   // an appended leaf-map row landed in another leaf after the rebuild
};

// ---------------------------------------------------------------------------------------------
// optional per-stage timing with CUDA events on the work stream (enabled by ol_forest_profile)
// ---------------------------------------------------------------------------------------------
struct Profiler {
    struct Rec {
        const char* name;
        cudaEvent_t a, b;
        double units;  // elements processed (for bytes-per-launch accounting)
    };
    bool enabled = false;
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t get_event() {
        if (!pool.empty()) {
            cudaEvent_t e = pool.back();
            pool.pop_back();
            return e;
        }
        cudaEvent_t e;
        cudaEventCreate(&e);
        return e;
    }
    void clear() {
        for (auto& r : recs) {
            pool.push_back(r.a);
            pool.push_back(r.b);
        }
        recs.clear();
    }
    ~Profiler() {
        clear();
        for (auto e : pool) cudaEventDestroy(e);
    }
};

// ---------------------------------------------------------------------------------------------
// Process-wide cache of the blocks obtained from a host allocator callback.  A pipeline step builds a fresh forest (the
// reference builds a fresh Grid), and without the cache every step went back into the host language for each arena
// chunk and each large buffer (Python: 5-10 us per torch.empty, ~30 calls per step, all of it time the GPU may have to
// wait for).  Blocks are keyed by (callbacks, user pointer, stream): work on ONE stream is ordered, so a block freed by
// one context may be handed to the next context on the same stream at once - the same rule torch's caching allocator
// applies.  A block leaves the cache through the callback it came from (ol_release_cached_memory, the byte cap, or an
// allocation failure); the host binding keeps its callbacks alive for the life of the process (forest.py).
// ---------------------------------------------------------------------------------------------
struct BlockCache {
    struct Key {
        ol_alloc_fn a;
        ol_free_fn f;
        void* user;
        cudaStream_t stream;
        bool operator<(const Key& o) const {
            if (a != o.a) return (uintptr_t)a < (uintptr_t)o.a;
            if (f != o.f) return (uintptr_t)f < (uintptr_t)o.f;
            if (user != o.user) return user < o.user;
            return stream < o.stream;
        }
    };
    std::mutex mu;
    std::map<Key, std::multimap<size_t, void*>> free_blocks;
    std::map<void*, size_t> sizes;  // every block that went through the cache: its true size
    size_t cached_bytes = 0;
    size_t cap_bytes = (size_t)-1;  // set on first use (OL_CACHE_BYTES, default 1/4 of the device memory)

    void init_cap() {
        if (cap_bytes != (size_t)-1) return;
        const char* e = getenv("OL_CACHE_BYTES");
        if (e && *e) {
            cap_bytes = (size_t)strtoull(e, nullptr, 10);
            return;
        }
        size_t fr = 0, tot = 0;
        cap_bytes = (cudaMemGetInfo(&fr, &tot) == cudaSuccess) ? tot / 4 : ((size_t)8 << 30);
    }
    // a cached block of at least `bytes` and at most bytes + bytes / 8 (the steps of a pipeline ask for the same sizes again)
    void* take(const Key& k, size_t bytes) {
        std::lock_guard<std::mutex> lock(mu);
        auto it = free_blocks.find(k);
        if (it == free_blocks.end()) return nullptr;
        auto b = it->second.lower_bound(bytes);
        if (b == it->second.end() || b->first > bytes + bytes / 8) return nullptr;
        void* p = b->second;
        cached_bytes -= b->first;
        it->second.erase(b);
        return p;
    }
    void note(void* p, size_t bytes) {
        std::lock_guard<std::mutex> lock(mu);
        sizes[p] = bytes;
    }
    // returns false if the block must be freed by the caller (unknown block, or the cache is full)
    bool put(const Key& k, void* p) {
        std::lock_guard<std::mutex> lock(mu);
        init_cap();
        auto s = sizes.find(p);
        if (s == sizes.end()) return false;
        if (cached_bytes + s->second > cap_bytes) {
            sizes.erase(s);
            return false;
        }
        free_blocks[k].emplace(s->second, p);
        cached_bytes += s->second;
        return true;
    }
    void forget(void* p) {
        std::lock_guard<std::mutex> lock(mu);
        sizes.erase(p);
    }
    // hands every cached block back to where it came from; returns the bytes released
    size_t release_all() {
        std::map<Key, std::multimap<size_t, void*>> drop;
        size_t bytes;
        {
            std::lock_guard<std::mutex> lock(mu);
            drop.swap(free_blocks);
            bytes = cached_bytes;
            cached_bytes = 0;
            for (auto& kv : drop)
                for (auto& b : kv.second) sizes.erase(b.second);
        }
        for (auto& kv : drop)
            for (auto& b : kv.second) {
                if (kv.first.f)
                    kv.first.f(kv.first.user, b.second);
                else
                    cudaFree(b.second);
            }
        return bytes;
    }
};
extern BlockCache g_block_cache;

// ---------------------------------------------------------------------------------------------
// execution context: stream + allocator callbacks (the host binding passes torch's caching
// allocator; NULL callbacks fall back to cudaMallocAsync / cudaFreeAsync on the stream).
// ---------------------------------------------------------------------------------------------
struct Ctx {
    cudaStream_t stream = nullptr;
    ol_alloc_fn alloc_fn = nullptr;
    ol_free_fn free_fn = nullptr;
    void* alloc_user = nullptr;
    uint32_t* d_err = nullptr;  // device error word
    Profiler* prof = nullptr;
    int num_sms = 148;
    size_t bytes_live = 0, bytes_peak = 0;

    // ---- device memory ---------------------------------------------------------------------------------------------
    // Every allocator callback is a trip into the host language (Python: ~5-10 us per torch.empty), and one pipeline step
    // makes several hundred short-lived allocations - measured as the largest part of the time the GPU spent waiting for
    // the host.  So:
    //   * requests up to ARENA_MAX_REQUEST bytes are served by a native best-fit ARENA that sub-allocates chunks obtained
    //     from the callback (4 MB doubling to 128 MB).  Everything runs on ONE stream, so a block may be reused the moment
    //     it is freed (stream order), exactly like torch's caching allocator on a single stream.  Chunks stay with the Ctx
    //     until it is destroyed (release_arena()).
    //   * larger requests go to the callback directly; inside one public call freed ones are parked in a small
    //     exact-size pool and handed out again (the level loops allocate the same sizes over and over).  trim_pool()
    //     returns them at the end of each C-ABI entry point.
    struct Parked {
        void* ptr;
        size_t bytes;
    };
    std::vector<Parked> pool;
    size_t pool_bytes = 0;
    static constexpr size_t POOL_MAX_ENTRIES = 64;
    static constexpr size_t ARENA_ALIGN = 512;
    static constexpr size_t ARENA_MAX_REQUEST = 32u << 20;
    static constexpr size_t ARENA_FIRST_CHUNK = 4u << 20;
    static constexpr size_t ARENA_MAX_CHUNK = 128u << 20;
    struct ArenaBlock {
        size_t size;
        int chunk;
    };
    std::map<char*, ArenaBlock> arena_free;             // by address (coalescing)
    std::multimap<size_t, char*> arena_by_size;         // best fit
    std::vector<std::pair<char*, size_t>> arena_chunks;
    size_t arena_next_chunk = ARENA_FIRST_CHUNK;
    size_t arena_bytes = 0;
    bool arena_enabled = true;

    static size_t arena_round(size_t b) { return (b + ARENA_ALIGN - 1) / ARENA_ALIGN * ARENA_ALIGN; }
    void arena_insert_free(char* p, size_t size, int chunk) {
        // merge with the free neighbours of the same chunk
        auto next = arena_free.lower_bound(p);
        if (next != arena_free.end() && next->second.chunk == chunk && p + size == next->first) {
            size += next->second.size;
            arena_erase_size(next->second.size, next->first);
            next = arena_free.erase(next);
        }
        if (next != arena_free.begin()) {
            auto prev = std::prev(next);
            if (prev->second.chunk == chunk && prev->first + prev->second.size == p) {
                arena_erase_size(prev->second.size, prev->first);
                p = prev->first;
                size += prev->second.size;
                arena_free.erase(prev);
            }
        }
        arena_free[p] = ArenaBlock{size, chunk};
        arena_by_size.emplace(size, p);
    }
    void arena_erase_size(size_t size, char* p) {
        auto range = arena_by_size.equal_range(size);
        for (auto it = range.first; it != range.second; ++it)
            if (it->second == p) {
                arena_by_size.erase(it);
                return;
            }
    }
    void* arena_alloc(size_t sz) {
        auto it = arena_by_size.lower_bound(sz);
        if (it == arena_by_size.end()) {
            size_t chunk = std::max(arena_next_chunk, sz);
            arena_next_chunk = std::min(arena_next_chunk * 2, ARENA_MAX_CHUNK);
            char* base = static_cast<char*>(raw_alloc(chunk));
            arena_chunks.emplace_back(base, chunk);
            arena_bytes += chunk;
            arena_insert_free(base, chunk, (int)arena_chunks.size() - 1);
            it = arena_by_size.lower_bound(sz);
        }
        char* p = it->second;
        const ArenaBlock blk = arena_free[p];
        arena_by_size.erase(it);
        arena_free.erase(p);
        if (blk.size > sz) {
            arena_free[p + sz] = ArenaBlock{blk.size - sz, blk.chunk};
            arena_by_size.emplace(blk.size - sz, p + sz);
        }
        return p;
    }
    void arena_free_block(char* p, size_t sz) {
        // the owning chunk: the last chunk whose base is <= p (few chunks: linear scan)
        int chunk = -1;
        for (size_t i = 0; i < arena_chunks.size(); ++i)
            if (p >= arena_chunks[i].first && p < arena_chunks[i].first + arena_chunks[i].second) chunk = (int)i;
        arena_insert_free(p, sz, chunk);
    }
    void release_arena() {
        for (auto& c : arena_chunks) raw_free(c.first);
        arena_chunks.clear();
        arena_free.clear();
        arena_by_size.clear();
        arena_bytes = 0;
        arena_next_chunk = ARENA_FIRST_CHUNK;
    }

    void* alloc(size_t bytes) {
        if (bytes == 0) bytes = 16;
        bytes_live += bytes;
        if (bytes_live > bytes_peak) bytes_peak = bytes_live;
        if (arena_enabled && bytes <= ARENA_MAX_REQUEST) return arena_alloc(arena_round(bytes));
        for (size_t i = pool.size(); i-- > 0;) {
            if (pool[i].bytes == bytes) {
                void* p = pool[i].ptr;
                pool[i] = pool.back();
                pool.pop_back();
                pool_bytes -= bytes;
                return p;
            }
        }
        return raw_alloc(bytes);
    }
    void free(void* p, size_t bytes) {
        if (!p) return;
        if (bytes == 0) bytes = 16;
        bytes_live -= bytes;
        if (arena_enabled && bytes <= ARENA_MAX_REQUEST) {
            arena_free_block(static_cast<char*>(p), arena_round(bytes));
            return;
        }
        if (pool_enabled && pool.size() < POOL_MAX_ENTRIES) {
            pool.push_back(Parked{p, bytes});
            pool_bytes += bytes;
            return;
        }
        raw_free(p);
    }
    void trim_pool() {
        for (auto& e : pool) raw_free(e.ptr);
        pool.clear();
        pool_bytes = 0;
    }
    bool pool_enabled = false;
    BlockCache::Key cache_key() const { return BlockCache::Key{alloc_fn, free_fn, alloc_user, stream}; }
    void* raw_alloc(size_t bytes) {
        void* p = g_block_cache.take(cache_key(), bytes);
        if (p) return p;
        if (alloc_fn) {
            p = alloc_fn(alloc_user, bytes);
            if (!p) {
                trim_pool();  // give the parked and the cached buffers back and retry once
                g_block_cache.release_all();
                p = alloc_fn(alloc_user, bytes);
            }
            if (!p) throw Error{OL_ERR_ALLOC, "host allocator callback returned NULL for " + std::to_string(bytes) + " bytes"};
        } else {
            cudaError_t e = cudaMallocAsync(&p, bytes, stream);
            if (e != cudaSuccess) {
                cudaGetLastError();
                g_block_cache.release_all();
                OL_CUDA(cudaMallocAsync(&p, bytes, stream));
            }
        }
        g_block_cache.note(p, bytes);
        return p;
    }
    void raw_free(void* p) {
        if (g_block_cache.put(cache_key(), p)) return;
        if (free_fn)
            free_fn(alloc_user, p);
        else
            cudaFreeAsync(p, stream);
    }
    void sync() { OL_CUDA(cudaStreamSynchronize(stream)); }

    // ---- status words of the single-pass scans (primitives.cuh) --------------------------------------------------------
    // A chained scan needs zeroed status words (two per tile + a ticket counter).  Instead of an allocation and a memset
    // per scan (13 per pipeline step, each a 2 us operation plus a 2 us bubble) the scans of a context take consecutive
    // slices of ONE region that is zeroed once, when the first scan asks; a scan that does not fit any more gets its own.
    static constexpr size_t STATUS_POOL_WORDS = (size_t)1 << 20;  // 8 MB: ~500 k tiles per context
    unsigned long long* status_pool = nullptr;
    size_t status_used = 0;
    unsigned long long* status_words(size_t words) {
        words = (words + 1) & ~(size_t)1;  // slices stay 16-byte aligned (vector loads of the status pairs)
        if (status_used + words > STATUS_POOL_WORDS) return nullptr;  // the caller allocates and zeroes its own
        if (!status_pool) {
            status_pool = static_cast<unsigned long long*>(alloc(STATUS_POOL_WORDS * 8));
            OL_CUDA(cudaMemsetAsync(status_pool, 0, STATUS_POOL_WORDS * 8, stream));
        }
        unsigned long long* p = status_pool + status_used;
        status_used += words;
        return p;
    }
    ~Ctx() {
        if (status_pool) free(status_pool, STATUS_POOL_WORDS * 8);
        trim_pool();
        release_arena();
    }
};

// enables the temporary pool for the duration of one public call
struct PoolScope {
    Ctx& c;
    explicit PoolScope(Ctx& ctx) : c(ctx) { c.pool_enabled = true; }
    ~PoolScope() {
        c.pool_enabled = false;
        c.trim_pool();
    }
};

// times everything enqueued on the stream between construction and destruction under `name`
struct ProfScope {
    Ctx& c;
    Profiler::Rec rec{};
    bool on;
    ProfScope(Ctx& ctx, const char* name, double units = 0.0) : c(ctx), on(ctx.prof && ctx.prof->enabled) {
        if (on) {
            rec.name = name;
            rec.units = units;
            rec.a = c.prof->get_event();
            rec.b = c.prof->get_event();
            cudaEventRecord(rec.a, c.stream);
        }
    }
    ~ProfScope() {
        if (on) {
            cudaEventRecord(rec.b, c.stream);
            c.prof->recs.push_back(rec);
        }
    }
};

// ---------------------------------------------------------------------------------------------
// Mail: a scalar result posted by a kernel straight into page-locked host memory (zero copy), so that the host learns a
// count the moment the producing kernel knows it - without a device-to-host copy, a stream synchronisation (each one left
// the GPU idle for 20-30 us: copy engine, host wake-up, next launch) or an event.  The kernels enqueued BEHIND the
// producer keep running while the host reads the slot, which is what makes speculative launches and lazily consumed
// counts possible (forest_host.inl: split_levels, build, ensure_blocks).
//   slot[0] = ticket (process-wide unique, written last after a system fence), slot[1] = the count,
//   slot[2] = the device error word, slot[3] = one auxiliary 32-bit device value.
// ---------------------------------------------------------------------------------------------
struct Mail {
    volatile unsigned long long* slot = nullptr;
    unsigned long long ticket = 0;
    const uint32_t* err = nullptr;  // device pointers whose current values ride along (may be NULL)
    const uint32_t* aux = nullptr;
};
struct MailResult {
    unsigned long long total = 0;
    uint32_t err = 0, aux = 0;
};
#ifdef __CUDACC__
__device__ __forceinline__ void mail_post(const Mail& m, unsigned long long total) {
    if (!m.slot) return;
    m.slot[1] = total;
    m.slot[2] = m.err ? (unsigned long long)*reinterpret_cast<const volatile uint32_t*>(m.err) : 0ull;
    m.slot[3] = m.aux ? (unsigned long long)*reinterpret_cast<const volatile uint32_t*>(m.aux) : 0ull;
    __threadfence_system();
    m.slot[0] = m.ticket;
}
#endif
extern unsigned long long g_mail_ticket;  // last ticket handed out (process-wide; 0 is never a ticket)
// waits for the ticket; `stream` is only queried now and then to notice a dead producer
MailResult mail_wait(const Mail& m, cudaStream_t stream);

#ifdef __CUDACC__
// Run index of a segmentation, kept by the caller after segment_runs: the head bit of every element (one word per 32)
// and the number of runs that start before every word.  8 B per 32 elements.
struct RunIndex {
    const uint32_t* words;
    const uint32_t* word_off;
    const unsigned long long* d_total;
    uint32_t n;
    // number of runs that start before element p (p <= n): the run of element p is runs_before(p + 1) - 1, and the runs
    // of the elements [p, q) are [runs_before(p), runs_before(q)) when p is a head
    __device__ __forceinline__ uint32_t runs_before(uint32_t p) const {
        if (p >= n) return (uint32_t)*d_total;
        return word_off[p >> 5] + __popc(words[p >> 5] & ((1u << (p & 31)) - 1u));
    }
};
#endif

// RAII device buffer of T, bound to a Ctx.
template <typename T>
struct DevBuf {
    Ctx* ctx = nullptr;
    T* ptr = nullptr;
    size_t count = 0;

    DevBuf() = default;
    DevBuf(Ctx& c, size_t n) { reset(c, n); }
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept { *this = std::move(o); }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            release();
            ctx = o.ctx;
            ptr = o.ptr;
            count = o.count;
            o.ptr = nullptr;
            o.count = 0;
        }
        return *this;
    }
    ~DevBuf() { release(); }
    void reset(Ctx& c, size_t n) {
        release();
        ctx = &c;
        count = n;
        ptr = static_cast<T*>(c.alloc(n * sizeof(T)));
    }
    void release() {
        if (ptr && ctx) ctx->free(ptr, count * sizeof(T));
        ptr = nullptr;
        count = 0;
    }
    void swap(DevBuf& o) {
        std::swap(ctx, o.ctx);
        std::swap(ptr, o.ptr);
        std::swap(count, o.count);
    }
    void zero() {
        if (count) OL_CUDA(cudaMemsetAsync(ptr, 0, count * sizeof(T), ctx->stream));
    }
    T* get() const { return ptr; }
    size_t size() const { return count; }
};

template <typename T>
inline void d2h(Ctx& c, T* host, const T* dev, size_t n) {
    if (n) OL_CUDA(cudaMemcpyAsync(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost, c.stream));
}
template <typename T>
inline void h2d(Ctx& c, T* dev, const T* host, size_t n) {
    if (n) OL_CUDA(cudaMemcpyAsync(dev, host, n * sizeof(T), cudaMemcpyHostToDevice, c.stream));
}
template <typename T>
inline void d2d(Ctx& c, T* dst, const T* src, size_t n) {
    if (n) OL_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToDevice, c.stream));
}

inline unsigned grid_for(size_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// ---------------------------------------------------------------------------------------------
// numpy float64 floor_divide, restated (numpy/core/src/npymath/npy_math_internal.h.src,
// npy_divmod): the arithmetic behind `(points - corner) // edge` in
// /root/reference/octreelib/grid/grid.py:72-76.  fmod is exact on host and device, the rest is
// plain IEEE add/sub/div (the library is compiled with -fmad=false), so host and device agree.
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline double npy_floor_divide_ref(double a, double b) {
    if (b == 0.0) return a / b;
    double mod = fmod(a, b);
    double div = (a - mod) / b;
    if (mod != 0.0) {
        if ((b < 0) != (mod < 0)) {
            div -= 1.0;
        }
    }
    double floordiv;
    if (div != 0.0) {
        floordiv = floor(div);
        if (div - floordiv > 0.5) floordiv += 1.0;
    } else {
        floordiv = copysign(0.0, a / b);
    }
    return floordiv;
}

// Fast path used by the kernels.  For finite a and finite b > 0 with |a / b| < 2^51 numpy's result above IS the
// exact mathematical floor(a / b) (fmod is exact, the rest only snaps (a - mod) / b back to the integer it
// approximates).  The same integer is obtained without the iterative fmod: q0 = floor(fl(a / b)) is either the
// exact floor k or k + 1 (rounding to nearest is monotone and k, k + 1 are representable, so k <= fl(a / b) <= k + 1),
// and it is k + 1 exactly when the residual a - q0 b is negative; the single-rounded fma keeps that sign.
// tests/test_cpu_native_host.py checks this against numpy on random and adversarial operands.
__host__ __device__ inline double npy_floor_divide(double a, double b) {
    if (!(b > 0.0) || !(fabs(a) < 1.7e308) || !(b < 1.7e308)) return npy_floor_divide_ref(a, b);
    double q = floor(a / b);
    if (!(fabs(q) < 2251799813685248.0)) return npy_floor_divide_ref(a, b);  // 2^51
    if (fma(-q, b, a) < 0.0) q -= 1.0;
    return q;
}

// The same with the divisor's reciprocal supplied: inv = 1 / b when b is a power of two, else 0.  Multiplying by an exact
// power of two and dividing by it are both the correctly rounded value of the same real number, so a * inv == a / b bit for
// bit (over- and underflow included) - and the software division sequence (~25 instructions on the FP64 pipe, three per
// point in the key pass) disappears for the usual edges (1, 0.5, 0.25, 2, 4 m).
__host__ __device__ inline double npy_floor_divide_inv(double a, double b, double inv) {
    if (inv == 0.0 || !(fabs(a) < 1.7e308)) return npy_floor_divide(a, b);
    double q = floor(a * inv);
    if (!(fabs(q) < 2251799813685248.0)) return npy_floor_divide(a, b);  // 2^51
    if (fma(-q, b, a) < 0.0) q -= 1.0;
    return q;
}
// 1 / b if b is a finite positive power of two whose reciprocal is a normal number, else 0
inline double pow2_reciprocal(double b) {
    int e = 0;
    if (!(b > 0.0) || !(b < 1.7e308) || frexp(b, &e) != 0.5 || e < -1000 || e > 1000) return 0.0;
    return ldexp(1.0, 1 - e);
}

// order-preserving map double -> int64 (for atomicMin/atomicMax on coordinates)
__host__ __device__ inline long long double_to_ordered(double v) {
    long long b;
#ifdef __CUDA_ARCH__
    b = __double_as_longlong(v);
#else
    memcpy(&b, &v, 8);
#endif
    return b < 0 ? (b ^ 0x7fffffffffffffffLL) : b;
}
__host__ __device__ inline double ordered_to_double(long long k) {
    long long b = k < 0 ? (k ^ 0x7fffffffffffffffLL) : k;
#ifdef __CUDA_ARCH__
    return __longlong_as_double(b);
#else
    double v;
    memcpy(&v, &b, 8);
    return v;
#endif
}

}  // namespace ol
