// Forest pipeline: K0 bounding box, K1 keygen, K2 sort (onesweep.cuh / primitives.cuh), K3 run segmentation into cells
// and (cell, pose) pairs, K4 level-synchronous subdivision (per-leaf digit histogram + fused stable partition),
// scheme replay for late poses, K5 leaf enumeration order + geometry, (pose, leaf) block table, K7 filter / mask
// compaction.  K6 (RANSAC) lives in ransac.cu, the multi-GPU routing in partition.cu.
#include <algorithm>
#include <climits>
#include <exception>
#include <mutex>

#include "forest.cuh"
#include "primitives.cuh"

namespace ol {

// =============================================================================================
// small device helpers
// =============================================================================================
// segment of global rank r: last s with seg_start[s] <= r   (seg_start has n_seg + 1 entries)
__device__ __forceinline__ int seg_of_rank(const uint32_t* __restrict__ seg_start, int n_seg, uint32_t r) {
    // poses have similar sizes, so an interpolated first guess is usually right or off by one; a few linear
    // probes, then plain bisection of whatever interval is left
    const uint32_t total = seg_start[n_seg];
    int s = (int)((float)r * __fdividef((float)n_seg, (float)(total ? total : 1u)));  // a guess: any value is corrected below
    s = s < 0 ? 0 : (s >= n_seg ? n_seg - 1 : s);
    int lo = 0, hi = n_seg;  // invariant: seg_start[lo] <= r < seg_start[hi]
#pragma unroll 1
    for (int probe = 0; probe < 3; ++probe) {
        if (seg_start[s] > r) {
            hi = s;
            s = s - 1;
        } else if (seg_start[s + 1] <= r) {
            lo = s + 1;
            s = s + 1;
        } else {
            return s;
        }
        if (s < lo || s >= hi) break;
    }
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (seg_start[mid] <= r)
            lo = mid;
        else
            hi = mid;
    }
    return lo;
}

// bits [lo, hi) of x (hi <= 64), safe for empty fields and lo >= 64
__device__ __forceinline__ uint64_t key_field(uint64_t x, int lo, int hi) {
    const int width = hi - lo;
    if (width <= 0 || lo >= 64) return 0ull;
    uint64_t v = x >> lo;
    if (width < 64) v &= (1ull << width) - 1ull;
    return v;
}

__device__ __forceinline__ void unpack_cell(const KeyParams& kp, uint64_t ckey, long long q[3]) {
    // ckey = packed key without the pose bits: [ x field | y field | z field ]
    const int s0 = kp.shift[0] - kp.pose_bits, s1 = kp.shift[1] - kp.pose_bits, s2 = kp.shift[2] - kp.pose_bits;
    q[0] = kp.qmin[0] + (long long)key_field(ckey, s0, 64);
    q[1] = kp.qmin[1] + (long long)key_field(ckey, s1, s0);
    q[2] = kp.qmin[2] + (long long)key_field(ckey, s2, s1);
}

// Batched insert: copies many device clouds into the raw point array in one launch AND folds them into the bounding
// box / non-finite check (K0) on the way, so the separate pass over the new points is not needed.  The host cuts the
// clouds into chunks of at most INSERT_CHUNK doubles (a multiple of 3, like every cloud and the thread count), so each
// thread of CTA c - which copies chunk c with a plain coalesced loop - only ever sees one axis.
constexpr unsigned INSERT_CHUNK = 3u * 10920u;
constexpr int INSERT_THREADS = 192;
struct InsertChunk {
    const double* src;
    unsigned long long dst;  // first destination double
    unsigned len;
    unsigned pad;
};
// one cloud of the batch; the chunk descriptors are derived from these on the device (a batch of 128 poses is ~2400 chunks:
// the host uploads 128 rows instead of building and staging the chunk table - host time in front of the first kernel)
struct InsertCloud {
    const double* src;
    unsigned long long dst;    // first destination double
    unsigned long long len;    // doubles
    unsigned first_chunk;
    unsigned pad;
};
__global__ void __launch_bounds__(INSERT_THREADS) insert_batch_kernel(const InsertCloud* __restrict__ clouds, int n_clouds,
                                                                      unsigned chunk_len, double* __restrict__ dst,
                                                                      long long* __restrict__ bbox, uint32_t* __restrict__ err) {
    __shared__ InsertChunk s_chunk;
    if (threadIdx.x == 0) {
        int lo = 0, hi = n_clouds;  // last cloud with first_chunk <= blockIdx.x (clouds without points own no chunk)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (clouds[mid].first_chunk <= blockIdx.x)
                lo = mid;
            else
                hi = mid;
        }
        const InsertCloud cl = clouds[lo];
        const unsigned long long off = (unsigned long long)(blockIdx.x - cl.first_chunk) * chunk_len;
        s_chunk.src = cl.src + off;
        s_chunk.dst = cl.dst + off;
        s_chunk.len = (unsigned)min((unsigned long long)chunk_len, cl.len - off);
        s_chunk.pad = 0u;
    }
    __syncthreads();
    const InsertChunk c = s_chunk;
    const double* __restrict__ s = c.src;
    double* __restrict__ d = dst + c.dst;
    long long mn = LLONG_MAX, mx = LLONG_MIN;
    bool bad = false;
    for (unsigned e = threadIdx.x; e < c.len; e += INSERT_THREADS) {
        const double v = s[e];
        d[e] = v;
        if (!isfinite(v)) bad = true;
        const long long k = double_to_ordered(v);
        mn = k < mn ? k : mn;
        mx = k > mx ? k : mx;
    }
    __shared__ long long s_mn[INSERT_THREADS], s_mx[INSERT_THREADS];
    s_mn[threadIdx.x] = mn;
    s_mx[threadIdx.x] = mx;
    __syncthreads();
    if (threadIdx.x < 3) {  // axis a = threadIdx.x (chunk starts are multiples of 3)
        long long lo = LLONG_MAX, hi = LLONG_MIN;
        for (int t = threadIdx.x; t < INSERT_THREADS; t += 3) {
            lo = s_mn[t] < lo ? s_mn[t] : lo;
            hi = s_mx[t] > hi ? s_mx[t] : hi;
        }
        if (lo != LLONG_MAX) atomicMin(&bbox[threadIdx.x], lo);
        if (hi != LLONG_MIN) atomicMax(&bbox[3 + threadIdx.x], hi);
    }
    if (bad) atomicOr(err, (uint32_t)DEVERR_NONFINITE);
}

// Morton codes are stored as 32-bit words while at most MORTON32_MAX_DEPTH levels are encoded (3 bits per level + the
// out-of-node flag in the top bit) and as 64-bit words after extend_morton(): the partition kernels move them, so the
// narrow form saves a quarter of their traffic.
template <typename MortT>
struct MortBits {
    static constexpr MortT bad = (MortT)1 << (sizeof(MortT) * 8 - 1);
};

// =============================================================================================
// K0: bounding box of a newly inserted cloud (ordered-int atomics), non-finite check
// =============================================================================================
// Flat, fully coalesced walk over the 3n doubles.  192 threads per block (a multiple of 3) make the grid stride a
// multiple of 3 as well, so every thread only ever sees ONE axis (tid % 3) and keeps a single min / max pair.
constexpr int BBOX_THREADS = 192;
__global__ void __launch_bounds__(BBOX_THREADS) bbox_kernel(const double* __restrict__ xyz, size_t n, long long* __restrict__ bbox,
                                                            uint32_t* __restrict__ err) {
    long long mn = LLONG_MAX, mx = LLONG_MIN;
    bool bad = false;
    const size_t total = n * 3, stride = (size_t)gridDim.x * BBOX_THREADS;
    for (size_t e = (size_t)blockIdx.x * BBOX_THREADS + threadIdx.x; e < total; e += stride) {
        const double v = xyz[e];
        if (!isfinite(v)) bad = true;
        const long long k = double_to_ordered(v);
        mn = k < mn ? k : mn;
        mx = k > mx ? k : mx;
    }
    __shared__ long long s_mn[BBOX_THREADS], s_mx[BBOX_THREADS];
    s_mn[threadIdx.x] = mn;
    s_mx[threadIdx.x] = mx;
    __syncthreads();
    if (threadIdx.x < 3) {  // axis a = threadIdx.x: combine the threads a, a + 3, a + 6, ...
        long long lo = LLONG_MAX, hi = LLONG_MIN;
        for (int t = threadIdx.x; t < BBOX_THREADS; t += 3) {
            lo = s_mn[t] < lo ? s_mn[t] : lo;
            hi = s_mx[t] > hi ? s_mx[t] : hi;
        }
        if (lo != LLONG_MAX) atomicMin(&bbox[threadIdx.x], lo);
        if (hi != LLONG_MIN) atomicMax(&bbox[3 + threadIdx.x], hi);
    }
    if (bad) atomicOr(err, (uint32_t)DEVERR_NONFINITE);
}

// =============================================================================================
// K1: packed cell key + in-cell Morton code per point (one pass over the raw cloud)
// =============================================================================================
// KeyT = uint32_t when the packed cell key (+ pose bits) fits 32 bits - every BASELINE configuration; the grid-wide
// sort then moves 4 + 4 bytes per pair and pass instead of 8 + 4.
template <typename KeyT, typename MortT>
__global__ void __launch_bounds__(256) keygen_kernel(const double* __restrict__ xyz, uint32_t n, KeyParams kp,
                                                     const uint32_t* __restrict__ seg_start,
                                                     const int32_t* __restrict__ seg_pose, int n_seg,
                                                     KeyT* __restrict__ keys, uint32_t* __restrict__ vals,
                                                     MortT* __restrict__ mort, uint32_t* __restrict__ err, int embed_levels) {
    // embed_levels > 0: the Morton code (3 x embed_levels bits) and the out-of-node flag (1 bit) ride in the LOW bits of the
    // sort key, below the packed cell key - the sort only looks at the bits above them, so the code arrives in sorted
    // order for free (no separate 4-byte array to write here and to gather through the permutation afterwards)
    uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double p[3] = {xyz[(size_t)r * 3 + 0], xyz[(size_t)r * 3 + 1], xyz[(size_t)r * 3 + 2]};
    long long q[3] = {0, 0, 0};
    uint64_t key = 0;
    uint32_t e = 0;
    if (!kp.single_cell) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            double qa = cell_coord_inv(p[a], kp.corner[a], kp.edge, kp.inv_edge);
            if (!(fabs(qa) < 4503599627370496.0)) {  // 2^52
                e |= DEVERR_CELL_RANGE;
                qa = 0.0;
            }
            q[a] = (long long)qa;
            long long rel = q[a] - kp.qmin[a];
            if (rel < 0) {
                e |= DEVERR_CELL_RANGE;
                rel = 0;
            }
            if (kp.shift[a] < 64) key |= ((uint64_t)rel) << kp.shift[a];
        }
    }
    if (kp.pose_bits) key |= (uint64_t)seg_pose[seg_of_rank(seg_start, n_seg, r)];
    double c[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) c[a] = cell_corner_coord(q[a], kp.corner[a], kp.edge, kp.single_cell);
    int bad;
    MortT m = (MortT)point_morton(p, c, kp.edge, kp.depth, &bad);
    if (embed_levels > 0) {
        key = (key << (3 * embed_levels + 1)) | ((uint64_t)(bad < kp.depth ? 1u : 0u) << (3 * embed_levels)) | (uint64_t)m;
    } else {
        if (bad < kp.depth) m |= MortBits<MortT>::bad;
        mort[r] = m;
    }
    keys[r] = (KeyT)key;
    vals[r] = r;  // the sort's payload: the point's rank
    if (e) atomicOr(err, e);
}

// Morton codes of already ordered points at a (deeper) depth: position i holds point perm[i] of cell
// cell_of[i] (or lcell[cell_of[i]] when lcell != nullptr, i.e. cell_of is the leaf index).
template <typename MortT>
__global__ void __launch_bounds__(256) remorton_kernel(const double* __restrict__ xyz, const uint32_t* __restrict__ perm,
                                                       const uint32_t* __restrict__ cell_of, const uint32_t* __restrict__ lcell,
                                                       const uint64_t* __restrict__ cell_key, KeyParams kp, uint32_t n,
                                                       MortT* __restrict__ mort) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t r = perm[i];
    uint32_t c = cell_of[i];
    if (lcell) c = lcell[c];
    long long q[3] = {0, 0, 0};
    if (!kp.single_cell) unpack_cell(kp, cell_key[c], q);
    const double p[3] = {xyz[r * 3], xyz[r * 3 + 1], xyz[r * 3 + 2]};
    double c0[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) c0[a] = cell_corner_coord(q[a], kp.corner[a], kp.edge, kp.single_cell);
    int bad;
    MortT m = (MortT)point_morton(p, c0, kp.edge, kp.depth, &bad);
    if (bad < kp.depth) m |= MortBits<MortT>::bad;
    mort[i] = m;
}

// =============================================================================================
// K3: run-length segmentation of the sorted keys
// =============================================================================================
// key / emit functors for segment_runs (primitives.cuh)
template <typename KeyT>
struct CellKeyFn {  // grid cell of a sorted position: the packed key without its pose bits
    const KeyT* keys;
    int pose_bits;
    __device__ uint64_t operator()(uint32_t i) const { return (uint64_t)(keys[i] >> pose_bits); }
};
// the same for keys that carry the Morton field in their low `fw` bits (keygen_kernel, embed_levels > 0): the field is
// peeled off into the 32-bit Morton array of the base order while the cell segmentation reads the key anyway
template <typename KeyT>
struct CellKeyEmbedFn {
    const KeyT* keys;
    int shift;  // pose bits + fw
    int fw;     // 3 x levels + 1
    uint32_t* mort_out;
    __device__ uint64_t operator()(uint32_t i) const {
        const KeyT k = keys[i];
        const uint32_t field = (uint32_t)k & ((1u << fw) - 1u);
        mort_out[i] = (field & ((1u << (fw - 1)) - 1u)) | ((field >> (fw - 1)) ? MortBits<uint32_t>::bad : 0u);
        return (uint64_t)(k >> shift);
    }
};
struct CellEmitFn {
    uint64_t* cell_key;
    uint32_t* cell_start;
    __device__ void operator()(uint32_t run, uint32_t i, uint64_t key) const {
        cell_key[run] = key;
        cell_start[run] = i;
    }
};
struct GroupPoseKeyFn {  // (group of the position, pose of its point): group = cell index or leaf index
    const uint32_t* group;
    const uint32_t* perm;
    const uint32_t* seg_start;
    const int32_t* seg_pose;
    int n_seg;
    // two stages (primitives.cuh: RunKey): (group, rank) from the coalesced arrays, then the pose of the rank
    __device__ __forceinline__ uint64_t load(uint32_t i) const { return ((uint64_t)group[i] << 32) | (uint64_t)perm[i]; }
    __device__ __forceinline__ uint64_t finish(uint64_t v) const {
        return (v & 0xffffffff00000000ull) | (uint64_t)(uint32_t)seg_pose[seg_of_rank(seg_start, n_seg, (uint32_t)v)];
    }
    __device__ uint64_t operator()(uint32_t i) const { return finish(load(i)); }
};
struct CellPoseEmitFn {  // (cell, pose) pairs that own an octree; the first pose of a cell created it (dict order, grid.py:56)
    uint32_t* cp_cell;
    int32_t* cp_pose;
    int32_t* cell_first_pose;
    const uint32_t* cellidx;
    __device__ void operator()(uint32_t run, uint32_t i, uint64_t key) const {
        const uint32_t cell = (uint32_t)(key >> 32);
        cp_cell[run] = cell;
        cp_pose[run] = (int32_t)(uint32_t)key;
        if (i == 0 || cellidx[i - 1] != cell) cell_first_pose[cell] = (int32_t)(uint32_t)key;
    }
};
struct BlockEmitFn {  // non-empty (pose, leaf) blocks
    uint32_t* blk_start;
    uint32_t* blk_leaf;
    int32_t* blk_pose;
    __device__ void operator()(uint32_t run, uint32_t i, uint64_t key) const {
        blk_start[run] = i;
        blk_leaf[run] = (uint32_t)(key >> 32);
        blk_pose[run] = (int32_t)(uint32_t)key;
    }
};

// =============================================================================================
// keep-flag compaction of the per-position arrays (K7: apply_keep, compact_base)
//   keep_bits_kernel     keep bytes -> one bit word per 32 positions + the kept count of every 2048-position tile
//   (exclusive scan of the tile counts; total = kept positions)
//   compact_move_kernel  ranks inside the tile from the bit words (64 words per tile), moves perm / mort / aux and
//                        leaves word_off[] = new position of every word's first kept element
//   remap_starts_kernel  new_start[k] = word_off[s >> 5] + popc(bits[s >> 5] below bit s & 31),  s = old_start[k]
// Traffic: 1 B + 12 B read per position, 12 B written per kept position, 8 B of tables per 32 positions.
// =============================================================================================
constexpr int CMP_THREADS = 256;
constexpr int CMP_TILE = 2048;
constexpr int CMP_WORDS = CMP_TILE / 32;

// keep bit of position i = keep[via ? via[i] : i]
__global__ void __launch_bounds__(CMP_THREADS) keep_bits_kernel(const uint8_t* __restrict__ keep, const uint32_t* __restrict__ via,
                                                                uint32_t n, uint32_t* __restrict__ bits,
                                                                uint32_t* __restrict__ tile_cnt) {
    __shared__ uint32_t s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const uint32_t base = blockIdx.x * CMP_TILE;
    const int lane = threadIdx.x & 31;
    uint32_t c = 0;
    // (every keep flag of the thread first, then the ballots: loads inside a warp-synchronous loop are issued one trip to
    // memory at a time)
    uint8_t flag[CMP_TILE / CMP_THREADS];
#pragma unroll
    for (int j = 0; j < CMP_TILE / CMP_THREADS; ++j) {
        const uint32_t i = base + j * CMP_THREADS + threadIdx.x;
        flag[j] = i < n ? keep[via ? via[i] : i] : (uint8_t)0;
    }
#pragma unroll
    for (int j = 0; j < CMP_TILE / CMP_THREADS; ++j) {
        const uint32_t i = base + j * CMP_THREADS + threadIdx.x;
        const bool k = flag[j] != 0;
        const uint32_t m = __ballot_sync(0xffffffffu, k);
        if (lane == 0 && i < n) {
            bits[i >> 5] = m;
            c += __popc(m);
        }
    }
    if (lane == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = s_cnt;
}

template <typename MortT>
__global__ void __launch_bounds__(CMP_THREADS) compact_move_kernel(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ tile_off,
                                                                   uint32_t n, const uint32_t* __restrict__ perm_in,
                                                                   const MortT* __restrict__ mort_in, const uint32_t* __restrict__ aux_in,
                                                                   uint32_t* __restrict__ perm_out, MortT* __restrict__ mort_out,
                                                                   uint32_t* __restrict__ aux_out, uint32_t* __restrict__ word_off) {
    __shared__ uint32_t s_mask[CMP_WORDS], s_off[CMP_WORDS], s_half;
    const uint32_t base = blockIdx.x * CMP_TILE;
    const uint32_t n_words = (n + 31) >> 5;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < CMP_WORDS) {  // warps 0 and 1: exclusive scan of the 64 word counts
        const uint32_t w = (base >> 5) + threadIdx.x;
        const uint32_t m = w < n_words ? bits[w] : 0u;
        const uint32_t c = __popc(m);
        uint32_t inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += v;
        }
        if (threadIdx.x == 31) s_half = inc;
        s_mask[threadIdx.x] = m;
        s_off[threadIdx.x] = inc - c;
    }
    __syncthreads();
    if (threadIdx.x < CMP_WORDS) {
        const uint32_t off = tile_off[blockIdx.x] + s_off[threadIdx.x] + (warp ? s_half : 0u);
        s_off[threadIdx.x] = off;
        const uint32_t w = (base >> 5) + threadIdx.x;
        if (w < n_words) word_off[w] = off;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < CMP_TILE / CMP_THREADS; ++j) {
        const uint32_t i = base + j * CMP_THREADS + threadIdx.x;
        const int w = j * (CMP_THREADS / 32) + warp;
        const uint32_t m = s_mask[w];
        if (i < n && ((m >> lane) & 1u)) {
            const uint32_t dst = s_off[w] + __popc(m & ((1u << lane) - 1u));
            perm_out[dst] = perm_in[i];
            mort_out[dst] = mort_in[i];
            aux_out[dst] = aux_in[i];
        }
    }
}

// new_start[k] = kept positions before old_start[k] (k < m), new_start[m] = total
__global__ void remap_starts_kernel(const uint32_t* __restrict__ old_start, const uint32_t* __restrict__ bits,
                                    const uint32_t* __restrict__ word_off, uint32_t m, uint32_t n_old, uint32_t total,
                                    uint32_t* __restrict__ new_start) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > m) return;
    if (k == m) {
        new_start[k] = total;
        return;
    }
    const uint32_t s = old_start[k];
    new_start[k] = (s < n_old) ? word_off[s >> 5] + __popc(bits[s >> 5] & ((1u << (s & 31u)) - 1u)) : total;
}

// alive_r[perm[i]] = 1 for the positions of the current order (ensure_alive)
__global__ void mark_alive_kernel(const uint32_t* __restrict__ perm, uint32_t n, uint8_t* __restrict__ alive_r) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) alive_r[perm[i]] = 1;
}

// =============================================================================================
// K4: level-synchronous subdivision
// =============================================================================================
}  // namespace ol
#include "geometry.cuh"
namespace ol {

__global__ void weighted_count_kernel(const uint32_t* __restrict__ leaf_of, const uint32_t* __restrict__ perm,
                                      const uint8_t* __restrict__ ldepth, int level,
                                      const uint32_t* __restrict__ seg_start, const int32_t* __restrict__ seg_pose,
                                      int n_seg, const uint8_t* __restrict__ listed, uint32_t n,
                                      uint32_t* __restrict__ wcount) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool on = false;
    uint32_t k = 0xffffffffu;
    if (i < n) {
        k = leaf_of[i];
        if (ldepth[k] == level) on = listed[seg_pose[seg_of_rank(seg_start, n_seg, perm[i])]] != 0;
    }
    uint32_t key = on ? k : 0xffffffffu;
    uint32_t peers = __match_any_sync(0xffffffffu, key);
    if (on && (threadIdx.x & 31) == (__ffs(peers) - 1)) atomicAdd(&wcount[k], __popc(peers));
}

// key of a tree node for the scheme replay: (cell index, depth <= REPLAY_MAX_DEPTH, Morton path)
constexpr int REPLAY_MAX_DEPTH = 9;
__host__ __device__ inline uint64_t replay_key(uint32_t cell, uint32_t depth, uint64_t path) {
    return ((uint64_t)cell << 32) | ((uint64_t)depth << 27) | (path & 0x7ffffffull);
}

// Split decision of one level as the INPUT functor of a scan over the leaves (transform_scan, primitives.cuh): the scan
// yields the index of every splitting leaf among the splitting leaves, and the output functor packs both into
//     sinfo[k] = (number of splitting leaves before k) << 1 | (k splits)
// which is all the partition kernels need: split index s = sinfo >> 1 (if the low bit is set), and the leaf's index in
// the next level's table = k + 7 * (sinfo >> 1) (every split replaces one leaf by eight).
// MODE: what decides (count threshold / count table / membership in a recorded shape); CAP = the level is the maximum
// depth: nothing may split, a leaf that wants to is an error.  Template parameters, so that the threshold and table
// instantiations are straight-line code without stores: the scan evaluates 16 leaves per thread back to back, and only
// then does the compiler issue the loads of all of them together (with the branches of the other modes in the way every
// leaf cost its own one or two round trips to memory: 25 us for a scan over 600 k leaves).  GEOM = the level also has
// geometric terms (geometry.cuh): a leaf splits if the count rule OR one of the terms says so, evaluated on the leaf's
// statistics in `geo`; the count-only instantiations never see those loads.
enum DecideMode { DECIDE_THRESHOLD = 0, DECIDE_TABLE = 1, DECIDE_REPLAY = 2 };
template <int MODE, bool CAP, bool GEOM = false>
struct DecideIn {
    const uint32_t* __restrict__ lstart;
    const uint8_t* __restrict__ ldepth;
    int level;
    const uint32_t* __restrict__ wcount;
    long long max_points;
    const uint8_t* __restrict__ table;
    long long table_len;
    int beyond;
    int max_depth;
    const uint64_t* replay_keys;
    uint32_t n_replay;
    const uint32_t* lcell;
    const uint64_t* lpath;
    uint32_t* err;
    const GeomLeaf* __restrict__ geo;
    const ol_geom_term* __restrict__ terms;
    int n_terms;
    __device__ __forceinline__ uint32_t operator()(size_t k) const {
        bool want = false;
        if (MODE == DECIDE_REPLAY) {
            // scheme replay (octree_manager.py:171 -> octree.py:222-227): split exactly the nodes of the recorded shape
            if (ldepth[k] == level && level < REPLAY_MAX_DEPTH) {
                const uint64_t key = replay_key(lcell[k], (uint32_t)level, lpath[k]);
                uint32_t lo = 0, hi = n_replay;
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (replay_keys[mid] < key)
                        lo = mid + 1;
                    else
                        hi = mid;
                }
                want = lo < n_replay && replay_keys[lo] == key;
            }
        } else {
            const uint32_t depth = ldepth[k];
            const uint32_t s0 = lstart[k], s1 = lstart[k + 1];
            const long long cnt = wcount ? (long long)wcount[k] : (long long)(s1 - s0);
            if (MODE == DECIDE_TABLE) {
                const long long at = cnt < table_len ? cnt : table_len - 1;  // always a valid entry: the load is unconditional
                const uint8_t t = table[at];
                want = cnt < table_len ? (t != 0) : (beyond != 0);
            } else {
                want = cnt > max_points;
            }
            if (GEOM) {
                const GeomLeaf g = geo[k];
                for (int t = 0; t < n_terms; ++t) want = want || geom_term_holds(terms[t], g.n, g.extent, g.thickness);
            }
            want = want && (int)depth == level;
            if (CAP) {
                if (want) atomicOr(err, (uint32_t)DEVERR_DEPTH_CAP);
                want = false;
            }
        }
        return want ? 1u : 0u;
    }
};
// input of the level's ONE scan: [ tile_hist (8 x tiles) | leaf_cnt[g][s], g < 8, s < n_split ] with leaf_cnt stored at
// stride `stride` >= n_split (speculative histogram pass: the stride is a bound fixed before n_split was known)
struct HistIn {
    const uint32_t* tile_hist;
    const uint32_t* leaf_cnt;
    uint32_t n_tile8, n_split, stride;
    __device__ uint32_t operator()(size_t i) const {
        const uint32_t j = i < n_tile8 ? 0u : (uint32_t)(i - n_tile8);
        const uint32_t g = j / n_split;
        const uint32_t* p = i < n_tile8 ? tile_hist + i : leaf_cnt + ((size_t)g * stride + (j - g * n_split));
        return *p;  // one unconditional load: the 16 elements of a thread are fetched together
    }
};
struct DecideOut {
    uint32_t* sinfo;
    __device__ void operator()(size_t k, uint32_t ex, uint32_t v) const { sinfo[k] = (ex << 1) | v; }
};

constexpr int PART_THREADS = 256;
constexpr int PART_ITEMS = 8;
constexpr int PART_TILE = PART_THREADS * PART_ITEMS;

template <typename MortT>
__device__ __forceinline__ uint32_t level_digit(MortT m, int shift) {
    return (uint32_t)(m >> shift) & 7u;
}

// per-tile histogram of the level digit over positions that belong to splitting leaves
template <typename MortT>
__global__ void __launch_bounds__(PART_THREADS) part_hist_kernel(const uint32_t* __restrict__ leaf_of,
                                                                  const MortT* __restrict__ mort,
                                                                  const uint32_t* __restrict__ sinfo, uint32_t n,
                                                                  uint32_t num_tiles, uint32_t n_split, int shift,
                                                                  uint32_t* __restrict__ tile_hist /*[8][tiles]*/,
                                                                  uint32_t* __restrict__ leaf_cnt /*[8][n_split]*/,
                                                                  const unsigned long long* __restrict__ d_nsplit) {
    // n_split = the STRIDE of leaf_cnt: the exact number of splitting leaves, or - when the pass was enqueued before the
    // host knew that number (d_nsplit != nullptr: speculative, forest_host.inl) - an upper bound.  A level that splits
    // nothing has nothing to count.
    if (d_nsplit && *d_nsplit == 0ull) return;
    __shared__ uint32_t h[8];
    if (threadIdx.x < 8) h[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t base = blockIdx.x * PART_TILE;
    const int lane = threadIdx.x & 31;
    // loads first, for all of the thread's positions (leaf and Morton word, then the dependent split info), and only then
    // the warp-synchronous counting: with the loads inside the loop every position paid its two round trips to memory
    // one after the other
    uint32_t lf[PART_ITEMS], keys[PART_ITEMS];
    MortT mo[PART_ITEMS];
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const uint32_t i = base + j * PART_THREADS + threadIdx.x;
        lf[j] = i < n ? leaf_of[i] : 0u;
        mo[j] = i < n ? mort[i] : (MortT)0;
    }
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const uint32_t i = base + j * PART_THREADS + threadIdx.x;
        const uint32_t si = i < n ? sinfo[lf[j]] : 0u;
        keys[j] = (si & 1u) ? (((si >> 1) << 3) | level_digit(mo[j], shift)) : 0xffffffffu;  // (split-leaf index << 3) | digit
    }
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const uint32_t key = keys[j];
        // positions are leaf-ordered, so a warp holds few distinct (leaf, digit) pairs: one atomic per pair
        const uint32_t peers = __match_any_sync(0xffffffffu, key);
        if (key != 0xffffffffu && lane == (__ffs(peers) - 1)) {
            const uint32_t c = (uint32_t)__popc(peers);
            atomicAdd(&h[key & 7u], c);
            atomicAdd(&leaf_cnt[(size_t)(key & 7u) * n_split + (key >> 3)], c);
        }
    }
    __syncthreads();
    if (threadIdx.x < 8) tile_hist[(size_t)threadIdx.x * num_tiles + blockIdx.x] = h[threadIdx.x];
}

struct Packed8 {
    unsigned long long lo, hi;  // 8 x 16-bit counters (digits 0..3 in lo, 4..7 in hi)
};
__device__ __forceinline__ uint32_t packed_get(const Packed8& p, uint32_t g) {
    return (uint32_t)(((g < 4 ? p.lo : p.hi) >> ((g & 3u) * 16)) & 0xffffull);
}
__device__ __forceinline__ void packed_inc(Packed8& p, uint32_t g) {
    unsigned long long one = 1ull << ((g & 3u) * 16);
    if (g < 4)
        p.lo += one;
    else
        p.hi += one;
}

// Stable 8-way partition of every splitting leaf's range in ONE pass (everything else is copied through).
// With S_g(i) = number of active positions before i whose digit is g (a global running count: the tile's offset from
// the scanned tile histograms plus a running count inside the tile), the destination of an active position i of leaf k
// (split index s) with digit g is
//     lstart[k] + sum_{c<g} leaf_cnt[c][s] + (S_g(i) - S_g(first position of k)),
// and S_g(first position of k) is the exclusive scan over the split leaves of leaf_cnt[g][.] (leaf_beg) because split
// leaves appear in position order.  Blocked arrangement (8 consecutive positions per thread): measured 4.2 ms for the
// three levels of the 100 M workload against 7.3 ms for a warp-striped variant with match-based ranking.
template <typename MortT>
__global__ void __launch_bounds__(PART_THREADS, 3) part_move_kernel(
    const uint32_t* __restrict__ leaf_of, const MortT* __restrict__ mort, const uint32_t* __restrict__ perm,
    const uint32_t* __restrict__ sinfo, const uint32_t* __restrict__ tile_off,
    const uint32_t* __restrict__ delta, uint32_t n, uint32_t num_tiles, int shift, int level,
    uint32_t* __restrict__ leaf_out, MortT* __restrict__ mort_out, uint32_t* __restrict__ perm_out,
    // for the out-of-node re-check
    const double* __restrict__ xyz, const uint32_t* __restrict__ lcell, const uint64_t* __restrict__ cell_key, KeyParams kp,
    uint32_t* __restrict__ err) {
    __shared__ unsigned long long wlo[8], whi[8];
    __shared__ uint32_t G[8];
    // Output staging: a leaf is partitioned inside its own range, so nearly every destination lies in the tile's own
    // range of positions.  Those go through shared memory and leave as 16-byte coalesced stores; only the pieces of a
    // splitting leaf that straddles a tile boundary are stored directly.  s_mask marks the staged positions.
    __shared__ __align__(16) uint32_t s_leaf[PART_TILE], s_perm[PART_TILE];
    __shared__ __align__(16) MortT s_mort[PART_TILE];
    __shared__ uint32_t s_mask[PART_TILE / 32];
    if (threadIdx.x < 8) G[threadIdx.x] = tile_off[(size_t)threadIdx.x * num_tiles + blockIdx.x];
    if (threadIdx.x < PART_TILE / 32) s_mask[threadIdx.x] = 0u;
    const uint32_t tile_base = blockIdx.x * PART_TILE;
    const uint32_t first = tile_base + threadIdx.x * PART_ITEMS;
    uint32_t leaf[PART_ITEMS];
    uint32_t g[PART_ITEMS];
    uint32_t pr[PART_ITEMS];
    MortT m[PART_ITEMS];
    Packed8 cnt{0ull, 0ull};
    static_assert(PART_ITEMS == 8, "vector loads below assume 8 items per thread");
    if (first + PART_ITEMS <= n) {
        // the thread's 8 consecutive elements are one or two aligned 32-byte segments: 16-byte vector loads
        const uint4 l0 = reinterpret_cast<const uint4*>(leaf_of + first)[0], l1 = reinterpret_cast<const uint4*>(leaf_of + first)[1];
        const uint4 p0 = reinterpret_cast<const uint4*>(perm + first)[0], p1 = reinterpret_cast<const uint4*>(perm + first)[1];
        leaf[0] = l0.x, leaf[1] = l0.y, leaf[2] = l0.z, leaf[3] = l0.w, leaf[4] = l1.x, leaf[5] = l1.y, leaf[6] = l1.z, leaf[7] = l1.w;
        pr[0] = p0.x, pr[1] = p0.y, pr[2] = p0.z, pr[3] = p0.w, pr[4] = p1.x, pr[5] = p1.y, pr[6] = p1.z, pr[7] = p1.w;
        if (sizeof(MortT) == 4) {
            const uint4 m0 = reinterpret_cast<const uint4*>(mort + first)[0], m1 = reinterpret_cast<const uint4*>(mort + first)[1];
            m[0] = (MortT)m0.x, m[1] = (MortT)m0.y, m[2] = (MortT)m0.z, m[3] = (MortT)m0.w;
            m[4] = (MortT)m1.x, m[5] = (MortT)m1.y, m[6] = (MortT)m1.z, m[7] = (MortT)m1.w;
        } else {
#pragma unroll
            for (int j = 0; j < PART_ITEMS; j += 2) {
                const ulonglong2 v = reinterpret_cast<const ulonglong2*>(mort + first)[j / 2];
                m[j] = (MortT)v.x;
                m[j + 1] = (MortT)v.y;
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < PART_ITEMS; ++j) {
            const uint32_t i = first + j;
            leaf[j] = i < n ? leaf_of[i] : 0u;
            pr[j] = i < n ? perm[i] : 0u;
            m[j] = i < n ? mort[i] : (MortT)0;
        }
    }
#pragma unroll
    uint32_t sp[PART_ITEMS];  // sinfo of the item's leaf
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        g[j] = 8u;
        sp[j] = first + j < n ? sinfo[leaf[j]] : 0u;  // (splits before) << 1 | splits
        if (sp[j] & 1u) {
            g[j] = level_digit(m[j], shift);
            packed_inc(cnt, g[j]);
        }
    }
    // block exclusive scan of the packed counters
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long ilo = cnt.lo, ihi = cnt.hi;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned long long tl = __shfl_up_sync(0xffffffffu, ilo, o);
        unsigned long long th = __shfl_up_sync(0xffffffffu, ihi, o);
        if (lane >= o) {
            ilo += tl;
            ihi += th;
        }
    }
    if (lane == 31) {
        wlo[warp] = ilo;
        whi[warp] = ihi;
    }
    __syncthreads();
    unsigned long long blo = 0, bhi = 0;
    for (int w = 0; w < warp; ++w) {
        blo += wlo[w];
        bhi += whi[w];
    }
    Packed8 run{blo + ilo - cnt.lo, bhi + ihi - cnt.hi};
#pragma unroll
    for (int j = 0; j < PART_ITEMS; ++j) {
        const uint32_t i = first + j;
        if (i >= n) break;
        const uint32_t k = leaf[j];
        uint32_t dst = i, nl = k + 7u * (sp[j] >> 1);
        if (g[j] < 8u) {
            const uint32_t S = G[g[j]] + packed_get(run, g[j]);
            packed_inc(run, g[j]);
            dst = S + delta[(size_t)(sp[j] >> 1) * 8 + g[j]];
            nl += g[j];
            if (m[j] & MortBits<MortT>::bad) {
                // the point left its node at some level: an error only if that level is being split
                const uint32_t r = pr[j];
                long long q[3] = {0, 0, 0};
                if (!kp.single_cell) unpack_cell(kp, cell_key[lcell[k]], q);
                double p[3] = {xyz[(size_t)r * 3], xyz[(size_t)r * 3 + 1], xyz[(size_t)r * 3 + 2]};
                double c0[3];
                for (int a = 0; a < 3; ++a) c0[a] = cell_corner_coord(q[a], kp.corner[a], kp.edge, kp.single_cell);
                int bad;
                point_morton(p, c0, kp.edge, kp.depth, &bad);
                if (bad <= level) atomicOr(err, (uint32_t)DEVERR_OUT_OF_NODE);
            }
        }
        const uint32_t rel = dst - tile_base;  // wraps to a huge value below the tile
        if (rel < (uint32_t)PART_TILE) {
            s_leaf[rel] = nl;
            s_mort[rel] = m[j];
            s_perm[rel] = pr[j];
            atomicOr(&s_mask[rel >> 5], 1u << (rel & 31u));
        } else {
            leaf_out[dst] = nl;
            mort_out[dst] = m[j];
            perm_out[dst] = pr[j];
        }
    }
    __syncthreads();
#pragma unroll
    for (int h = 0; h < PART_TILE / (PART_THREADS * 4); ++h) {
        const uint32_t o = (uint32_t)h * PART_THREADS * 4 + threadIdx.x * 4;  // 4 consecutive positions, lane-consecutive
        const uint32_t nib = (s_mask[o >> 5] >> (o & 31u)) & 0xfu;
        const uint32_t gpos = tile_base + o;
        if (nib == 0xfu) {
            *reinterpret_cast<uint4*>(leaf_out + gpos) = *reinterpret_cast<const uint4*>(&s_leaf[o]);
            *reinterpret_cast<uint4*>(perm_out + gpos) = *reinterpret_cast<const uint4*>(&s_perm[o]);
            if (sizeof(MortT) == 4) {
                *reinterpret_cast<uint4*>(mort_out + gpos) = *reinterpret_cast<const uint4*>(&s_mort[o]);
            } else {
                reinterpret_cast<ulonglong2*>(mort_out + gpos)[0] = reinterpret_cast<const ulonglong2*>(&s_mort[o])[0];
                reinterpret_cast<ulonglong2*>(mort_out + gpos)[1] = reinterpret_cast<const ulonglong2*>(&s_mort[o])[1];
            }
        } else if (nib) {
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                if ((nib >> b) & 1u) {
                    leaf_out[gpos + b] = s_leaf[o + b];
                    mort_out[gpos + b] = s_mort[o + b];
                    perm_out[gpos + b] = s_perm[o + b];
                }
            }
        }
    }
}

// New leaf / internal tables of a level, plus the partition deltas.  `scanned` is the exclusive scan of the level's flat
// histogram buffer [ tile_hist (8 x tiles) | leaf_cnt (8 x n_split) ], `*total` its grand total:
//   leaf_beg[g][s] = scanned[8 tiles + g n_split + s] - scanned[8 tiles]   (running count of digit g before split leaf s)
//   leaf_cnt[g][s] = difference to the next entry
//   delta[s][g]    = (first destination of the leaf's digit-g child) - leaf_beg[g][s], so that the move kernel needs ONE
//                    4-byte gather per point.
__global__ void expand_leaves_kernel(uint32_t L, uint32_t A, uint32_t I_old, const uint32_t* __restrict__ sinfo,
                                     const uint32_t* __restrict__ scanned, const unsigned long long* __restrict__ total,
                                     uint32_t num_tiles, uint32_t n_split,
                                     const uint32_t* __restrict__ lstart, const uint32_t* __restrict__ lcell,
                                     const int32_t* __restrict__ lparent, const uint64_t* __restrict__ lpath,
                                     const uint8_t* __restrict__ ldepth, const uint8_t* __restrict__ lchild,
                                     uint32_t L_new, uint32_t* __restrict__ lstart_n, uint32_t* __restrict__ lcell_n,
                                     int32_t* __restrict__ lparent_n, uint64_t* __restrict__ lpath_n,
                                     uint8_t* __restrict__ ldepth_n, uint8_t* __restrict__ lchild_n,
                                     uint32_t* __restrict__ istart, uint32_t* __restrict__ icell,
                                     uint8_t* __restrict__ idepth, uint64_t* __restrict__ ipath, int32_t* __restrict__ iparent,
                                     uint8_t* __restrict__ ichild, uint32_t* __restrict__ delta /*[n_split][8]*/) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= L) return;
    const uint32_t si = sinfo[k];
    const uint32_t s = si >> 1;
    const uint32_t j0 = k + 7u * s;
    if (!(si & 1u)) {
        lstart_n[j0] = lstart[k];
        lcell_n[j0] = lcell[k];
        lparent_n[j0] = lparent[k];
        lpath_n[j0] = lpath[k];
        ldepth_n[j0] = ldepth[k];
        lchild_n[j0] = lchild[k];
    } else {
        const uint32_t id = I_old + s;
        istart[id] = lstart[k];
        icell[id] = lcell[k];
        idepth[id] = ldepth[k];
        ipath[id] = lpath[k];
        iparent[id] = lparent[k];
        ichild[id] = lchild[k];
        const size_t flat_len = (size_t)8 * num_tiles + (size_t)8 * n_split;
        const uint32_t t_tiles = scanned[(size_t)8 * num_tiles];
        uint32_t run = lstart[k];
        // the sixteen scanned counts of the eight children first (strided gathers, all in flight), then the stores
        uint32_t e0s[8], e1s[8];
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) {
            const size_t idx = (size_t)8 * num_tiles + (size_t)c * n_split + s;
            e0s[c] = scanned[idx];
            e1s[c] = idx + 1 < flat_len ? scanned[idx + 1] : (uint32_t)*total;
        }
        const uint32_t cell_k = lcell[k];
        const uint64_t path_k = lpath[k];
        const uint8_t depth_k = ldepth[k];
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) {
            const uint32_t e0 = e0s[c], e1 = e1s[c];
            delta[(size_t)s * 8 + c] = run - (e0 - t_tiles);
            const uint32_t j = j0 + c;
            lstart_n[j] = run;
            run += e1 - e0;
            lcell_n[j] = cell_k;
            lparent_n[j] = (int32_t)id;
            lpath_n[j] = (path_k << 3) | (uint64_t)c;
            ldepth_n[j] = (uint8_t)(depth_k + 1);
            lchild_n[j] = (uint8_t)c;
        }
    }
    if (k == L - 1) lstart_n[L_new] = A;
}

// bounding box (6 ordered-int words) + error word -> the host mailbox (8 words: ticket, box, error); common.cuh: Mail
__global__ void post_bbox_kernel(const long long* __restrict__ bbox, const Mail m) {
    if (threadIdx.x != 0) return;
    for (int a = 0; a < 6; ++a) m.slot[1 + a] = (unsigned long long)bbox[a];
    m.slot[7] = (unsigned long long)*reinterpret_cast<const volatile uint32_t*>(m.err);
    __threadfence_system();
    m.slot[0] = m.ticket;
}

// current shape := one leaf per cell (reset_shape)
__global__ void init_leaves_kernel(uint32_t L, uint32_t* __restrict__ lcell, int32_t* __restrict__ lparent, uint64_t* __restrict__ lpath,
                                   uint8_t* __restrict__ ldepth, uint8_t* __restrict__ lchild) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= L) return;
    lcell[k] = k;
    lparent[k] = -1;
    lpath[k] = 0ull;
    ldepth[k] = 0;
    lchild[k] = 0;
}

// ---- scheme replay: record the split nodes by cell COORDINATES (the packed key changes when the grid is rebuilt) ----
__global__ void save_shape_kernel(uint32_t I, const uint32_t* __restrict__ icell, const uint8_t* __restrict__ idepth,
                                  const uint64_t* __restrict__ ipath, const uint64_t* __restrict__ cell_key, KeyParams kp,
                                  long long* __restrict__ q_out /*[I][3]*/, uint32_t* __restrict__ depth_out,
                                  uint64_t* __restrict__ path_out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= I) return;
    long long q[3] = {0, 0, 0};
    if (!kp.single_cell) unpack_cell(kp, cell_key[icell[i]], q);
    q_out[(size_t)i * 3 + 0] = q[0];
    q_out[(size_t)i * 3 + 1] = q[1];
    q_out[(size_t)i * 3 + 2] = q[2];
    depth_out[i] = idepth[i];
    path_out[i] = ipath[i];
}

// epoch of every internal node of a rebuilt shape: carried over from the recorded shape where the node existed
// (bisection of its replay key), `epoch` (the current subdivide call) where it is new
__global__ void assign_epochs_kernel(uint32_t I, const uint32_t* __restrict__ icell, const uint8_t* __restrict__ idepth,
                                     const uint64_t* __restrict__ ipath, const uint64_t* __restrict__ sorted_keys,
                                     const uint32_t* __restrict__ sorted_vals, const uint32_t* __restrict__ saved_epoch,
                                     uint32_t n_saved, uint32_t epoch, uint32_t* __restrict__ iepoch) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= I) return;
    uint32_t out = epoch;
    if (n_saved) {
        const uint64_t key = replay_key(icell[i], idepth[i], ipath[i]);
        uint32_t lo = 0, hi = n_saved;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (sorted_keys[mid] < key)
                lo = mid + 1;
            else
                hi = mid;
        }
        if (lo < n_saved && sorted_keys[lo] == key) out = saved_epoch ? saved_epoch[sorted_vals[lo]] : 1u;
    }
    iepoch[i] = out;
}

// recorded split node -> key under the NEW cell table (binary search of the packed cell key); ~0 if the cell is gone.
// A node of a cell outside the key's range is dropped: below qmin, or with a field that spills into the next one (or past
// bit 63), its packed key could equal that of a cell the forest holds.  The key is valid only if it unpacks to the node's q.
__global__ void replay_keys_kernel(uint32_t n, const long long* __restrict__ q_in, const uint32_t* __restrict__ depth_in,
                                   const uint64_t* __restrict__ path_in, const uint64_t* __restrict__ cell_key, uint32_t C,
                                   KeyParams kp, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t out = ~0ull;
    uint64_t packed = 0;
    bool ok = true;
    if (!kp.single_cell) {
        long long q[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            q[a] = q_in[(size_t)i * 3 + a];
            const long long rel = q[a] - kp.qmin[a];
            if (rel < 0) ok = false;
            const int s = kp.shift[a] - kp.pose_bits;
            if (ok && s < 64) packed |= ((uint64_t)rel) << s;
        }
        long long back[3];
        unpack_cell(kp, packed, back);
        ok = ok && back[0] == q[0] && back[1] == q[1] && back[2] == q[2];
    }
    if (ok) {
        uint32_t lo = 0, hi = C;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (cell_key[mid] < packed)
                lo = mid + 1;
            else
                hi = mid;
        }
        if (lo < C && cell_key[lo] == packed) out = replay_key(lo, depth_in[i], path_in[i]);
    }
    keys[i] = out;
    vals[i] = i;
}

// =============================================================================================
// K5: leaf enumeration order (reference `_cached_leaves` order) and leaf geometry
// =============================================================================================
// The order needs no sort.  Internal nodes are created level by level (ids of depth d are the contiguous range
// [begin[d], begin[d + 1])) in depth-first leaf order, so inside a level (cell, path) ascends strictly.  The pre-order
// rank of node i (cell c, depth d, path p) is a sum of bisections, one per level:
//   levels above d: nodes whose (cell, path) is <= (c, prefix of p at that depth)   - ancestors come first,
//   its own level : i - begin[d],
//   levels below d: nodes whose (cell, prefix of their path at depth d) is < (c, p) - descendants come after.
// (Keyed by the PATH, not by the range start: nodes without points - uniform refinement with MaxDepth / MinEdge splits
// them too - share their range start with their neighbours.)
// With imask[p] = set of children of p that are internal, node p emits 8 - popc(imask[p]) leaves; an exclusive scan of
// these counts in rank order (leafbase) gives, for a leaf with parent p and child id c,
//   cache position = first leaf of the cell + leafbase[rank p] - leafbase[rank of the cell's root] + popc(~imask[p] & below c)
// (the cell's leaves occupy the same index range in depth-first and in enumeration order).
struct LevelBegins {
    uint32_t b[OL_MAX_DEPTH + 2];
    int n;  // levels
};

__global__ void internal_mask_kernel(uint32_t I, const int32_t* __restrict__ iparent, const uint8_t* __restrict__ ichild,
                                     uint32_t* __restrict__ imask) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= I) return;
    const int32_t p = iparent[i];
    if (p >= 0) atomicOr(&imask[p], 1u << ichild[i]);
}

__global__ void internal_rank_kernel(uint32_t I, const uint8_t* __restrict__ idepth, const uint32_t* __restrict__ icell,
                                     const uint64_t* __restrict__ ipath, const uint32_t* __restrict__ imask, LevelBegins lv,
                                     uint32_t* __restrict__ irank, uint32_t* __restrict__ nlc_r, uint32_t* __restrict__ cell_ifirst) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= I) return;
    const uint32_t c = icell[i];
    const uint64_t p = ipath[i];
    const int d = idepth[i];
    uint32_t rank = 0;
    for (int dd = 0; dd < lv.n; ++dd) {
        const uint32_t b0 = lv.b[dd], b1 = lv.b[dd + 1];
        if (dd == d) {
            rank += i - b0;
            continue;
        }
        // first id in [b0, b1) that does NOT precede node i in pre-order
        const int up = dd < d ? 3 * (d - dd) : 0, down = dd > d ? 3 * (dd - d) : 0;
        const uint64_t want = p >> up;
        uint32_t lo = b0, hi = b1;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            const uint32_t cm = icell[mid];
            const uint64_t pm = ipath[mid] >> down;
            const bool before = cm != c ? (cm < c) : (dd < d ? pm <= want : pm < want);
            if (before)
                lo = mid + 1;
            else
                hi = mid;
        }
        rank += lo - b0;
    }
    irank[i] = rank;
    nlc_r[rank] = 8u - (uint32_t)__popc(imask[i]);
    if (d == 0) cell_ifirst[c] = rank;
}

// first leaf of every cell (every cell owns at least one leaf; the range is the same in both leaf orders)
__global__ void cell_first_leaf_kernel(uint32_t L, const uint32_t* __restrict__ lcell, uint32_t* __restrict__ cell_leaf_begin) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= L) return;
    const uint32_t c = lcell[k];
    if (k == 0 || lcell[k - 1] != c) cell_leaf_begin[c] = k;
}

__global__ void leaf_order_geometry_kernel(uint32_t L, const uint32_t* __restrict__ lcell, const int32_t* __restrict__ lparent,
                                           const uint8_t* __restrict__ lchild, const uint64_t* __restrict__ lpath,
                                           const uint8_t* __restrict__ ldepth, const uint32_t* __restrict__ irank,
                                           const uint32_t* __restrict__ imask, const uint32_t* __restrict__ leafbase,
                                           const uint32_t* __restrict__ cell_ifirst, const uint32_t* __restrict__ cell_leaf_begin,
                                           const uint64_t* __restrict__ cell_key, KeyParams kp, uint32_t* __restrict__ cache_rank,
                                           uint32_t* __restrict__ leaf_by_cache, double* __restrict__ corner,
                                           double* __restrict__ edge) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= L) return;
    const uint32_t c = lcell[k];
    uint32_t j = cell_leaf_begin[c];
    const int32_t p = lparent[k];
    if (p >= 0) {
        const uint32_t ch = lchild[k];
        j += leafbase[irank[p]] - leafbase[cell_ifirst[c]] + (uint32_t)__popc(~imask[p] & ((1u << ch) - 1u));
    }
    cache_rank[k] = j;
    leaf_by_cache[j] = k;
    long long q[3] = {0, 0, 0};
    if (!kp.single_cell) unpack_cell(kp, cell_key[c], q);
    double co[3];
    for (int a = 0; a < 3; ++a) co[a] = cell_corner_coord(q[a], kp.corner[a], kp.edge, kp.single_cell);
    double e = kp.edge;
    const int depth = ldepth[k];
    const uint64_t path = lpath[k];
    for (int d = 0; d < depth; ++d) {
        const double h = e * 0.5;  // octree.py:181
        const uint32_t dig = (uint32_t)(path >> (3 * (depth - 1 - d))) & 7u;
        if (dig & 4u) co[0] = co[0] + h;  // octree.py:186
        if (dig & 2u) co[1] = co[1] + h;
        if (dig & 1u) co[2] = co[2] + h;
        e = h;
    }
    corner[(size_t)j * 3 + 0] = co[0];
    corner[(size_t)j * 3 + 1] = co[1];
    corner[(size_t)j * 3 + 2] = co[2];
    edge[j] = e;
}

// =============================================================================================
// (pose, leaf) blocks
// =============================================================================================
// largest block: grid-stride walk, one atomic per CTA (one per warp on a single address cost 0.85 ms for 41 M blocks)
__global__ void __launch_bounds__(256) block_max_kernel(const uint32_t* __restrict__ blk_start, const unsigned long long* __restrict__ d_nb,
                                                        uint32_t* __restrict__ out_max) {
    __shared__ uint32_t s_w[8];
    const uint32_t nb = (uint32_t)*d_nb;  // device-side count: the host has not read it yet
    uint32_t v = 0;
    for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += gridDim.x * blockDim.x) {
        const uint32_t sz = blk_start[b + 1] - blk_start[b];
        v = sz > v ? sz : v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        uint32_t t = __shfl_xor_sync(0xffffffffu, v, o);
        v = t > v ? t : v;
    }
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) v = s_w[w] > v ? s_w[w] : v;
        if (v) atomicMax(out_max, v);
    }
}

__global__ void block_keep_kernel(uint32_t nb, const uint32_t* __restrict__ blk_start, const int32_t* __restrict__ blk_pose,
                                  const uint8_t* __restrict__ listed, const uint8_t* __restrict__ table,
                                  long long table_len, uint8_t* __restrict__ keep_blk) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    uint8_t keep = 1;
    if (!listed || listed[blk_pose[b]]) {
        long long sz = (long long)(blk_start[b + 1] - blk_start[b]);
        if (sz > table_len - 1) sz = table_len - 1;
        keep = table[sz];
    }
    keep_blk[b] = keep;
}

__global__ void run_of_pos_kernel(RunIndex ri, uint32_t n, uint32_t* __restrict__ run_of_pos) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) run_of_pos[i] = ri.runs_before(i + 1) - 1u;
}

__global__ void pos_keep_from_block_kernel(uint32_t n, const uint32_t* __restrict__ blk_of_pos,
                                           const uint8_t* __restrict__ keep_blk, uint8_t* __restrict__ keep_pos) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keep_pos[i] = keep_blk[blk_of_pos[i]];
}

}  // namespace ol

#include "leaf_maps.cuh"
#include "locate.cuh"
#include "forest_host.inl"
#include "forest_host2.inl"
