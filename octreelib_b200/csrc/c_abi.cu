// extern "C" entry points of liboctreelib_b200 (declared in include/octreelib_b200.h).
#include <atomic>
#include <cfloat>
#include <algorithm>
#include <new>

#include "exchange.cuh"
#include "forest.cuh"
#include "primitives.cuh"

struct ol_forest {
    ol::Forest impl;
    explicit ol_forest(const ol_forest_config& c) : impl(c) {}
};

struct ol_exchange {
    ol::Exchange impl;
    ol_exchange(int world, int rank, int n_poses, int64_t rows_cap, int nbuf, void* const* ctrl, void* const* data, int device)
        : impl(world, rank, n_poses, rows_cap, nbuf, ctrl, data, device) {}
};

namespace ol {
unsigned long long g_launch_count = 0;
int g_debug_sync = -1;
bool g_force_legacy_sort = false;
BlockCache g_block_cache;
unsigned long long g_mail_ticket = 0;

MailResult mail_wait(const Mail& m, cudaStream_t stream) {
    MailResult r;
    if (!m.slot) return r;
    unsigned long long spins = 0;
    bool drained = false;
    while (m.slot[0] != m.ticket) {
        if (drained) throw Error{OL_ERR_INTERNAL, "a kernel finished without posting its result to the host mailbox"};
        if ((++spins & 0x3fffu) == 0) {  // every ~16 k polls: is the producer still alive?
            const cudaError_t q = cudaStreamQuery(stream);
            if (q == cudaSuccess)
                drained = true;  // everything has run: the slot must hold the ticket on the next look
            else if (q != cudaErrorNotReady)
                throw Error{OL_ERR_CUDA, std::string("waiting for a kernel result: ") + cudaGetErrorString(q)};
        }
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    r.total = m.slot[1];
    r.err = (uint32_t)m.slot[2];
    r.aux = (uint32_t)m.slot[3];
    return r;
}
int g_os_variant = 0;
static thread_local std::string g_last_error;
void set_last_error(int code, const std::string& msg) { g_last_error = "[ol_status " + std::to_string(code) + "] " + msg; }
}  // namespace ol

#define OL_API_BEGIN try {
#define OL_API_END                                                     \
    }                                                                  \
    catch (const ol::Error& e) {                                       \
        ol::set_last_error(e.code, e.msg);                             \
        return e.code;                                                 \
    }                                                                  \
    catch (const std::bad_alloc&) {                                    \
        ol::set_last_error(OL_ERR_ALLOC, "host out of memory");        \
        return OL_ERR_ALLOC;                                           \
    }                                                                  \
    catch (const std::exception& e) {                                  \
        ol::set_last_error(OL_ERR_INVALID, e.what());                  \
        return OL_ERR_INVALID;                                         \
    }                                                                  \
    return OL_OK;

#define OL_NEED(p)                                                                       \
    if (!(p)) {                                                                          \
        ol::set_last_error(OL_ERR_INVALID, "NULL argument: " #p);                        \
        return OL_ERR_INVALID;                                                           \
    }

// every forest entry point: counts whose kernels were enqueued by an earlier call are read first (forest.cuh: resolve_pending),
// and large temporaries are parked for the duration of the call
struct ForestScope {
    ol::PoolScope pool;
    explicit ForestScope(ol::Forest& f) : pool(f.ctx) { f.resolve_pending(); }
};

extern "C" {

int ol_abi_version(void) { return OL_ABI_VERSION; }
const char* ol_last_error(void) { return ol::g_last_error.c_str(); }

int ol_forest_create(const ol_forest_config* config, ol_forest** out) {
    OL_NEED(config);
    OL_NEED(out);
    OL_API_BEGIN
    *out = new ol_forest(*config);
    OL_API_END
}

int ol_forest_destroy(ol_forest* f) {
    OL_API_BEGIN
    delete f;
    OL_API_END
}

int ol_forest_insert(ol_forest* f, const double* xyz, int64_t n, int32_t src_on_device, int32_t* out_pose_index) {
    OL_NEED(f);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    int p = f->impl.insert(xyz, n, src_on_device != 0, nullptr, nullptr, nullptr, 0, 0);
    if (out_pose_index) *out_pose_index = p;
    OL_API_END
}

int ol_forest_insert_batch(ol_forest* f, const double* const* xyz_dev_ptrs_host, const int64_t* sizes_host, int32_t count,
                           int32_t* out_first_pose_index) {
    OL_NEED(f);
    OL_API_BEGIN
    OL_REQUIRE(count == 0 || (xyz_dev_ptrs_host && sizes_host), OL_ERR_INVALID, "NULL batch tables");
    ForestScope scope(f->impl);
    int p = f->impl.insert_batch(xyz_dev_ptrs_host, sizes_host, count);
    if (out_first_pose_index) *out_first_pose_index = p;
    OL_API_END
}

int ol_forest_insert_segments(ol_forest* f, const double* xyz, int64_t n, int32_t src_on_device, const int64_t* seg_sizes,
                              const int32_t* seg_pose, const int64_t* seg_first, int32_t n_segments, int32_t n_poses_total) {
    OL_NEED(f);
    OL_NEED(seg_sizes);
    OL_NEED(seg_pose);
    OL_API_BEGIN
    OL_REQUIRE(n_segments > 0, OL_ERR_INVALID, "n_segments must be positive");
    ForestScope scope(f->impl);
    f->impl.insert(xyz, n, src_on_device != 0, seg_sizes, seg_pose, seg_first, n_segments, n_poses_total);
    OL_API_END
}

int64_t ol_exchange_ctrl_bytes(int32_t world, int32_t n_poses) { return (int64_t)ol::XchgCtrl::bytes(world, n_poses); }

int ol_exchange_create(int32_t world, int32_t rank, int32_t n_poses, int64_t rows_cap, int32_t n_buffers, void* const* ctrl_ptrs_host,
                       void* const* data_ptrs_host, int32_t device, ol_exchange** out) {
    OL_NEED(ctrl_ptrs_host);
    OL_NEED(data_ptrs_host);
    OL_NEED(out);
    OL_API_BEGIN
    *out = new ol_exchange(world, rank, n_poses, rows_cap, n_buffers, ctrl_ptrs_host, data_ptrs_host, device);
    OL_API_END
}

int ol_exchange_destroy(ol_exchange* x) {
    OL_API_BEGIN
    delete x;
    OL_API_END
}

int ol_exchange_run(ol_exchange* x, ol_forest* f, const double* const* clouds_dev_ptrs_host, const int64_t* sizes_host,
                    const int32_t* poses_host, int32_t count, int32_t slabs, int32_t buffer, int64_t* info_out, int64_t* bounds_out,
                    uint32_t* pose_sizes_out) {
    OL_NEED(x);
    OL_NEED(f);
    OL_API_BEGIN
    OL_REQUIRE(count == 0 || (clouds_dev_ptrs_host && sizes_host && poses_host), OL_ERR_INVALID, "NULL cloud tables");
    ForestScope scope(f->impl);
    x->impl.run(f->impl, clouds_dev_ptrs_host, sizes_host, poses_host, count, slabs, buffer, info_out, bounds_out, pose_sizes_out);
    OL_API_END
}

int ol_forest_disown_points(ol_forest* f) {
    OL_NEED(f);
    OL_API_BEGIN
    f->impl.disown_points();
    OL_API_END
}

int ol_forest_subdivide(ol_forest* f, int64_t max_points, const int32_t* pose_indices, int32_t n_poses) {
    OL_NEED(f);
    OL_API_BEGIN
    OL_REQUIRE(max_points >= 0, OL_ERR_INVALID, "max_points must be >= 0 (an empty node would split forever)");
    ForestScope scope(f->impl);
    ol::Forest::SplitRule rule;
    rule.first_level = {0};
    rule.max_points = {max_points};
    f->impl.subdivide(rule, pose_indices, n_poses);
    OL_API_END
}

int ol_forest_subdivide_table(ol_forest* f, const uint8_t* split_table_host, int64_t table_len, int32_t split_beyond,
                              const int32_t* pose_indices, int32_t n_poses) {
    OL_NEED(f);
    OL_NEED(split_table_host);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    ol::Forest::SplitRule rule;
    rule.first_level = {0};
    rule.tables_host = split_table_host;
    rule.table_len = table_len;
    rule.beyond = {split_beyond};
    f->impl.subdivide(rule, pose_indices, n_poses);
    OL_API_END
}

// the count part of a level-dependent split rule (ol_forest_subdivide_levels / _geometric)
static ol::Forest::SplitRule level_rule(const int32_t* first_level, int32_t n_entries, const int64_t* level_max_points,
                                        const uint8_t* split_tables_host, int64_t table_len, const int32_t* split_beyond) {
    OL_REQUIRE(n_entries >= 1 && n_entries <= 64, OL_ERR_INVALID, "split rule needs 1..64 level entries");
    OL_REQUIRE(split_tables_host ? split_beyond != nullptr : level_max_points != nullptr, OL_ERR_INVALID,
               "split rule needs thresholds or tables");
    ol::Forest::SplitRule rule;
    for (int e = 0; e < n_entries; ++e) {
        rule.first_level.push_back(first_level[e]);
        if (split_tables_host) {
            rule.beyond.push_back(split_beyond[e]);
        } else {
            // -1 = "every node of these levels splits, empty ones included" (MaxDepth / MinEdge: uniform refinement);
            // it ends at the next entry's first level or at the depth cap
            OL_REQUIRE(level_max_points[e] >= -1, OL_ERR_INVALID, "level_max_points must be >= -1");
            rule.max_points.push_back(level_max_points[e]);
        }
    }
    rule.tables_host = split_tables_host;
    rule.table_len = split_tables_host ? table_len : 0;
    return rule;
}

static void check_geom_terms(const ol_geom_term* terms, int32_t n) {
    OL_REQUIRE(n >= 0 && n <= OL_GEOM_MAX_TERMS, OL_ERR_INVALID,
               "at most " + std::to_string(OL_GEOM_MAX_TERMS) + " geometric terms per rule entry");
    OL_REQUIRE(n == 0 || terms, OL_ERR_INVALID, "NULL geometric terms");
    for (int32_t t = 0; t < n; ++t) {
        OL_REQUIRE(terms[t].stat == OL_GEOM_EXTENT || terms[t].stat == OL_GEOM_THICKNESS, OL_ERR_INVALID, "unknown geometric statistic");
        OL_REQUIRE(terms[t].op == OL_GEOM_GT || terms[t].op == OL_GEOM_LE, OL_ERR_INVALID, "unknown geometric comparison");
        OL_REQUIRE(terms[t].min_points >= 0, OL_ERR_INVALID, "min_points must be >= 0");
        OL_REQUIRE(terms[t].value >= 0.0 && terms[t].value <= DBL_MAX, OL_ERR_INVALID, "a geometric threshold must be finite and >= 0");
    }
}

int ol_forest_subdivide_levels(ol_forest* f, const int32_t* first_level, int32_t n_entries, const int64_t* level_max_points,
                               const uint8_t* split_tables_host, int64_t table_len, const int32_t* split_beyond,
                               const int32_t* pose_indices, int32_t n_poses) {
    OL_NEED(f);
    OL_NEED(first_level);
    OL_API_BEGIN
    ol::Forest::SplitRule rule = level_rule(first_level, n_entries, level_max_points, split_tables_host, table_len, split_beyond);
    ForestScope scope(f->impl);
    f->impl.subdivide(rule, pose_indices, n_poses);
    OL_API_END
}

int ol_forest_subdivide_geometric(ol_forest* f, const int32_t* first_level, int32_t n_entries, const int64_t* level_max_points,
                                  const uint8_t* split_tables_host, int64_t table_len, const int32_t* split_beyond,
                                  const ol_geom_term* terms, const int32_t* n_terms, const int32_t* pose_indices,
                                  int32_t n_poses) {
    OL_NEED(f);
    OL_NEED(first_level);
    OL_NEED(n_terms);
    OL_API_BEGIN
    ol::Forest::SplitRule rule = level_rule(first_level, n_entries, level_max_points, split_tables_host, table_len, split_beyond);
    rule.term_begin.push_back(0);
    for (int e = 0; e < n_entries; ++e) {
        check_geom_terms(terms ? terms + rule.term_begin.back() : nullptr, n_terms[e]);
        rule.terms.insert(rule.terms.end(), terms + rule.term_begin.back(), terms + rule.term_begin.back() + n_terms[e]);
        rule.term_begin.push_back(rule.term_begin.back() + n_terms[e]);
    }
    ForestScope scope(f->impl);
    f->impl.subdivide(rule, pose_indices, n_poses);
    OL_API_END
}

int ol_forest_export_shape(ol_forest* f, int64_t* q, uint32_t* depth, uint64_t* path, int64_t* out_n) {
    OL_NEED(f);
    OL_NEED(out_n);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    *out_n = (int64_t)f->impl.export_shape(reinterpret_cast<long long*>(q), depth, reinterpret_cast<unsigned long long*>(path));
    OL_API_END
}

int ol_forest_impose_shape(ol_forest* f, const int64_t* q, const uint32_t* depth, const uint64_t* path, int64_t n) {
    OL_NEED(f);
    OL_API_BEGIN
    OL_REQUIRE(n >= 0 && n < (1ll << 29), OL_ERR_INVALID, "bad node count");
    OL_REQUIRE(n == 0 || (q && depth && path), OL_ERR_INVALID, "NULL shape arrays");
    ForestScope scope(f->impl);
    f->impl.impose_shape(reinterpret_cast<const long long*>(q), depth, reinterpret_cast<const unsigned long long*>(path), (uint32_t)n);
    OL_API_END
}

int ol_forest_filter(ol_forest* f, const uint8_t* keep_table_host, int64_t table_len, const int32_t* pose_indices,
                     int32_t n_poses) {
    OL_NEED(f);
    OL_NEED(keep_table_host);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.filter(keep_table_host, table_len, pose_indices, n_poses);
    OL_API_END
}

int ol_forest_filter_geometric(ol_forest* f, const uint8_t* keep_table_host, int64_t table_len, const ol_geom_term* terms,
                               int32_t n_terms, const int32_t* pose_indices, int32_t n_poses) {
    OL_NEED(f);
    OL_NEED(keep_table_host);
    OL_API_BEGIN
    check_geom_terms(terms, n_terms);
    ForestScope scope(f->impl);
    f->impl.filter(keep_table_host, table_len, pose_indices, n_poses, terms, n_terms);
    OL_API_END
}

int ol_forest_ransac(ol_forest* f, const double* table_host, int32_t H, int32_t K, double threshold, const int32_t* pose_rank,
                     int32_t poses_per_batch, int32_t apply, uint32_t flags, const int64_t* pose_start) {
    OL_NEED(f);
    OL_NEED(table_host);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.ransac(table_host, H, K, threshold, pose_rank, poses_per_batch, apply != 0, flags, pose_start);
    OL_API_END
}

int ol_forest_pose_point_counts(ol_forest* f, int64_t* out_host) {
    OL_NEED(f);
    OL_NEED(out_host);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.pose_point_counts(out_host);
    OL_API_END
}

int ol_forest_apply_mask(ol_forest* f) {
    OL_NEED(f);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.apply_mask();
    OL_API_END
}

int ol_forest_apply_pose_mask(ol_forest* f, const int32_t* pose_rank, int32_t pose_index, const uint8_t* mask_host, int64_t n) {
    OL_NEED(f);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.apply_pose_mask(pose_rank, pose_index, mask_host, n);
    OL_API_END
}

int ol_forest_profile(ol_forest* f, int32_t enable) {
    OL_NEED(f);
    OL_API_BEGIN
    f->impl.ctx.sync();
    f->impl.prof.clear();
    f->impl.prof.enabled = enable != 0;
    OL_API_END
}

int ol_forest_profile_read(ol_forest* f, char* buf, int64_t buf_len, int64_t* out_len) {
    OL_NEED(f);
    OL_API_BEGIN
    std::string rep = f->impl.profile_report();
    if (out_len) *out_len = (int64_t)rep.size();
    if (buf && buf_len > 0) {
        size_t n = std::min<size_t>(rep.size(), (size_t)buf_len - 1);
        memcpy(buf, rep.data(), n);
        buf[n] = 0;
    }
    OL_API_END
}

uint64_t ol_launch_count(void) { return ol::g_launch_count; }
uint64_t ol_release_cached_memory(void) { return (uint64_t)ol::g_block_cache.release_all(); }

int ol_forest_stats_light(ol_forest* f, ol_forest_stats* out) {
    OL_NEED(f);
    OL_NEED(out);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.stats(out, true);
    OL_API_END
}

int ol_forest_stats_get(ol_forest* f, ol_forest_stats* out) {
    OL_NEED(f);
    OL_NEED(out);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.stats(out);
    OL_API_END
}

int ol_forest_pose_counts(ol_forest* f, int64_t* out_host) {
    OL_NEED(f);
    OL_NEED(out_host);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.pose_counts(out_host);
    OL_API_END
}

int ol_forest_export_cells(ol_forest* f, int64_t* q, double* corner, int32_t* first_pose, int64_t* n_nodes, int64_t* leaf_begin) {
    OL_NEED(f);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.export_cells(q, corner, first_pose, n_nodes, leaf_begin);
    OL_API_END
}

int ol_forest_export_cell_poses(ol_forest* f, int32_t* cell, int32_t* pose) {
    OL_NEED(f);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.export_cell_poses(cell, pose);
    OL_API_END
}

int ol_forest_export_leaves(ol_forest* f, double* corner, double* edge, int32_t* cell, int32_t* depth, int32_t* parent_epoch) {
    OL_NEED(f);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.export_leaves(corner, edge, cell, depth, parent_epoch);
    OL_API_END
}

int ol_forest_export_blocks(ol_forest* f, const int32_t* pose_rank, int32_t* pose, int32_t* leaf, int32_t* size) {
    OL_NEED(f);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    f->impl.export_blocks(pose_rank, pose, leaf, size);
    OL_API_END
}

int ol_forest_export_block_stats(ol_forest* f, const int32_t* pose_rank, int32_t pose_index, int32_t* pose, int64_t* n,
                                 double* mean, double* cov, double* extent, int64_t* out_n) {
    OL_NEED(f);
    OL_NEED(out_n);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    *out_n = f->impl.export_block_stats(pose_rank, pose_index, pose, n, mean, cov, extent);
    OL_API_END
}

int ol_forest_export_ransac(ol_forest* f, int32_t scored_only, int32_t* pose, int32_t* leaf, int32_t* size, float* plane,
                            int32_t* best, int32_t* best_count, int64_t* out_n) {
    OL_NEED(f);
    OL_API_BEGIN
    const bool count_only = !pose && !leaf && !size && !plane && !best && !best_count;
    ForestScope scope(f->impl);
    int64_t n = f->impl.export_ransac(scored_only != 0, count_only, pose, leaf, size, plane, best, best_count);
    if (out_n) *out_n = n;
    OL_API_END
}

int ol_forest_export_points(ol_forest* f, const int32_t* pose_rank, int32_t pose_index, int32_t order, double* xyz, int64_t* idx,
                            int32_t* cell, uint8_t* mask, int64_t* out_n) {
    OL_NEED(f);
    OL_API_BEGIN
    ForestScope scope(f->impl);
    int64_t n = f->impl.export_points(pose_rank, pose_index, order, xyz, idx, cell, mask);
    if (out_n) *out_n = n;
    OL_API_END
}

// ---- kernel-level RANSAC boundary (CudaRansac.evaluate, ransac/cuda_ransac.py:43-81) -----------
namespace {
__global__ void sizes_to_u32_kernel(const int32_t* sizes, uint32_t n, int K, uint32_t* out, uint32_t* wflags, uint32_t* maxsz) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    int s = sizes[b];
    out[b] = s > 0 ? (uint32_t)s : 0u;
    wflags[b] = s >= K ? 1u : 0u;
    if (s > 0) atomicMax(maxsz, (uint32_t)s);
}
__global__ void starts_to_i64_kernel(const uint32_t* starts, uint32_t n, long long* out) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < n) out[b] = (long long)starts[b];
}
__global__ void work_emit2_kernel(uint32_t nb, const uint32_t* flags, const uint32_t* scan_ex, uint32_t* work) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < nb && flags[b]) work[scan_ex[b]] = b;
}
ol::Ctx make_ctx(void* stream, ol_alloc_fn alloc, ol_free_fn free_fn, void* user) {
    ol::Ctx c;
    c.stream = (cudaStream_t)stream;
    c.alloc_fn = alloc;
    c.free_fn = free_fn;
    c.alloc_user = user;
    c.pool_enabled = true;  // trimmed by ~Ctx when the entry point returns
    return c;
}
}  // namespace

int ol_ransac_evaluate(void* stream, const double* points_dev, int64_t n, const int32_t* block_sizes_dev, int64_t B,
                       const double* table_dev, int32_t H, int32_t K, double threshold, uint8_t* mask_dev, float* plane_dev,
                       int32_t* best_dev, int32_t* best_count_dev, uint32_t flags, ol_alloc_fn alloc, ol_free_fn free_fn,
                       void* alloc_user) {
    OL_API_BEGIN
    using namespace ol;
    OL_REQUIRE(threshold > 0, OL_ERR_INVALID, "Threshold must be positive");
    OL_REQUIRE(H >= 1 && H <= 1024, OL_ERR_INVALID, "hypotheses_number must be in 1..1024");
    OL_REQUIRE(K >= 1 && K <= 64, OL_ERR_INVALID, "initial_points_number must be in 1..64");
    OL_REQUIRE(n >= 0 && n < (1ll << 31) && B >= 0 && B < (1ll << 31), OL_ERR_INVALID, "sizes out of range");
    Ctx c = make_ctx(stream, alloc, free_fn, alloc_user);
    if (n) OL_CUDA(cudaMemsetAsync(mask_dev, 0, (size_t)n, c.stream));
    if (B == 0) return OL_OK;
    const uint32_t nb = (uint32_t)B;
    DevBuf<uint32_t> err(c, 1), sizes(c, nb), starts(c, nb), wflags(c, nb), wscan(c, nb), maxsz(c, 1);
    DevBuf<long long> ref(c, nb);
    DevBuf<unsigned long long> d_total(c, 2);
    err.zero();
    maxsz.zero();
    c.d_err = err.get();
    const unsigned g = (nb + 255) / 256;
    sizes_to_u32_kernel<<<g, 256, 0, c.stream>>>(block_sizes_dev, nb, K, sizes.get(), wflags.get(), maxsz.get());
    OL_CHECK_LAUNCH();
    exclusive_scan_u32(c, sizes.get(), starts.get(), nb, d_total.get());  // cuda_ransac.py:65-67
    exclusive_scan_u32(c, wflags.get(), wscan.get(), nb, d_total.get() + 1);
    starts_to_i64_kernel<<<g, 256, 0, c.stream>>>(starts.get(), nb, ref.get());
    OL_CHECK_LAUNCH();
    unsigned long long tot[2];
    uint32_t mx;
    OL_CUDA(cudaMemcpyAsync(tot, d_total.get(), 16, cudaMemcpyDeviceToHost, c.stream));
    OL_CUDA(cudaMemcpyAsync(&mx, maxsz.get(), 4, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    OL_REQUIRE((int64_t)tot[0] == n, OL_ERR_INVALID, "block_sizes do not add up to the number of points");
    if (plane_dev) OL_CUDA(cudaMemsetAsync(plane_dev, 0, (size_t)nb * 16, c.stream));
    if (best_count_dev) OL_CUDA(cudaMemsetAsync(best_count_dev, 0, (size_t)nb * 4, c.stream));
    if (best_dev) {
        fill_kernel<int32_t><<<g, 256, 0, c.stream>>>(best_dev, nb, -1);
        OL_CHECK_LAUNCH();
    }
    const uint32_t n_work = (uint32_t)tot[1];
    DevBuf<uint32_t> work(c, n_work);
    work_emit2_kernel<<<g, 256, 0, c.stream>>>(nb, wflags.get(), wscan.get(), work.get());
    OL_CHECK_LAUNCH();
    launch_ransac(c, points_dev, n, starts.get(), block_sizes_dev, ref.get(), work.get(), nullptr, n_work, mx, table_dev, H, K, threshold,
                  mask_dev, plane_dev, best_dev, best_count_dev, flags);
    uint32_t herr = 0;
    OL_CUDA(cudaMemcpyAsync(&herr, err.get(), 4, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    OL_REQUIRE(!(herr & DEVERR_FILTER_BOUND), OL_ERR_INTERNAL, "RANSAC verify: an exact inlier count left its pre-filter interval");
    OL_API_END
}

int ol_ransac_stats_read(uint64_t out[16], int32_t reset) {
    OL_NEED(out);
    OL_API_BEGIN
    unsigned long long tmp[16];
    ol::ransac_stats_read(tmp, reset != 0);
    for (int i = 0; i < 16; ++i) out[i] = tmp[i];
    OL_API_END
}

// ---- arithmetic pipe peaks (roofline denominators of the RANSAC kernel, SURVEY.md 8(d)) -----------------------------
extern "C++" {
namespace {
// 8 independent fused multiply-add chains per thread, `iters` rounds: 16 flops per thread and round
template <typename T>
__global__ void __launch_bounds__(256) fma_peak_kernel(T* __restrict__ out, int iters, T seed) {
    T a0 = seed, a1 = seed + (T)1, a2 = seed + (T)2, a3 = seed + (T)3, a4 = seed + (T)4, a5 = seed + (T)5, a6 = seed + (T)6,
      a7 = seed + (T)7;
    const T m = (T)0.999999, b = (T)1e-6 * (T)(threadIdx.x + 1);
#pragma unroll 4
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, b);
        a1 = fma(a1, m, b);
        a2 = fma(a2, m, b);
        a3 = fma(a3, m, b);
        a4 = fma(a4, m, b);
        a5 = fma(a5, m, b);
        a6 = fma(a6, m, b);
        a7 = fma(a7, m, b);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

template <typename T>
double measure_fma(cudaStream_t stream, int sms) {
    const int blocks = sms * 8, threads = 256, iters = sizeof(T) == 8 ? 4096 : 16384;
    T* out = nullptr;
    OL_CUDA(cudaMalloc(&out, (size_t)blocks * threads * sizeof(T)));
    cudaEvent_t e0, e1;
    OL_CUDA(cudaEventCreate(&e0));
    OL_CUDA(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {  // first repetition = warm-up
        OL_CUDA(cudaEventRecord(e0, stream));
        fma_peak_kernel<T><<<blocks, threads, 0, stream>>>(out, iters, (T)1);
        OL_CUDA(cudaEventRecord(e1, stream));
        OL_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        OL_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double tflops = 16.0 * iters * (double)blocks * threads / (ms * 1e-3) / 1e12;
        if (rep > 0 && tflops > best) best = tflops;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    return best;
}
}  // namespace
}  // extern "C++"

int ol_measure_fma_peak(void* stream, double* out_fp64_tflops, double* out_fp32_tflops) {
    OL_API_BEGIN
    int dev = 0, sms = 148;
    OL_CUDA(cudaGetDevice(&dev));
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (out_fp64_tflops) *out_fp64_tflops = measure_fma<double>((cudaStream_t)stream, sms);
    if (out_fp32_tflops) *out_fp32_tflops = measure_fma<float>((cudaStream_t)stream, sms);
    OL_API_END
}

// ---- primitives ---------------------------------------------------------------------------------
int ol_debug_sort_variant(int32_t variant) {
    ol::g_os_variant = variant;
    return OL_OK;
}

int ol_debug_force_legacy_sort(int32_t on) {
    ol::g_force_legacy_sort = on != 0;
    return OL_OK;
}

int ol_sort_pairs_u64(void* stream, uint64_t* keys_dev, uint32_t* vals_dev, int64_t n, int32_t begin_bit, int32_t end_bit,
                      ol_alloc_fn alloc, ol_free_fn free_fn, void* alloc_user) {
    OL_API_BEGIN
    using namespace ol;
    OL_REQUIRE(n >= 0 && begin_bit >= 0 && end_bit <= 64 && begin_bit <= end_bit, OL_ERR_INVALID, "bad sort arguments");
    Ctx c = make_ctx(stream, alloc, free_fn, alloc_user);
    DevBuf<uint64_t> k1(c, (size_t)n);
    DevBuf<uint32_t> v1(c, (size_t)n);
    int w = radix_sort_pairs<uint64_t>(c, keys_dev, k1.get(), vals_dev, v1.get(), (size_t)n, begin_bit, end_bit);
    if (w) {
        d2d(c, keys_dev, k1.get(), (size_t)n);
        d2d(c, vals_dev, v1.get(), (size_t)n);
    }
    c.sync();
    OL_API_END
}

int ol_sort_pairs_u32(void* stream, uint32_t* keys_dev, uint32_t* vals_dev, int64_t n, int32_t begin_bit, int32_t end_bit,
                      ol_alloc_fn alloc, ol_free_fn free_fn, void* alloc_user) {
    OL_API_BEGIN
    using namespace ol;
    OL_REQUIRE(n >= 0 && begin_bit >= 0 && end_bit <= 32 && begin_bit <= end_bit, OL_ERR_INVALID, "bad sort arguments");
    Ctx c = make_ctx(stream, alloc, free_fn, alloc_user);
    DevBuf<uint32_t> k1(c, (size_t)n), v1(c, (size_t)n);
    int w = radix_sort_pairs<uint32_t>(c, keys_dev, k1.get(), vals_dev, v1.get(), (size_t)n, begin_bit, end_bit);
    if (w) {
        d2d(c, keys_dev, k1.get(), (size_t)n);
        d2d(c, vals_dev, v1.get(), (size_t)n);
    }
    c.sync();
    OL_API_END
}

int ol_exclusive_scan_u32(void* stream, const uint32_t* in_dev, uint32_t* out_dev, int64_t n, uint64_t* total_host,
                          ol_alloc_fn alloc, ol_free_fn free_fn, void* alloc_user) {
    OL_API_BEGIN
    using namespace ol;
    OL_REQUIRE(n >= 0, OL_ERR_INVALID, "negative length");
    Ctx c = make_ctx(stream, alloc, free_fn, alloc_user);
    DevBuf<unsigned long long> d_total(c, 1);
    exclusive_scan_u32(c, in_dev, out_dev, (size_t)n, d_total.get());
    if (total_host) {
        unsigned long long t;
        OL_CUDA(cudaMemcpyAsync(&t, d_total.get(), 8, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
        *total_host = t;
    } else {
        c.sync();
    }
    OL_API_END
}

// (what the kernels evaluate: the reciprocal fast path for power-of-two divisors, the division otherwise)
double ol_host_floor_divide(double a, double b) { return ol::npy_floor_divide_inv(a, b, ol::pow2_reciprocal(b)); }

int ol_host_point_key(double edge, const double corner[3], int32_t single_cell, int32_t depth, const double p[3], int64_t q[3],
                      uint64_t* morton, int32_t* bad_level) {
    OL_API_BEGIN
    OL_REQUIRE(depth >= 0 && depth <= OL_MAX_DEPTH, OL_ERR_INVALID, "depth out of range");
    double c0[3];
    for (int a = 0; a < 3; ++a) {
        long long qa = single_cell ? 0 : (long long)ol::cell_coord_inv(p[a], corner[a], edge, ol::pow2_reciprocal(edge));
        q[a] = qa;
        c0[a] = ol::cell_corner_coord(qa, corner[a], edge, single_cell);
    }
    int bad;
    unsigned long long m = ol::point_morton(p, c0, edge, depth, &bad);
    if (morton) *morton = m;
    if (bad_level) *bad_level = bad;
    OL_API_END
}

}  // extern "C"
