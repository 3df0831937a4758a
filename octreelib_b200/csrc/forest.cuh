// Forest: the device-resident state behind one Grid (many cells x many poses) or one
// OctreeManager / Octree (a single cell).  See DESIGN.md for the data layout.
#pragma once
#include <initializer_list>
#include <vector>

#include "common.cuh"
#include "pointkey.cuh"

namespace ol {

constexpr int MORTON_INITIAL_DEPTH = 8;
constexpr int MORTON32_MAX_DEPTH = 10;  // 30 digit bits + the out-of-node flag fit a 32-bit word

struct Forest {
    Ctx ctx;
    ol_forest_config cfg{};
    int max_depth = OL_MAX_DEPTH;

    // ---- raw input, indexed by the global point rank r (insertion order) -----------------------
    DevBuf<double> P64;          // [cap][3]
    size_t cap = 0, N = 0;
    size_t bbox_done = 0;        // points already folded into d_bbox / checked for NaN
    // multi-GPU exchange (exchange.cu): P64 may be a receive buffer the forest does not own (DevBuf without a context), and
    // the cell-coordinate range of its points is then known without a bounding-box pass
    bool q_known = false;
    long long q_lo[3] = {0, 0, 0}, q_hi[3] = {0, 0, 0};
    bool points_external() const { return P64.ptr != nullptr && P64.ctx == nullptr; }
    void adopt_points(double* ext, size_t n, const int64_t* seg_sizes, const int32_t* seg_pose_in, const int64_t* seg_first_in,
                      int n_segments, int n_poses_total, const long long qlo[3], const long long qhi[3]);
    void disown_points();        // copy an adopted point array into memory of the forest's own
    DevBuf<uint8_t> alive_r;     // [cap] 1 = point still stored; allocated by the first removal (filter / RANSAC mask)
    bool any_dead = false;
    bool alive_stale = false;    // alive_r lags behind the current order (apply_keep); see ensure_alive
    bool base_dirty = false;     // base order still contains dead points
    std::vector<uint32_t> seg_start;  // host: first rank of every segment (+ sentinel N)
    std::vector<int32_t> seg_pose;    // host: pose index of every segment
    std::vector<int64_t> seg_first;   // host: index of the segment's first point inside its pose's cloud
    bool segs_pose_monotone = true;
    int n_poses = 0;
    DevBuf<uint8_t> seg_blob;    // the three segment tables in one allocation (upload_segments); d_seg_* are views
    DevBuf<uint32_t> d_seg_start;
    DevBuf<int32_t> d_seg_pose;
    DevBuf<int64_t> d_seg_first;
    DevBuf<long long> d_bbox;    // [6] ordered-int min xyz, max xyz
    DevBuf<uint32_t> d_err;      // [1]
    bool uploads_pending = false;  // copies of pinned host clouds in flight on the upload streams (forest_host.inl)
    int upload_turn = 0;
    cudaStream_t upload_stream();
    void join_uploads();
    void* pinned = nullptr;      // small pinned scratch for read-backs (256 B)
    // Results posted by kernels straight into page-locked memory (common.cuh: Mail): 8 slots of 4 words.  A count whose
    // producer has been enqueued may stay unread until somebody needs it (`*_pending`): the eager parts of the pipeline
    // (build after an exchange, leaf order + block table after a subdivide) return to the host language while the GPU
    // still works, and every C-ABI entry point starts with resolve_pending().
    void* mailbox = nullptr;
    enum MailSlot { MAIL_CELLS = 0, MAIL_BLOCKS = 1, MAIL_LEVEL = 2, MAIL_WORK = 3, MAIL_COMPACT = 4, MAIL_MISC = 5 };
    Mail mail_open(int slot, const uint32_t* aux = nullptr);
    MailResult mail_take(const Mail& m) { return mail_wait(m, ctx.stream); }
    bool cells_pending = false, blocks_pending = false;
    Mail cells_mail{}, blocks_mail{};
    DevBuf<unsigned long long> d_nb;  // [1] number of blocks (device copy, read by block_max_kernel)
    void resolve_cells();
    void resolve_blocks();
    void resolve_pending() {
        resolve_cells();
        resolve_blocks();
    }
    void build_enqueue();          // K1-K3 enqueued, C not read yet
    void ensure_blocks_enqueue();  // block table enqueued, NB not read yet
    void prefetch_tables();        // leaf order + block table enqueued right after a subdivide (no wait)

    // ---- base structure: points grouped by cell, (pose, input index) order inside a cell --------
    bool built = false;
    KeyParams kp{};
    int key_bits = 0;
    int key_embed = 0;           // Morton levels carried in the low bits of the 32-bit sort key (0: separate Morton array)
    uint32_t A0 = 0;             // alive points in the base order
    DevBuf<uint32_t> perm0;      // [A0] base position -> r
    DevBuf<uint64_t> mort0;      // [A0] Morton code of the point (top bit: out-of-node somewhere); 32-bit words packed two
                                 // per element while mort32 is set (kp.depth <= MORTON32_MAX_DEPTH), 64-bit words after
    bool mort32 = true;
    size_t mort_len(size_t n) const { return mort32 ? (n + 1) / 2 : n; }  // DevBuf<uint64_t> elements for n codes
    DevBuf<uint32_t> cellidx0;   // [A0] base position -> cell index
    uint32_t C = 0;
    DevBuf<uint64_t> cell_key;   // [C] packed cell key (without pose bits)
    DevBuf<uint32_t> cell_start0;// [C+1]
    uint32_t CP = 0;
    bool cp_valid = false;       // cp_* / cell_first_pose built (lazily: ensure_cell_poses)
    DevBuf<uint32_t> cp_cell;    // [CP]
    DevBuf<int32_t> cp_pose;     // [CP]
    DevBuf<int32_t> cell_first_pose;  // [C]

    // ---- current tree shape and point order -----------------------------------------------------
    bool shaped = false;         // current arrays valid
    bool order_virgin = false;   // perm / mort / leaf_of not copied from the base order yet (see reset_shape)
    uint32_t A = 0;
    uint32_t A_shape = 0;        // A when the shape was built (istart[] positions refer to that order)
    DevBuf<uint32_t> perm;       // [A] position -> r ; order = (cell, leaf DFS, pose, input index)
    DevBuf<uint64_t> mort;       // [A]
    DevBuf<uint32_t> leaf_of;    // [A] position -> leaf (DFS index)
    uint32_t L = 0;
    DevBuf<uint32_t> lstart;     // [L+1]
    DevBuf<uint32_t> lcell;      // [L]
    DevBuf<int32_t> lparent;     // [L] internal node id, -1 for an unsplit cell root
    DevBuf<uint64_t> lpath;      // [L] Morton digits from the root (3 bits per level)
    DevBuf<uint8_t> ldepth;      // [L]
    DevBuf<uint8_t> lchild;      // [L]
    uint32_t I = 0;
    size_t icap = 0;             // capacity of the internal-node arrays (grown geometrically: no copy per level)
    DevBuf<uint32_t> istart;     // [I] first position of the internal node's range
    DevBuf<uint32_t> icell;      // [I]
    DevBuf<uint8_t> idepth;      // [I]
    DevBuf<uint64_t> ipath;      // [I] Morton digits from the cell root
    DevBuf<int32_t> iparent;     // [I] parent internal node, -1 for a cell root
    DevBuf<uint8_t> ichild;      // [I] child id under the parent
    std::vector<uint32_t> level_ibegin;  // host: internal ids of depth d are [level_ibegin[d], level_ibegin[d + 1])
    int depth_reached = 0;

    // ---- derived tables (rebuilt lazily after the shape or the point set changes) ---------------
    bool order_valid = false;    // leaf enumeration order + geometry
    DevBuf<uint32_t> cache_rank; // [L] DFS leaf -> position in the reference's leaf order
    DevBuf<uint32_t> leaf_by_cache;  // [L] inverse
    DevBuf<double> leaf_corner;  // [L][3] in cache order
    DevBuf<double> leaf_edge;    // [L]   in cache order
    DevBuf<uint32_t> cell_leaf_begin;  // [C+1] in cache order

    // scheme replay (insert after a subdivision, octree_manager.py:161-171): the split nodes of the last shape,
    // by cell coordinates, imposed again on the rebuilt grid the next time the shape is needed
    bool replay_pending = false;
    uint32_t sp_n = 0;
    DevBuf<long long> sp_q;      // [sp_n][3]
    DevBuf<uint32_t> sp_depth;   // [sp_n]
    DevBuf<uint64_t> sp_path;    // [sp_n]
    DevBuf<uint32_t> sp_epoch;   // [sp_n] (only while epochs_valid)

    // Leaf enumeration order across SEVERAL subdivide calls.  Every pose octree of the reference keeps its leaf list across
    // calls (octree_base.py:48-49, octree.py:183-191): with node_epoch(v) = first subdivide call whose scheme split v and
    // pose_epoch(p) = calls made before pose p was created, the leaves of pose p inside a cell are enumerated by
    // (max(node_epoch(parent), pose_epoch(p)), one-call order).  One call (every BASELINE configuration): all epochs are 1
    // and nothing below is touched.  From the second call on the epoch of every internal node is carried over from the
    // previous shape (matched by cell coordinates, depth, path) and the block order adds the epoch to its sort key.
    int n_subdivide_calls = 0;
    std::vector<int> pose_epoch;   // host, per pose index
    bool epochs_valid = false;     // iepoch[] holds the epochs (false: every internal node has epoch 1)
    DevBuf<uint32_t> iepoch;       // [I]
    bool history_active() const { return n_subdivide_calls >= 2 && epochs_valid && I > 0; }
    void assign_epochs(int epoch, const uint64_t* sorted_keys, const uint32_t* sorted_vals, uint32_t n_saved);

    bool blocks_valid = false;
    uint32_t NB = 0;
    DevBuf<uint32_t> blk_start;  // [NB+1] position of the block's first point
    DevBuf<uint32_t> blk_leaf;   // [NB] DFS leaf index
    DevBuf<int32_t> blk_pose;    // [NB]
    DevBuf<uint32_t> blk_words;     // [(A + 31) / 32] block-head bit of every position
    DevBuf<uint32_t> blk_word_off;  // [(A + 31) / 32] blocks that start before every word of blk_words
    RunIndex blk_index() const { return RunIndex{blk_words.get(), blk_word_off.get(), d_nb.get(), A}; }
    DevBuf<uint32_t> blk_of_pos; // [A] position -> block, derived from the run index on demand (ensure_blk_of_pos)
    bool blk_of_pos_valid = false;
    void ensure_blk_of_pos();
    uint32_t max_block = 0;
    bool max_block_known = false;  // max_block holds the size of the largest block
    bool max_block_enqueued = false;  // ... or a kernel that leaves it in d_max_block has been launched
    void enqueue_max_block();
    DevBuf<uint32_t> d_max_block;  // [1]

    // ---- RANSAC results of the last ol_forest_ransac call ----------------------------------------
    bool ransac_valid = false;   // `mask` is aligned with the current point order (not applied yet)
    DevBuf<uint8_t> mask;        // [A at the time of the call] inlier mask per position
    uint32_t mask_n = 0;
    uint32_t res_n = 0;          // snapshot of the block table in reference order, with the planes
    DevBuf<int32_t> res_pose, res_leaf, res_size, res_best, res_count;  // [res_n]
    DevBuf<float> res_plane;     // [res_n][4]
    bool snap_pending = false;   // res_* not gathered yet: raw per-block arrays of the last run (block-table order)
    DevBuf<uint32_t> sn_ref_order, sn_leaf;
    DevBuf<uint32_t> sn_arr_rank, sn_arr_blk;  // sort-free batch layout: (pose rank, block) in arranged order, sorted on demand
    int sn_rank_bits = 0;
    int sn_K = 0;            // blocks with fewer points were not fitted: their result rows are undefined
    DevBuf<int32_t> sn_pose, sn_size, sn_best, sn_count;
    DevBuf<float> sn_plane;
    bool sample_oob_seen = false;
    uint32_t last_ransac_work = 0;  // blocks scored by the last RANSAC launch
    Profiler prof;

    explicit Forest(const ol_forest_config& c);
    ~Forest();

    // pipeline stages
    int insert(const double* xyz, int64_t n, bool on_device, const int64_t* seg_sizes, const int32_t* seg_pose_in,
               const int64_t* seg_first_in, int n_segments, int n_poses_total);
    int insert_batch(const double* const* xyz_dev, const int64_t* sizes, int count);  // many device clouds, one copy kernel
    void build();            // K1-K3: keygen, sort, cells
    void ensure_cell_poses();  // (cell, pose) pairs of the base order
    void compact_base();     // drop dead points from the base order
    struct CompactTables {
        DevBuf<uint32_t> bits, word_off, tile_off;
    };
    uint32_t compact_tables(const uint8_t* keep, const uint32_t* via, uint32_t n, CompactTables& t);
    void compact_move(CompactTables& t, uint32_t n, const uint32_t* perm_in, const uint64_t* mort_in, const uint32_t* aux_in,
                      uint32_t* perm_out, uint64_t* mort_out, uint32_t* aux_out);
    void ensure_alive();     // alive_r := membership in the current order, if apply_keep left it stale
    void extend_morton();    // Morton codes at the full depth (lazy: MORTON_INITIAL_DEPTH levels first)
    void reset_shape();      // current := base (every cell one leaf)
    // Split rule of K4, piecewise constant in the octree level (node-size thresholds: criteria.py): entry e applies to the
    // levels [first_level[e], first_level[e + 1]); threshold form (count > max_points[e]) or table form
    // (tables[e][count], counts >= table_len use beyond[e]).
    struct SplitRule {
        std::vector<int> first_level;
        std::vector<int64_t> max_points;
        const uint8_t* tables_host = nullptr;  // [entries][table_len]
        int64_t table_len = 0;
        std::vector<int> beyond;
        // geometric terms (geometry.cuh), OR-ed with the count rule: entry e owns terms[term_begin[e] .. term_begin[e + 1])
        std::vector<ol_geom_term> terms;
        std::vector<int> term_begin;  // empty: no entry has terms
        int n_terms(int e) const { return term_begin.empty() ? 0 : term_begin[e + 1] - term_begin[e]; }
        bool needs_cov(int e) const {
            for (int t = 0; t < n_terms(e); ++t)
                if (terms[term_begin[e] + t].stat == OL_GEOM_THICKNESS) return true;
            return false;
        }
        // fewest points of a node on which a term of entry e can hold (a "> value" term needs at least one point)
        int64_t geom_min_points(int e) const {
            int64_t m = INT64_MAX;
            for (int t = 0; t < n_terms(e); ++t) {
                const ol_geom_term& g = terms[term_begin[e] + t];
                m = std::min<int64_t>(m, g.op == OL_GEOM_GT ? std::max<int64_t>(g.min_points, 1) : g.min_points);
            }
            return m;
        }
        int entry_for(int level) const {
            int e = 0;
            for (size_t i = 0; i < first_level.size(); ++i)
                if (first_level[i] <= level) e = (int)i;
            return e;
        }
    };
    void subdivide(const SplitRule& rule, const int32_t* poses, int n_poses_listed);  // K4
    void split_levels(const SplitRule* rule, const uint8_t* d_tables, const uint8_t* d_listed, int n_listed,
                      const uint64_t* replay_keys, uint32_t n_replay, const ol_geom_term* d_terms = nullptr);  // the level loop of K4
    void reserve_internal(size_t need);
    void ensure_max_block();
    // copies up to 8 small device objects into the pinned scratch block back to back with ONE stream synchronisation
    struct ReadItem {
        const void* src;
        size_t bytes;
        void* dst;
    };
    void read_back(std::initializer_list<ReadItem> items);
    void throw_device_errors(uint32_t e);
    void note_ransac_flags(uint32_t e);
    uint32_t export_shape(long long* q_host, uint32_t* depth_host, unsigned long long* path_host);  // NULL: count only
    void impose_shape(const long long* q_host, const uint32_t* depth_host, const unsigned long long* path_host, uint32_t n);
    void save_shape();       // record the split nodes before a rebuild
    void replay_shape();     // impose the recorded shape on the rebuilt grid
    void ensure_shape();
    void materialize_order();  // perm / mort / leaf_of := base order, if reset_shape deferred the copy
    void ensure_order();     // K5: leaf enumeration order + geometry
    void ensure_blocks();    // (pose, leaf) runs
    void filter(const uint8_t* keep_table, int64_t table_len, const int32_t* poses, int n_poses_listed,
                const ol_geom_term* terms = nullptr, int n_terms = 0);
    int64_t export_block_stats(const int32_t* pose_rank, int pose, int32_t* o_pose, int64_t* o_n, double* o_mean, double* o_cov,
                               double* o_ext);
    void apply_keep(const uint8_t* keep_pos);  // K7: drop positions with keep == 0
    void compute_ref_order(const int32_t* pose_rank_host, DevBuf<uint32_t>& ref_order, DevBuf<int32_t>& d_pose_rank,
                           DevBuf<uint32_t>* sorted_rank = nullptr);
    void ransac(const double* table_host, int H, int K, double threshold, const int32_t* pose_rank, int ppb, bool apply,
                uint32_t flags, const int64_t* pose_start = nullptr);
    void pose_point_counts(int64_t* out_host);
    void apply_mask();
    void materialize_snapshot();
    void drop_snapshot();
    void apply_pose_mask(const int32_t* pose_rank, int pose, const uint8_t* mask_host, int64_t n);
    void pose_counts(int64_t* out_host);
    void stats(ol_forest_stats* s, bool light = false);
    std::string profile_report();  // "name count total_ms" per line; clears the records
    void export_cells(int64_t* q, double* corner, int32_t* first_pose, int64_t* n_nodes, int64_t* leaf_begin);
    void export_cell_poses(int32_t* cell, int32_t* pose);
    void export_leaves(double* corner, double* edge, int32_t* cell, int32_t* depth, int32_t* parent_epoch);
    void export_blocks(const int32_t* pose_rank, int32_t* pose, int32_t* leaf, int32_t* size);
    int64_t export_ransac(bool scored_only, bool count_only, int32_t* pose, int32_t* leaf, int32_t* size, float* plane,
                          int32_t* best, int32_t* count);
    int64_t export_points(const int32_t* pose_rank, int pose, int order, double* xyz, int64_t* idx, int32_t* cell,
                          uint8_t* mask_out);
    void check_device_errors();
    void upload_segments();
    uint32_t read_u32(const uint32_t* dptr);
    unsigned long long read_u64(const unsigned long long* dptr);
};

// ransac.cu
void launch_ransac(Ctx& c, const double* points, int64_t n_points, const uint32_t* blk_phys_start,
                   const int32_t* blk_size, const long long* blk_ref_start, const uint32_t* work_list, const uint32_t* pk_start,
                   uint32_t n_work, uint32_t max_block, const double* table, int H, int K, double threshold, uint8_t* mask, float* plane,
                   int32_t* best, int32_t* best_count, uint32_t flags);

void ransac_stats_read(unsigned long long out[16], bool reset);

}  // namespace ol
