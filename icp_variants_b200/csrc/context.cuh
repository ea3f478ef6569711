// context.cuh -- private to the host side of the icp_gpu_* C ABI (include/icp_gpu.h): the context, its device buffers and the
// steps the entry points share.  Host code only; the entry points live in one file per subsystem (context.cu, clouds.cu, ...) and
// take their C linkage from the declarations in icp_gpu.h.
#pragma once
#include "icp_internal.cuh"
#include <string.h>
#include <vector>

#define DESC_QUERY (ICP_MAX_ITERS)       // descriptor slot used by icp_gpu_query_matches
#define DESC_TOTAL (ICP_MAX_ITERS + 1)

// A device allocation of the context, grown by ensure() and freed with the context.
struct DeviceBuf {
    void* p = nullptr; size_t cap = 0;
    DeviceBuf() = default;
    DeviceBuf(DeviceBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    ~DeviceBuf() { if (p) cudaFree(p); }
};

struct icp_gpu_ctx {
    int device = 0, n_sms = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_stream = nullptr;                      // host uploads run here and overlap the previous cloud's build
    // The part of buildIndex that reads only the library's own data (tree levels, boxes, adjacency lists) runs on aux_stream, so that
    // whatever the caller enqueues next on `stream` (normally the source's pack + sort) overlaps it; consumers of the index join first.
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_index_ready = nullptr;
    MatchChunks chunks;                                      // streams + events of the chunked search (created with the context)
    bool index_pending = false;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr};           // [target, source]: staging filled
    cudaEvent_t ev_xyz[2] = {nullptr, nullptr};              // the points of the upload are there (normals and colours follow)
    IcpLatePack late[2]; bool late_pending[2] = {false, false};   // normal records still to be packed by the sort
    cudaEvent_t ev_packed[2] = {nullptr, nullptr};           // staging consumed by the pack kernel
    bool packed_once[2] = {false, false};
    DeviceBuf stage2;                                        // the source's staging area (the target uses `stage`)
    icp_gpu_config cfg;
    float K[9]; uint32_t width = 0, height = 0; bool have_camera = false;
    // clouds
    DeviceBuf stage, src_raw_pts, src_raw_nrm, src_pts, src_nrm, tgt_pts, tgt_nrm, tgt_pts_sorted, tgt_nrm_sorted;
    int n_src = -1, n_tgt = -1;
    std::vector<uint8_t> src_finite;   // host copy of "point and normal finite" per ORIGINAL source index
    bool src_finite_valid = false;
    std::vector<int> src_rank;         // host copy: original source index -> position in the sorted source
    bool src_rank_valid = false;
    // target grid
    DeviceBuf grid, bbox, bvh_box, bvh_desc, leaf_start, leaf_rank, node_rank, child_start, adj, adj_box, adj1, adj1_box, adj_gap;
    // sort / tree scratch, one set per cloud (the two builds run on different streams)
    struct SortBufs { DeviceBuf keys_a, keys_b, idx_a, idx_b, hist, msd; unsigned int* keys_sorted = nullptr; int msd_shift = 0; };
    SortBufs tsort, ssort;
    DeviceBuf lv_flags, lv_tiles, delta_a, delta_b;
    int adj1_capacity = 0;
    int adj_capacity = 0;
    int T = 0; bool grid_built = false; double index_ms = 0.0;
    bool nn_stale = true;                                    // a new cloud made the remembered neighbours (nn_pos / nn_leaf) meaningless
    // source grid: only its sort order is used (consecutive queries are spatial neighbours: coherent tree walks)
    DeviceBuf sgrid, sbbox, order_dev, voxel_table;
    int Ts = 0;
    // loop state
    DeviceBuf state, desc, mask, match_pos, match_w, match_idx, nn_pos, nn_leaf, qbuf, seedbuf, partials, pose_dev, history;
    DeviceBuf nrm_out_dev;
    DeviceBuf prep_in, prep_tmp, prep_out, gt_src, gt_ref, met_partial, met_out;
    DeviceBuf scratch[16];                                   // operands of the value-level entry points (transform, weights, solve)
    DeviceBuf batch_io, batch_scratch, batch_plan;           // batched registration: uploaded operands + results, match slices, configs + pair lists + masks
    DeviceBuf ms_io, ms_nn, ms_scratch, ms_desc, ms_mask;    // multi-start registration: operands + results, per-(start, query) neighbours and match slices, plan
    DeviceBuf bi_io, bi_arena, bi_scratch, bi_plan;          // indexed batch: operands + results, per-pair clouds and indices, build scratch, plans + pair table
    DeviceBuf vox_io, vox_tmp;                               // voxel downsampling: operands + results, voxel records + sort + compaction
    long long n_gt = 0; int last_iters = 0;
    float* h_pose = nullptr; float* h_history = nullptr; DevState* h_state = nullptr;   // pinned
    IterDesc* h_desc = nullptr;                                                       // pinned, DESC_TOTAL
    int n_reduce_blocks = 1;
    // graph cache
    cudaGraphExec_t graph_exec = nullptr;
    std::vector<long long> graph_key;
    uint64_t graph_launches = 0;
    // async call state
    bool pending = false; int pending_iters = 0;
    // shard iteration state
    bool shard_open = false; int shard_algo = 0, shard_iters = 0;
    // point-sharded registration over peer memory (icp_gpu_peer_*)
    void* peer_box = nullptr;                               // own mailbox (plain cudaMalloc: exportable through CUDA IPC)
    void* peer_ptr[ICP_MAX_PEERS] = {nullptr};              // every rank's mailbox as mapped here
    bool peer_ipc[ICP_MAX_PEERS] = {false};                 // opened with cudaIpcOpenMemHandle (to be closed)
    int peer_world = 0, peer_rank = 0, peer_plan_check = 0;
    uint64_t peer_epoch = 0;                                // part of the graph key: a new attachment is a new graph
    icp_gpu_stats stats;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    char err[512];
};

// Sets the context's last error message (when there is a context) and returns `code`.
int fail(icp_gpu_ctx* c, int code, const char* fmt, ...);

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) return fail(ctx, ICP_GPU_E_CUDA, "%s: %s", #call, cudaGetErrorString(e__)); \
    } while (0)

// graph_reads = false: a buffer no captured graph refers to (the batch entry points'), so growing it keeps the cached graph
int ensure(icp_gpu_ctx* ctx, DeviceBuf& b, size_t bytes, bool graph_reads = true);
// Entry prologue: a null context is ICP_GPU_E_ARG; with `idle`, a pending registration is refused; the context's device is made current.
int enter(icp_gpu_ctx* ctx, bool idle = true);
// Consumers of the target index (and anything that overwrites it) first wait for the part of its build that runs on aux_stream.
int join_index(icp_gpu_ctx* ctx);
// The pose up through the pinned staging, then the loop state reset to it.  Only the registration loop has early-stop thresholds.
int upload_pose(icp_gpu_ctx* ctx, const float pose[16], float stop_rot = 0.f, float stop_trans = 0.f);
// DevState.status of a finished loop as the return code and message.  `iteration` (-1: none) is named in the message; `no_match` is
// the printf format of the ICP_GPU_E_NO_MATCHES message, given the iteration.
int status_error(icp_gpu_ctx* ctx, int status, int iteration, const char* no_match);
// Offsets of segments of the given byte sizes laid out one after the other in one allocation, each 256-byte aligned; returns the total.
size_t pack_segments(const size_t* sizes, int n, size_t* off);

// The iterations of one registration (make_plan, registration.cu).
struct Plan {
    int n_iters = 0;
    std::vector<IterDesc> desc;         // n_iters entries
    std::vector<uint32_t> mask;         // concatenated selection masks, one bit per original source index (mt19937 mode)
    std::vector<int> voxel_depth;       // voxel pyramid: grid depth of every mask slot built on the device
};

// 32-bit words of a selection mask over n source points (one word at least)
inline size_t mask_words(long long n) { return ((size_t)(n > 0 ? n : 1) + 31) / 32; }

// The query set "every point": stride 1, no mask, no finite filter, no device selection stream.
inline IterDesc all_points_desc() {
    IterDesc d; memset(&d, 0, sizeof(d));
    d.stride = 1; d.mask_word_offset = -1; d.proba = -1.0f;
    return d;
}

// "Point and normal finite" (PointCloud.h:335) of the xyz triples p and m; without normals (m null) the point alone.
inline bool point_finite(const float* p, const float* m) {
    return isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]) && (!m || (isfinite(m[0]) && isfinite(m[1]) && isfinite(m[2])));
}

// Where one cloud's build writes: the packed records, the grid and the sort, and for a target its index (grid.cu's launchers).  The
// context's clouds point it at their own buffers; the indexed batch at one pair's slices of its arena and at scratch the pairs share.
struct CloudBufs {
    float4 *pts, *nrm;                                       // packed records, upload order
    unsigned int* bbox; GridParams* grid;                    // 8 words ([7]: points with a non-finite coordinate); the grid
    unsigned int *keys_a, *keys_b, *idx_a, *idx_b, *hist, *msd;   // the sort (msd null: no MSD table)
    float4 *pts_sorted, *nrm_sorted;
    unsigned char* lv_flags; unsigned int* lv_tiles; int *delta_a, *delta_b;    // the index: tree scratch, then the tree
    unsigned int *leaf_start, *leaf_rank, *node_rank, *child_start; BvhDesc* bvh_desc; float4* bvh_box;
    unsigned int *adj, *adj1; float4 *adj_box, *adj1_box; float* adj_gap; int adj_capacity, adj1_capacity;
    unsigned int* keys_sorted; int msd_shift;                // set by sort_cloud: keys_a or keys_b, and the MSD table's shift
};
// Adjacency capacities of a target of n points: lists for up to n/4 leaves (a healthy tree has ~n/20) and n/32 level-1 nodes; a
// cloud with more simply gets no shortcut for the rest.
inline int adj_capacity_for(int n) { return (n > 0 ? n : 1) / 4 + 64; }
inline int adj1_capacity_for(int n) { return (n > 0 ? n : 1) / 32 + 64; }

int pick_T(int n, bool source);                                                                                            // clouds.cu
// AoS3 (device arrays; n = 0: nothing) -> b.pts / b.nrm, b.bbox, b.grid; clears b.hist for the sort.  with_normals = false: the
// normal records follow through the sort's IcpLatePack.
int pack_cloud(icp_gpu_ctx* ctx, CloudBufs& b, const float* xyz, const float* nrm, const uint8_t* rgba, int n, int T, bool with_normals); // clouds.cu
int sort_cloud(icp_gpu_ctx* ctx, CloudBufs& b, int n, int T, const IcpLatePack* late, int* launches);                     // clouds.cu
int build_tree(icp_gpu_ctx* ctx, const CloudBufs& b, int n, int T, cudaStream_t s, int* launches);                        // clouds.cu
int check_config(icp_gpu_ctx* ctx, const icp_gpu_config* c, const char* who);                                          // context.cu
int set_cloud(icp_gpu_ctx* ctx, bool target, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n, bool dev);  // clouds.cu
int fetch_src_rank(icp_gpu_ctx* ctx);                                                                                      // clouds.cu
int fetch_src_finite(icp_gpu_ctx* ctx);                                                                                    // clouds.cu
void draw_selection_masks(const icp_gpu_config& cfg, const IcpSchedule& sch, long long n, const uint8_t* finite, uint32_t* out);  // registration.cu
int choose_algorithm(const icp_gpu_ctx* c);                                                                                // registration.cu
int check_ready(icp_gpu_ctx* ctx);                                                                                         // registration.cu
void fill_match_args(icp_gpu_ctx* c, MatchArgs& a, int algo, int desc_index, bool want_idx);                               // registration.cu
void fill_reduce_args(icp_gpu_ctx* c, ReduceArgs& r, int algo, int solve);                                                 // registration.cu
int refresh_seeds(icp_gpu_ctx* ctx, int algo, bool allow_seed);                                                            // registration.cu
// The plan of a registration with cfg of a source of n points whose grid has depth Ts; finite: its "point and normal finite" flags
// per original index (read with mt19937 selection and multires only).
int plan_iterations(icp_gpu_ctx* ctx, const icp_gpu_config& cfg, int n, int Ts, const uint8_t* finite, Plan& plan);    // registration.cu
int make_plan(icp_gpu_ctx* ctx, Plan& plan);                                                                               // registration.cu
int upload_plan(icp_gpu_ctx* ctx, const Plan& plan, IterDesc* desc, DeviceBuf& mask, bool graph_reads);                   // registration.cu
// The plan's voxel pyramid levels of the sorted source (src_pts / src_nrm, its grid of depth Ts) into mask (slot j at j * words);
// table: scratch of 2^(deepest level) entries.
int build_voxel_levels(icp_gpu_ctx* ctx, const Plan& plan, const float4* src_pts, const float4* src_nrm, int n, const GridParams* grid, int Ts,
                       unsigned int* table, unsigned int* mask, size_t words);                                             // registration.cu
void peer_close(icp_gpu_ctx* ctx);                                                                                         // sharded.cu
