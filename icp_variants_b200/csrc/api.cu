// api.cu -- the icp_gpu_* C ABI (include/icp_gpu.h): context, device buffers, iteration planning,
// CUDA-graph replay of the registration loop.  Host code only; the kernels live in grid.cu,
// match.cu, solve.cu and lm.cu.
//
// What runs where: the host plans the iterations (level strides, selection masks) and enqueues
// them; every iteration is {match kernel, reduction(+solve) kernel(s)} on one stream with no host
// synchronisation in between -- the loop state (pose, iteration counter, status) lives in DevState
// on the device.  The only host<->device traffic of estimate_pose is the iteration descriptors and
// the 16-float pose up, and the pose, pose history and DevState down.
//
// Reference: ICPOptimizer.h:185-349 / :493-663 (the loop), NearestNeighbor.h:12-36 (matcher API).
#include "icp_internal.cuh"
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <map>
#include <new>
#include <string>
#include <vector>

#define DESC_QUERY (ICP_MAX_ITERS)       // descriptor slot used by icp_gpu_query_matches
#define DESC_TOTAL (ICP_MAX_ITERS + 1)

namespace {

// std::mt19937 + libstdc++ generate_canonical<double,53> (selection.h:88-104, contract D7)
struct Mt19937 {
    uint32_t mt[624]; int idx;
    void seed(uint32_t s) {
        mt[0] = s;
        for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
        idx = 624;
    }
    uint32_t next() {
        if (idx >= 624) {
            for (int i = 0; i < 624; ++i) {
                const uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
                mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
            idx = 0;
        }
        uint32_t y = mt[idx++];
        y ^= (y >> 11); y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= (y >> 18);
        return y;
    }
    double canonical() {
        const double lo = (double)next(), hi = (double)next();
        double v = (lo + hi * 4294967296.0) / 18446744073709551616.0;
        if (v >= 1.0) v = nextafter(1.0, 0.0);
        return v;
    }
};

long long __float_as_int_host(float f) { int32_t i; memcpy(&i, &f, 4); return (long long)i; }

struct DeviceBuf {
    void* p = nullptr; size_t cap = 0;
};

struct Plan {
    int n_iters = 0;
    std::vector<IterDesc> desc;         // n_iters entries
    std::vector<uint32_t> mask;         // concatenated selection masks, one bit per original source index (mt19937 mode)
    std::vector<int> voxel_depth;       // voxel pyramid: grid depth of every mask slot built on the device
};

}  // namespace

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

namespace {

int fail(icp_gpu_ctx* c, int code, const char* fmt, ...) {
    if (c) {
        va_list ap; va_start(ap, fmt);
        vsnprintf(c->err, sizeof(c->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) return fail(ctx, ICP_GPU_E_CUDA, "%s: %s", #call, cudaGetErrorString(e__)); \
    } while (0)

// graph_reads = false: a buffer no captured graph refers to (the batch entry points'), so growing it keeps the cached graph
int ensure(icp_gpu_ctx* ctx, DeviceBuf& b, size_t bytes, bool graph_reads = true) {
    if (bytes <= b.cap && b.p) return 0;
    if (graph_reads && ctx->graph_exec) { cudaGraphExecDestroy(ctx->graph_exec); ctx->graph_exec = nullptr; ctx->graph_key.clear(); }
    if (b.p) { cudaStreamSynchronize(ctx->stream); if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream); if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream); cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    CU(cudaMalloc(&b.p, want));
    b.cap = want;
    return 0;
}

int bind(icp_gpu_ctx* ctx) {
    CU(cudaSetDevice(ctx->device));
    return 0;
}

int pick_T(int n, bool source = false) {
    // Target: the finest grid the 32-bit keys hold (10 bits per axis) -- the radix sort costs the same for any T, and fine
    // cells give compact leaves.  Source: 4 cells per point; its grid also defines the voxel pyramid levels, which the
    // oracle restates (oracle/icp_oracle.c:orc_pick_T).
    if (!source) {
        int T = 3 * ICP_MAX_BITS_PER_AXIS;
        if (const char* e = getenv("ICP_GPU_TARGET_GRID_BITS")) { const int v = atoi(e); if (v >= 3 && v <= 3 * ICP_MAX_BITS_PER_AXIS) T = v; }   // tuning knob
        return T;
    }
    int T = 3;
    while (T < 24 && (1ll << T) < (long long)ICP_SOURCE_CELLS_PER_POINT * (long long)(n > 0 ? n : 1)) ++T;
    if (T > 3 * ICP_MAX_BITS_PER_AXIS) T = 3 * ICP_MAX_BITS_PER_AXIS;
    return T;
}

int choose_algorithm(const icp_gpu_ctx* c) {   // 0 grid, 1 brute, 2 projective
    if (c->cfg.matching == ICP_GPU_MATCH_PROJECTIVE) return 2;
    if (c->cfg.nn_algorithm == ICP_GPU_NN_BRUTE || c->cfg.nn_algorithm == ICP_GPU_NN_BRUTE_NORM) return 1;
    if (c->cfg.nn_algorithm == ICP_GPU_NN_GRID) return 0;
    return c->n_tgt <= 2048 ? 1 : 0;
}

// Consumers of the target index (and anything that overwrites it) first wait for the part of its build that runs on aux_stream.
int join_index(icp_gpu_ctx* ctx) {
    if (!ctx->index_pending) return 0;
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_index_ready, 0));
    ctx->index_pending = false;
    return 0;
}

int ensure_sort(icp_gpu_ctx* ctx, icp_gpu_ctx::SortBufs& sb, int n, int T) {
    const size_t n1 = (size_t)(n > 0 ? n : 1);
    if (ensure(ctx, sb.keys_a, n1 * 4) || ensure(ctx, sb.keys_b, n1 * 4) || ensure(ctx, sb.idx_a, n1 * 4) || ensure(ctx, sb.idx_b, n1 * 4) ||
        ensure(ctx, sb.hist, icp_radix_hist_words(n, T) * 4) || ensure(ctx, sb.msd, ICP_MSD_WORDS * 4)) return ICP_GPU_E_CUDA;
    return 0;
}

int upload_cloud(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n, bool device_ptrs,
                 DeviceBuf& pts, DeviceBuf& nrmb, int kind /*0 target, 1 source*/) {
    const size_t n1 = (size_t)(n > 0 ? n : 1);
    DeviceBuf& bbox = kind == 0 ? ctx->bbox : ctx->sbbox;
    DeviceBuf& grid = kind == 0 ? ctx->grid : ctx->sgrid;
    icp_gpu_ctx::SortBufs& sb = kind == 0 ? ctx->tsort : ctx->ssort;
    // the pack kernel also derives the grid parameters and clears the histograms of the sort that follows
    const int T = pick_T((int)n, kind == 1);
    if (kind == 0) ctx->T = T; else ctx->Ts = T;
    if (ensure(ctx, pts, n1 * sizeof(float4)) || ensure(ctx, nrmb, n1 * sizeof(float4)) || ensure(ctx, bbox, 64) || ensure(ctx, grid, sizeof(GridParams)) ||
        ensure_sort(ctx, sb, (int)n, T)) return ICP_GPU_E_CUDA;
    const long long hist_words = (long long)icp_radix_hist_words((int)n, T);
    if (n == 0) {
        CU(icp_launch_pack_cloud(nullptr, nullptr, nullptr, 0, (float4*)pts.p, (float4*)nrmb.p, (unsigned int*)bbox.p, T, (GridParams*)grid.p,
                                 (unsigned int*)sb.hist.p, hist_words, 1, ctx->stream));
        ctx->late_pending[kind] = false;
        return 0;
    }
    const float* dx = xyz; const float* dn = nrm; const uint8_t* dc = rgba;
    if (!device_ptrs) {
        // Host arrays go through a per-cloud staging area on the copy stream, so that the upload of one cloud overlaps
        // the index build of the other on the compute stream.
        DeviceBuf& stage = kind == 0 ? ctx->stage : ctx->stage2;
        const size_t bx = (size_t)n * 12, bc = (size_t)n * 4;
        const size_t ox = 0, on = (bx + 255) / 256 * 256, oc = on + (nrm ? (bx + 255) / 256 * 256 : 0);
        if (ensure(ctx, stage, oc + (rgba ? bc : 0) + 256)) return ICP_GPU_E_CUDA;
        char* st = (char*)stage.p;
        if (ctx->packed_once[kind]) CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_packed[kind], 0));   // staging still being read?
        CU(cudaMemcpyAsync(st + ox, xyz, bx, cudaMemcpyHostToDevice, ctx->copy_stream));
        CU(cudaEventRecord(ctx->ev_xyz[kind], ctx->copy_stream));       // the sort starts from the points alone
        dx = (const float*)(st + ox);
        if (nrm) { CU(cudaMemcpyAsync(st + on, nrm, bx, cudaMemcpyHostToDevice, ctx->copy_stream)); dn = (const float*)(st + on); }
        if (rgba) { CU(cudaMemcpyAsync(st + oc, rgba, bc, cudaMemcpyHostToDevice, ctx->copy_stream)); dc = (const uint8_t*)(st + oc); }
        CU(cudaEventRecord(ctx->ev_copied[kind], ctx->copy_stream));
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_xyz[kind], 0));
        // the normal / colour records are packed by the sort just before its last pass (the only one that moves them)
        ctx->late[kind].nrm = dn; ctx->late[kind].rgba = dc; ctx->late[kind].nrmo = (float4*)nrmb.p; ctx->late[kind].ready = ctx->ev_copied[kind];
    }
    ctx->late_pending[kind] = !device_ptrs;
    CU(icp_launch_pack_cloud(dx, dn, dc, (int)n, (float4*)pts.p, (float4*)nrmb.p, (unsigned int*)bbox.p, T, (GridParams*)grid.p,
                             (unsigned int*)sb.hist.p, hist_words, device_ptrs ? 1 : 0, ctx->stream));
    ctx->stats.n_kernel_launches += 1;
    return 0;
}

// buildIndex: radix sort by cell code, leaves and upper levels from the sorted keys, tight boxes, adjacency lists.
int build_grid(icp_gpu_ctx* ctx) {
    const int n = ctx->n_tgt;
    const size_t n1 = (size_t)(n > 0 ? n : 1);
    if (ensure(ctx, ctx->tgt_pts_sorted, n1 * sizeof(float4)) || ensure(ctx, ctx->tgt_nrm_sorted, n1 * sizeof(float4)) ||
        ensure(ctx, ctx->lv_flags, n1 + 64) || ensure(ctx, ctx->lv_tiles, (n1 / 1024 + 2) * 4) ||
        ensure(ctx, ctx->delta_a, (n1 + 2) * 4) || ensure(ctx, ctx->delta_b, (n1 + 2) * 4) ||
        ensure(ctx, ctx->leaf_start, (n1 + 2) * 4) || ensure(ctx, ctx->leaf_rank, (n1 + 2) * 4) || ensure(ctx, ctx->bvh_desc, sizeof(BvhDesc)) ||
        ensure(ctx, ctx->bvh_box, icp_bvh_max_nodes(n) * 2 * sizeof(float4)) ||
        ensure(ctx, ctx->node_rank, (icp_bvh_max_nodes(n) + ICP_BVH_MAX_LEVELS) * 4) ||
        ensure(ctx, ctx->child_start, (icp_bvh_max_nodes(n) + ICP_BVH_MAX_LEVELS) * 4))
        return ICP_GPU_E_CUDA;
    // adjacency lists for up to n/4 leaves (a healthy tree has ~n/20); a cloud with more leaves simply gets no shortcut for the rest
    ctx->adj_capacity = (int)(n1 / 4 + 64);
    ctx->adj1_capacity = (int)(n1 / 32 + 64);
    if (ensure(ctx, ctx->adj, (size_t)ctx->adj_capacity * 32 * 4) || ensure(ctx, ctx->adj_gap, (size_t)ctx->adj_capacity * 32 * 4) ||
        ensure(ctx, ctx->adj_box, (size_t)ctx->adj_capacity * 2 * sizeof(float4)) ||
        ensure(ctx, ctx->adj1, (size_t)ctx->adj1_capacity * 32 * 4) || ensure(ctx, ctx->adj1_box, (size_t)ctx->adj1_capacity * 2 * sizeof(float4)))
        return ICP_GPU_E_CUDA;
    int launches = 0;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;              // a build still running on aux_stream reads what this one overwrites
    CU(cudaEventRecord(ctx->ev[0], ctx->stream));
    CU(icp_launch_cloud_sort((const float4*)ctx->tgt_pts.p, (const float4*)ctx->tgt_nrm.p, n, ctx->T, (const GridParams*)ctx->grid.p,
                             (unsigned int*)ctx->tsort.keys_a.p, (unsigned int*)ctx->tsort.keys_b.p, (unsigned int*)ctx->tsort.idx_a.p,
                             (unsigned int*)ctx->tsort.idx_b.p, (unsigned int*)ctx->tsort.hist.p, (float4*)ctx->tgt_pts_sorted.p,
                             (float4*)ctx->tgt_nrm_sorted.p, (unsigned int*)ctx->tsort.msd.p, &ctx->tsort.keys_sorted, &ctx->tsort.msd_shift,
                             ctx->late_pending[0] ? &ctx->late[0] : nullptr, ctx->stream, &launches));
    if (ctx->late_pending[0]) { CU(cudaEventRecord(ctx->ev_packed[0], ctx->stream)); ctx->packed_once[0] = true; ctx->late_pending[0] = false; }
    cudaStream_t ts = getenv("ICP_GPU_NO_AUX_STREAM") ? ctx->stream : ctx->aux_stream;       // tuning knob (A/B measurement)
    if (ts != ctx->stream) { CU(cudaEventRecord(ctx->ev_fork, ctx->stream)); CU(cudaStreamWaitEvent(ts, ctx->ev_fork, 0)); }
    CU(icp_launch_bvh_build((float4*)ctx->tgt_pts_sorted.p, (float4*)ctx->tgt_nrm_sorted.p, n, ctx->T, ctx->tsort.keys_sorted,
                            (const unsigned int*)ctx->bbox.p + 7, (unsigned char*)ctx->lv_flags.p, (unsigned int*)ctx->lv_tiles.p, (int*)ctx->delta_a.p,
                            (int*)ctx->delta_b.p, (unsigned int*)ctx->leaf_rank.p, (unsigned int*)ctx->leaf_start.p, (unsigned int*)ctx->node_rank.p,
                            (unsigned int*)ctx->child_start.p, (BvhDesc*)ctx->bvh_desc.p, (float4*)ctx->bvh_box.p, ctx->n_sms, ts, &launches));
    const bool bottom_up = !getenv("ICP_GPU_ADJ_FROM_ROOT");                                  // tuning knob (A/B measurement)
    CU(icp_launch_leaf_adjacency((const BvhDesc*)ctx->bvh_desc.p, (const float4*)ctx->bvh_box.p, (const unsigned int*)ctx->child_start.p,
                                 (unsigned int*)ctx->adj1.p, (float4*)ctx->adj1_box.p, ctx->adj1_capacity, 1, nullptr, nullptr, nullptr, 0, ctx->n_sms, ts, &launches));
    CU(icp_launch_leaf_adjacency((const BvhDesc*)ctx->bvh_desc.p, (const float4*)ctx->bvh_box.p, (const unsigned int*)ctx->child_start.p,
                                 (unsigned int*)ctx->adj.p, (float4*)ctx->adj_box.p, ctx->adj_capacity, 0, (const unsigned int*)ctx->node_rank.p,
                                 bottom_up ? (const unsigned int*)ctx->adj1.p : nullptr, (const float4*)ctx->adj1_box.p, ctx->adj1_capacity, ctx->n_sms, ts, &launches,
                                 (float*)ctx->adj_gap.p));
    CU(cudaEventRecord(ctx->ev[1], ts));
    if (ts != ctx->stream) { CU(cudaEventRecord(ctx->ev_index_ready, ts)); ctx->index_pending = true; }
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    ctx->grid_built = true;
    return 0;
}

// Sorts the source into the cell order of its own grid (Morton order); points with a non-finite coordinate keep a slot at the end.
int build_source(icp_gpu_ctx* ctx) {
    const int n = ctx->n_src;
    const size_t n1 = (size_t)(n > 0 ? n : 1);
    if (ensure(ctx, ctx->src_pts, n1 * sizeof(float4)) || ensure(ctx, ctx->src_nrm, n1 * sizeof(float4))) return ICP_GPU_E_CUDA;
    int launches = 0;
    CU(icp_launch_cloud_sort((const float4*)ctx->src_raw_pts.p, (const float4*)ctx->src_raw_nrm.p, n, ctx->Ts, (const GridParams*)ctx->sgrid.p,
                             (unsigned int*)ctx->ssort.keys_a.p, (unsigned int*)ctx->ssort.keys_b.p, (unsigned int*)ctx->ssort.idx_a.p,
                             (unsigned int*)ctx->ssort.idx_b.p, (unsigned int*)ctx->ssort.hist.p, (float4*)ctx->src_pts.p,
                             (float4*)ctx->src_nrm.p, nullptr, &ctx->ssort.keys_sorted, &ctx->ssort.msd_shift,
                             ctx->late_pending[1] ? &ctx->late[1] : nullptr, ctx->stream, &launches));
    if (ctx->late_pending[1]) { CU(cudaEventRecord(ctx->ev_packed[1], ctx->stream)); ctx->packed_once[1] = true; ctx->late_pending[1] = false; }
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    return 0;
}

int set_cloud(icp_gpu_ctx* ctx, bool target, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n, bool dev) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (n < 0 || n > 0x7fffffff / 4 || (n > 0 && !xyz)) return fail(ctx, ICP_GPU_E_ARG, "bad cloud (n=%lld, xyz=%p)", (long long)n, (const void*)xyz);
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending; call icp_gpu_estimate_pose_finish first");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    if (target) {
        if (join_index(ctx)) return ICP_GPU_E_CUDA;      // the previous build's tail (aux_stream) still reads the scratch this upload resets
        if (upload_cloud(ctx, xyz, nrm, rgba, n, dev, ctx->tgt_pts, ctx->tgt_nrm, 0)) return ICP_GPU_E_CUDA;
        ctx->n_tgt = (int)n;
        // buildIndex: the grid is always built (cheap), the matcher choice is made per call
        if (build_grid(ctx)) return ICP_GPU_E_CUDA;
    } else {
        if (upload_cloud(ctx, xyz, nrm, rgba, n, dev, ctx->src_raw_pts, ctx->src_raw_nrm, 1)) return ICP_GPU_E_CUDA;
        ctx->n_src = (int)n;
        ctx->src_finite_valid = false; ctx->src_rank_valid = false;     // fetched lazily from the device when a plan needs them
        const size_t n1 = (size_t)(n > 0 ? n : 1);
        if (ensure(ctx, ctx->match_pos, n1 * 4) || ensure(ctx, ctx->match_w, n1 * 4) || ensure(ctx, ctx->match_idx, n1 * 4) ||
            ensure(ctx, ctx->nn_pos, n1 * 4) || ensure(ctx, ctx->nn_leaf, n1 * 4) || ensure(ctx, ctx->qbuf, n1 * sizeof(float4)) ||
            ensure(ctx, ctx->seedbuf, n1 * sizeof(float4))) return ICP_GPU_E_CUDA;
        ctx->n_reduce_blocks = icp_reduce_blocks((int)n, ctx->n_sms);
        if (ensure(ctx, ctx->partials, (size_t)ctx->n_reduce_blocks * ICP_NRED * sizeof(double))) return ICP_GPU_E_CUDA;
        if (build_source(ctx)) return ICP_GPU_E_CUDA;
    }
    // a new cloud invalidates the neighbours remembered from earlier searches: the next search resets them (seed kernel or fill)
    ctx->nn_stale = true;
    // Host arrays are only borrowed for the duration of the call: wait for the copies (not for the index build, which
    // keeps running on the compute stream).  The device-pointer forms are fully asynchronous.
    if (!dev && n > 0) CU(cudaEventSynchronize(ctx->ev_copied[target ? 0 : 1]));
    return ICP_GPU_OK;
}

// original index -> sorted position (host copy), fetched lazily: only the host-drawn selection
// masks and the query_matches output order need it
int fetch_src_rank(icp_gpu_ctx* ctx) {
    if (ctx->src_rank_valid) return 0;
    const size_t n = (size_t)ctx->n_src;
    std::vector<int> order(n);
    if (n > 0) {
        if (ensure(ctx, ctx->order_dev, n * 4)) return ICP_GPU_E_CUDA;
        CU(icp_launch_extract_order((const float4*)ctx->src_pts.p, (int)n, (int*)ctx->order_dev.p, ctx->stream));
        CU(cudaMemcpyAsync(order.data(), ctx->order_dev.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    ctx->src_rank.assign(n, 0);
    for (size_t p = 0; p < n; ++p) ctx->src_rank[(size_t)order[p]] = (int)p;
    ctx->src_rank_valid = true;
    return 0;
}

// "point and normal finite" flags of a device-resident source, fetched lazily (mt19937 + multires only)
int fetch_src_finite(icp_gpu_ctx* ctx) {
    if (ctx->src_finite_valid) return 0;
    const size_t n = (size_t)ctx->n_src;
    std::vector<float4> p(n), m(n);
    CU(cudaMemcpyAsync(p.data(), ctx->src_raw_pts.p, n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(m.data(), ctx->src_raw_nrm.p, n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->src_finite.resize(n);
    for (size_t i = 0; i < n; ++i)
        ctx->src_finite[i] = (isfinite(p[i].x) && isfinite(p[i].y) && isfinite(p[i].z) && isfinite(m[i].x) && isfinite(m[i].y) && isfinite(m[i].z)) ? 1 : 0;
    ctx->src_finite_valid = true;
    return 0;
}

// The mt19937 selection masks of one registration (selection.h:88-104, contract D7): iteration i's mask is out[i * words ..),
// words = ceil(max(n, 1) / 32), one bit per original source index, zero-filled by the caller.  resample() draws once per point of the
// level cloud, in order: every stride-th point, with multires only those whose point and normal are finite (finite[k], PointCloud.h:335).
// One PointSelection per level (:652), seeded with seed + level (initSampler); its stream runs on across the stride-1 iterations.
void draw_selection_masks(const icp_gpu_config& cfg, const IcpSchedule& sch, long long n, const uint8_t* finite, uint32_t* out) {
    const size_t words = ((size_t)(n > 0 ? n : 1) + 31) / 32;
    Mt19937 rng; int level = -1;
    for (int i = 0; i < sch.n_iters; ++i) {
        const int lv = icp_schedule_level(sch, i), stride = icp_schedule_stride(sch, i);
        if (lv != level) { rng.seed(cfg.seed + (uint32_t)lv); level = lv; }
        uint32_t* m = out + (size_t)i * words;
        for (long long k = 0; k < n; k += stride) {
            if (cfg.multires && !finite[(size_t)k]) continue;
            if (rng.canonical() < cfg.proba) m[k >> 5] |= 1u << (k & 31);
        }
    }
}

// The iteration schedule of estimatePose (ICPOptimizer.h:503-525, :540, :549-550, :634-655; Appendix A of SURVEY.md).
int make_plan(icp_gpu_ctx* ctx, Plan& plan) {
    const icp_gpu_config& cfg = ctx->cfg;
    const int n = ctx->n_src;
    const bool host_rng = cfg.selection == ICP_GPU_SELECT_RANDOM && cfg.selection_rng == ICP_GPU_RNG_MT19937;
    const bool dev_rng = cfg.selection == ICP_GPU_SELECT_RANDOM && cfg.selection_rng == ICP_GPU_RNG_DEVICE;
    if (host_rng && cfg.multires && fetch_src_finite(ctx)) return ICP_GPU_E_CUDA;
    const size_t mask_words = ((size_t)(n > 0 ? n : 1) + 31) / 32;
    const bool voxel = cfg.multires && cfg.pyramid_mode == ICP_GPU_PYRAMID_VOXEL;
    const IcpSchedule sch = icp_schedule(cfg.n_iterations, cfg.multires, n);
    if (sch.n_iters > ICP_MAX_ITERS) return fail(ctx, ICP_GPU_E_ARG, "more than %d iterations", ICP_MAX_ITERS);
    if (host_rng) {
        plan.mask.assign((size_t)sch.n_iters * mask_words, 0u);
        draw_selection_masks(cfg, sch, n, ctx->src_finite.data(), plan.mask.data());
    }
    for (int i = 0; i < sch.n_iters; ++i) {
        const int stride = icp_schedule_stride(sch, i);
        IterDesc d; memset(&d, 0, sizeof(d));
        d.stride = stride; d.mask_word_offset = -1; d.filter_finite = cfg.multires ? 1 : 0; d.proba = -1.0f;
        if (voxel && stride > 1) {
            // level = one point per occupied source-grid cell at depth Ts' - ceil(1.5 log2 stride)
            int k = 0; while ((1 << k) < stride) ++k;
            int D = (ctx->Ts < 22 ? ctx->Ts : 22) - (3 * k + 1) / 2; if (D < 0) D = 0;
            int slot = -1;
            for (size_t j = 0; j < plan.voxel_depth.size(); ++j) if (plan.voxel_depth[j] == D) slot = (int)j;
            if (slot < 0) { slot = (int)plan.voxel_depth.size(); plan.voxel_depth.push_back(D); }
            d.stride = 1; d.mask_word_offset = (int)((size_t)slot * mask_words);
        }
        if (dev_rng) { d.proba = (float)cfg.proba; d.rng_key = cfg.seed * 2654435761u + (uint32_t)(i + 1) * 0x9E3779B9u; }
        if (host_rng) d.mask_word_offset = (int)((size_t)i * mask_words);
        plan.desc.push_back(d);
    }
    plan.n_iters = sch.n_iters;
    return 0;
}

// Field checks of a configuration (icp_gpu_set_config, and every entry of icp_gpu_estimate_pose_batch_configs); `who` prefixes the
// message ("config 3: ").
int check_config(icp_gpu_ctx* ctx, const icp_gpu_config* c, const char* who) {
    if (c->metric < 0 || c->metric > 2) return fail(ctx, ICP_GPU_E_ARG, "%smetric %d", who, c->metric);
    if (c->minimizer < 0 || c->minimizer > 1) return fail(ctx, ICP_GPU_E_ARG, "%sminimizer %d", who, c->minimizer);
    if (c->matching < 0 || c->matching > 1) return fail(ctx, ICP_GPU_E_ARG, "%smatching %d", who, c->matching);
    if (c->selection < 0 || c->selection > 1) return fail(ctx, ICP_GPU_E_ARG, "%sselection %d", who, c->selection);
    if (c->selection_rng < 0 || c->selection_rng > 1) return fail(ctx, ICP_GPU_E_ARG, "%sselection_rng %d", who, c->selection_rng);
    if (c->weighting < 0 || c->weighting > 3) return fail(ctx, ICP_GPU_E_ARG, "%sweighting %d", who, c->weighting);
    if (c->nn_algorithm < 0 || c->nn_algorithm > 3) return fail(ctx, ICP_GPU_E_ARG, "%snn_algorithm %d", who, c->nn_algorithm);
    if (c->nn_algorithm == ICP_GPU_NN_BRUTE_NORM && c->color_icp) return fail(ctx, ICP_GPU_E_ARG, "%sthe norm-thresholded brute-force matcher is 3-D only (NearestNeighbor.h:63-69)", who);
    if (c->pyramid_mode != ICP_GPU_PYRAMID_STRIDE && c->pyramid_mode != ICP_GPU_PYRAMID_VOXEL) return fail(ctx, ICP_GPU_E_ARG, "%spyramid_mode %d", who, c->pyramid_mode);
    if (c->multires && c->pyramid_mode == ICP_GPU_PYRAMID_VOXEL && c->selection == ICP_GPU_SELECT_RANDOM && c->selection_rng == ICP_GPU_RNG_MT19937)
        return fail(ctx, ICP_GPU_E_ARG, "%svoxel pyramid levels are built on the device: use the device selection stream with them", who);
    if (c->n_iterations < 0 || c->n_iterations > ICP_MAX_ITERS) return fail(ctx, ICP_GPU_E_ARG, "%sn_iterations %d (max %d)", who, c->n_iterations, ICP_MAX_ITERS);
    if (c->lm_max_iterations < 0 || c->lm_max_iterations > 64) return fail(ctx, ICP_GPU_E_ARG, "%slm_max_iterations %d", who, c->lm_max_iterations);
    if (!(c->early_stop_rotation >= 0.f) || !(c->early_stop_translation >= 0.f)) return fail(ctx, ICP_GPU_E_ARG, "%searly-stop thresholds must be >= 0", who);
    if (!(c->weight_max_distance_sq >= 0.f)) return fail(ctx, ICP_GPU_E_ARG, "%sweight_max_distance_sq %g", who, (double)c->weight_max_distance_sq);
    if (c->matching == ICP_GPU_MATCH_PROJECTIVE && c->color_icp) return fail(ctx, ICP_GPU_E_ARG, "%scolour ICP is a k-NN variant (main.cpp:240-243)", who);
    return 0;
}

int check_ready(icp_gpu_ctx* ctx) {
    if (ctx->n_src < 0) return fail(ctx, ICP_GPU_E_STATE, "no source cloud set");
    if (ctx->n_tgt < 0) return fail(ctx, ICP_GPU_E_STATE, "no target cloud set (buildIndex)");
    if (ctx->cfg.matching == ICP_GPU_MATCH_PROJECTIVE) {
        // NearestNeighbor.h:335-349
        if (!ctx->have_camera) return fail(ctx, ICP_GPU_E_STATE, "projective matching needs icp_gpu_set_camera");
        if ((long long)ctx->width * ctx->height != (long long)ctx->n_tgt || ctx->height == 0)
            return fail(ctx, ICP_GPU_E_STATE, "projective matching: target size %d != width*height %u*%u", ctx->n_tgt, ctx->width, ctx->height);
    }
    return 0;
}

// Projective matching of a full-frame source (one point per pixel of the camera the target was taken with): the kernels
// then address the source in its original pixel order (the unsorted upload) instead of the Morton order.
bool proj_tiled(const icp_gpu_ctx* c, int algo) {
    return algo == 2 && c->n_src > 0 && (long long)c->width * c->height == (long long)c->n_src && !getenv("ICP_GPU_NO_PROJ_TILES");
}

void fill_match_args(icp_gpu_ctx* c, MatchArgs& a, int algo, int desc_index, bool want_idx) {
    memset(&a, 0, sizeof(a));
    const bool grid_order = (algo == 0);
    a.src_pts = (const float4*)c->src_pts.p; a.src_nrm = (const float4*)c->src_nrm.p; a.n_src = c->n_src;
    a.mask = (const unsigned int*)c->mask.p; a.desc = (const IterDesc*)c->desc.p;
    a.state_ro = (const DevState*)c->state.p; a.state = (DevState*)c->state.p;
    a.tgt_pts = (const float4*)(grid_order ? c->tgt_pts_sorted.p : c->tgt_pts.p);
    a.tgt_nrm = (const float4*)(grid_order ? c->tgt_nrm_sorted.p : c->tgt_nrm.p);
    a.n_tgt = c->n_tgt;
    a.bvh_box = (const float4*)c->bvh_box.p; a.bvh = (const BvhDesc*)c->bvh_desc.p; a.leaf_start = (const unsigned int*)c->leaf_start.p;
    a.leaf_rank = (const unsigned int*)c->leaf_rank.p; a.child_start = (const unsigned int*)c->child_start.p;
    a.adj = (const unsigned int*)c->adj.p; a.adj_box = (const float4*)c->adj_box.p; a.adj_capacity = c->adj_capacity;
    a.adj_gap = getenv("ICP_GPU_NO_ADJ_GAP") ? nullptr : (const float*)c->adj_gap.p;   // tuning knob (A/B measurement)
    a.nn_leaf = (int*)c->nn_leaf.p;
    a.adj1 = (const unsigned int*)c->adj1.p; a.adj1_box = (const float4*)c->adj1_box.p; a.adj1_capacity = c->adj1_capacity;
    a.node_rank = (const unsigned int*)c->node_rank.p;
    if (getenv("ICP_GPU_NO_ADJACENCY1")) a.adj1_capacity = 0;   // tuning knob
    if (getenv("ICP_GPU_NO_ADJACENCY")) a.adj_capacity = 0;   // tuning knob
    if (c->have_camera) { a.fx = c->K[0]; a.fy = c->K[4]; a.cx = c->K[6]; a.cy = c->K[7]; }   // column-major Matrix3f
    a.width = c->width; a.height = c->height;
    a.weighting = c->cfg.weighting; a.rejection = c->cfg.rejection; a.color_icp = c->cfg.color_icp;
    a.max_d2 = c->cfg.max_distance_sq;
    a.weight_max_d2 = c->cfg.weight_max_distance_sq > 0.f ? c->cfg.weight_max_distance_sq : c->cfg.max_distance_sq;
    a.match_pos = (int*)c->match_pos.p; a.match_w = (float*)c->match_w.p; a.match_idx = want_idx ? (int*)c->match_idx.p : nullptr;
    a.nn_pos = (int*)c->nn_pos.p; a.qbuf = (float4*)c->qbuf.p; a.seedbuf = (float4*)c->seedbuf.p;
    a.desc_index = desc_index;
    a.q_begin = 0; a.q_end = c->n_src;
    a.use_seed = grid_order ? 1 : 0;
    a.brute_norm = c->cfg.nn_algorithm == ICP_GPU_NN_BRUTE_NORM ? 1 : 0;
    if (proj_tiled(c, algo)) { a.src_pts = (const float4*)c->src_raw_pts.p; a.src_nrm = (const float4*)c->src_raw_nrm.p; a.proj_tiled = 1; }
    a.fast_path = getenv("ICP_GPU_NO_FASTPATH") ? 0 : 1;   // tuning knob (A/B measurement)
    a.collect_stats = c->cfg.collect_stats;
}

void fill_reduce_args(icp_gpu_ctx* c, ReduceArgs& r, int algo, int solve) {
    memset(&r, 0, sizeof(r));
    const bool grid_order = (algo == 0);
    r.src_pts = (const float4*)c->src_pts.p; r.src_nrm = (const float4*)c->src_nrm.p; r.n_src = c->n_src;
    r.state = (DevState*)c->state.p;
    r.tgt_pts = (const float4*)(grid_order ? c->tgt_pts_sorted.p : c->tgt_pts.p);
    r.tgt_nrm = (const float4*)(grid_order ? c->tgt_nrm_sorted.p : c->tgt_nrm.p);
    r.match_pos = (const int*)c->match_pos.p; r.match_w = (const float*)c->match_w.p;
    r.partials = (double*)c->partials.p; r.pose_history = (float*)c->history.p;
    r.metric = c->cfg.metric; r.solve = solve;
    r.fused = 0; r.nn_pos = (const int*)c->nn_pos.p; r.n_tgt = c->n_tgt; r.mask = (const unsigned int*)c->mask.p;
    r.desc = (const IterDesc*)c->desc.p; r.desc_index = -1;
    r.weighting = c->cfg.weighting; r.rejection = c->cfg.rejection; r.max_d2 = c->cfg.max_distance_sq;
    r.weight_max_d2 = c->cfg.weight_max_distance_sq > 0.f ? c->cfg.weight_max_distance_sq : c->cfg.max_distance_sq;
    if (proj_tiled(c, algo)) { r.src_pts = (const float4*)c->src_raw_pts.p; r.src_nrm = (const float4*)c->src_raw_nrm.p; }
    r.profile = getenv("ICP_GPU_REDUCE_PROFILE") ? 1 : 0;   // diagnostic
    if (solve && c->peer_world > 1) {
        r.peer.world = c->peer_world; r.peer.rank = c->peer_rank;
        unsigned long long ms = 2000;
        if (const char* e = getenv("ICP_GPU_PEER_TIMEOUT_MS")) { const long long v = atoll(e); if (v >= 1 && v <= 600000) ms = (unsigned long long)v; }
        r.peer.timeout_ns = ms * 1000000ull;
        for (int j = 0; j < c->peer_world; ++j) r.peer.box[j] = (PeerBox*)c->peer_ptr[j];
        r.peer.plan_check = c->peer_plan_check;
    }
}

// Every query starts its search from the neighbour it had the last time it was searched (nn_pos / nn_leaf).  After a new
// cloud those are meaningless (nn_stale): they are replaced by seeds read off the target's sorted keys at the current pose
// (grid.cu; queries that still have a neighbour keep it), or reset to "none".
int refresh_seeds(icp_gpu_ctx* ctx, int algo, bool allow_seed) {
    if (algo != 0 || ctx->n_src <= 0 || !ctx->nn_pos.p) return 0;
    const bool seed = allow_seed && ctx->n_tgt > 0 && ctx->grid_built && !getenv("ICP_GPU_NO_GRID_SEED");
    if (seed) {
        CU(icp_launch_seed_from_keys((const float4*)ctx->src_pts.p, ctx->n_src, (const DevState*)ctx->state.p, (const GridParams*)ctx->grid.p,
                                     ctx->tsort.keys_sorted, ctx->n_tgt, (const unsigned int*)ctx->bbox.p + 7, (const unsigned int*)ctx->tsort.msd.p,
                                     ctx->tsort.msd_shift, (const unsigned int*)ctx->leaf_rank.p, (int*)ctx->nn_pos.p, (int*)ctx->nn_leaf.p,
                                     ctx->nn_stale ? 1 : 0, ctx->stream));
        ctx->stats.n_kernel_launches += 1;
    } else if (ctx->nn_stale) {
        CU(icp_launch_fill_int((int*)ctx->nn_pos.p, ctx->n_src, -1, ctx->stream));
        ctx->stats.n_kernel_launches += 1;
    }
    ctx->nn_stale = false;
    return 0;
}

// Enqueue the whole loop.  ev_marks (nullable): events recorded around each stage for the timings report.
int enqueue_iterations(icp_gpu_ctx* ctx, const Plan& plan, int algo, std::vector<cudaEvent_t>* ev_marks) {
    MatchArgs ma; ReduceArgs ra;
    fill_match_args(ctx, ma, algo, -1, false);
    fill_reduce_args(ctx, ra, algo, 1);
    // Without work counters the linear minimiser reads the search result directly: weighting and rejection are
    // evaluated inside the reduction and the match records (and their launch) are skipped.
    if (algo == 0 && ctx->cfg.minimizer == ICP_GPU_MIN_LINEAR && !ctx->cfg.collect_stats) { ma.skip_finish = 1; ra.fused = 1; }
    int launches = 0;
    const int nb = ctx->n_reduce_blocks;
    // Two chunks of >= 64k queries (tuning knob: ICP_GPU_MATCH_CHUNKS).  Measured at 370k queries: 1 / 2 / 3 / 4 chunks
    // 4.78 / 4.54 / 4.58 / 4.69 ms per 30-iteration registration.
    MatchChunks mc = ctx->chunks;
    mc.n = ctx->n_src >= 131072 ? 2 : 1;
    if (const char* e = getenv("ICP_GPU_MATCH_CHUNKS")) { const int v = atoi(e); if (v >= 1 && v <= ICP_MAX_MATCH_CHUNKS) mc.n = v; }
    for (int i = 0; i < plan.n_iters; ++i) {
        if (ev_marks) CU(cudaEventRecord((*ev_marks)[2 * i], ctx->stream));
        CU(icp_launch_match(ma, algo, ctx->n_sms, ctx->stream, &launches, (ev_marks && algo == 0) ? (*ev_marks)[2 * plan.n_iters + 1 + i] : nullptr, &mc));
        if (ev_marks) CU(cudaEventRecord((*ev_marks)[2 * i + 1], ctx->stream));
        if (ctx->cfg.minimizer == ICP_GPU_MIN_LM) CU(icp_launch_lm(ra, nb, ctx->cfg.lm_max_iterations, ctx->stream, &launches));
        else CU(icp_launch_reduce(ra, nb, ctx->stream, &launches));
    }
    if (ev_marks) CU(cudaEventRecord((*ev_marks)[2 * plan.n_iters], ctx->stream));
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    return 0;
}

int start_registration(icp_gpu_ctx* ctx, const float pose_in[16], icp_gpu_timings* timings) {
    if (!ctx || !pose_in) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is already pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    int rc = check_ready(ctx); if (rc) return rc;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    if (ctx->peer_world > 1 && ctx->cfg.multires)
        return fail(ctx, ICP_GPU_E_ARG, "point-sharded registration: the multi-resolution schedule is derived from the local shard (level strides and count "
                                        "differ between ranks and from the unsharded cloud); run it with multires off");
    Plan plan;
    rc = make_plan(ctx, plan); if (rc) return rc;
    // what every rank must agree on for the exchanges to pair up; checked inside the first exchange (icp_internal.cuh: peer_exchange_row)
    ctx->peer_plan_check = plan.n_iters * 64 + ctx->cfg.metric * 16 + ctx->cfg.minimizer * 8 + (ctx->cfg.lm_max_iterations & 7);
    const int algo = choose_algorithm(ctx);
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    // descriptors + selection lists + pose up (pinned staging, stream-ordered)
    memcpy(ctx->h_desc, plan.desc.data(), sizeof(IterDesc) * (size_t)plan.n_iters);
    if (plan.n_iters > 0) CU(cudaMemcpyAsync(ctx->desc.p, ctx->h_desc, sizeof(IterDesc) * (size_t)plan.n_iters, cudaMemcpyHostToDevice, ctx->stream));
    if (!plan.voxel_depth.empty()) {
        const size_t mask_words = ((size_t)(ctx->n_src > 0 ? ctx->n_src : 1) + 31) / 32;
        int dmax = 0; for (int D : plan.voxel_depth) dmax = D > dmax ? D : dmax;
        if (ensure(ctx, ctx->mask, plan.voxel_depth.size() * mask_words * sizeof(uint32_t)) ||
            ensure(ctx, ctx->voxel_table, sizeof(unsigned int) * ((size_t)1 << dmax))) return ICP_GPU_E_CUDA;
        int launches = 0;
        for (size_t j = 0; j < plan.voxel_depth.size(); ++j)
            CU(icp_launch_voxel_level((const float4*)ctx->src_pts.p, (const float4*)ctx->src_nrm.p, ctx->n_src, (const GridParams*)ctx->sgrid.p,
                                      ctx->Ts, plan.voxel_depth[j], (unsigned int*)ctx->voxel_table.p, (unsigned int*)ctx->mask.p + j * mask_words,
                                      mask_words, ctx->stream, &launches));
        ctx->stats.n_kernel_launches += (uint64_t)launches;
    }
    if (!plan.mask.empty()) {
        if (ensure(ctx, ctx->mask, plan.mask.size() * sizeof(uint32_t))) return ICP_GPU_E_CUDA;
        CU(cudaMemcpyAsync(ctx->mask.p, plan.mask.data(), plan.mask.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));   // plan.mask is pageable and dies with this frame
    }
    memcpy(ctx->h_pose, pose_in, 16 * sizeof(float));
    CU(cudaMemcpyAsync(ctx->pose_dev.p, ctx->h_pose, 16 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CU(icp_launch_pose_init((DevState*)ctx->state.p, (const float*)ctx->pose_dev.p, ctx->stream, ctx->cfg.early_stop_rotation, ctx->cfg.early_stop_translation));
    ctx->stats.n_kernel_launches += 1;
    rc = refresh_seeds(ctx, algo, true); if (rc) return rc;

    std::vector<cudaEvent_t> marks;
    if (timings) {
        memset(timings, 0, sizeof(*timings));
        marks.resize((size_t)3 * plan.n_iters + 1);   // 2 per iteration + end, then one per iteration between the two search kernels
        for (auto& e : marks) CU(cudaEventCreate(&e));
        rc = enqueue_iterations(ctx, plan, algo, &marks);
    } else if (ctx->cfg.use_graph && plan.n_iters > 0) {
        // The graph depends only on launch shapes and pointers, not on descriptor contents.
        std::vector<long long> key;
        key.push_back(algo); key.push_back(ctx->cfg.metric); key.push_back(ctx->cfg.minimizer); key.push_back(ctx->cfg.lm_max_iterations);
        key.push_back(ctx->cfg.weighting); key.push_back(ctx->cfg.rejection); key.push_back(ctx->cfg.color_icp); key.push_back(ctx->cfg.collect_stats);
        key.push_back((long long)__float_as_int_host(ctx->cfg.max_distance_sq)); key.push_back((long long)__float_as_int_host(ctx->cfg.weight_max_distance_sq));
        key.push_back(ctx->n_src); key.push_back(ctx->n_tgt); key.push_back(ctx->T); key.push_back(ctx->width); key.push_back(ctx->height);
        for (int k = 0; k < 9; ++k) key.push_back((long long)__float_as_int_host(ctx->have_camera ? ctx->K[k] : 0.f));
        key.push_back((long long)(uintptr_t)ctx->mask.p); key.push_back((long long)(uintptr_t)ctx->stream);
        key.push_back(plan.n_iters);
        key.push_back(ctx->peer_world); key.push_back(ctx->peer_rank); key.push_back((long long)ctx->peer_epoch);
        if (!ctx->graph_exec || key != ctx->graph_key) {
            cudaGraph_t g = nullptr;
            CU(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
            const uint64_t before = ctx->stats.n_kernel_launches;
            rc = enqueue_iterations(ctx, plan, algo, nullptr);
            cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
            if (rc) { if (g) cudaGraphDestroy(g); return rc; }
            if (ce != cudaSuccess) return fail(ctx, ICP_GPU_E_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(ce));
            // A new cloud size (every frame of a sequence) changes launch shapes and arguments, not the graph's topology: the
            // instantiated graph is updated in place, which is several times cheaper than instantiating a new one.
            bool updated = false;
            if (ctx->graph_exec) {
                cudaGraphExecUpdateResultInfo info;
                updated = cudaGraphExecUpdate(ctx->graph_exec, g, &info) == cudaSuccess;
                if (!updated) { cudaGetLastError(); cudaGraphExecDestroy(ctx->graph_exec); ctx->graph_exec = nullptr; }
            }
            ce = updated ? cudaSuccess : cudaGraphInstantiate(&ctx->graph_exec, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) { ctx->graph_exec = nullptr; return fail(ctx, ICP_GPU_E_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ce)); }
            ctx->graph_key = key;
            ctx->graph_launches = ctx->stats.n_kernel_launches - before;
        } else {
            ctx->stats.n_kernel_launches += ctx->graph_launches;
        }
        CU(cudaGraphLaunch(ctx->graph_exec, ctx->stream));
    } else {
        rc = enqueue_iterations(ctx, plan, algo, nullptr);
    }
    if (rc) return rc;
    // results down
    CU(cudaMemcpyAsync(ctx->h_state, ctx->state.p, sizeof(DevState), cudaMemcpyDeviceToHost, ctx->stream));
    if (plan.n_iters > 0) CU(cudaMemcpyAsync(ctx->h_history, ctx->history.p, sizeof(float) * 16 * (size_t)plan.n_iters, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->pending = true; ctx->pending_iters = plan.n_iters;
    if (timings) {
        CU(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < plan.n_iters; ++i) {
            float a = 0.f, b = 0.f;
            cudaEventElapsedTime(&a, marks[2 * i], marks[2 * i + 1]);
            cudaEventElapsedTime(&b, marks[2 * i + 1], marks[2 * i + 2]);
            timings->matching_ms += a; timings->solver_ms += b;
            float c = 0.f;
            if (algo == 0 && cudaEventElapsedTime(&c, marks[2 * i], marks[2 * plan.n_iters + 1 + i]) == cudaSuccess) timings->search_prep_ms += c; else cudaGetLastError();
        }
        float tot = 0.f;
        if (plan.n_iters > 0) cudaEventElapsedTime(&tot, marks[0], marks[2 * plan.n_iters]);
        float idx_ms = 0.f;
        if (ctx->grid_built && cudaEventElapsedTime(&idx_ms, ctx->ev[0], ctx->ev[1]) == cudaSuccess) ctx->index_ms = idx_ms; else cudaGetLastError();
        timings->total_ms = tot; timings->index_ms = ctx->index_ms; timings->n_iterations = plan.n_iters;
        const int per_match = algo == 0 ? ((ctx->cfg.minimizer == ICP_GPU_MIN_LINEAR && !ctx->cfg.collect_stats) ? 2 : 3) : 1;
        timings->n_match_launches = plan.n_iters * per_match;
        timings->n_solver_launches = (int)ctx->stats.n_kernel_launches - 1 - plan.n_iters * per_match;
        for (auto& e : marks) cudaEventDestroy(e);
    }
    return ICP_GPU_OK;
}

void copy_counters(icp_gpu_ctx* ctx) {
    const DevState& st = *ctx->h_state;
    ctx->stats.n_queries = st.n_queries; ctx->stats.n_matched = st.n_matched;
    ctx->stats.n_distance_evals = st.n_evals; ctx->stats.n_nodes_visited = st.n_nodes;
    for (int k = 0; k < 6; ++k) ctx->stats.reduce_profile_ns[k] = st.prof[k];
}

int finish_registration(icp_gpu_ctx* ctx, float pose_out[16], float* pose_history, int32_t* n_iterations_out) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (!ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "no registration pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    ctx->pending = false;
    CU(cudaStreamSynchronize(ctx->stream));
    const DevState& st = *ctx->h_state;
    if (pose_out) memcpy(pose_out, st.pose, 16 * sizeof(float));
    if (pose_history && st.iters_done > 0) memcpy(pose_history, ctx->h_history, sizeof(float) * 16 * (size_t)st.iters_done);
    if (n_iterations_out) *n_iterations_out = st.iters_done;
    ctx->last_iters = st.iters_done;
    copy_counters(ctx);
    if (st.status == ICP_GPU_E_NO_MATCHES)
        return fail(ctx, ICP_GPU_E_NO_MATCHES, "iteration %d had no surviving correspondence (the reference hangs in ASSERT here)", st.iters_done);
    if (st.status == ICP_GPU_E_PEER)
        return fail(ctx, ICP_GPU_E_PEER, "point-sharded registration: a peer's row did not arrive in time (iteration %d; rank %d of %d)", st.iters_done, ctx->peer_rank, ctx->peer_world);
    if (st.status != 0) return fail(ctx, st.status, "iteration %d: singular / non-finite normal equations", st.iters_done);
    return ICP_GPU_OK;
}

void peer_close(icp_gpu_ctx* ctx) {
    for (int j = 0; j < ICP_MAX_PEERS; ++j) {
        if (ctx->peer_ipc[j] && ctx->peer_ptr[j]) { if (cudaIpcCloseMemHandle(ctx->peer_ptr[j]) != cudaSuccess) cudaGetLastError(); }
        ctx->peer_ptr[j] = nullptr; ctx->peer_ipc[j] = false;
    }
    ctx->peer_world = 0; ctx->peer_rank = 0; ctx->peer_epoch += 1;
}

// (Re)creates the mailbox in its initial state: no row received, exchange counter 0.
int peer_reset_box(icp_gpu_ctx* ctx) {
    CU(cudaStreamSynchronize(ctx->stream));
    peer_close(ctx);
    if (!ctx->peer_box) CU(cudaMalloc(&ctx->peer_box, sizeof(PeerBox)));
    CU(cudaMemsetAsync(ctx->peer_box, 0, sizeof(PeerBox), ctx->stream));
    CU(cudaMemsetAsync(&((DevState*)ctx->state.p)->xchg_seq, 0, sizeof(unsigned int), ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

}  // namespace

// ============================================================================ C ABI
extern "C" {

int icp_gpu_abi_version(void) { return ICP_GPU_ABI_VERSION; }

int icp_gpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void icp_gpu_default_config(icp_gpu_config* cfg) {
    if (!cfg) return;
    memset(cfg, 0, sizeof(*cfg));
    cfg->metric = ICP_GPU_METRIC_P2P; cfg->minimizer = ICP_GPU_MIN_LINEAR; cfg->matching = ICP_GPU_MATCH_KNN;
    cfg->selection = ICP_GPU_SELECT_ALL; cfg->proba = 1.0; cfg->seed = 0; cfg->selection_rng = ICP_GPU_RNG_MT19937;
    cfg->weighting = ICP_GPU_WEIGHT_CONSTANT; cfg->rejection = 1; cfg->max_distance_sq = 0.0003f;
    cfg->color_icp = 0; cfg->multires = 0; cfg->pyramid_mode = ICP_GPU_PYRAMID_STRIDE; cfg->n_iterations = 20;
    cfg->lm_max_iterations = 10; cfg->nn_algorithm = ICP_GPU_NN_AUTO; cfg->use_graph = 1; cfg->collect_stats = 1;
    cfg->weight_max_distance_sq = 0.0f; cfg->early_stop_rotation = 0.0f; cfg->early_stop_translation = 0.0f;
}

int icp_gpu_create(icp_gpu_ctx** out, int device) {
    if (!out) return ICP_GPU_E_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { cudaGetLastError(); return ICP_GPU_E_CUDA; }   // no CPU fallback
    if (device < 0 || device >= n) return ICP_GPU_E_ARG;
    icp_gpu_ctx* ctx = new (std::nothrow) icp_gpu_ctx();
    if (!ctx) return ICP_GPU_E_CUDA;
    ctx->err[0] = 0; ctx->device = device;
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    icp_gpu_default_config(&ctx->cfg);
    cudaDeviceProp prop;
    bool ok = cudaSetDevice(device) == cudaSuccess && cudaGetDeviceProperties(&prop, device) == cudaSuccess;
    if (ok && prop.major < 10) ok = false;   // the kernels are built for sm_100a only
    if (ok) ctx->n_sms = prop.multiProcessorCount;
    ok = ok && cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) == cudaSuccess;
    ctx->stream = ctx->own_stream;
    ok = ok && cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&ctx->ev_index_ready, cudaEventDisableTiming) == cudaSuccess;
    for (int c = 0; c < ICP_MAX_MATCH_CHUNKS - 1; ++c)
        ok = ok && cudaStreamCreateWithFlags(&ctx->chunks.stream[c], cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&ctx->chunks.done[c], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->chunks.fork, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok && i < 4; ++i) ok = cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
    for (int i = 0; ok && i < 2; ++i) ok = cudaEventCreateWithFlags(&ctx->ev_xyz[i], cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming) == cudaSuccess &&
                                           cudaEventCreateWithFlags(&ctx->ev_packed[i], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaMallocHost((void**)&ctx->h_pose, 16 * sizeof(float)) == cudaSuccess;
    ok = ok && cudaMallocHost((void**)&ctx->h_history, 16 * sizeof(float) * ICP_MAX_ITERS) == cudaSuccess;
    ok = ok && cudaMallocHost((void**)&ctx->h_state, sizeof(DevState)) == cudaSuccess;
    ok = ok && cudaMallocHost((void**)&ctx->h_desc, sizeof(IterDesc) * DESC_TOTAL) == cudaSuccess;
    ok = ok && ensure(ctx, ctx->state, sizeof(DevState)) == 0 && ensure(ctx, ctx->desc, sizeof(IterDesc) * DESC_TOTAL) == 0 &&
         ensure(ctx, ctx->pose_dev, 64) == 0 && ensure(ctx, ctx->history, 16 * sizeof(float) * ICP_MAX_ITERS) == 0 &&
         ensure(ctx, ctx->mask, 256) == 0;
    if (ok) ok = cudaMemsetAsync(ctx->state.p, 0, sizeof(DevState), ctx->stream) == cudaSuccess && cudaStreamSynchronize(ctx->stream) == cudaSuccess;
    if (!ok) { cudaGetLastError(); icp_gpu_destroy(ctx); return ICP_GPU_E_CUDA; }
    *out = ctx;
    return ICP_GPU_OK;
}

int icp_gpu_destroy(icp_gpu_ctx* ctx) {
    if (!ctx) return ICP_GPU_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
    if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
    peer_close(ctx);
    if (ctx->peer_box) cudaFree(ctx->peer_box);
    DeviceBuf* bufs[] = {&ctx->stage, &ctx->stage2, &ctx->src_pts, &ctx->src_nrm, &ctx->tgt_pts, &ctx->tgt_nrm, &ctx->tgt_pts_sorted, &ctx->tgt_nrm_sorted,
                         &ctx->grid, &ctx->bbox, &ctx->sbbox, &ctx->lv_flags, &ctx->lv_tiles, &ctx->delta_a, &ctx->delta_b, &ctx->tsort.keys_a, &ctx->tsort.keys_b, &ctx->tsort.idx_a, &ctx->tsort.idx_b, &ctx->tsort.hist, &ctx->tsort.msd, &ctx->ssort.keys_a, &ctx->ssort.keys_b, &ctx->ssort.idx_a, &ctx->ssort.idx_b, &ctx->ssort.hist, &ctx->ssort.msd, &ctx->state, &ctx->desc, &ctx->mask,
                         &ctx->match_pos, &ctx->match_w, &ctx->match_idx, &ctx->partials, &ctx->pose_dev, &ctx->history,
                         &ctx->src_raw_pts, &ctx->src_raw_nrm, &ctx->sgrid, &ctx->order_dev,
                         &ctx->nn_pos, &ctx->bvh_box, &ctx->bvh_desc, &ctx->leaf_start, &ctx->leaf_rank, &ctx->node_rank, &ctx->child_start, &ctx->qbuf, &ctx->adj, &ctx->adj_box, &ctx->adj_gap, &ctx->adj1, &ctx->adj1_box, &ctx->voxel_table, &ctx->nn_leaf, &ctx->seedbuf,
                         &ctx->nrm_out_dev, &ctx->batch_io, &ctx->batch_scratch, &ctx->batch_plan, &ctx->prep_in, &ctx->prep_tmp, &ctx->prep_out, &ctx->gt_src, &ctx->gt_ref, &ctx->met_partial, &ctx->met_out};
    for (DeviceBuf* b : bufs) if (b->p) cudaFree(b->p);
    for (DeviceBuf& b : ctx->scratch) if (b.p) cudaFree(b.p);
    if (ctx->h_pose) cudaFreeHost(ctx->h_pose);
    if (ctx->h_history) cudaFreeHost(ctx->h_history);
    if (ctx->h_state) cudaFreeHost(ctx->h_state);
    if (ctx->h_desc) cudaFreeHost(ctx->h_desc);
    for (int i = 0; i < 4; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < 2; ++i) { if (ctx->ev_xyz[i]) cudaEventDestroy(ctx->ev_xyz[i]); if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]); if (ctx->ev_packed[i]) cudaEventDestroy(ctx->ev_packed[i]); }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    for (int c = 0; c < ICP_MAX_MATCH_CHUNKS - 1; ++c)
        if (ctx->chunks.stream[c]) { cudaStreamSynchronize(ctx->chunks.stream[c]); cudaStreamDestroy(ctx->chunks.stream[c]); }
    for (int c = 0; c < ICP_MAX_MATCH_CHUNKS - 1; ++c) if (ctx->chunks.done[c]) cudaEventDestroy(ctx->chunks.done[c]);
    if (ctx->chunks.fork) cudaEventDestroy(ctx->chunks.fork);
    if (ctx->ev_index_ready) cudaEventDestroy(ctx->ev_index_ready);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return ICP_GPU_OK;
}

const char* icp_gpu_last_error(const icp_gpu_ctx* ctx) { return ctx ? ctx->err : "null context"; }

int icp_gpu_set_stream(icp_gpu_ctx* ctx, void* cuda_stream) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaStreamSynchronize(ctx->aux_stream));
    ctx->index_pending = false;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return ICP_GPU_OK;
}

int icp_gpu_synchronize(icp_gpu_ctx* ctx) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_set_config(icp_gpu_ctx* ctx, const icp_gpu_config* c) {
    if (!ctx || !c) return ICP_GPU_E_ARG;
    const int rc = check_config(ctx, c, "");
    if (rc) return rc;
    ctx->cfg = *c;
    return ICP_GPU_OK;
}

// PointCloud(depthMap, colorFrame, depthIntrinsics, depthExtrinsics, width, height, keepOriginalSize, downsampleFactor,
// maxDistance) -- PointCloud.h:78-165 -- on the device; the result can become the context's target or source directly.
int icp_gpu_cloud_from_depth(icp_gpu_ctx* ctx, const float* depth, const uint8_t* rgbx, const float K[9], const float E[16],
                             uint32_t width, uint32_t height, int keep_original_size, uint32_t downsample, float max_distance, int role,
                             float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* n_out) {
    if (!ctx || !K) return ICP_GPU_E_ARG;
    if (!depth || width == 0 || height == 0 || downsample == 0 || (long long)width * height > 0x7fffffff / 4)
        return fail(ctx, ICP_GPU_E_ARG, "bad depth map (%p, %ux%u, downsample %u)", (const void*)depth, width, height, downsample);
    if (role < ICP_GPU_CLOUD_TARGET || role > ICP_GPU_CLOUD_ONLY) return fail(ctx, ICP_GPU_E_ARG, "role %d", role);
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending; call icp_gpu_estimate_pose_finish first");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    const long long npx = (long long)width * height;
    DepthArgs a; memset(&a, 0, sizeof(a));
    a.width = width; a.height = height; a.downsample = downsample; a.keep_original_size = keep_original_size ? 1 : 0;
    a.n_candidates = (npx + downsample - 1) / downsample;
    a.fovX = K[0]; a.fovY = K[4]; a.cX = K[6]; a.cY = K[7];          // column-major Matrix3f: (0,0), (1,1), (0,2), (1,2)
    a.half_max_distance = max_distance / 2.f;
    for (int i = 0; i < 16; ++i) a.Einv[i] = (i % 5 == 0) ? 1.f : 0.f;
    if (E) {   // inverse in fp64, rounded to fp32 (the reference's drivers only pass the identity, VirtualSensor.h:52)
        double m[4][8];
        for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) { m[r][c] = E[r + 4 * c]; m[r][4 + c] = (r == c) ? 1.0 : 0.0; }
        for (int k = 0; k < 4; ++k) {
            int p = k; for (int i = k + 1; i < 4; ++i) if (fabs(m[i][k]) > fabs(m[p][k])) p = i;
            if (m[p][k] == 0.0) return fail(ctx, ICP_GPU_E_ARG, "singular depth extrinsics");
            if (p != k) for (int j = 0; j < 8; ++j) { const double t = m[k][j]; m[k][j] = m[p][j]; m[p][j] = t; }
            const double d = m[k][k];
            for (int j = 0; j < 8; ++j) m[k][j] /= d;
            for (int i = 0; i < 4; ++i) if (i != k) { const double f = m[i][k]; if (f != 0.0) for (int j = 0; j < 8; ++j) m[i][j] -= f * m[k][j]; }
        }
        for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) a.Einv[r + 4 * c] = (float)m[r][4 + c];
    }
    const size_t nc = (size_t)a.n_candidates, nb = (nc + 255) / 256;
    const size_t depth_bytes = (size_t)npx * 4, color_bytes = rgbx ? (size_t)npx + 3 : 0;
    const size_t o_color = (depth_bytes + 255) / 256 * 256;
    // staging: points, normals, colours, flags, block counts (+ total) ; outputs: points, normals, colours
    const size_t t_nrm = (nc * 12 + 255) / 256 * 256, t_rgba = 2 * t_nrm, t_flag = t_rgba + (nc * 4 + 255) / 256 * 256,
                 t_cnt = t_flag + (nc * 4 + 255) / 256 * 256, t_end = t_cnt + (nb + 2) * 4;
    if (ensure(ctx, ctx->prep_in, o_color + color_bytes + 256) || ensure(ctx, ctx->prep_tmp, t_end + 256) || ensure(ctx, ctx->prep_out, 2 * t_nrm + nc * 4 + 256))
        return ICP_GPU_E_CUDA;
    char* in = (char*)ctx->prep_in.p; char* tmp = (char*)ctx->prep_tmp.p; char* out = (char*)ctx->prep_out.p;
    CU(cudaMemcpyAsync(in, depth, depth_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (rgbx) CU(cudaMemcpyAsync(in + o_color, rgbx, color_bytes, cudaMemcpyHostToDevice, ctx->stream));
    int launches = 0;
    unsigned int* total = (unsigned int*)(tmp + t_cnt) + nb;
    CU(icp_launch_depth_cloud((const float*)in, rgbx ? (const unsigned char*)(in + o_color) : nullptr, a, (float*)tmp, (float*)(tmp + t_nrm),
                              (unsigned char*)(tmp + t_rgba), (unsigned int*)(tmp + t_flag), (unsigned int*)(tmp + t_cnt), total,
                              (float*)out, (float*)(out + t_nrm), (unsigned char*)(out + 2 * t_nrm), ctx->stream, &launches));
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    unsigned int n = 0;
    CU(cudaMemcpyAsync(&n, total, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));    // the host arrays were pageable: all copies are done; n is known
    if (n_out) *n_out = (int64_t)n;
    if (n > 0) {
        if (xyz_out) CU(cudaMemcpyAsync(xyz_out, out, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
        if (nrm_out) CU(cudaMemcpyAsync(nrm_out, out + t_nrm, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
        if (rgba_out) CU(cudaMemcpyAsync(rgba_out, out + 2 * t_nrm, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    int rc = ICP_GPU_OK;
    if (role != ICP_GPU_CLOUD_ONLY)
        rc = set_cloud(ctx, role == ICP_GPU_CLOUD_TARGET, (const float*)out, (const float*)(out + t_nrm), (const uint8_t*)(out + 2 * t_nrm), (int64_t)n, true);
    if (xyz_out || nrm_out || rgba_out) CU(cudaStreamSynchronize(ctx->stream));
    return rc;
}

// PointCloud(pcl::PointCloud<pcl::PointXYZ>::Ptr) (PointCloud.h:41-76): k-NN PCA normals (pcl::NormalEstimation, setKSearch(k)) of the
// context's TARGET cloud, computed with the index set_target built.  The normals replace the target's own (used by the next
// registrations) and are returned in the caller's point order.
int icp_gpu_target_normals(icp_gpu_ctx* ctx, int32_t k, const float viewpoint[3], float* nrm_out, float* curvature_out) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (k < 3 || k > 8) return fail(ctx, ICP_GPU_E_ARG, "k %d (3..8)", k);
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending; call icp_gpu_estimate_pose_finish first");
    if (!ctx->grid_built) return fail(ctx, ICP_GPU_E_STATE, "no target cloud set");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    const int n = ctx->n_tgt;
    if (n <= 0) return ICP_GPU_OK;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    if (ensure(ctx, ctx->nrm_out_dev, (size_t)n * 16 + 256)) return ICP_GPU_E_CUDA;
    NormalArgs a; memset(&a, 0, sizeof(a));
    a.pts = (const float4*)ctx->tgt_pts_sorted.p; a.n = n;
    a.bvh_box = (const float4*)ctx->bvh_box.p; a.bvh = (const BvhDesc*)ctx->bvh_desc.p; a.leaf_start = (const unsigned int*)ctx->leaf_start.p;
    a.leaf_rank = (const unsigned int*)ctx->leaf_rank.p; a.child_start = (const unsigned int*)ctx->child_start.p;
    a.adj = (const unsigned int*)ctx->adj.p; a.adj_box = (const float4*)ctx->adj_box.p; a.adj_capacity = ctx->adj_capacity;
    a.k = k;
    for (int i = 0; i < 3; ++i) a.vp[i] = viewpoint ? viewpoint[i] : 0.f;
    a.out_nrm = (float*)ctx->nrm_out_dev.p; a.out_curv = (float*)ctx->nrm_out_dev.p + 3 * (size_t)n;
    a.nrm_sorted = (float4*)ctx->tgt_nrm_sorted.p; a.nrm_orig = (float4*)ctx->tgt_nrm.p;
    CU(cudaMemsetAsync(ctx->nrm_out_dev.p, 0xFF, (size_t)n * 16, ctx->stream));     // NaN: points the index does not hold (non-finite ones)
    CU(icp_launch_pca_normals(a, ctx->stream));
    ctx->stats.n_kernel_launches += 1;
    if (nrm_out) CU(cudaMemcpyAsync(nrm_out, a.out_nrm, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    if (curvature_out) CU(cudaMemcpyAsync(curvature_out, a.out_curv, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (nrm_out || curvature_out) CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

// ConvergenceMeasure(sourcePoints, unchangedPoints) (ConvergenceMeasure.h:32-41): the known correspondences.
int icp_gpu_set_correspondences(icp_gpu_ctx* ctx, const float* src_xyz, const float* ref_xyz, int64_t m) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (m < 0 || (m > 0 && (!src_xyz || !ref_xyz))) return fail(ctx, ICP_GPU_E_ARG, "bad correspondences (m=%lld)", (long long)m);
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    ctx->n_gt = 0;
    if (m == 0) return ICP_GPU_OK;
    if (ensure(ctx, ctx->gt_src, (size_t)m * 12) || ensure(ctx, ctx->gt_ref, (size_t)m * 12)) return ICP_GPU_E_CUDA;
    CU(cudaMemcpyAsync(ctx->gt_src.p, src_xyz, (size_t)m * 12, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->gt_ref.p, ref_xyz, (size_t)m * 12, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->n_gt = m;
    return ICP_GPU_OK;
}

// The same with the correspondences reconstructRoom builds (main.cpp:300-307): every point of the resident source
// against itself under a ground-truth pose, gtTargetPoints = transformPoints(source.getPoints(), gt_pose).
int icp_gpu_set_correspondences_pose(icp_gpu_ctx* ctx, const float gt_pose[16]) {
    if (!ctx || !gt_pose) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending; call icp_gpu_estimate_pose_finish first");
    if (ctx->n_src <= 0 || !ctx->src_raw_pts.p) return fail(ctx, ICP_GPU_E_STATE, "no source cloud set");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    ctx->n_gt = 0;
    const size_t m = (size_t)ctx->n_src;
    if (ensure(ctx, ctx->gt_src, m * 12) || ensure(ctx, ctx->gt_ref, m * 12) || ensure(ctx, ctx->met_out, 256)) return ICP_GPU_E_CUDA;
    CU(cudaMemcpyAsync(ctx->met_out.p, gt_pose, 64, cudaMemcpyHostToDevice, ctx->stream));
    CU(icp_launch_gt_from_source((const float4*)ctx->src_raw_pts.p, (long long)m, (const float*)ctx->met_out.p, (float*)ctx->gt_src.p, (float*)ctx->gt_ref.p, ctx->stream));
    ctx->stats.n_kernel_launches += 1;
    CU(cudaStreamSynchronize(ctx->stream));     // gt_pose is the caller's (pageable) memory; met_out is reused by icp_gpu_convergence_errors
    ctx->n_gt = (long long)m;
    return ICP_GPU_OK;
}

// recordAlignmentError after every iteration of the last registration (ICPOptimizer.h:629-631), evaluated on the device
// from the per-iteration poses the loop left there.
int icp_gpu_convergence_errors(icp_gpu_ctx* ctx, float* rmse_out, double* benchmark_out, int32_t capacity, int32_t* n_out) {
    if (!ctx || !rmse_out) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending; call icp_gpu_estimate_pose_finish first");
    if (ctx->n_gt <= 0) return fail(ctx, ICP_GPU_E_STATE, "no correspondences set (icp_gpu_set_correspondences)");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    const int n = ctx->last_iters < capacity ? ctx->last_iters : capacity;
    if (n_out) *n_out = n;
    if (n <= 0) return ICP_GPU_OK;
    const int nb = icp_metrics_blocks(ctx->n_gt, ctx->n_sms);
    if (ensure(ctx, ctx->met_partial, (size_t)n * nb * 6 * sizeof(double)) || ensure(ctx, ctx->met_out, (size_t)n * (4 + 12 + 8) + 64)) return ICP_GPU_E_CUDA;
    double* bench = (double*)ctx->met_out.p;                       // n doubles, then n rmse floats, then 3n centroid floats
    float* rmse = (float*)(bench + n); float* centroid = rmse + n;
    int launches = 0;
    CU(icp_launch_metrics((const float*)ctx->gt_src.p, (const float*)ctx->gt_ref.p, ctx->n_gt, (const float*)ctx->history.p, n, nb,
                          (double*)ctx->met_partial.p, rmse, centroid, benchmark_out ? bench : nullptr, ctx->stream, &launches));
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    CU(cudaMemcpyAsync(rmse_out, rmse, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (benchmark_out) CU(cudaMemcpyAsync(benchmark_out, bench, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

// rmseAlignmentError(pose) / benchmarkError(pose) (ConvergenceMeasure.h:50-66, :104-151) of ONE pose the caller supplies, over the
// correspondences set before: the metrics kernels with a one-entry pose history.
int icp_gpu_alignment_error(icp_gpu_ctx* ctx, const float pose[16], float* rmse_out, double* benchmark_out) {
    if (!ctx || !pose || !rmse_out) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending; call icp_gpu_estimate_pose_finish first");
    if (ctx->n_gt <= 0) return fail(ctx, ICP_GPU_E_STATE, "no correspondences set (icp_gpu_set_correspondences)");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    const int nb = icp_metrics_blocks(ctx->n_gt, ctx->n_sms);
    if (ensure(ctx, ctx->met_partial, (size_t)nb * 6 * sizeof(double)) || ensure(ctx, ctx->met_out, (4 + 12 + 8) + 64) || ensure(ctx, ctx->scratch[15], 64)) return ICP_GPU_E_CUDA;
    CU(cudaMemcpyAsync(ctx->scratch[15].p, pose, 64, cudaMemcpyHostToDevice, ctx->stream));
    double* bench = (double*)ctx->met_out.p; float* rmse = (float*)(bench + 1); float* centroid = rmse + 1;
    int launches = 0;
    CU(icp_launch_metrics((const float*)ctx->gt_src.p, (const float*)ctx->gt_ref.p, ctx->n_gt, (const float*)ctx->scratch[15].p, 1, nb,
                          (double*)ctx->met_partial.p, rmse, centroid, benchmark_out ? bench : nullptr, ctx->stream, &launches));
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    CU(cudaMemcpyAsync(rmse_out, rmse, 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (benchmark_out) CU(cudaMemcpyAsync(benchmark_out, bench, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_get_config(const icp_gpu_ctx* ctx, icp_gpu_config* c) {
    if (!ctx || !c) return ICP_GPU_E_ARG;
    *c = ctx->cfg;
    return ICP_GPU_OK;
}

int icp_gpu_set_camera(icp_gpu_ctx* ctx, const float K[9], uint32_t width, uint32_t height) {
    if (!ctx || !K) return ICP_GPU_E_ARG;
    memcpy(ctx->K, K, 9 * sizeof(float));
    ctx->width = width; ctx->height = height; ctx->have_camera = true;
    return ICP_GPU_OK;
}

int icp_gpu_set_target(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n) { return set_cloud(ctx, true, xyz, nrm, rgba, n, false); }
int icp_gpu_set_source(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n) { return set_cloud(ctx, false, xyz, nrm, rgba, n, false); }
int icp_gpu_set_target_dev(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n) { return set_cloud(ctx, true, xyz, nrm, rgba, n, true); }
int icp_gpu_set_source_dev(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n) { return set_cloud(ctx, false, xyz, nrm, rgba, n, true); }

int icp_gpu_query_matches(icp_gpu_ctx* ctx, const float pose[16], const int32_t* sel_idx, int64_t n_sel, int32_t* idx_out, float* weight_out) {
    if (!ctx || !pose || !idx_out || !weight_out) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    int rc = check_ready(ctx); if (rc) return rc;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    const int n = ctx->n_src;
    const int nq = sel_idx ? (int)n_sel : n;
    if (sel_idx && (n_sel < 0 || n_sel > n)) return fail(ctx, ICP_GPU_E_ARG, "n_sel %lld", (long long)n_sel);
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    if (fetch_src_rank(ctx)) return ICP_GPU_E_CUDA;
    IterDesc d; memset(&d, 0, sizeof(d));
    d.stride = 1; d.mask_word_offset = -1; d.filter_finite = 0; d.proba = -1.0f;
    std::vector<uint32_t> mask;
    if (sel_idx) {
        mask.assign(((size_t)(n > 0 ? n : 1) + 31) / 32, 0u);
        for (int64_t k = 0; k < n_sel; ++k) {
            if (sel_idx[k] < 0 || sel_idx[k] >= n) return fail(ctx, ICP_GPU_E_ARG, "sel_idx[%lld] out of range", (long long)k);
            mask[(size_t)sel_idx[k] >> 5] |= 1u << (sel_idx[k] & 31);
        }
        if (ensure(ctx, ctx->mask, mask.size() * 4)) return ICP_GPU_E_CUDA;
        CU(cudaMemcpyAsync(ctx->mask.p, mask.data(), mask.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        d.mask_word_offset = 0;
    }
    ctx->h_desc[DESC_QUERY] = d;
    CU(cudaMemcpyAsync((IterDesc*)ctx->desc.p + DESC_QUERY, &ctx->h_desc[DESC_QUERY], sizeof(IterDesc), cudaMemcpyHostToDevice, ctx->stream));
    memcpy(ctx->h_pose, pose, 16 * sizeof(float));
    CU(cudaMemcpyAsync(ctx->pose_dev.p, ctx->h_pose, 16 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CU(icp_launch_pose_init((DevState*)ctx->state.p, (const float*)ctx->pose_dev.p, ctx->stream));
    const int algo = choose_algorithm(ctx);
    rc = refresh_seeds(ctx, algo, false); if (rc) return rc;       // stages 2-4 at one pose: an unseeded search unless a registration left neighbours
    MatchArgs ma; fill_match_args(ctx, ma, algo, DESC_QUERY, true);
    int launches = 1;
    CU(icp_launch_match(ma, algo, ctx->n_sms, ctx->stream, &launches));
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    std::vector<int> idx_s((size_t)n); std::vector<float> w_s((size_t)n);
    if (n > 0) {
        CU(cudaMemcpyAsync(idx_s.data(), ctx->match_idx.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(w_s.data(), ctx->match_w.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaMemcpyAsync(ctx->h_state, ctx->state.p, sizeof(DevState), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    // device results are in sorted-source order; the caller gets its own order back
    for (int k = 0; k < nq; ++k) {
        const int o = sel_idx ? sel_idx[k] : k;
        const int p = ma.proj_tiled ? o : ctx->src_rank[(size_t)o];
        idx_out[k] = idx_s[(size_t)p]; weight_out[k] = w_s[(size_t)p];
    }
    copy_counters(ctx);
    return ICP_GPU_OK;
}

int icp_gpu_iterations_bound(const icp_gpu_config* cfg, int64_t n_source) {
    if (!cfg || n_source < 0 || n_source > 0x7fffffff) return ICP_GPU_E_ARG;
    return icp_schedule(cfg->n_iterations, cfg->multires, n_source).n_iters;
}

int icp_gpu_max_iterations(const icp_gpu_ctx* ctx) {
    if (!ctx) return ICP_GPU_E_ARG;
    return icp_gpu_iterations_bound(&ctx->cfg, ctx->n_src > 0 ? ctx->n_src : 0);
}

int icp_gpu_estimate_pose_async(icp_gpu_ctx* ctx, const float pose_in[16]) { return start_registration(ctx, pose_in, nullptr); }

int icp_gpu_estimate_pose_finish(icp_gpu_ctx* ctx, float pose_out[16], float* pose_history, int32_t* n_iterations_out) {
    return finish_registration(ctx, pose_out, pose_history, n_iterations_out);
}

int icp_gpu_estimate_pose(icp_gpu_ctx* ctx, float pose_inout[16], float* pose_history, int32_t* n_iterations_out, icp_gpu_timings* timings) {
    int rc = start_registration(ctx, pose_inout, timings);
    if (rc) return rc;
    return finish_registration(ctx, pose_inout, pose_history, n_iterations_out);
}

int icp_gpu_measure_fp32_peak(icp_gpu_ctx* ctx, int32_t mode, double* tflops_out) {
    if (!ctx || !tflops_out || mode < 0 || mode > 1) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    CU(icp_measure_fp32_peak(mode, ctx->n_sms, ctx->stream, tflops_out));
    return ICP_GPU_OK;
}

int icp_gpu_get_stats(icp_gpu_ctx* ctx, icp_gpu_stats* out) {
    if (!ctx || !out) return ICP_GPU_E_ARG;
    *out = ctx->stats;
    return ICP_GPU_OK;
}

// ---------------------------------------------------------------------------- point-sharded iteration
int icp_gpu_iteration_phases(const icp_gpu_ctx* ctx) {
    if (!ctx) return ICP_GPU_E_ARG;
    return ctx->cfg.metric == ICP_GPU_METRIC_SYMMETRIC ? 2 : 1;
}

static int shard_values(int metric, int phase) {
    if (metric == ICP_GPU_METRIC_P2P) return 23;
    if (metric == ICP_GPU_METRIC_SYMMETRIC && phase == 0) return 7;
    return 28;
}

int icp_gpu_iteration_begin(icp_gpu_ctx* ctx, const float pose_in[16]) {
    if (!ctx || !pose_in) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (ctx->cfg.minimizer != ICP_GPU_MIN_LINEAR) return fail(ctx, ICP_GPU_E_ARG, "the point-sharded path supports the linear minimiser only");
    if (ctx->peer_world > 1) return fail(ctx, ICP_GPU_E_STATE, "peers are attached: icp_gpu_estimate_pose is the point-sharded registration (icp_gpu_peer_detach first)");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    int rc = check_ready(ctx); if (rc) return rc;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    IterDesc d; memset(&d, 0, sizeof(d));
    d.stride = 1; d.mask_word_offset = -1; d.filter_finite = 0; d.proba = -1.0f;
    for (int i = 0; i < ICP_MAX_ITERS; ++i) ctx->h_desc[i] = d;      // every iteration of the shard loop: all points
    CU(cudaMemcpyAsync(ctx->desc.p, ctx->h_desc, sizeof(IterDesc) * ICP_MAX_ITERS, cudaMemcpyHostToDevice, ctx->stream));
    memcpy(ctx->h_pose, pose_in, 16 * sizeof(float));
    CU(cudaMemcpyAsync(ctx->pose_dev.p, ctx->h_pose, 16 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CU(icp_launch_pose_init((DevState*)ctx->state.p, (const float*)ctx->pose_dev.p, ctx->stream));
    ctx->shard_open = true; ctx->shard_algo = choose_algorithm(ctx); ctx->shard_iters = 0;
    rc = refresh_seeds(ctx, ctx->shard_algo, true); if (rc) return rc;
    return ICP_GPU_OK;
}

int icp_gpu_iteration_local_dev(icp_gpu_ctx* ctx, int phase, double** partials_dev, int32_t* n_values) {
    if (!ctx || !partials_dev || !n_values) return ICP_GPU_E_ARG;
    if (!ctx->shard_open) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_iteration_begin not called");
    if (phase < 0 || phase >= icp_gpu_iteration_phases(ctx)) return fail(ctx, ICP_GPU_E_ARG, "phase %d", phase);
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    const int algo = ctx->shard_algo;
    int launches = 0;
    if (phase == 0) {
        if (ctx->shard_iters >= ICP_MAX_ITERS) return fail(ctx, ICP_GPU_E_ARG, "more than %d iterations since icp_gpu_iteration_begin", ICP_MAX_ITERS);
        ctx->shard_iters += 1;
        MatchArgs ma; fill_match_args(ctx, ma, algo, -1, false);
        CU(icp_launch_match(ma, algo, ctx->n_sms, ctx->stream, &launches));
    }
    ReduceArgs ra; fill_reduce_args(ctx, ra, algo, 0);
    CU(icp_launch_reduce_phase(ra, ctx->n_reduce_blocks, phase, ctx->stream, &launches));
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    *partials_dev = ((DevState*)ctx->state.p)->shard_partials;
    *n_values = shard_values(ctx->cfg.metric, phase);
    return ICP_GPU_OK;
}

int icp_gpu_iteration_local(icp_gpu_ctx* ctx, int phase, double* partials_out, int32_t* n_values) {
    if (!partials_out) return ICP_GPU_E_ARG;
    double* dev = nullptr;
    int rc = icp_gpu_iteration_local_dev(ctx, phase, &dev, n_values);
    if (rc) return rc;
    CU(cudaMemcpyAsync(partials_out, dev, sizeof(double) * (size_t)*n_values, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_iteration_apply_dev(icp_gpu_ctx* ctx, int phase) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (!ctx->shard_open) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_iteration_begin not called");
    if (phase < 0 || phase >= icp_gpu_iteration_phases(ctx)) return fail(ctx, ICP_GPU_E_ARG, "phase %d", phase);
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    const int mode = ctx->cfg.metric == ICP_GPU_METRIC_SYMMETRIC ? (phase == 0 ? 3 : 2) : ctx->cfg.metric;
    CU(icp_launch_shard_apply((DevState*)ctx->state.p, mode, (float*)ctx->history.p, ctx->stream));
    ctx->stats.n_kernel_launches += 1;
    return ICP_GPU_OK;
}

int icp_gpu_iteration_apply(icp_gpu_ctx* ctx, int phase, const double* reduced_in, int32_t n_values) {
    if (!ctx || !reduced_in) return ICP_GPU_E_ARG;
    if (n_values < 0 || n_values > ICP_GPU_MAX_PARTIALS) return fail(ctx, ICP_GPU_E_ARG, "n_values %d", n_values);
    if (!ctx->shard_open) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_iteration_begin not called");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    CU(cudaMemcpyAsync(((DevState*)ctx->state.p)->shard_partials, reduced_in, sizeof(double) * (size_t)n_values, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));   // reduced_in is pageable caller memory
    return icp_gpu_iteration_apply_dev(ctx, phase);
}

int icp_gpu_iteration_end(icp_gpu_ctx* ctx, float pose_out[16]) {
    if (!ctx || !pose_out) return ICP_GPU_E_ARG;
    if (!ctx->shard_open) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_iteration_begin not called");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    ctx->shard_open = false;
    CU(cudaMemcpyAsync(ctx->h_state, ctx->state.p, sizeof(DevState), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    memcpy(pose_out, ctx->h_state->pose, 16 * sizeof(float));
    if (ctx->h_state->status == ICP_GPU_E_NO_MATCHES) return fail(ctx, ICP_GPU_E_NO_MATCHES, "no surviving correspondence on any rank");
    if (ctx->h_state->status != 0) return fail(ctx, ctx->h_state->status, "singular / non-finite normal equations");
    return ICP_GPU_OK;
}

// ---------------------------------------------------------------------------- point-sharded registration over peer memory
int icp_gpu_peer_export(icp_gpu_ctx* ctx, void* handle_out) {
    if (!ctx || !handle_out) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    static_assert(sizeof(cudaIpcMemHandle_t) == ICP_GPU_PEER_HANDLE_BYTES, "handle size");
    if (peer_reset_box(ctx)) return ICP_GPU_E_CUDA;
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, ctx->peer_box));
    memcpy(handle_out, &h, sizeof(h));
    return ICP_GPU_OK;
}

int icp_gpu_peer_address(icp_gpu_ctx* ctx, void** mailbox_dev) {
    if (!ctx || !mailbox_dev) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    if (peer_reset_box(ctx)) return ICP_GPU_E_CUDA;
    *mailbox_dev = ctx->peer_box;
    return ICP_GPU_OK;
}

static int peer_attach_common(icp_gpu_ctx* ctx, int32_t rank, int32_t world, const void* handles, void* const* ptrs) {
    if (!ctx || (!handles && !ptrs)) return ICP_GPU_E_ARG;
    if (world < 1 || world > ICP_MAX_PEERS || rank < 0 || rank >= world) return fail(ctx, ICP_GPU_E_ARG, "rank %d of world %d (max %d)", rank, world, ICP_MAX_PEERS);
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (!ctx->peer_box) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_peer_export / icp_gpu_peer_address not called");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    CU(cudaStreamSynchronize(ctx->stream));
    peer_close(ctx);
    for (int j = 0; j < world; ++j) {
        if (j == rank) { ctx->peer_ptr[j] = ctx->peer_box; continue; }
        if (ptrs) {
            if (!ptrs[j]) { peer_close(ctx); return fail(ctx, ICP_GPU_E_ARG, "mailbox %d is null", j); }
            ctx->peer_ptr[j] = ptrs[j];
        } else {
            cudaIpcMemHandle_t h;
            memcpy(&h, (const char*)handles + (size_t)j * ICP_GPU_PEER_HANDLE_BYTES, sizeof(h));
            void* p = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) { cudaGetLastError(); peer_close(ctx); return fail(ctx, ICP_GPU_E_CUDA, "cudaIpcOpenMemHandle(rank %d): %s", j, cudaGetErrorString(e)); }
            ctx->peer_ptr[j] = p; ctx->peer_ipc[j] = true;
        }
    }
    ctx->peer_world = world; ctx->peer_rank = rank;
    return ICP_GPU_OK;
}

int icp_gpu_peer_attach(icp_gpu_ctx* ctx, int32_t rank, int32_t world, const void* handles) {
    if (!handles) return ICP_GPU_E_ARG;
    return peer_attach_common(ctx, rank, world, handles, nullptr);
}

int icp_gpu_peer_attach_ptrs(icp_gpu_ctx* ctx, int32_t rank, int32_t world, void* const* mailboxes_dev) {
    if (!mailboxes_dev) return ICP_GPU_E_ARG;
    return peer_attach_common(ctx, rank, world, nullptr, mailboxes_dev);
}

int icp_gpu_peer_detach(icp_gpu_ctx* ctx) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    CU(cudaStreamSynchronize(ctx->stream));
    peer_close(ctx);
    return ICP_GPU_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------- value-level operations outside the loop
namespace {
// host array -> scratch slot k of the context (nullable in, nullptr out)
int up(icp_gpu_ctx* ctx, int k, const void* host, size_t bytes, void** dev) {
    *dev = nullptr;
    if (!host || bytes == 0) return 0;
    if (ensure(ctx, ctx->scratch[k], bytes)) return ICP_GPU_E_CUDA;
    CU(cudaMemcpyAsync(ctx->scratch[k].p, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dev = ctx->scratch[k].p;
    return 0;
}
}  // namespace

static int transform_common(icp_gpu_ctx* ctx, const float pose[16], const float* in, int64_t n, float* out, int normals) {
    if (!ctx || !pose || n < 0 || (n > 0 && (!in || !out))) return ICP_GPU_E_ARG;
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    if (n == 0) return ICP_GPU_OK;
    void* din = nullptr;
    if (up(ctx, 0, in, (size_t)n * 12, &din) || ensure(ctx, ctx->scratch[1], (size_t)n * 12)) return ICP_GPU_E_CUDA;
    CU(icp_launch_transform((const float*)din, (long long)n, pose, normals, (float*)ctx->scratch[1].p, ctx->stream));
    ctx->stats.n_kernel_launches += 1;
    CU(cudaMemcpyAsync(out, ctx->scratch[1].p, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

extern "C" {

int icp_gpu_transform_points(icp_gpu_ctx* ctx, const float pose[16], const float* xyz_in, int64_t n, float* xyz_out) {
    return transform_common(ctx, pose, xyz_in, n, xyz_out, 0);
}
int icp_gpu_transform_normals(icp_gpu_ctx* ctx, const float pose[16], const float* nrm_in, int64_t n, float* nrm_out) {
    return transform_common(ctx, pose, nrm_in, n, nrm_out, 1);
}

int icp_gpu_apply_weights(icp_gpu_ctx* ctx, int32_t weighting, float max_distance_sq, const float* src_xyz, const float* src_nrm, const uint8_t* src_rgba,
                          int64_t n_src, const float* tgt_xyz, const float* tgt_nrm, const uint8_t* tgt_rgba, int64_t n_tgt, const int32_t* idx,
                          float* weight_inout) {
    if (!ctx || n_src < 0 || n_tgt < 0 || (n_src > 0 && (!src_xyz || !idx || !weight_inout)) || (n_tgt > 0 && !tgt_xyz)) return ICP_GPU_E_ARG;
    if (weighting < 0 || weighting > 3) return fail(ctx, ICP_GPU_E_ARG, "weighting %d", weighting);
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    if (n_src == 0 || weighting == ICP_GPU_WEIGHT_CONSTANT) return ICP_GPU_OK;      // weighting.h:44
    void *sp, *sn, *sc, *tp, *tn, *tc, *di, *dw;
    if (up(ctx, 0, src_xyz, (size_t)n_src * 12, &sp) || up(ctx, 1, src_nrm, (size_t)n_src * 12, &sn) || up(ctx, 2, src_rgba, (size_t)n_src * 4, &sc) ||
        up(ctx, 3, tgt_xyz, (size_t)n_tgt * 12, &tp) || up(ctx, 4, tgt_nrm, (size_t)n_tgt * 12, &tn) || up(ctx, 5, tgt_rgba, (size_t)n_tgt * 4, &tc) ||
        up(ctx, 6, idx, (size_t)n_src * 4, &di) || up(ctx, 7, weight_inout, (size_t)n_src * 4, &dw)) return ICP_GPU_E_CUDA;
    CU(icp_launch_apply_weights(weighting, max_distance_sq, (const float*)sp, (const float*)sn, (const unsigned int*)sc, (const float*)tp, (const float*)tn,
                                (const unsigned int*)tc, (long long)n_tgt, (const int*)di, (float*)dw, (long long)n_src, ctx->stream));
    ctx->stats.n_kernel_launches += 1;
    CU(cudaMemcpyAsync(weight_inout, dw, (size_t)n_src * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_solve_linear(icp_gpu_ctx* ctx, int32_t metric, const float* src_xyz, const float* src_nrm, const float* tgt_xyz, const float* tgt_nrm,
                         const float* weights, int64_t n, float pose_out[16]) {
    if (!ctx || !pose_out || n < 0 || n > 0x7fffffff / 4 || (n > 0 && (!src_xyz || !tgt_xyz))) return ICP_GPU_E_ARG;
    if (metric < 0 || metric > 2) return fail(ctx, ICP_GPU_E_ARG, "metric %d", metric);
    if (metric == ICP_GPU_METRIC_P2PLANE && n > 0 && !tgt_nrm) return fail(ctx, ICP_GPU_E_ARG, "point-to-plane needs the target normals");
    if (metric == ICP_GPU_METRIC_SYMMETRIC && n > 0 && (!tgt_nrm || !src_nrm)) return fail(ctx, ICP_GPU_E_ARG, "the symmetric metric needs both normals");
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending");
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    for (int i = 0; i < 16; ++i) pose_out[i] = (i % 5 == 0) ? 1.f : 0.f;
    if (n == 0) return fail(ctx, ICP_GPU_E_NO_MATCHES, "no correspondences (the reference hangs in ASSERT here, ICPOptimizer.h:668,680,788)");
    void *s, *sn, *t, *tn, *w;
    const size_t n1 = (size_t)n;
    if (up(ctx, 0, src_xyz, n1 * 12, &s) || up(ctx, 1, src_nrm, n1 * 12, &sn) || up(ctx, 2, tgt_xyz, n1 * 12, &t) || up(ctx, 3, tgt_nrm, n1 * 12, &tn) ||
        up(ctx, 4, weights, n1 * 4, &w)) return ICP_GPU_E_CUDA;
    for (int k = 8; k < 14; ++k) if (ensure(ctx, ctx->scratch[k], n1 * (k < 12 ? sizeof(float4) : 4))) return ICP_GPU_E_CUDA;
    const int nb = icp_reduce_blocks((int)n, ctx->n_sms);
    if (ensure(ctx, ctx->scratch[14], (size_t)nb * ICP_NRED * sizeof(double))) return ICP_GPU_E_CUDA;
    CU(icp_launch_pack_pairs((const float*)s, (const float*)sn, (const float*)t, (const float*)tn, (const float*)w, (int)n, (float4*)ctx->scratch[8].p,
                             (float4*)ctx->scratch[9].p, (float4*)ctx->scratch[10].p, (float4*)ctx->scratch[11].p, (int*)ctx->scratch[12].p,
                             (float*)ctx->scratch[13].p, ctx->stream));
    // the pairs are already in a common frame: the loop state starts at the identity, the "estimated pose" it ends with is the increment
    const float eye[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    memcpy(ctx->h_pose, eye, sizeof(eye));
    CU(cudaMemcpyAsync(ctx->pose_dev.p, ctx->h_pose, 16 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CU(icp_launch_pose_init((DevState*)ctx->state.p, (const float*)ctx->pose_dev.p, ctx->stream));
    ReduceArgs ra; memset(&ra, 0, sizeof(ra));
    ra.src_pts = (const float4*)ctx->scratch[8].p; ra.src_nrm = (const float4*)ctx->scratch[9].p; ra.n_src = (int)n;
    ra.tgt_pts = (const float4*)ctx->scratch[10].p; ra.tgt_nrm = (const float4*)ctx->scratch[11].p; ra.n_tgt = (int)n;
    ra.match_pos = (const int*)ctx->scratch[12].p; ra.match_w = (const float*)ctx->scratch[13].p;
    ra.state = (DevState*)ctx->state.p; ra.partials = (double*)ctx->scratch[14].p; ra.pose_history = nullptr;
    ra.metric = metric; ra.solve = 1; ra.fused = 0; ra.desc_index = -1;
    int launches = 2;
    CU(icp_launch_reduce(ra, nb, ctx->stream, &launches));
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    CU(cudaMemcpyAsync(ctx->h_state, ctx->state.p, sizeof(DevState), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    const DevState& st = *ctx->h_state;
    if (st.status == ICP_GPU_E_NO_MATCHES) return fail(ctx, ICP_GPU_E_NO_MATCHES, "no finite correspondence");
    if (st.status != 0) return fail(ctx, st.status, "singular / non-finite system");
    memcpy(pose_out, st.pose, 16 * sizeof(float));
    return ICP_GPU_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------- batched registration of small pairs (batch.cu)
namespace {
// dev = false: every array is a host array, uploaded into batch_io and the results copied back; dev = true: every per-pair array is a
// device array on the context's device, read and written in place.  Either way the call waits for the batch.  config_index null:
// every pair runs with configs[0] (icp_gpu_estimate_pose_batch).
int estimate_pose_batch_configs(icp_gpu_ctx* ctx, int32_t n_configs, const icp_gpu_config* configs, int32_t n_pairs, const int32_t* config_index,
                                const float* src_xyz, const float* src_nrm, const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm,
                                const int64_t* tgt_off, const float* poses_in, float* poses_out, int32_t* n_iterations_out, int32_t* status_out,
                                float* pose_history, int32_t history_rows, bool dev) {
    if (n_configs < 1 || !configs) return fail(ctx, ICP_GPU_E_ARG, "batch: %d configs (at least one is needed)", n_configs);
    char who[32];
    for (int k = 0; k < n_configs; ++k) {
        const icp_gpu_config& c = configs[k];
        snprintf(who, sizeof(who), "batch: config %d: ", k);
        const int rc = check_config(ctx, &c, who);
        if (rc) return rc;
        if (c.matching != ICP_GPU_MATCH_KNN) return fail(ctx, ICP_GPU_E_ARG, "%sk-NN matching only (projective matching runs through icp_gpu_estimate_pose)", who);
        if (c.color_icp) return fail(ctx, ICP_GPU_E_ARG, "%s3-D matching only (colour ICP runs through icp_gpu_estimate_pose)", who);
        if (c.nn_algorithm == ICP_GPU_NN_BRUTE_NORM) return fail(ctx, ICP_GPU_E_ARG, "%ssquared-distance matching only (no norm-thresholded brute force)", who);
        if (c.multires && c.pyramid_mode == ICP_GPU_PYRAMID_VOXEL) return fail(ctx, ICP_GPU_E_ARG, "%sthe STRIDE pyramid only (the VOXEL pyramid runs through icp_gpu_estimate_pose)", who);
    }
    if (history_rows < 0) return fail(ctx, ICP_GPU_E_ARG, "batch: history_rows %d", history_rows);
    if (bind(ctx)) return ICP_GPU_E_CUDA;
    if (n_pairs == 0) return ICP_GPU_OK;
    const size_t B = (size_t)n_pairs;
    std::vector<int64_t> so(B + 1), to(B + 1);
    std::vector<int32_t> ci(B, 0);
    if (dev) {
        CU(cudaMemcpyAsync(so.data(), src_off, (B + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(to.data(), tgt_off, (B + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (config_index) CU(cudaMemcpyAsync(ci.data(), config_index, B * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    } else {
        memcpy(so.data(), src_off, (B + 1) * 8); memcpy(to.data(), tgt_off, (B + 1) * 8);
        if (config_index) memcpy(ci.data(), config_index, B * 4);
    }
    if (so[0] != 0 || to[0] != 0) return fail(ctx, ICP_GPU_E_ARG, "batch: the offsets must start at 0 (src %lld, tgt %lld)", (long long)so[0], (long long)to[0]);
    // pairs grouped by (minimiser, metric): group 3 * lm + metric
    std::vector<int> groups[6]; int group_tgt[6] = {0, 0, 0, 0, 0, 0};
    int max_rows = 0; bool need_scratch = false, need_finite = false, any_mask = false;
    for (size_t b = 0; b < B; ++b) {
        if (so[b + 1] < so[b] || to[b + 1] < to[b]) return fail(ctx, ICP_GPU_E_ARG, "batch: offsets of pair %zu are not monotone", b);
        const int64_t nt = to[b + 1] - to[b];
        if (nt > ICP_BATCH_MAX_TARGET)
            return fail(ctx, ICP_GPU_E_ARG, "batch: pair %zu has %lld target points, more than the %d a block stages; register it with icp_gpu_estimate_pose",
                        b, (long long)nt, ICP_BATCH_MAX_TARGET);
        if (ci[b] < 0 || ci[b] >= n_configs) return fail(ctx, ICP_GPU_E_ARG, "batch: pair %zu: config_index %d outside [0, %d)", b, ci[b], n_configs);
        const icp_gpu_config& c = configs[ci[b]];
        const int g = 3 * (c.minimizer == ICP_GPU_MIN_LM ? 1 : 0) + c.metric;
        groups[g].push_back((int)b);
        if (nt > group_tgt[g]) group_tgt[g] = (int)nt;
        const int rows = icp_schedule(c.n_iterations, c.multires, so[b + 1] - so[b]).n_iters;
        if (rows > max_rows) max_rows = rows;
        need_scratch = need_scratch || c.minimizer == ICP_GPU_MIN_LM || c.metric == ICP_GPU_METRIC_SYMMETRIC;
        const bool mt = c.selection == ICP_GPU_SELECT_RANDOM && c.selection_rng == ICP_GPU_RNG_MT19937;
        any_mask = any_mask || mt;
        need_finite = need_finite || (mt && c.multires);
    }
    const int64_t ns = so[B], nt = to[B];
    if (ns > 0x7fffffff / 4 || nt > 0x7fffffff / 4) return fail(ctx, ICP_GPU_E_ARG, "batch: %lld source / %lld target points in all", (long long)ns, (long long)nt);
    if ((ns > 0 && !src_xyz) || (nt > 0 && !tgt_xyz)) return fail(ctx, ICP_GPU_E_ARG, "batch: null point array");
    if (pose_history && history_rows < max_rows)
        return fail(ctx, ICP_GPU_E_ARG, "batch: history_rows %d, a pair of the batch runs up to %d iterations", history_rows, max_rows);
    const size_t hist_floats = pose_history ? B * (size_t)history_rows * 16 : 0;

    // mt19937 selection masks, drawn on the host (draw_selection_masks, as make_plan does); a mask set depends on the configuration,
    // the source size and, with multires, the source's finite flags: pairs that share those share one copy
    std::vector<uint32_t> masks; std::vector<long long> mask_off(any_mask ? B : 0, 0);
    if (any_mask) {
        std::vector<float> hp, hn;                       // the sources' points and normals, read back for the finite flags (_dev)
        const float* sp = src_xyz; const float* sn = src_nrm;
        if (need_finite && dev) {
            hp.resize((size_t)ns * 3); if (src_nrm) hn.resize((size_t)ns * 3);
            CU(cudaMemcpyAsync(hp.data(), src_xyz, (size_t)ns * 12, cudaMemcpyDeviceToHost, ctx->stream));
            if (src_nrm) CU(cudaMemcpyAsync(hn.data(), src_nrm, (size_t)ns * 12, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));
            sp = hp.data(); sn = src_nrm ? hn.data() : nullptr;
        }
        std::map<std::string, long long> shared;
        std::vector<uint8_t> finite;
        for (size_t b = 0; b < B; ++b) {
            const icp_gpu_config& c = configs[ci[b]];
            if (!(c.selection == ICP_GPU_SELECT_RANDOM && c.selection_rng == ICP_GPU_RNG_MT19937)) continue;
            const long long n = so[b + 1] - so[b];
            std::string key((const char*)&ci[b], 4); key.append((const char*)&n, 8);
            if (c.multires) {
                finite.assign((size_t)n, 0);
                for (long long k = 0; k < n; ++k) {
                    const float* p = sp + 3 * (so[b] + k); const float* m = sn ? sn + 3 * (so[b] + k) : nullptr;
                    finite[(size_t)k] = (isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]) && (!m || (isfinite(m[0]) && isfinite(m[1]) && isfinite(m[2])))) ? 1 : 0;
                }
                key.append((const char*)finite.data(), finite.size());
            }
            auto it = shared.find(key);
            if (it != shared.end()) { mask_off[b] = it->second; continue; }
            const IcpSchedule sch = icp_schedule(c.n_iterations, c.multires, n);
            const size_t words = ((size_t)(n > 0 ? n : 1) + 31) / 32;
            mask_off[b] = (long long)masks.size();
            masks.resize(masks.size() + (size_t)sch.n_iters * words, 0u);
            draw_selection_masks(c, sch, n, finite.data(), masks.data() + mask_off[b]);
            shared.emplace(std::move(key), mask_off[b]);
        }
    }

    BatchArgs a; memset(&a, 0, sizeof(a));
    a.src_xyz = src_xyz; a.src_nrm = src_nrm; a.src_off = (const long long*)src_off;
    a.tgt_xyz = tgt_xyz; a.tgt_nrm = tgt_nrm; a.tgt_off = (const long long*)tgt_off;
    a.poses_in = poses_in; a.poses_out = poses_out; a.n_iter_out = n_iterations_out; a.status_out = status_out; a.history = pose_history;
    a.history_rows = history_rows;
    if (!dev) {
        // one upload area, segments 256-byte aligned: inputs, then the results the kernel writes
        const size_t sizes[] = {(size_t)ns * 12, src_nrm ? (size_t)ns * 12 : 0, (size_t)nt * 12, tgt_nrm ? (size_t)nt * 12 : 0, (B + 1) * 8, (B + 1) * 8,
                                B * 64, B * 64, B * 4, B * 4, hist_floats * 4};
        const void* host_in[] = {src_xyz, src_nrm, tgt_xyz, tgt_nrm, src_off, tgt_off, poses_in};
        size_t off[11], total = 0;
        for (int k = 0; k < 11; ++k) { off[k] = total; total += (sizes[k] + 255) / 256 * 256; }
        if (ensure(ctx, ctx->batch_io, total, false)) return ICP_GPU_E_CUDA;
        char* base = (char*)ctx->batch_io.p;
        for (int k = 0; k < 7; ++k) if (sizes[k]) CU(cudaMemcpyAsync(base + off[k], host_in[k], sizes[k], cudaMemcpyHostToDevice, ctx->stream));
        a.src_xyz = (const float*)(base + off[0]); a.src_nrm = src_nrm ? (const float*)(base + off[1]) : nullptr;
        a.tgt_xyz = (const float*)(base + off[2]); a.tgt_nrm = tgt_nrm ? (const float*)(base + off[3]) : nullptr;
        a.src_off = (const long long*)(base + off[4]); a.tgt_off = (const long long*)(base + off[5]); a.poses_in = (const float*)(base + off[6]);
        a.poses_out = (float*)(base + off[7]); a.n_iter_out = (int*)(base + off[8]); a.status_out = (int*)(base + off[9]);
        a.history = pose_history ? (float*)(base + off[10]) : nullptr;
    }
    // the plan: configuration table, per-pair config index, the groups' pair lists, masks and their offsets
    std::vector<BatchCfg> tab((size_t)n_configs);
    for (int k = 0; k < n_configs; ++k) {
        const icp_gpu_config& c = configs[k];
        BatchCfg& t = tab[(size_t)k]; memset(&t, 0, sizeof(t));
        t.n_iterations = c.n_iterations; t.multires = c.multires ? 1 : 0; t.weighting = c.weighting; t.rejection = c.rejection;
        t.lm_max_iterations = c.lm_max_iterations;
        t.mt_mask = c.selection == ICP_GPU_SELECT_RANDOM && c.selection_rng == ICP_GPU_RNG_MT19937;
        t.max_d2 = c.max_distance_sq;
        t.weight_max_d2 = c.weight_max_distance_sq > 0.f ? c.weight_max_distance_sq : c.max_distance_sq;
        t.proba = c.selection == ICP_GPU_SELECT_RANDOM && c.selection_rng == ICP_GPU_RNG_DEVICE ? (float)c.proba : -1.0f;
        t.seed = c.seed;
        t.stop_rot = c.early_stop_rotation; t.stop_trans = c.early_stop_translation;
    }
    std::vector<int> pair_list; pair_list.reserve(B);
    size_t group_at[6];
    for (int g = 0; g < 6; ++g) { group_at[g] = pair_list.size(); pair_list.insert(pair_list.end(), groups[g].begin(), groups[g].end()); }
    {
        const size_t sizes[] = {tab.size() * sizeof(BatchCfg), B * 4, B * 4, masks.size() * 4, mask_off.size() * 8};
        const void* host_in[] = {tab.data(), ci.data(), pair_list.data(), masks.data(), mask_off.data()};
        size_t off[5], total = 0;
        for (int k = 0; k < 5; ++k) { off[k] = total; total += (sizes[k] + 255) / 256 * 256; }
        if (ensure(ctx, ctx->batch_plan, total, false)) return ICP_GPU_E_CUDA;
        char* base = (char*)ctx->batch_plan.p;
        for (int k = 0; k < 5; ++k) if (sizes[k]) CU(cudaMemcpyAsync(base + off[k], host_in[k], sizes[k], cudaMemcpyHostToDevice, ctx->stream));
        a.cfgs = (const BatchCfg*)(base + off[0]); a.cfg_index = (const int*)(base + off[1]); a.pairs = (const int*)(base + off[2]);
        a.mask = (const unsigned int*)(base + off[3]); a.mask_off = (const long long*)(base + off[4]);
    }
    if (a.history && hist_floats) CU(cudaMemsetAsync(a.history, 0, hist_floats * 4, ctx->stream));   // rows past a pair's last iteration read 0
    if (need_scratch) {
        if (ensure(ctx, ctx->batch_scratch, (size_t)(ns > 0 ? ns : 1) * sizeof(int2), false)) return ICP_GPU_E_CUDA;
        a.scratch = (int2*)ctx->batch_scratch.p;
    }
    // one launch per non-empty group; the groups after the first run on the auxiliary streams between a fork and a join event, so
    // that a small group does not wait behind a large one
    const int* pairs_dev = a.pairs;
    int n_aux = 0; bool first = true;
    CU(cudaEventRecord(ctx->chunks.fork, ctx->stream));
    for (int g = 0; g < 6; ++g) {
        if (groups[g].empty()) continue;
        a.pairs = pairs_dev + group_at[g];
        cudaStream_t st = ctx->stream;
        if (!first) { st = ctx->chunks.stream[n_aux]; CU(cudaStreamWaitEvent(st, ctx->chunks.fork, 0)); }
        CU(icp_launch_batch(a, g % 3, g / 3, (int)groups[g].size(), group_tgt[g], st));
        if (!first) CU(cudaEventRecord(ctx->chunks.done[n_aux++], st));
        first = false;
    }
    for (int k = 0; k < n_aux; ++k) CU(cudaStreamWaitEvent(ctx->stream, ctx->chunks.done[k], 0));
    if (!dev) {
        CU(cudaMemcpyAsync(poses_out, a.poses_out, B * 64, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(n_iterations_out, a.n_iter_out, B * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(status_out, a.status_out, B * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (hist_floats) CU(cudaMemcpyAsync(pose_history, a.history, hist_floats * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int batch_common_checks(icp_gpu_ctx* ctx, int32_t n_pairs, const int64_t* src_off, const int64_t* tgt_off, const float* poses_in, float* poses_out,
                        int32_t* n_iterations_out, int32_t* status_out) {
    if (n_pairs < 0) return fail(ctx, ICP_GPU_E_ARG, "n_pairs %d", n_pairs);
    if (!src_off || !tgt_off || !poses_in || !poses_out || !n_iterations_out || !status_out)
        return fail(ctx, ICP_GPU_E_ARG, "batch: offsets, poses_in, poses_out, n_iterations_out and status_out are required");
    if (ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending; call icp_gpu_estimate_pose_finish first");
    return 0;
}

// The context's configuration for every pair, with the refusals this entry point has always had.
int estimate_pose_batch(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                        const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in, float* poses_out,
                        int32_t* n_iterations_out, int32_t* status_out, float* pose_history, bool dev) {
    if (!ctx) return ICP_GPU_E_ARG;
    int rc = batch_common_checks(ctx, n_pairs, src_off, tgt_off, poses_in, poses_out, n_iterations_out, status_out);
    if (rc) return rc;
    const icp_gpu_config& cfg = ctx->cfg;
    if (cfg.minimizer != ICP_GPU_MIN_LINEAR) return fail(ctx, ICP_GPU_E_ARG, "batch: the linear minimiser only (Levenberg-Marquardt runs through icp_gpu_estimate_pose_batch_configs)");
    if (cfg.multires) return fail(ctx, ICP_GPU_E_ARG, "batch: no multi-resolution schedule (run it through icp_gpu_estimate_pose_batch_configs)");
    if (cfg.matching != ICP_GPU_MATCH_KNN) return fail(ctx, ICP_GPU_E_ARG, "batch: k-NN matching only (projective matching runs through icp_gpu_estimate_pose)");
    if (cfg.color_icp) return fail(ctx, ICP_GPU_E_ARG, "batch: 3-D matching only (colour ICP runs through icp_gpu_estimate_pose)");
    if (cfg.nn_algorithm == ICP_GPU_NN_BRUTE_NORM) return fail(ctx, ICP_GPU_E_ARG, "batch: squared-distance matching only (no norm-thresholded brute force)");
    if (cfg.selection == ICP_GPU_SELECT_RANDOM && cfg.selection_rng != ICP_GPU_RNG_DEVICE)
        return fail(ctx, ICP_GPU_E_ARG, "batch: random selection needs the device stream (selection_rng = ICP_GPU_RNG_DEVICE); mt19937 selection runs through icp_gpu_estimate_pose_batch_configs");
    return estimate_pose_batch_configs(ctx, 1, &ctx->cfg, n_pairs, nullptr, src_xyz, src_nrm, src_off, tgt_xyz, tgt_nrm, tgt_off, poses_in, poses_out,
                                       n_iterations_out, status_out, pose_history, cfg.n_iterations, dev);
}

int estimate_pose_batch_configs_entry(icp_gpu_ctx* ctx, int32_t n_configs, const icp_gpu_config* configs, int32_t n_pairs, const int32_t* config_index,
                                      const float* src_xyz, const float* src_nrm, const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm,
                                      const int64_t* tgt_off, const float* poses_in, float* poses_out, int32_t* n_iterations_out, int32_t* status_out,
                                      float* pose_history, int32_t history_rows, bool dev) {
    if (!ctx) return ICP_GPU_E_ARG;
    int rc = batch_common_checks(ctx, n_pairs, src_off, tgt_off, poses_in, poses_out, n_iterations_out, status_out);
    if (rc) return rc;
    if (!config_index) return fail(ctx, ICP_GPU_E_ARG, "batch: config_index is required");
    return estimate_pose_batch_configs(ctx, n_configs, configs, n_pairs, config_index, src_xyz, src_nrm, src_off, tgt_xyz, tgt_nrm, tgt_off, poses_in,
                                       poses_out, n_iterations_out, status_out, pose_history, history_rows, dev);
}
}  // namespace

extern "C" {

int icp_gpu_estimate_pose_batch(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                                const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in, float* poses_out,
                                int32_t* n_iterations_out, int32_t* status_out, float* pose_history) {
    return estimate_pose_batch(ctx, n_pairs, src_xyz, src_nrm, src_off, tgt_xyz, tgt_nrm, tgt_off, poses_in, poses_out, n_iterations_out,
                               status_out, pose_history, false);
}

int icp_gpu_estimate_pose_batch_dev(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                                    const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in, float* poses_out,
                                    int32_t* n_iterations_out, int32_t* status_out, float* pose_history) {
    return estimate_pose_batch(ctx, n_pairs, src_xyz, src_nrm, src_off, tgt_xyz, tgt_nrm, tgt_off, poses_in, poses_out, n_iterations_out,
                               status_out, pose_history, true);
}

int icp_gpu_estimate_pose_batch_configs(icp_gpu_ctx* ctx, int32_t n_configs, const icp_gpu_config* configs, int32_t n_pairs,
                                        const int32_t* config_index, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                                        const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in,
                                        float* poses_out, int32_t* n_iterations_out, int32_t* status_out, float* pose_history,
                                        int32_t history_rows) {
    return estimate_pose_batch_configs_entry(ctx, n_configs, configs, n_pairs, config_index, src_xyz, src_nrm, src_off, tgt_xyz, tgt_nrm, tgt_off,
                                             poses_in, poses_out, n_iterations_out, status_out, pose_history, history_rows, false);
}

int icp_gpu_estimate_pose_batch_configs_dev(icp_gpu_ctx* ctx, int32_t n_configs, const icp_gpu_config* configs, int32_t n_pairs,
                                            const int32_t* config_index, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                                            const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in,
                                            float* poses_out, int32_t* n_iterations_out, int32_t* status_out, float* pose_history,
                                            int32_t history_rows) {
    return estimate_pose_batch_configs_entry(ctx, n_configs, configs, n_pairs, config_index, src_xyz, src_nrm, src_off, tgt_xyz, tgt_nrm, tgt_off,
                                             poses_in, poses_out, n_iterations_out, status_out, pose_history, history_rows, true);
}

}  // extern "C"
