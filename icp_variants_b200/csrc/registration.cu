// registration.cu -- the registration loop (icp_gpu_estimate_pose[_async/_finish]): iteration planning, CUDA-graph replay of the
// loop, and the matches at one pose (icp_gpu_query_matches).  Host code only; the kernels live in grid.cu, match.cu, solve.cu and lm.cu.
//
// What runs where: the host plans the iterations (level strides, selection masks) and enqueues
// them; every iteration is {match kernel, reduction(+solve) kernel(s)} on one stream with no host
// synchronisation in between -- the loop state (pose, iteration counter, status) lives in DevState
// on the device.  The only host<->device traffic of estimate_pose is the iteration descriptors and
// the 16-float pose up, and the pose, pose history and DevState down.
//
// Reference: ICPOptimizer.h:185-349 / :493-663 (the loop), NearestNeighbor.h:12-36 (matcher API).
#include "context.cuh"
#include <stdlib.h>

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

struct Plan {
    int n_iters = 0;
    std::vector<IterDesc> desc;         // n_iters entries
    std::vector<uint32_t> mask;         // concatenated selection masks, one bit per original source index (mt19937 mode)
    std::vector<int> voxel_depth;       // voxel pyramid: grid depth of every mask slot built on the device
};

struct KernelClouds { const float4 *src_pts, *src_nrm, *tgt_pts, *tgt_nrm; bool tiled; };   // kernel_clouds

}  // namespace

// The mt19937 selection masks of one registration (selection.h:88-104, contract D7): iteration i's mask is out[i * words ..),
// words = mask_words(n), one bit per original source index, zero-filled by the caller.  resample() draws once per point of the
// level cloud, in order: every stride-th point, with multires only those whose point and normal are finite (finite[k], PointCloud.h:335).
// One PointSelection per level (:652), seeded with seed + level (initSampler); its stream runs on across the stride-1 iterations.
void draw_selection_masks(const icp_gpu_config& cfg, const IcpSchedule& sch, long long n, const uint8_t* finite, uint32_t* out) {
    const size_t words = mask_words(n);
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

int choose_algorithm(const icp_gpu_ctx* c) {   // 0 grid, 1 brute, 2 projective
    if (c->cfg.matching == ICP_GPU_MATCH_PROJECTIVE) return 2;
    if (c->cfg.nn_algorithm == ICP_GPU_NN_BRUTE || c->cfg.nn_algorithm == ICP_GPU_NN_BRUTE_NORM) return 1;
    if (c->cfg.nn_algorithm == ICP_GPU_NN_GRID) return 0;
    return c->n_tgt <= 2048 ? 1 : 0;
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

// The iteration schedule of estimatePose (ICPOptimizer.h:503-525, :540, :549-550, :634-655; Appendix A of SURVEY.md).
static int make_plan(icp_gpu_ctx* ctx, Plan& plan) {
    const icp_gpu_config& cfg = ctx->cfg;
    const int n = ctx->n_src;
    const bool host_rng = cfg.selection == ICP_GPU_SELECT_RANDOM && cfg.selection_rng == ICP_GPU_RNG_MT19937;
    const bool dev_rng = cfg.selection == ICP_GPU_SELECT_RANDOM && cfg.selection_rng == ICP_GPU_RNG_DEVICE;
    if (host_rng && cfg.multires && fetch_src_finite(ctx)) return ICP_GPU_E_CUDA;
    const size_t words = mask_words(n);
    const bool voxel = cfg.multires && cfg.pyramid_mode == ICP_GPU_PYRAMID_VOXEL;
    const IcpSchedule sch = icp_schedule(cfg.n_iterations, cfg.multires, n);
    if (sch.n_iters > ICP_MAX_ITERS) return fail(ctx, ICP_GPU_E_ARG, "more than %d iterations", ICP_MAX_ITERS);
    if (host_rng) {
        plan.mask.assign((size_t)sch.n_iters * words, 0u);
        draw_selection_masks(cfg, sch, n, ctx->src_finite.data(), plan.mask.data());
    }
    for (int i = 0; i < sch.n_iters; ++i) {
        const int stride = icp_schedule_stride(sch, i);
        IterDesc d = all_points_desc();
        d.stride = stride; d.filter_finite = cfg.multires ? 1 : 0;
        if (voxel && stride > 1) {
            // level = one point per occupied source-grid cell at depth Ts' - ceil(1.5 log2 stride)
            int k = 0; while ((1 << k) < stride) ++k;
            int D = (ctx->Ts < 22 ? ctx->Ts : 22) - (3 * k + 1) / 2; if (D < 0) D = 0;
            int slot = -1;
            for (size_t j = 0; j < plan.voxel_depth.size(); ++j) if (plan.voxel_depth[j] == D) slot = (int)j;
            if (slot < 0) { slot = (int)plan.voxel_depth.size(); plan.voxel_depth.push_back(D); }
            d.stride = 1; d.mask_word_offset = (int)((size_t)slot * words);
        }
        if (dev_rng) { d.proba = (float)cfg.proba; d.rng_key = cfg.seed * 2654435761u + (uint32_t)(i + 1) * 0x9E3779B9u; }
        if (host_rng) d.mask_word_offset = (int)((size_t)i * words);
        plan.desc.push_back(d);
    }
    plan.n_iters = sch.n_iters;
    return 0;
}

// Projective matching of a full-frame source (one point per pixel of the camera the target was taken with): the kernels
// then address the source in its original pixel order (the unsorted upload) instead of the Morton order.
static bool proj_tiled(const icp_gpu_ctx* c, int algo) {
    return algo == 2 && c->n_src > 0 && (long long)c->width * c->height == (long long)c->n_src;
}

// The clouds the search and the reduction read: the target in grid order for the BVH search, else in upload order; the source in
// Morton order, or in pixel order when proj_tiled.
static KernelClouds kernel_clouds(const icp_gpu_ctx* c, int algo) {
    const bool grid_order = algo == 0, tiled = proj_tiled(c, algo);
    return {(const float4*)(tiled ? c->src_raw_pts.p : c->src_pts.p), (const float4*)(tiled ? c->src_raw_nrm.p : c->src_nrm.p),
            (const float4*)(grid_order ? c->tgt_pts_sorted.p : c->tgt_pts.p), (const float4*)(grid_order ? c->tgt_nrm_sorted.p : c->tgt_nrm.p), tiled};
}

void fill_match_args(icp_gpu_ctx* c, MatchArgs& a, int algo, int desc_index, bool want_idx) {
    memset(&a, 0, sizeof(a));
    const KernelClouds k = kernel_clouds(c, algo);
    a.src_pts = k.src_pts; a.src_nrm = k.src_nrm; a.n_src = c->n_src; a.proj_tiled = k.tiled ? 1 : 0;
    a.mask = (const unsigned int*)c->mask.p; a.desc = (const IterDesc*)c->desc.p;
    a.state_ro = (const DevState*)c->state.p; a.state = (DevState*)c->state.p;
    a.tgt_pts = k.tgt_pts; a.tgt_nrm = k.tgt_nrm; a.n_tgt = c->n_tgt;
    a.bvh_box = (const float4*)c->bvh_box.p; a.bvh = (const BvhDesc*)c->bvh_desc.p; a.leaf_start = (const unsigned int*)c->leaf_start.p;
    a.leaf_rank = (const unsigned int*)c->leaf_rank.p; a.child_start = (const unsigned int*)c->child_start.p;
    a.adj = (const unsigned int*)c->adj.p; a.adj_box = (const float4*)c->adj_box.p; a.adj_capacity = c->adj_capacity;
    a.adj_gap = (const float*)c->adj_gap.p;
    a.nn_leaf = (int*)c->nn_leaf.p;
    a.adj1 = (const unsigned int*)c->adj1.p; a.adj1_box = (const float4*)c->adj1_box.p; a.adj1_capacity = c->adj1_capacity;
    a.node_rank = (const unsigned int*)c->node_rank.p;
    if (c->have_camera) { a.fx = c->K[0]; a.fy = c->K[4]; a.cx = c->K[6]; a.cy = c->K[7]; }   // column-major Matrix3f
    a.width = c->width; a.height = c->height;
    a.weighting = c->cfg.weighting; a.rejection = c->cfg.rejection; a.color_icp = c->cfg.color_icp;
    a.max_d2 = c->cfg.max_distance_sq;
    a.weight_max_d2 = c->cfg.weight_max_distance_sq > 0.f ? c->cfg.weight_max_distance_sq : c->cfg.max_distance_sq;
    a.match_pos = (int*)c->match_pos.p; a.match_w = (float*)c->match_w.p; a.match_idx = want_idx ? (int*)c->match_idx.p : nullptr;
    a.nn_pos = (int*)c->nn_pos.p; a.qbuf = (float4*)c->qbuf.p; a.seedbuf = (float4*)c->seedbuf.p;
    a.desc_index = desc_index;
    a.q_begin = 0; a.q_end = c->n_src;
    a.brute_norm = c->cfg.nn_algorithm == ICP_GPU_NN_BRUTE_NORM ? 1 : 0;
    a.collect_stats = c->cfg.collect_stats;
}

void fill_reduce_args(icp_gpu_ctx* c, ReduceArgs& r, int algo, int solve) {
    memset(&r, 0, sizeof(r));
    const KernelClouds k = kernel_clouds(c, algo);
    r.src_pts = k.src_pts; r.src_nrm = k.src_nrm; r.n_src = c->n_src;
    r.state = (DevState*)c->state.p;
    r.tgt_pts = k.tgt_pts; r.tgt_nrm = k.tgt_nrm;
    r.match_pos = (const int*)c->match_pos.p; r.match_w = (const float*)c->match_w.p;
    r.partials = (double*)c->partials.p; r.pose_history = (float*)c->history.p;
    r.metric = c->cfg.metric; r.solve = solve;
    r.fused = 0; r.nn_pos = (const int*)c->nn_pos.p; r.n_tgt = c->n_tgt; r.mask = (const unsigned int*)c->mask.p;
    r.desc = (const IterDesc*)c->desc.p; r.desc_index = -1;
    r.weighting = c->cfg.weighting; r.rejection = c->cfg.rejection; r.max_d2 = c->cfg.max_distance_sq;
    r.weight_max_d2 = c->cfg.weight_max_distance_sq > 0.f ? c->cfg.weight_max_distance_sq : c->cfg.max_distance_sq;
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
    const bool seed = allow_seed && ctx->n_tgt > 0 && ctx->grid_built;
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
static int enqueue_iterations(icp_gpu_ctx* ctx, const Plan& plan, int algo, std::vector<cudaEvent_t>* ev_marks) {
    MatchArgs ma; ReduceArgs ra;
    fill_match_args(ctx, ma, algo, -1, false);
    fill_reduce_args(ctx, ra, algo, 1);
    // Without work counters the linear minimiser reads the search result directly: weighting and rejection are
    // evaluated inside the reduction and the match records (and their launch) are skipped.
    if (algo == 0 && ctx->cfg.minimizer == ICP_GPU_MIN_LINEAR && !ctx->cfg.collect_stats) { ma.skip_finish = 1; ra.fused = 1; }
    int launches = 0;
    const int nb = ctx->n_reduce_blocks;
    // Two chunks of >= 64k queries (test hook: ICP_GPU_MATCH_CHUNKS).  Measured at 370k queries: 1 / 2 / 3 / 4 chunks
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

static int start_registration(icp_gpu_ctx* ctx, const float pose_in[16], icp_gpu_timings* timings) {
    if (!pose_in) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
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
        const size_t words = mask_words(ctx->n_src);
        int dmax = 0; for (int D : plan.voxel_depth) dmax = D > dmax ? D : dmax;
        if (ensure(ctx, ctx->mask, plan.voxel_depth.size() * words * sizeof(uint32_t)) ||
            ensure(ctx, ctx->voxel_table, sizeof(unsigned int) * ((size_t)1 << dmax))) return ICP_GPU_E_CUDA;
        int launches = 0;
        for (size_t j = 0; j < plan.voxel_depth.size(); ++j)
            CU(icp_launch_voxel_level((const float4*)ctx->src_pts.p, (const float4*)ctx->src_nrm.p, ctx->n_src, (const GridParams*)ctx->sgrid.p,
                                      ctx->Ts, plan.voxel_depth[j], (unsigned int*)ctx->voxel_table.p, (unsigned int*)ctx->mask.p + j * words,
                                      words, ctx->stream, &launches));
        ctx->stats.n_kernel_launches += (uint64_t)launches;
    }
    if (!plan.mask.empty()) {
        if (ensure(ctx, ctx->mask, plan.mask.size() * sizeof(uint32_t))) return ICP_GPU_E_CUDA;
        CU(cudaMemcpyAsync(ctx->mask.p, plan.mask.data(), plan.mask.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));   // plan.mask is pageable and dies with this frame
    }
    if (upload_pose(ctx, pose_in, ctx->cfg.early_stop_rotation, ctx->cfg.early_stop_translation)) return ICP_GPU_E_CUDA;
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

static void copy_counters(icp_gpu_ctx* ctx) {
    const DevState& st = *ctx->h_state;
    ctx->stats.n_queries = st.n_queries; ctx->stats.n_matched = st.n_matched;
    ctx->stats.n_distance_evals = st.n_evals; ctx->stats.n_nodes_visited = st.n_nodes;
    for (int k = 0; k < 6; ++k) ctx->stats.reduce_profile_ns[k] = st.prof[k];
}

int icp_gpu_estimate_pose_finish(icp_gpu_ctx* ctx, float pose_out[16], float* pose_history, int32_t* n_iterations_out) {
    if (int rc = enter(ctx, false)) return rc;
    if (!ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "no registration pending");
    ctx->pending = false;
    CU(cudaStreamSynchronize(ctx->stream));
    const DevState& st = *ctx->h_state;
    if (pose_out) memcpy(pose_out, st.pose, 16 * sizeof(float));
    if (pose_history && st.iters_done > 0) memcpy(pose_history, ctx->h_history, sizeof(float) * 16 * (size_t)st.iters_done);
    if (n_iterations_out) *n_iterations_out = st.iters_done;
    ctx->last_iters = st.iters_done;
    copy_counters(ctx);
    return status_error(ctx, st.status, st.iters_done, "iteration %d had no surviving correspondence (the reference hangs in ASSERT here)");
}

int icp_gpu_query_matches(icp_gpu_ctx* ctx, const float pose[16], const int32_t* sel_idx, int64_t n_sel, int32_t* idx_out, float* weight_out) {
    if (!pose || !idx_out || !weight_out) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    int rc = check_ready(ctx); if (rc) return rc;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    const int n = ctx->n_src;
    const int nq = sel_idx ? (int)n_sel : n;
    if (sel_idx && (n_sel < 0 || n_sel > n)) return fail(ctx, ICP_GPU_E_ARG, "n_sel %lld", (long long)n_sel);
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    if (fetch_src_rank(ctx)) return ICP_GPU_E_CUDA;
    IterDesc d = all_points_desc();
    std::vector<uint32_t> mask;
    if (sel_idx) {
        mask.assign(mask_words(n), 0u);
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
    if (upload_pose(ctx, pose)) return ICP_GPU_E_CUDA;
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

int icp_gpu_estimate_pose(icp_gpu_ctx* ctx, float pose_inout[16], float* pose_history, int32_t* n_iterations_out, icp_gpu_timings* timings) {
    if (int rc = start_registration(ctx, pose_inout, timings)) return rc;
    return icp_gpu_estimate_pose_finish(ctx, pose_inout, pose_history, n_iterations_out);
}
