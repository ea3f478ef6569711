// batch_indexed_api.cu -- the host side of indexed batched registration (icp_gpu_estimate_pose_batch_indexed[_dev]): B pairs of any
// size, each against an index of its own target built in the call, all registered in one launch of multistart.cu's kernel with one
// thread-block cluster per pair.  Host code only.
//
//   inputs   the concatenated clouds (one upload each, or read in place), the offsets read back and checked
//   build    pair by pair on the context's stream: the source packed and sorted, the target packed, sorted and indexed -- the steps
//            and launchers of set_source / set_target (clouds.cu) -- into the pair's slices of one arena; the sort and tree scratch is
//            shared, as the builds run one after another
//   plan     plan_iterations per pair (registration.cu): descriptors into one table, mt19937 masks drawn on the host, VOXEL levels
//            built on the pair's own source grid
//   launch   one cluster per pair, the largest sources first (a shorter tail on mixed sizes; no result depends on the order)
#include "context.cuh"
#include <algorithm>
#include <numeric>

namespace {

// Byte sizes of one pair's arena segments (ns source, nt target points).
enum { A_SRC_PTS, A_SRC_NRM, A_TGT_PTS, A_TGT_NRM, A_KEYS_A, A_KEYS_B, A_MSD, A_GRID, A_BBOX, A_LEAF_START, A_LEAF_RANK, A_BVH_DESC, A_BVH_BOX,
       A_CHILD_START, A_ADJ, A_ADJ_BOX, A_SEGMENTS };

void arena_sizes(int ns, int nt, size_t* sz) {
    const size_t s1 = (size_t)(ns > 0 ? ns : 1), t1 = (size_t)(nt > 0 ? nt : 1);
    const size_t nodes = icp_bvh_max_nodes(nt), cap = (size_t)adj_capacity_for(nt);
    sz[A_SRC_PTS] = sz[A_SRC_NRM] = s1 * sizeof(float4);
    sz[A_TGT_PTS] = sz[A_TGT_NRM] = t1 * sizeof(float4);
    sz[A_KEYS_A] = sz[A_KEYS_B] = t1 * 4;
    sz[A_MSD] = ICP_MSD_WORDS * 4; sz[A_GRID] = sizeof(GridParams); sz[A_BBOX] = 64;
    sz[A_LEAF_START] = sz[A_LEAF_RANK] = (t1 + 2) * 4;
    sz[A_BVH_DESC] = sizeof(BvhDesc); sz[A_BVH_BOX] = nodes * 2 * sizeof(float4);
    sz[A_CHILD_START] = (nodes + ICP_BVH_MAX_LEVELS) * 4;
    sz[A_ADJ] = cap * 32 * 4; sz[A_ADJ_BOX] = cap * 2 * sizeof(float4);
}

// Scratch the builds share, sized for the largest source (ms) and target (mt) of the batch: packed records, the source's bbox and
// grid, the sort's ping-pong buffers and histograms, the tree's scratch, the level-1 lists and the VOXEL table.
enum { S_PTS, S_NRM, S_SBBOX, S_SGRID, S_SKEYS_A, S_SKEYS_B, S_IDX_A, S_IDX_B, S_HIST, S_LV_FLAGS, S_LV_TILES, S_DELTA_A, S_DELTA_B, S_NODE_RANK,
       S_ADJ1, S_ADJ1_BOX, S_ADJ_GAP, S_VOXEL, S_SEGMENTS };

}  // namespace

static int estimate_pose_batch_indexed(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const uint8_t* src_rgba,
                                       const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm, const uint8_t* tgt_rgba, const int64_t* tgt_off,
                                       const float* poses_in, float* poses_out, int32_t* n_iterations_out, int32_t* status_out, int64_t* inliers_out,
                                       double* rmse_out, float* pose_history, int32_t history_rows, int32_t* match_idx_out, float* match_w_out, bool dev) {
    if (int rc = enter(ctx)) return rc;
    if (n_pairs < 0) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: n_pairs %d", n_pairs);
    if (!src_off || !tgt_off || !poses_in || !poses_out || !n_iterations_out || !status_out || !inliers_out || !rmse_out)
        return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: the offsets, poses_in, poses_out, n_iterations_out, status_out, inliers_out and rmse_out are required");
    if ((match_idx_out == nullptr) != (match_w_out == nullptr)) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: match_idx_out and match_w_out go together");
    const icp_gpu_config& cfg = ctx->cfg;
    if (cfg.matching != ICP_GPU_MATCH_KNN) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: k-NN matching only (projective matching runs through icp_gpu_estimate_pose)");
    if (cfg.nn_algorithm == ICP_GPU_NN_BRUTE_NORM) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: squared-distance matching only (no norm-thresholded brute force)");
    if (ctx->peer_world > 1) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: the context has attached peers (point-sharded registration runs through icp_gpu_estimate_pose)");
    if (n_pairs == 0) return ICP_GPU_OK;
    const size_t B = (size_t)n_pairs;
    std::vector<int64_t> so(B + 1), to(B + 1);
    if (dev) {
        CU(cudaMemcpyAsync(so.data(), src_off, (B + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(to.data(), tgt_off, (B + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    } else {
        memcpy(so.data(), src_off, (B + 1) * 8); memcpy(to.data(), tgt_off, (B + 1) * 8);
    }
    if (so[0] != 0 || to[0] != 0) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: the offsets must start at 0 (src %lld, tgt %lld)", (long long)so[0], (long long)to[0]);
    int max_s = 0, max_t = 0, max_rows = 0;
    for (size_t b = 0; b < B; ++b) {
        if (so[b + 1] < so[b] || to[b + 1] < to[b]) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: offsets of pair %zu are not monotone", b);
        const int64_t ns = so[b + 1] - so[b], nt = to[b + 1] - to[b];
        if (ns > 0x7fffffff / 4 || nt > 0x7fffffff / 4)
            return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: pair %zu has %lld source / %lld target points, above a cloud's limit of %d", b, (long long)ns,
                        (long long)nt, 0x7fffffff / 4);
        max_s = std::max(max_s, (int)ns); max_t = std::max(max_t, (int)nt);
        max_rows = std::max(max_rows, icp_schedule(cfg.n_iterations, cfg.multires, ns).n_iters);
    }
    const int64_t ns_all = so[B], nt_all = to[B];
    if (ns_all > 0x7fffffff) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: %lld source points in all exceed INT32_MAX", (long long)ns_all);
    if ((ns_all > 0 && !src_xyz) || (nt_all > 0 && !tgt_xyz)) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: null point array");
    if (max_rows > ICP_MAX_ITERS) return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: a pair of the batch runs more than %d iterations", ICP_MAX_ITERS);
    if (pose_history && history_rows < max_rows)
        return fail(ctx, ICP_GPU_E_ARG, "batch_indexed: history_rows %d, a pair of the batch runs up to %d iterations", history_rows, max_rows);

    // inputs: the host form uploads each concatenated array once, then the results the kernel writes
    const size_t hist_floats = pose_history ? B * (size_t)history_rows * 16 : 0;
    const size_t match_n = match_idx_out ? (size_t)ns_all : 0;
    const float *sx = src_xyz, *sn = src_nrm, *tx = tgt_xyz, *tn = tgt_nrm; const uint8_t *sc = src_rgba, *tc = tgt_rgba;
    const float* pin = poses_in; float* pout = poses_out; int* n_it = n_iterations_out; int* st = status_out;
    long long* inl = (long long*)inliers_out; double* rmse = rmse_out; float* hist = pose_history; int* midx = match_idx_out; float* mw = match_w_out;
    if (!dev) {
        const size_t sizes[] = {(size_t)ns_all * 12, src_nrm ? (size_t)ns_all * 12 : 0, src_rgba ? (size_t)ns_all * 4 : 0, (size_t)nt_all * 12,
                                tgt_nrm ? (size_t)nt_all * 12 : 0, tgt_rgba ? (size_t)nt_all * 4 : 0, B * 64,
                                B * 64, B * 4, B * 4, B * 8, B * 8, hist_floats * 4, match_n * 4, match_n * 4};
        const void* host_in[] = {src_xyz, src_nrm, src_rgba, tgt_xyz, tgt_nrm, tgt_rgba, poses_in};
        size_t off[15];
        if (ensure(ctx, ctx->bi_io, pack_segments(sizes, 15, off), false)) return ICP_GPU_E_CUDA;
        char* base = (char*)ctx->bi_io.p;
        for (int k = 0; k < 7; ++k) if (sizes[k]) CU(cudaMemcpyAsync(base + off[k], host_in[k], sizes[k], cudaMemcpyHostToDevice, ctx->stream));
        sx = (const float*)(base + off[0]); sn = src_nrm ? (const float*)(base + off[1]) : nullptr; sc = src_rgba ? (const uint8_t*)(base + off[2]) : nullptr;
        tx = (const float*)(base + off[3]); tn = tgt_nrm ? (const float*)(base + off[4]) : nullptr; tc = tgt_rgba ? (const uint8_t*)(base + off[5]) : nullptr;
        pin = (const float*)(base + off[6]); pout = (float*)(base + off[7]); n_it = (int*)(base + off[8]); st = (int*)(base + off[9]);
        inl = (long long*)(base + off[10]); rmse = (double*)(base + off[11]); hist = pose_history ? (float*)(base + off[12]) : nullptr;
        midx = match_n ? (int*)(base + off[13]) : nullptr; mw = match_n ? (float*)(base + off[14]) : nullptr;
    }

    // the plans; mt19937 with multires reads the sources' finite flags (the _dev form reads the sources back for them)
    const bool host_rng = cfg.selection == ICP_GPU_SELECT_RANDOM && cfg.selection_rng == ICP_GPU_RNG_MT19937;
    std::vector<float> hp, hn;
    const float* fp = src_xyz; const float* fn = src_nrm;
    if (host_rng && cfg.multires && dev && ns_all > 0) {
        hp.resize((size_t)ns_all * 3); if (src_nrm) hn.resize((size_t)ns_all * 3);
        CU(cudaMemcpyAsync(hp.data(), src_xyz, (size_t)ns_all * 12, cudaMemcpyDeviceToHost, ctx->stream));
        if (src_nrm) CU(cudaMemcpyAsync(hn.data(), src_nrm, (size_t)ns_all * 12, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        fp = hp.data(); fn = src_nrm ? hn.data() : nullptr;
    }
    std::vector<Plan> plans(B);
    std::vector<size_t> desc_at(B), mask_at(B);
    size_t n_desc = 0, n_mask_words = 0; int dmax = 0;
    std::vector<uint8_t> finite;
    for (size_t b = 0; b < B; ++b) {
        const int ns = (int)(so[b + 1] - so[b]);
        if (host_rng && cfg.multires) {
            finite.assign((size_t)ns, 0);
            for (int k = 0; k < ns; ++k) finite[(size_t)k] = point_finite(fp + 3 * (so[b] + k), fn ? fn + 3 * (so[b] + k) : nullptr) ? 1 : 0;
        }
        if (int rc = plan_iterations(ctx, cfg, ns, pick_T(ns, true), finite.data(), plans[b])) return rc;
        const Plan& p = plans[b];
        desc_at[b] = n_desc; n_desc += (size_t)p.n_iters;
        mask_at[b] = n_mask_words;
        n_mask_words += std::max(p.mask.size(), p.voxel_depth.size() * mask_words(ns));
        for (int D : p.voxel_depth) dmax = std::max(dmax, D);
    }
    std::vector<IterDesc> descs(n_desc > 0 ? n_desc : 1);
    std::vector<uint32_t> masks;
    if (host_rng) masks.assign(n_mask_words, 0u);
    for (size_t b = 0; b < B; ++b) {
        std::copy(plans[b].desc.begin(), plans[b].desc.end(), descs.begin() + (long)desc_at[b]);
        if (host_rng) std::copy(plans[b].mask.begin(), plans[b].mask.end(), masks.begin() + (long)mask_at[b]);
    }

    // the arena (every pair's clouds and index), the shared build scratch and the plan area
    std::vector<size_t> asz(B * A_SEGMENTS), aoff(B * A_SEGMENTS);
    for (size_t b = 0; b < B; ++b) arena_sizes((int)(so[b + 1] - so[b]), (int)(to[b + 1] - to[b]), &asz[b * A_SEGMENTS]);
    if (ensure(ctx, ctx->bi_arena, pack_segments(asz.data(), (int)asz.size(), aoff.data()), false)) return ICP_GPU_E_CUDA;
    const int Ts_max = pick_T(max_s, true), T_t = pick_T(max_t, false);
    const size_t m1 = (size_t)std::max(std::max(max_s, max_t), 1), t1 = (size_t)std::max(max_t, 1), nodes = icp_bvh_max_nodes(max_t);
    const size_t hist_words = std::max(icp_radix_hist_words(max_s, Ts_max), icp_radix_hist_words(max_t, T_t));
    const int cap = adj_capacity_for(max_t), cap1 = adj1_capacity_for(max_t);
    size_t ssz[S_SEGMENTS], soff[S_SEGMENTS];
    ssz[S_PTS] = ssz[S_NRM] = m1 * sizeof(float4); ssz[S_SBBOX] = 64; ssz[S_SGRID] = sizeof(GridParams);
    ssz[S_SKEYS_A] = ssz[S_SKEYS_B] = (size_t)std::max(max_s, 1) * 4; ssz[S_IDX_A] = ssz[S_IDX_B] = m1 * 4; ssz[S_HIST] = hist_words * 4;
    ssz[S_LV_FLAGS] = t1 + 64; ssz[S_LV_TILES] = (t1 / 1024 + 2) * 4; ssz[S_DELTA_A] = ssz[S_DELTA_B] = (t1 + 2) * 4;
    ssz[S_NODE_RANK] = (nodes + ICP_BVH_MAX_LEVELS) * 4; ssz[S_ADJ1] = (size_t)cap1 * 32 * 4; ssz[S_ADJ1_BOX] = (size_t)cap1 * 2 * sizeof(float4);
    ssz[S_ADJ_GAP] = (size_t)cap * 32 * 4; ssz[S_VOXEL] = sizeof(unsigned int) * ((size_t)1 << dmax);
    if (ensure(ctx, ctx->bi_scratch, pack_segments(ssz, S_SEGMENTS, soff), false)) return ICP_GPU_E_CUDA;
    const bool need_scratch = cfg.minimizer == ICP_GPU_MIN_LM || cfg.metric == ICP_GPU_METRIC_SYMMETRIC;
    const size_t q1 = (size_t)(ns_all > 0 ? ns_all : 1);
    const size_t psz[] = {descs.size() * sizeof(IterDesc), n_mask_words * 4, B * sizeof(MsPair), B * 4, q1 * 4, need_scratch ? q1 * sizeof(int2) : 0};
    size_t poff[6];
    if (ensure(ctx, ctx->bi_plan, pack_segments(psz, 6, poff), false)) return ICP_GPU_E_CUDA;
    char* arena = (char*)ctx->bi_arena.p; char* scr = (char*)ctx->bi_scratch.p; char* plan = (char*)ctx->bi_plan.p;
    IterDesc* desc_dev = (IterDesc*)(plan + poff[0]); unsigned int* mask_dev = (unsigned int*)(plan + poff[1]);

    // per pair: the source packed and sorted (and its VOXEL levels), the target packed, sorted and indexed
    CloudBufs sb; memset(&sb, 0, sizeof(sb));
    sb.pts = (float4*)(scr + soff[S_PTS]); sb.nrm = (float4*)(scr + soff[S_NRM]); sb.bbox = (unsigned int*)(scr + soff[S_SBBOX]);
    sb.grid = (GridParams*)(scr + soff[S_SGRID]); sb.keys_a = (unsigned int*)(scr + soff[S_SKEYS_A]); sb.keys_b = (unsigned int*)(scr + soff[S_SKEYS_B]);
    sb.idx_a = (unsigned int*)(scr + soff[S_IDX_A]); sb.idx_b = (unsigned int*)(scr + soff[S_IDX_B]); sb.hist = (unsigned int*)(scr + soff[S_HIST]);
    CloudBufs tb = sb;
    tb.bbox = nullptr; tb.grid = nullptr; tb.keys_a = tb.keys_b = nullptr;
    tb.lv_flags = (unsigned char*)(scr + soff[S_LV_FLAGS]); tb.lv_tiles = (unsigned int*)(scr + soff[S_LV_TILES]);
    tb.delta_a = (int*)(scr + soff[S_DELTA_A]); tb.delta_b = (int*)(scr + soff[S_DELTA_B]); tb.node_rank = (unsigned int*)(scr + soff[S_NODE_RANK]);
    tb.adj1 = (unsigned int*)(scr + soff[S_ADJ1]); tb.adj1_box = (float4*)(scr + soff[S_ADJ1_BOX]); tb.adj_gap = (float*)(scr + soff[S_ADJ_GAP]);
    std::vector<MsPair> pairs(B);
    int launches = 0;
    for (size_t b = 0; b < B; ++b) {
        const int ns = (int)(so[b + 1] - so[b]), nt = (int)(to[b + 1] - to[b]);
        const size_t* o = &aoff[b * A_SEGMENTS];
        const int Ts = pick_T(ns, true), T = pick_T(nt, false);
        sb.pts_sorted = (float4*)(arena + o[A_SRC_PTS]); sb.nrm_sorted = (float4*)(arena + o[A_SRC_NRM]);
        if (pack_cloud(ctx, sb, sx + 3 * so[b], sn ? sn + 3 * so[b] : nullptr, sc ? sc + 4 * so[b] : nullptr, ns, Ts, true) ||
            sort_cloud(ctx, sb, ns, Ts, nullptr, &launches))
            return ICP_GPU_E_CUDA;
        if (!plans[b].voxel_depth.empty() &&
            build_voxel_levels(ctx, plans[b], sb.pts_sorted, sb.nrm_sorted, ns, sb.grid, Ts, (unsigned int*)(scr + soff[S_VOXEL]), mask_dev + mask_at[b],
                               mask_words(ns)))
            return ICP_GPU_E_CUDA;
        tb.bbox = (unsigned int*)(arena + o[A_BBOX]); tb.grid = (GridParams*)(arena + o[A_GRID]);
        tb.keys_a = (unsigned int*)(arena + o[A_KEYS_A]); tb.keys_b = (unsigned int*)(arena + o[A_KEYS_B]); tb.msd = (unsigned int*)(arena + o[A_MSD]);
        tb.pts_sorted = (float4*)(arena + o[A_TGT_PTS]); tb.nrm_sorted = (float4*)(arena + o[A_TGT_NRM]);
        tb.leaf_start = (unsigned int*)(arena + o[A_LEAF_START]); tb.leaf_rank = (unsigned int*)(arena + o[A_LEAF_RANK]);
        tb.bvh_desc = (BvhDesc*)(arena + o[A_BVH_DESC]); tb.bvh_box = (float4*)(arena + o[A_BVH_BOX]); tb.child_start = (unsigned int*)(arena + o[A_CHILD_START]);
        tb.adj = (unsigned int*)(arena + o[A_ADJ]); tb.adj_box = (float4*)(arena + o[A_ADJ_BOX]);
        tb.adj_capacity = adj_capacity_for(nt); tb.adj1_capacity = adj1_capacity_for(nt);
        if (pack_cloud(ctx, tb, tx + 3 * to[b], tn ? tn + 3 * to[b] : nullptr, tc ? tc + 4 * to[b] : nullptr, nt, T, true) ||
            sort_cloud(ctx, tb, nt, T, nullptr, &launches) || build_tree(ctx, tb, nt, T, ctx->stream, &launches))
            return ICP_GPU_E_CUDA;
        launches += 2;                                    // the two packs
        MsPair& v = pairs[b]; memset(&v, 0, sizeof(v));
        v.src_pts = sb.pts_sorted; v.src_nrm = sb.nrm_sorted; v.n_src = ns;
        v.tgt_pts = tb.pts_sorted; v.tgt_nrm = tb.nrm_sorted; v.n_tgt = nt;
        v.bvh_box = tb.bvh_box; v.bvh = tb.bvh_desc; v.leaf_start = tb.leaf_start; v.leaf_rank = tb.leaf_rank; v.child_start = tb.child_start;
        v.adj = tb.adj; v.adj_box = tb.adj_box; v.adj_capacity = tb.adj_capacity;
        v.grid = tb.grid; v.keys = tb.keys_sorted; v.msd_start = tb.msd; v.msd_shift = tb.msd_shift; v.nonfinite = tb.bbox + 7;
        v.desc = desc_dev + desc_at[b]; v.mask = mask_dev + mask_at[b]; v.n_iters = plans[b].n_iters;
        v.q_off = so[b]; v.max_d2 = cfg.max_distance_sq;
    }
    ctx->stats.n_kernel_launches += (uint64_t)launches;

    // the plan area: descriptors, mt19937 masks (after the VOXEL levels, as upload_plan orders them), pair table, launch order
    std::vector<int> order(B);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return so[x + 1] - so[x] > so[y + 1] - so[y]; });
    {
        const void* host_in[] = {descs.data(), masks.data(), pairs.data(), order.data()};
        const size_t sizes[] = {n_desc * sizeof(IterDesc), masks.size() * 4, B * sizeof(MsPair), B * 4};
        for (int k = 0; k < 4; ++k) if (sizes[k]) CU(cudaMemcpyAsync(plan + poff[k], host_in[k], sizes[k], cudaMemcpyHostToDevice, ctx->stream));
    }
    if (ns_all > 0) CU(cudaMemsetAsync(plan + poff[4], 0xFF, (size_t)ns_all * 4, ctx->stream));     // no remembered neighbour: -1
    if (hist_floats) CU(cudaMemsetAsync(hist, 0, hist_floats * 4, ctx->stream));                   // rows past a pair's last iteration read 0

    MsArgs a; memset(&a, 0, sizeof(a));
    a.weighting = cfg.weighting; a.rejection = cfg.rejection; a.lm_max_iterations = cfg.lm_max_iterations;
    a.weight_max_d2 = cfg.weight_max_distance_sq > 0.f ? cfg.weight_max_distance_sq : cfg.max_distance_sq;
    a.stop_rot = cfg.early_stop_rotation; a.stop_trans = cfg.early_stop_translation;
    a.poses_in = pin; a.poses_out = pout; a.n_iter_out = n_it; a.status_out = st; a.inliers_out = inl; a.rmse_out = rmse;
    a.history = hist; a.history_rows = history_rows; a.match_idx = midx; a.match_w = mw;
    a.nn_pos = (int*)(plan + poff[4]); a.scratch = need_scratch ? (int2*)(plan + poff[5]) : nullptr;
    a.pairs = (const MsPair*)(plan + poff[2]); a.order = (const int*)(plan + poff[3]);
    int cluster = 1;
    CU(icp_launch_multistart(a, true, cfg.minimizer == ICP_GPU_MIN_LM ? 1 : 0, cfg.metric, cfg.color_icp ? 1 : 0, n_pairs, max_s, ctx->n_sms, ctx->stream,
                             &cluster));
    ctx->stats.n_kernel_launches += 1;
    if (!dev) {
        CU(cudaMemcpyAsync(poses_out, pout, B * 64, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(n_iterations_out, n_it, B * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(status_out, st, B * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(inliers_out, inl, B * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(rmse_out, rmse, B * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (hist_floats) CU(cudaMemcpyAsync(pose_history, hist, hist_floats * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (match_n) {
            CU(cudaMemcpyAsync(match_idx_out, midx, match_n * 4, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaMemcpyAsync(match_w_out, mw, match_n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        }
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_estimate_pose_batch_indexed(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const uint8_t* src_rgba,
                                        const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm, const uint8_t* tgt_rgba, const int64_t* tgt_off,
                                        const float* poses_in, float* poses_out, int32_t* n_iterations_out, int32_t* status_out, int64_t* inliers_out,
                                        double* rmse_out, float* pose_history, int32_t history_rows, int32_t* match_idx_out, float* match_w_out) {
    return estimate_pose_batch_indexed(ctx, n_pairs, src_xyz, src_nrm, src_rgba, src_off, tgt_xyz, tgt_nrm, tgt_rgba, tgt_off, poses_in, poses_out,
                                       n_iterations_out, status_out, inliers_out, rmse_out, pose_history, history_rows, match_idx_out, match_w_out, false);
}

int icp_gpu_estimate_pose_batch_indexed_dev(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const uint8_t* src_rgba,
                                            const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm, const uint8_t* tgt_rgba,
                                            const int64_t* tgt_off, const float* poses_in, float* poses_out, int32_t* n_iterations_out,
                                            int32_t* status_out, int64_t* inliers_out, double* rmse_out, float* pose_history, int32_t history_rows,
                                            int32_t* match_idx_out, float* match_w_out) {
    return estimate_pose_batch_indexed(ctx, n_pairs, src_xyz, src_nrm, src_rgba, src_off, tgt_xyz, tgt_nrm, tgt_rgba, tgt_off, poses_in, poses_out,
                                       n_iterations_out, status_out, inliers_out, rmse_out, pose_history, history_rows, match_idx_out, match_w_out, true);
}
