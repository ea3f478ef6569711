// multistart_api.cu -- the host side of multi-start registration (icp_gpu_estimate_pose_multistart[_dev]): the checks, the plan and
// the one launch.  Host code only; the kernel lives in multistart.cu.
#include "context.cuh"

// dev = false: every array is a host array, the poses uploaded into ms_io and the results copied back; dev = true: every array is a
// device array on the context's device, read and written in place.  Either way the call waits for the launch.
static int estimate_pose_multistart(icp_gpu_ctx* ctx, int32_t n_starts, const float* poses_in, float* poses_out, int32_t* n_iterations_out,
                                    int32_t* status_out, int64_t* inliers_out, double* rmse_out, float* pose_history, int32_t* match_idx_out,
                                    float* match_w_out, bool dev) {
    if (int rc = enter(ctx)) return rc;
    if (n_starts < 0) return fail(ctx, ICP_GPU_E_ARG, "multistart: n_starts %d", n_starts);
    if (n_starts > 0 && (!poses_in || !poses_out || !n_iterations_out || !status_out || !inliers_out || !rmse_out))
        return fail(ctx, ICP_GPU_E_ARG, "multistart: poses_in, poses_out, n_iterations_out, status_out, inliers_out and rmse_out are required");
    if ((match_idx_out == nullptr) != (match_w_out == nullptr)) return fail(ctx, ICP_GPU_E_ARG, "multistart: match_idx_out and match_w_out go together");
    const icp_gpu_config& cfg = ctx->cfg;
    if (cfg.matching != ICP_GPU_MATCH_KNN) return fail(ctx, ICP_GPU_E_ARG, "multistart: k-NN matching only (projective matching runs through icp_gpu_estimate_pose)");
    if (cfg.nn_algorithm == ICP_GPU_NN_BRUTE_NORM) return fail(ctx, ICP_GPU_E_ARG, "multistart: squared-distance matching only (no norm-thresholded brute force)");
    if (ctx->peer_world > 1) return fail(ctx, ICP_GPU_E_ARG, "multistart: the context has attached peers (point-sharded registration runs through icp_gpu_estimate_pose)");
    if (int rc = check_ready(ctx)) return rc;
    const int n = ctx->n_src;
    if ((long long)n_starts * n > 0x7fffffffll)
        return fail(ctx, ICP_GPU_E_ARG, "multistart: %d starts x %d source points exceed INT32_MAX (query, start) pairs", n_starts, n);
    if (n_starts == 0) return ICP_GPU_OK;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    Plan plan;
    if (int rc = make_plan(ctx, plan)) return rc;
    if (ensure(ctx, ctx->ms_desc, sizeof(IterDesc) * (size_t)(plan.n_iters > 0 ? plan.n_iters : 1), false)) return ICP_GPU_E_CUDA;
    if (int rc = upload_plan(ctx, plan, (IterDesc*)ctx->ms_desc.p, ctx->ms_mask, false)) return rc;
    const size_t K = (size_t)n_starts, pairs = K * (size_t)n;
    const bool lm = cfg.minimizer == ICP_GPU_MIN_LM;
    const bool need_scratch = lm || cfg.metric == ICP_GPU_METRIC_SYMMETRIC;
    if (ensure(ctx, ctx->ms_nn, (pairs > 0 ? pairs : 1) * 4, false)) return ICP_GPU_E_CUDA;
    if (need_scratch && ensure(ctx, ctx->ms_scratch, (pairs > 0 ? pairs : 1) * sizeof(int2), false)) return ICP_GPU_E_CUDA;
    if (pairs > 0) CU(cudaMemsetAsync(ctx->ms_nn.p, 0xFF, pairs * 4, ctx->stream));      // no remembered neighbour: -1

    MsArgs a; memset(&a, 0, sizeof(a));
    a.src_pts = (const float4*)ctx->src_pts.p; a.src_nrm = (const float4*)ctx->src_nrm.p; a.n_src = n;
    a.tgt_pts = (const float4*)ctx->tgt_pts_sorted.p; a.tgt_nrm = (const float4*)ctx->tgt_nrm_sorted.p; a.n_tgt = ctx->n_tgt;
    a.bvh_box = (const float4*)ctx->bvh_box.p; a.bvh = (const BvhDesc*)ctx->bvh_desc.p; a.leaf_start = (const unsigned int*)ctx->leaf_start.p;
    a.leaf_rank = (const unsigned int*)ctx->leaf_rank.p; a.child_start = (const unsigned int*)ctx->child_start.p;
    a.adj = (const unsigned int*)ctx->adj.p; a.adj_box = (const float4*)ctx->adj_box.p; a.adj_capacity = ctx->adj_capacity;
    a.grid = (const GridParams*)ctx->grid.p; a.keys = ctx->tsort.keys_sorted; a.msd_start = (const unsigned int*)ctx->tsort.msd.p;
    a.msd_shift = ctx->tsort.msd_shift; a.nonfinite = (const unsigned int*)ctx->bbox.p + 7;
    a.desc = (const IterDesc*)ctx->ms_desc.p; a.mask = (const unsigned int*)ctx->ms_mask.p; a.n_iters = plan.n_iters;
    a.weighting = cfg.weighting; a.rejection = cfg.rejection; a.lm_max_iterations = cfg.lm_max_iterations;
    a.max_d2 = cfg.max_distance_sq;
    a.weight_max_d2 = cfg.weight_max_distance_sq > 0.f ? cfg.weight_max_distance_sq : cfg.max_distance_sq;
    a.stop_rot = cfg.early_stop_rotation; a.stop_trans = cfg.early_stop_translation;
    a.history_rows = plan.n_iters;
    a.nn_pos = (int*)ctx->ms_nn.p; a.scratch = need_scratch ? (int2*)ctx->ms_scratch.p : nullptr;
    const size_t hist_floats = pose_history ? K * (size_t)plan.n_iters * 16 : 0;
    const size_t match_n = match_idx_out ? pairs : 0;
    if (dev) {
        a.poses_in = poses_in; a.poses_out = poses_out; a.n_iter_out = n_iterations_out; a.status_out = status_out;
        a.inliers_out = (long long*)inliers_out; a.rmse_out = rmse_out; a.history = pose_history;
        a.match_idx = match_idx_out; a.match_w = match_w_out;
    } else {
        // one area: the poses in, then the results the kernel writes
        const size_t sizes[] = {K * 64, K * 64, K * 4, K * 4, K * 8, K * 8, hist_floats * 4, match_n * 4, match_n * 4};
        size_t off[9];
        if (ensure(ctx, ctx->ms_io, pack_segments(sizes, 9, off), false)) return ICP_GPU_E_CUDA;
        char* base = (char*)ctx->ms_io.p;
        CU(cudaMemcpyAsync(base + off[0], poses_in, sizes[0], cudaMemcpyHostToDevice, ctx->stream));
        a.poses_in = (const float*)(base + off[0]); a.poses_out = (float*)(base + off[1]); a.n_iter_out = (int*)(base + off[2]);
        a.status_out = (int*)(base + off[3]); a.inliers_out = (long long*)(base + off[4]); a.rmse_out = (double*)(base + off[5]);
        a.history = pose_history ? (float*)(base + off[6]) : nullptr;
        a.match_idx = match_n ? (int*)(base + off[7]) : nullptr; a.match_w = match_n ? (float*)(base + off[8]) : nullptr;
    }
    if (hist_floats) CU(cudaMemsetAsync(a.history, 0, hist_floats * 4, ctx->stream));   // rows past a start's last iteration read 0
    int cluster = 1;
    CU(icp_launch_multistart(a, false, lm ? 1 : 0, cfg.metric, cfg.color_icp ? 1 : 0, n_starts, n, ctx->n_sms, ctx->stream, &cluster));
    ctx->stats.n_kernel_launches += 1;
    if (!dev) {
        CU(cudaMemcpyAsync(poses_out, a.poses_out, K * 64, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(n_iterations_out, a.n_iter_out, K * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(status_out, a.status_out, K * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(inliers_out, a.inliers_out, K * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(rmse_out, a.rmse_out, K * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (hist_floats) CU(cudaMemcpyAsync(pose_history, a.history, hist_floats * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (match_n) {
            CU(cudaMemcpyAsync(match_idx_out, a.match_idx, match_n * 4, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaMemcpyAsync(match_w_out, a.match_w, match_n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        }
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_estimate_pose_multistart(icp_gpu_ctx* ctx, int32_t n_starts, const float* poses_in, float* poses_out, int32_t* n_iterations_out,
                                     int32_t* status_out, int64_t* inliers_out, double* rmse_out, float* pose_history, int32_t* match_idx_out,
                                     float* match_w_out) {
    return estimate_pose_multistart(ctx, n_starts, poses_in, poses_out, n_iterations_out, status_out, inliers_out, rmse_out, pose_history,
                                    match_idx_out, match_w_out, false);
}

int icp_gpu_estimate_pose_multistart_dev(icp_gpu_ctx* ctx, int32_t n_starts, const float* poses_in, float* poses_out, int32_t* n_iterations_out,
                                         int32_t* status_out, int64_t* inliers_out, double* rmse_out, float* pose_history, int32_t* match_idx_out,
                                         float* match_w_out) {
    return estimate_pose_multistart(ctx, n_starts, poses_in, poses_out, n_iterations_out, status_out, inliers_out, rmse_out, pose_history,
                                    match_idx_out, match_w_out, true);
}
