// sharded.cu -- point-sharded registration: one iteration at a time with the reduction left to the caller (icp_gpu_iteration_*), and
// the mailboxes through which the ranks' reductions exchange rows over peer memory (icp_gpu_peer_*).  Host code only.
#include "context.cuh"

void peer_close(icp_gpu_ctx* ctx) {
    for (int j = 0; j < ICP_MAX_PEERS; ++j) {
        if (ctx->peer_ipc[j] && ctx->peer_ptr[j]) { if (cudaIpcCloseMemHandle(ctx->peer_ptr[j]) != cudaSuccess) cudaGetLastError(); }
        ctx->peer_ptr[j] = nullptr; ctx->peer_ipc[j] = false;
    }
    ctx->peer_world = 0; ctx->peer_rank = 0; ctx->peer_epoch += 1;
}

// (Re)creates the mailbox in its initial state: no row received, exchange counter 0.
static int peer_reset_box(icp_gpu_ctx* ctx) {
    CU(cudaStreamSynchronize(ctx->stream));
    peer_close(ctx);
    if (!ctx->peer_box) CU(cudaMalloc(&ctx->peer_box, sizeof(PeerBox)));
    CU(cudaMemsetAsync(ctx->peer_box, 0, sizeof(PeerBox), ctx->stream));
    CU(cudaMemsetAsync(&((DevState*)ctx->state.p)->xchg_seq, 0, sizeof(unsigned int), ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int shard_values(int metric, int phase) {
    if (metric == ICP_GPU_METRIC_P2P) return 23;
    if (metric == ICP_GPU_METRIC_SYMMETRIC && phase == 0) return 7;
    return 28;
}

static int peer_attach_common(icp_gpu_ctx* ctx, int32_t rank, int32_t world, const void* handles, void* const* ptrs) {
    if (world < 1 || world > ICP_MAX_PEERS || rank < 0 || rank >= world) return fail(ctx, ICP_GPU_E_ARG, "rank %d of world %d (max %d)", rank, world, ICP_MAX_PEERS);
    if (int rc = enter(ctx)) return rc;
    if (!ctx->peer_box) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_peer_export / icp_gpu_peer_address not called");
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

int icp_gpu_iteration_phases(const icp_gpu_ctx* ctx) {
    if (!ctx) return ICP_GPU_E_ARG;
    return ctx->cfg.metric == ICP_GPU_METRIC_SYMMETRIC ? 2 : 1;
}

int icp_gpu_iteration_begin(icp_gpu_ctx* ctx, const float pose_in[16]) {
    if (!pose_in) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    if (ctx->cfg.minimizer != ICP_GPU_MIN_LINEAR) return fail(ctx, ICP_GPU_E_ARG, "the point-sharded path supports the linear minimiser only");
    if (ctx->peer_world > 1) return fail(ctx, ICP_GPU_E_STATE, "peers are attached: icp_gpu_estimate_pose is the point-sharded registration (icp_gpu_peer_detach first)");
    int rc = check_ready(ctx); if (rc) return rc;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    const IterDesc d = all_points_desc();
    for (int i = 0; i < ICP_MAX_ITERS; ++i) ctx->h_desc[i] = d;      // every iteration of the shard loop: all points
    CU(cudaMemcpyAsync(ctx->desc.p, ctx->h_desc, sizeof(IterDesc) * ICP_MAX_ITERS, cudaMemcpyHostToDevice, ctx->stream));
    if (upload_pose(ctx, pose_in)) return ICP_GPU_E_CUDA;
    ctx->shard_open = true; ctx->shard_algo = choose_algorithm(ctx); ctx->shard_iters = 0;
    rc = refresh_seeds(ctx, ctx->shard_algo, true); if (rc) return rc;
    return ICP_GPU_OK;
}

int icp_gpu_iteration_local_dev(icp_gpu_ctx* ctx, int phase, double** partials_dev, int32_t* n_values) {
    if (!partials_dev || !n_values) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx, false)) return rc;
    if (!ctx->shard_open) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_iteration_begin not called");
    if (phase < 0 || phase >= icp_gpu_iteration_phases(ctx)) return fail(ctx, ICP_GPU_E_ARG, "phase %d", phase);
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
    if (int rc = icp_gpu_iteration_local_dev(ctx, phase, &dev, n_values)) return rc;
    CU(cudaMemcpyAsync(partials_out, dev, sizeof(double) * (size_t)*n_values, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_iteration_apply_dev(icp_gpu_ctx* ctx, int phase) {
    if (int rc = enter(ctx, false)) return rc;
    if (!ctx->shard_open) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_iteration_begin not called");
    if (phase < 0 || phase >= icp_gpu_iteration_phases(ctx)) return fail(ctx, ICP_GPU_E_ARG, "phase %d", phase);
    const int mode = ctx->cfg.metric == ICP_GPU_METRIC_SYMMETRIC ? (phase == 0 ? 3 : 2) : ctx->cfg.metric;
    CU(icp_launch_shard_apply((DevState*)ctx->state.p, mode, (float*)ctx->history.p, ctx->stream));
    ctx->stats.n_kernel_launches += 1;
    return ICP_GPU_OK;
}

int icp_gpu_iteration_apply(icp_gpu_ctx* ctx, int phase, const double* reduced_in, int32_t n_values) {
    if (!reduced_in) return ICP_GPU_E_ARG;
    if (n_values < 0 || n_values > ICP_GPU_MAX_PARTIALS) return fail(ctx, ICP_GPU_E_ARG, "n_values %d", n_values);
    if (int rc = enter(ctx, false)) return rc;
    if (!ctx->shard_open) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_iteration_begin not called");
    CU(cudaMemcpyAsync(((DevState*)ctx->state.p)->shard_partials, reduced_in, sizeof(double) * (size_t)n_values, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));   // reduced_in is pageable caller memory
    return icp_gpu_iteration_apply_dev(ctx, phase);
}

int icp_gpu_iteration_end(icp_gpu_ctx* ctx, float pose_out[16]) {
    if (!pose_out) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx, false)) return rc;
    if (!ctx->shard_open) return fail(ctx, ICP_GPU_E_STATE, "icp_gpu_iteration_begin not called");
    ctx->shard_open = false;
    CU(cudaMemcpyAsync(ctx->h_state, ctx->state.p, sizeof(DevState), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    memcpy(pose_out, ctx->h_state->pose, 16 * sizeof(float));
    return status_error(ctx, ctx->h_state->status, -1, "no surviving correspondence on any rank");
}

int icp_gpu_peer_export(icp_gpu_ctx* ctx, void* handle_out) {
    if (!handle_out) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    static_assert(sizeof(cudaIpcMemHandle_t) == ICP_GPU_PEER_HANDLE_BYTES, "handle size");
    if (peer_reset_box(ctx)) return ICP_GPU_E_CUDA;
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, ctx->peer_box));
    memcpy(handle_out, &h, sizeof(h));
    return ICP_GPU_OK;
}

int icp_gpu_peer_address(icp_gpu_ctx* ctx, void** mailbox_dev) {
    if (!mailbox_dev) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    if (peer_reset_box(ctx)) return ICP_GPU_E_CUDA;
    *mailbox_dev = ctx->peer_box;
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
    if (int rc = enter(ctx)) return rc;
    CU(cudaStreamSynchronize(ctx->stream));
    peer_close(ctx);
    return ICP_GPU_OK;
}
