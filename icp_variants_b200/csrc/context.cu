// context.cu -- the context (icp_gpu_create / _destroy, streams, configuration, camera, statistics) and the steps every entry
// point shares (context.cuh).  Host code only.
#include "context.cuh"
#include <stdarg.h>
#include <stdio.h>
#include <new>

int fail(icp_gpu_ctx* c, int code, const char* fmt, ...) {
    if (c) {
        va_list ap; va_start(ap, fmt);
        vsnprintf(c->err, sizeof(c->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

int ensure(icp_gpu_ctx* ctx, DeviceBuf& b, size_t bytes, bool graph_reads) {
    if (bytes <= b.cap && b.p) return 0;
    if (graph_reads && ctx->graph_exec) { cudaGraphExecDestroy(ctx->graph_exec); ctx->graph_exec = nullptr; ctx->graph_key.clear(); }
    if (b.p) { cudaStreamSynchronize(ctx->stream); if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream); if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream); cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    CU(cudaMalloc(&b.p, want));
    b.cap = want;
    return 0;
}

int enter(icp_gpu_ctx* ctx, bool idle) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (idle && ctx->pending) return fail(ctx, ICP_GPU_E_STATE, "a registration is pending; call icp_gpu_estimate_pose_finish first");
    CU(cudaSetDevice(ctx->device));
    return 0;
}

int join_index(icp_gpu_ctx* ctx) {
    if (!ctx->index_pending) return 0;
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_index_ready, 0));
    ctx->index_pending = false;
    return 0;
}

int upload_pose(icp_gpu_ctx* ctx, const float pose[16], float stop_rot, float stop_trans) {
    memcpy(ctx->h_pose, pose, 16 * sizeof(float));
    CU(cudaMemcpyAsync(ctx->pose_dev.p, ctx->h_pose, 16 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CU(icp_launch_pose_init((DevState*)ctx->state.p, (const float*)ctx->pose_dev.p, ctx->stream, stop_rot, stop_trans));
    return 0;
}

int status_error(icp_gpu_ctx* ctx, int status, int iteration, const char* no_match) {
    if (status == 0) return ICP_GPU_OK;
    if (status == ICP_GPU_E_NO_MATCHES) return fail(ctx, status, no_match, iteration);
    if (status == ICP_GPU_E_PEER)
        return fail(ctx, status, "point-sharded registration: a peer's row did not arrive in time (iteration %d; rank %d of %d)", iteration, ctx->peer_rank, ctx->peer_world);
    if (iteration < 0) return fail(ctx, status, "singular / non-finite normal equations");
    return fail(ctx, status, "iteration %d: singular / non-finite normal equations", iteration);
}

size_t pack_segments(const size_t* sizes, int n, size_t* off) {
    size_t total = 0;
    for (int k = 0; k < n; ++k) { off[k] = total; total += (sizes[k] + 255) / 256 * 256; }
    return total;
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
    delete ctx;                                              // the DeviceBufs free themselves
    return ICP_GPU_OK;
}

const char* icp_gpu_last_error(const icp_gpu_ctx* ctx) { return ctx ? ctx->err : "null context"; }

int icp_gpu_set_stream(icp_gpu_ctx* ctx, void* cuda_stream) {
    if (int rc = enter(ctx)) return rc;
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaStreamSynchronize(ctx->aux_stream));
    ctx->index_pending = false;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return ICP_GPU_OK;
}

int icp_gpu_synchronize(icp_gpu_ctx* ctx) {
    if (int rc = enter(ctx, false)) return rc;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_set_config(icp_gpu_ctx* ctx, const icp_gpu_config* c) {
    if (!ctx || !c) return ICP_GPU_E_ARG;
    if (int rc = check_config(ctx, c, "")) return rc;
    ctx->cfg = *c;
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

int icp_gpu_get_stats(icp_gpu_ctx* ctx, icp_gpu_stats* out) {
    if (!ctx || !out) return ICP_GPU_E_ARG;
    *out = ctx->stats;
    return ICP_GPU_OK;
}

int icp_gpu_measure_fp32_peak(icp_gpu_ctx* ctx, int32_t mode, double* tflops_out) {
    if (!tflops_out || mode < 0 || mode > 1) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    CU(icp_measure_fp32_peak(mode, ctx->n_sms, ctx->stream, tflops_out));
    return ICP_GPU_OK;
}
