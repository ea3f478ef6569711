// values.cu -- the reference API's value-level operations outside the loop (transforms, correspondence weights, one linear solve)
// and the convergence metrics (ConvergenceMeasure) over known correspondences.  Host code only.
#include "context.cuh"

// host array -> scratch slot k of the context (nullable in, nullptr out)
static int up(icp_gpu_ctx* ctx, int k, const void* host, size_t bytes, void** dev) {
    *dev = nullptr;
    if (!host || bytes == 0) return 0;
    if (ensure(ctx, ctx->scratch[k], bytes)) return ICP_GPU_E_CUDA;
    CU(cudaMemcpyAsync(ctx->scratch[k].p, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dev = ctx->scratch[k].p;
    return 0;
}

static int transform_common(icp_gpu_ctx* ctx, const float pose[16], const float* in, int64_t n, float* out, int normals) {
    if (!pose || n < 0 || (n > 0 && (!in || !out))) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    if (n == 0) return ICP_GPU_OK;
    void* din = nullptr;
    if (up(ctx, 0, in, (size_t)n * 12, &din) || ensure(ctx, ctx->scratch[1], (size_t)n * 12)) return ICP_GPU_E_CUDA;
    CU(icp_launch_transform((const float*)din, (long long)n, pose, normals, (float*)ctx->scratch[1].p, ctx->stream));
    ctx->stats.n_kernel_launches += 1;
    CU(cudaMemcpyAsync(out, ctx->scratch[1].p, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ICP_GPU_OK;
}

int icp_gpu_transform_points(icp_gpu_ctx* ctx, const float pose[16], const float* xyz_in, int64_t n, float* xyz_out) {
    return transform_common(ctx, pose, xyz_in, n, xyz_out, 0);
}
int icp_gpu_transform_normals(icp_gpu_ctx* ctx, const float pose[16], const float* nrm_in, int64_t n, float* nrm_out) {
    return transform_common(ctx, pose, nrm_in, n, nrm_out, 1);
}

int icp_gpu_apply_weights(icp_gpu_ctx* ctx, int32_t weighting, float max_distance_sq, const float* src_xyz, const float* src_nrm, const uint8_t* src_rgba,
                          int64_t n_src, const float* tgt_xyz, const float* tgt_nrm, const uint8_t* tgt_rgba, int64_t n_tgt, const int32_t* idx,
                          float* weight_inout) {
    if (n_src < 0 || n_tgt < 0 || (n_src > 0 && (!src_xyz || !idx || !weight_inout)) || (n_tgt > 0 && !tgt_xyz)) return ICP_GPU_E_ARG;
    if (weighting < 0 || weighting > 3) return fail(ctx, ICP_GPU_E_ARG, "weighting %d", weighting);
    if (int rc = enter(ctx)) return rc;
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
    if (!pose_out || n < 0 || n > 0x7fffffff / 4 || (n > 0 && (!src_xyz || !tgt_xyz))) return ICP_GPU_E_ARG;
    if (metric < 0 || metric > 2) return fail(ctx, ICP_GPU_E_ARG, "metric %d", metric);
    if (metric == ICP_GPU_METRIC_P2PLANE && n > 0 && !tgt_nrm) return fail(ctx, ICP_GPU_E_ARG, "point-to-plane needs the target normals");
    if (metric == ICP_GPU_METRIC_SYMMETRIC && n > 0 && (!tgt_nrm || !src_nrm)) return fail(ctx, ICP_GPU_E_ARG, "the symmetric metric needs both normals");
    if (int rc = enter(ctx)) return rc;
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
    if (upload_pose(ctx, eye)) return ICP_GPU_E_CUDA;
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
    if (int rc = status_error(ctx, ctx->h_state->status, -1, "no finite correspondence")) return rc;
    memcpy(pose_out, ctx->h_state->pose, 16 * sizeof(float));
    return ICP_GPU_OK;
}

// ConvergenceMeasure(sourcePoints, unchangedPoints) (ConvergenceMeasure.h:32-41): the known correspondences.
int icp_gpu_set_correspondences(icp_gpu_ctx* ctx, const float* src_xyz, const float* ref_xyz, int64_t m) {
    if (m < 0 || (m > 0 && (!src_xyz || !ref_xyz))) return fail(ctx, ICP_GPU_E_ARG, "bad correspondences (m=%lld)", (long long)m);
    if (int rc = enter(ctx, false)) return rc;
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
    if (!gt_pose) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    if (ctx->n_src <= 0 || !ctx->src_raw_pts.p) return fail(ctx, ICP_GPU_E_STATE, "no source cloud set");
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
    if (!rmse_out) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    if (ctx->n_gt <= 0) return fail(ctx, ICP_GPU_E_STATE, "no correspondences set (icp_gpu_set_correspondences)");
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
    if (!pose || !rmse_out) return ICP_GPU_E_ARG;
    if (int rc = enter(ctx)) return rc;
    if (ctx->n_gt <= 0) return fail(ctx, ICP_GPU_E_STATE, "no correspondences set (icp_gpu_set_correspondences)");
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
