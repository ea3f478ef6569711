// batch_api.cu -- the host side of batched registration of small pairs (icp_gpu_estimate_pose_batch[_configs][_dev]): the checks,
// the mt19937 masks, the upload and the one launch per (minimiser, metric) group.  Host code only; the kernels live in batch.cu.
#include "context.cuh"
#include <stdio.h>
#include <map>
#include <string>

// dev = false: every array is a host array, uploaded into batch_io and the results copied back; dev = true: every per-pair array is a
// device array on the context's device, read and written in place.  Either way the call waits for the batch.  config_index null:
// every pair runs with configs[0] (icp_gpu_estimate_pose_batch).
static int estimate_pose_batch_configs(icp_gpu_ctx* ctx, int32_t n_configs, const icp_gpu_config* configs, int32_t n_pairs, const int32_t* config_index,
                                const float* src_xyz, const float* src_nrm, const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm,
                                const int64_t* tgt_off, const float* poses_in, float* poses_out, int32_t* n_iterations_out, int32_t* status_out,
                                float* pose_history, int32_t history_rows, bool dev) {
    if (n_configs < 1 || !configs) return fail(ctx, ICP_GPU_E_ARG, "batch: %d configs (at least one is needed)", n_configs);
    char who[32];
    for (int k = 0; k < n_configs; ++k) {
        const icp_gpu_config& c = configs[k];
        snprintf(who, sizeof(who), "batch: config %d: ", k);
        if (int rc = check_config(ctx, &c, who)) return rc;
        if (c.matching != ICP_GPU_MATCH_KNN) return fail(ctx, ICP_GPU_E_ARG, "%sk-NN matching only (projective matching runs through icp_gpu_estimate_pose)", who);
        if (c.color_icp) return fail(ctx, ICP_GPU_E_ARG, "%s3-D matching only (colour ICP runs through icp_gpu_estimate_pose)", who);
        if (c.nn_algorithm == ICP_GPU_NN_BRUTE_NORM) return fail(ctx, ICP_GPU_E_ARG, "%ssquared-distance matching only (no norm-thresholded brute force)", who);
        if (c.multires && c.pyramid_mode == ICP_GPU_PYRAMID_VOXEL) return fail(ctx, ICP_GPU_E_ARG, "%sthe STRIDE pyramid only (the VOXEL pyramid runs through icp_gpu_estimate_pose)", who);
    }
    if (history_rows < 0) return fail(ctx, ICP_GPU_E_ARG, "batch: history_rows %d", history_rows);
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
                for (long long k = 0; k < n; ++k) finite[(size_t)k] = point_finite(sp + 3 * (so[b] + k), sn ? sn + 3 * (so[b] + k) : nullptr) ? 1 : 0;
                key.append((const char*)finite.data(), finite.size());
            }
            auto it = shared.find(key);
            if (it != shared.end()) { mask_off[b] = it->second; continue; }
            const IcpSchedule sch = icp_schedule(c.n_iterations, c.multires, n);
            mask_off[b] = (long long)masks.size();
            masks.resize(masks.size() + (size_t)sch.n_iters * mask_words(n), 0u);
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
        // one upload area: inputs, then the results the kernel writes
        const size_t sizes[] = {(size_t)ns * 12, src_nrm ? (size_t)ns * 12 : 0, (size_t)nt * 12, tgt_nrm ? (size_t)nt * 12 : 0, (B + 1) * 8, (B + 1) * 8,
                                B * 64, B * 64, B * 4, B * 4, hist_floats * 4};
        const void* host_in[] = {src_xyz, src_nrm, tgt_xyz, tgt_nrm, src_off, tgt_off, poses_in};
        size_t off[11];
        if (ensure(ctx, ctx->batch_io, pack_segments(sizes, 11, off), false)) return ICP_GPU_E_CUDA;
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
        size_t off[5];
        if (ensure(ctx, ctx->batch_plan, pack_segments(sizes, 5, off), false)) return ICP_GPU_E_CUDA;
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

static int batch_common_checks(icp_gpu_ctx* ctx, int32_t n_pairs, const int64_t* src_off, const int64_t* tgt_off, const float* poses_in, float* poses_out,
                        int32_t* n_iterations_out, int32_t* status_out) {
    if (n_pairs < 0) return fail(ctx, ICP_GPU_E_ARG, "n_pairs %d", n_pairs);
    if (!src_off || !tgt_off || !poses_in || !poses_out || !n_iterations_out || !status_out)
        return fail(ctx, ICP_GPU_E_ARG, "batch: offsets, poses_in, poses_out, n_iterations_out and status_out are required");
    return enter(ctx);
}

// The context's configuration for every pair, with the refusals this entry point has always had.
static int estimate_pose_batch(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                        const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in, float* poses_out,
                        int32_t* n_iterations_out, int32_t* status_out, float* pose_history, bool dev) {
    if (int rc = batch_common_checks(ctx, n_pairs, src_off, tgt_off, poses_in, poses_out, n_iterations_out, status_out)) return rc;
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

static int estimate_pose_batch_configs_entry(icp_gpu_ctx* ctx, int32_t n_configs, const icp_gpu_config* configs, int32_t n_pairs, const int32_t* config_index,
                                      const float* src_xyz, const float* src_nrm, const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm,
                                      const int64_t* tgt_off, const float* poses_in, float* poses_out, int32_t* n_iterations_out, int32_t* status_out,
                                      float* pose_history, int32_t history_rows, bool dev) {
    if (int rc = batch_common_checks(ctx, n_pairs, src_off, tgt_off, poses_in, poses_out, n_iterations_out, status_out)) return rc;
    if (!config_index) return fail(ctx, ICP_GPU_E_ARG, "batch: config_index is required");
    return estimate_pose_batch_configs(ctx, n_configs, configs, n_pairs, config_index, src_xyz, src_nrm, src_off, tgt_xyz, tgt_nrm, tgt_off, poses_in,
                                       poses_out, n_iterations_out, status_out, pose_history, history_rows, dev);
}

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
