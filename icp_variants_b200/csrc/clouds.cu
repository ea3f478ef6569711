// clouds.cu -- the context's clouds: upload, the target's index build (buildIndex) and the source's sort, clouds from depth maps
// and PCA normals of the target.  Host code only; the kernels live in grid.cu, prep.cu and normals.cu.
#include "context.cuh"

int pick_T(int n, bool source) {
    // Target: the finest grid the 32-bit keys hold (10 bits per axis) -- the radix sort costs the same for any T, and fine
    // cells give compact leaves.  Source: 4 cells per point; its grid also defines the voxel pyramid levels, which the
    // oracle restates (oracle/icp_oracle.c:orc_pick_T).
    if (!source) return 3 * ICP_MAX_BITS_PER_AXIS;
    int T = 3;
    while (T < 24 && (1ll << T) < (long long)ICP_SOURCE_CELLS_PER_POINT * (long long)(n > 0 ? n : 1)) ++T;
    if (T > 3 * ICP_MAX_BITS_PER_AXIS) T = 3 * ICP_MAX_BITS_PER_AXIS;
    return T;
}

static int ensure_sort(icp_gpu_ctx* ctx, icp_gpu_ctx::SortBufs& sb, int n, int T) {
    const size_t n1 = (size_t)(n > 0 ? n : 1);
    if (ensure(ctx, sb.keys_a, n1 * 4) || ensure(ctx, sb.keys_b, n1 * 4) || ensure(ctx, sb.idx_a, n1 * 4) || ensure(ctx, sb.idx_b, n1 * 4) ||
        ensure(ctx, sb.hist, icp_radix_hist_words(n, T) * 4) || ensure(ctx, sb.msd, ICP_MSD_WORDS * 4)) return ICP_GPU_E_CUDA;
    return 0;
}

// The context's buffers of one cloud as a CloudBufs (kind 0: the target with its index, 1: the source).
static CloudBufs context_bufs(icp_gpu_ctx* ctx, int kind) {
    CloudBufs b; memset(&b, 0, sizeof(b));
    icp_gpu_ctx::SortBufs& sb = kind == 0 ? ctx->tsort : ctx->ssort;
    b.pts = (float4*)(kind == 0 ? ctx->tgt_pts.p : ctx->src_raw_pts.p); b.nrm = (float4*)(kind == 0 ? ctx->tgt_nrm.p : ctx->src_raw_nrm.p);
    b.bbox = (unsigned int*)(kind == 0 ? ctx->bbox.p : ctx->sbbox.p); b.grid = (GridParams*)(kind == 0 ? ctx->grid.p : ctx->sgrid.p);
    b.keys_a = (unsigned int*)sb.keys_a.p; b.keys_b = (unsigned int*)sb.keys_b.p; b.idx_a = (unsigned int*)sb.idx_a.p; b.idx_b = (unsigned int*)sb.idx_b.p;
    b.hist = (unsigned int*)sb.hist.p; b.msd = kind == 0 ? (unsigned int*)sb.msd.p : nullptr;
    b.pts_sorted = (float4*)(kind == 0 ? ctx->tgt_pts_sorted.p : ctx->src_pts.p); b.nrm_sorted = (float4*)(kind == 0 ? ctx->tgt_nrm_sorted.p : ctx->src_nrm.p);
    if (kind == 0) {
        b.lv_flags = (unsigned char*)ctx->lv_flags.p; b.lv_tiles = (unsigned int*)ctx->lv_tiles.p; b.delta_a = (int*)ctx->delta_a.p; b.delta_b = (int*)ctx->delta_b.p;
        b.leaf_start = (unsigned int*)ctx->leaf_start.p; b.leaf_rank = (unsigned int*)ctx->leaf_rank.p; b.node_rank = (unsigned int*)ctx->node_rank.p;
        b.child_start = (unsigned int*)ctx->child_start.p; b.bvh_desc = (BvhDesc*)ctx->bvh_desc.p; b.bvh_box = (float4*)ctx->bvh_box.p;
        b.adj = (unsigned int*)ctx->adj.p; b.adj_box = (float4*)ctx->adj_box.p; b.adj_gap = (float*)ctx->adj_gap.p; b.adj_capacity = ctx->adj_capacity;
        b.adj1 = (unsigned int*)ctx->adj1.p; b.adj1_box = (float4*)ctx->adj1_box.p; b.adj1_capacity = ctx->adj1_capacity;
    }
    b.keys_sorted = sb.keys_sorted; b.msd_shift = sb.msd_shift;
    return b;
}

int pack_cloud(icp_gpu_ctx* ctx, CloudBufs& b, const float* xyz, const float* nrm, const uint8_t* rgba, int n, int T, bool with_normals) {
    const long long hist_words = (long long)icp_radix_hist_words(n, T);
    if (n == 0) CU(icp_launch_pack_cloud(nullptr, nullptr, nullptr, 0, b.pts, b.nrm, b.bbox, T, b.grid, b.hist, hist_words, 1, ctx->stream));
    else CU(icp_launch_pack_cloud(xyz, nrm, rgba, n, b.pts, b.nrm, b.bbox, T, b.grid, b.hist, hist_words, with_normals ? 1 : 0, ctx->stream));
    return 0;
}

int sort_cloud(icp_gpu_ctx* ctx, CloudBufs& b, int n, int T, const IcpLatePack* late, int* launches) {
    CU(icp_launch_cloud_sort(b.pts, b.nrm, n, T, b.grid, b.keys_a, b.keys_b, b.idx_a, b.idx_b, b.hist, b.pts_sorted, b.nrm_sorted, b.msd,
                             &b.keys_sorted, &b.msd_shift, late, ctx->stream, launches));
    return 0;
}

// The index over a sorted target (after sort_cloud): tree levels, tight boxes, adjacency lists, on stream s.
int build_tree(icp_gpu_ctx* ctx, const CloudBufs& b, int n, int T, cudaStream_t s, int* launches) {
    CU(icp_launch_bvh_build(b.pts_sorted, b.nrm_sorted, n, T, b.keys_sorted, b.bbox + 7, b.lv_flags, b.lv_tiles, b.delta_a, b.delta_b, b.leaf_rank,
                            b.leaf_start, b.node_rank, b.child_start, b.bvh_desc, b.bvh_box, ctx->n_sms, s, launches));
    CU(icp_launch_leaf_adjacency(b.bvh_desc, b.bvh_box, b.child_start, b.adj1, b.adj1_box, b.adj1_capacity, 1, nullptr, nullptr, nullptr, 0, ctx->n_sms, s,
                                 launches, nullptr));
    CU(icp_launch_leaf_adjacency(b.bvh_desc, b.bvh_box, b.child_start, b.adj, b.adj_box, b.adj_capacity, 0, b.node_rank, b.adj1, b.adj1_box,
                                 b.adj1_capacity, ctx->n_sms, s, launches, b.adj_gap));
    return 0;
}

static int upload_cloud(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n, bool device_ptrs,
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
    CloudBufs b = context_bufs(ctx, kind);
    if (n == 0) {
        if (pack_cloud(ctx, b, nullptr, nullptr, nullptr, 0, T, true)) return ICP_GPU_E_CUDA;
        ctx->late_pending[kind] = false;
        return 0;
    }
    const float* dx = xyz; const float* dn = nrm; const uint8_t* dc = rgba;
    if (!device_ptrs) {
        // Host arrays go through a per-cloud staging area on the copy stream, so that the upload of one cloud overlaps
        // the index build of the other on the compute stream.
        DeviceBuf& stage = kind == 0 ? ctx->stage : ctx->stage2;
        const size_t sizes[] = {(size_t)n * 12, nrm ? (size_t)n * 12 : 0, rgba ? (size_t)n * 4 : 0};   // points, normals, colours
        size_t off[3];
        if (ensure(ctx, stage, pack_segments(sizes, 3, off))) return ICP_GPU_E_CUDA;
        char* st = (char*)stage.p;
        if (ctx->packed_once[kind]) CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_packed[kind], 0));   // staging still being read?
        CU(cudaMemcpyAsync(st + off[0], xyz, sizes[0], cudaMemcpyHostToDevice, ctx->copy_stream));
        CU(cudaEventRecord(ctx->ev_xyz[kind], ctx->copy_stream));       // the sort starts from the points alone
        dx = (const float*)(st + off[0]);
        if (nrm) { CU(cudaMemcpyAsync(st + off[1], nrm, sizes[1], cudaMemcpyHostToDevice, ctx->copy_stream)); dn = (const float*)(st + off[1]); }
        if (rgba) { CU(cudaMemcpyAsync(st + off[2], rgba, sizes[2], cudaMemcpyHostToDevice, ctx->copy_stream)); dc = (const uint8_t*)(st + off[2]); }
        CU(cudaEventRecord(ctx->ev_copied[kind], ctx->copy_stream));
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_xyz[kind], 0));
        // the normal / colour records are packed by the sort just before its last pass (the only one that moves them)
        ctx->late[kind].nrm = dn; ctx->late[kind].rgba = dc; ctx->late[kind].nrmo = (float4*)nrmb.p; ctx->late[kind].ready = ctx->ev_copied[kind];
    }
    ctx->late_pending[kind] = !device_ptrs;
    if (pack_cloud(ctx, b, dx, dn, dc, (int)n, T, device_ptrs)) return ICP_GPU_E_CUDA;
    ctx->stats.n_kernel_launches += 1;
    return 0;
}

// buildIndex: radix sort by cell code, leaves and upper levels from the sorted keys, tight boxes, adjacency lists.
static int build_grid(icp_gpu_ctx* ctx) {
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
    ctx->adj_capacity = adj_capacity_for(n);
    ctx->adj1_capacity = adj1_capacity_for(n);
    if (ensure(ctx, ctx->adj, (size_t)ctx->adj_capacity * 32 * 4) || ensure(ctx, ctx->adj_gap, (size_t)ctx->adj_capacity * 32 * 4) ||
        ensure(ctx, ctx->adj_box, (size_t)ctx->adj_capacity * 2 * sizeof(float4)) ||
        ensure(ctx, ctx->adj1, (size_t)ctx->adj1_capacity * 32 * 4) || ensure(ctx, ctx->adj1_box, (size_t)ctx->adj1_capacity * 2 * sizeof(float4)))
        return ICP_GPU_E_CUDA;
    int launches = 0;
    if (join_index(ctx)) return ICP_GPU_E_CUDA;              // a build still running on aux_stream reads what this one overwrites
    CU(cudaEventRecord(ctx->ev[0], ctx->stream));
    CloudBufs b = context_bufs(ctx, 0);
    if (sort_cloud(ctx, b, n, ctx->T, ctx->late_pending[0] ? &ctx->late[0] : nullptr, &launches)) return ICP_GPU_E_CUDA;
    ctx->tsort.keys_sorted = b.keys_sorted; ctx->tsort.msd_shift = b.msd_shift;
    if (ctx->late_pending[0]) { CU(cudaEventRecord(ctx->ev_packed[0], ctx->stream)); ctx->packed_once[0] = true; ctx->late_pending[0] = false; }
    cudaStream_t ts = ctx->aux_stream;
    CU(cudaEventRecord(ctx->ev_fork, ctx->stream)); CU(cudaStreamWaitEvent(ts, ctx->ev_fork, 0));
    if (build_tree(ctx, b, n, ctx->T, ts, &launches)) return ICP_GPU_E_CUDA;
    CU(cudaEventRecord(ctx->ev[1], ts));
    CU(cudaEventRecord(ctx->ev_index_ready, ts)); ctx->index_pending = true;
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    ctx->grid_built = true;
    return 0;
}

// Sorts the source into the cell order of its own grid (Morton order); points with a non-finite coordinate keep a slot at the end.
static int build_source(icp_gpu_ctx* ctx) {
    const int n = ctx->n_src;
    const size_t n1 = (size_t)(n > 0 ? n : 1);
    if (ensure(ctx, ctx->src_pts, n1 * sizeof(float4)) || ensure(ctx, ctx->src_nrm, n1 * sizeof(float4))) return ICP_GPU_E_CUDA;
    int launches = 0;
    CloudBufs b = context_bufs(ctx, 1);
    if (sort_cloud(ctx, b, n, ctx->Ts, ctx->late_pending[1] ? &ctx->late[1] : nullptr, &launches)) return ICP_GPU_E_CUDA;
    ctx->ssort.keys_sorted = b.keys_sorted; ctx->ssort.msd_shift = b.msd_shift;
    if (ctx->late_pending[1]) { CU(cudaEventRecord(ctx->ev_packed[1], ctx->stream)); ctx->packed_once[1] = true; ctx->late_pending[1] = false; }
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    return 0;
}

int set_cloud(icp_gpu_ctx* ctx, bool target, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n, bool dev) {
    if (n < 0 || n > 0x7fffffff / 4 || (n > 0 && !xyz)) return fail(ctx, ICP_GPU_E_ARG, "bad cloud (n=%lld, xyz=%p)", (long long)n, (const void*)xyz);
    if (int rc = enter(ctx)) return rc;
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
    for (size_t i = 0; i < n; ++i) ctx->src_finite[i] = point_finite(&p[i].x, &m[i].x) ? 1 : 0;
    ctx->src_finite_valid = true;
    return 0;
}

int icp_gpu_set_target(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n) { return set_cloud(ctx, true, xyz, nrm, rgba, n, false); }
int icp_gpu_set_source(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n) { return set_cloud(ctx, false, xyz, nrm, rgba, n, false); }
int icp_gpu_set_target_dev(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n) { return set_cloud(ctx, true, xyz, nrm, rgba, n, true); }
int icp_gpu_set_source_dev(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n) { return set_cloud(ctx, false, xyz, nrm, rgba, n, true); }

// PointCloud(depthMap, colorFrame, depthIntrinsics, depthExtrinsics, width, height, keepOriginalSize, downsampleFactor,
// maxDistance) -- PointCloud.h:78-165 -- on the device; the result can become the context's target or source directly.
int icp_gpu_cloud_from_depth(icp_gpu_ctx* ctx, const float* depth, const uint8_t* rgbx, const float K[9], const float E[16],
                             uint32_t width, uint32_t height, int keep_original_size, uint32_t downsample, float max_distance, int role,
                             float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* n_out) {
    if (!K) return ICP_GPU_E_ARG;
    if (!depth || width == 0 || height == 0 || downsample == 0 || (long long)width * height > 0x7fffffff / 4)
        return fail(ctx, ICP_GPU_E_ARG, "bad depth map (%p, %ux%u, downsample %u)", (const void*)depth, width, height, downsample);
    if (role < ICP_GPU_CLOUD_TARGET || role > ICP_GPU_CLOUD_ONLY) return fail(ctx, ICP_GPU_E_ARG, "role %d", role);
    if (int rc = enter(ctx)) return rc;
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
    // input: depth, colours; staging: points, normals, colours, flags, block counts (+ total); the outputs use the first three
    const size_t in_sizes[] = {depth_bytes, color_bytes}, sizes[] = {nc * 12, nc * 12, nc * 4, nc * 4, (nb + 2) * 4};
    size_t in_off[2], t[5];
    const size_t in_total = pack_segments(in_sizes, 2, in_off), t_end = pack_segments(sizes, 5, t);
    if (ensure(ctx, ctx->prep_in, in_total) || ensure(ctx, ctx->prep_tmp, t_end) || ensure(ctx, ctx->prep_out, t[3])) return ICP_GPU_E_CUDA;
    char* in = (char*)ctx->prep_in.p; char* tmp = (char*)ctx->prep_tmp.p; char* out = (char*)ctx->prep_out.p;
    CU(cudaMemcpyAsync(in, depth, depth_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (rgbx) CU(cudaMemcpyAsync(in + in_off[1], rgbx, color_bytes, cudaMemcpyHostToDevice, ctx->stream));
    int launches = 0;
    unsigned int* total = (unsigned int*)(tmp + t[4]) + nb;
    CU(icp_launch_depth_cloud((const float*)in, rgbx ? (const unsigned char*)(in + in_off[1]) : nullptr, a, (float*)tmp, (float*)(tmp + t[1]),
                              (unsigned char*)(tmp + t[2]), (unsigned int*)(tmp + t[3]), (unsigned int*)(tmp + t[4]), total,
                              (float*)out, (float*)(out + t[1]), (unsigned char*)(out + t[2]), ctx->stream, &launches));
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    unsigned int n = 0;
    CU(cudaMemcpyAsync(&n, total, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));    // the host arrays were pageable: all copies are done; n is known
    if (n_out) *n_out = (int64_t)n;
    if (n > 0) {
        if (xyz_out) CU(cudaMemcpyAsync(xyz_out, out, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
        if (nrm_out) CU(cudaMemcpyAsync(nrm_out, out + t[1], (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
        if (rgba_out) CU(cudaMemcpyAsync(rgba_out, out + t[2], (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    int rc = ICP_GPU_OK;
    if (role != ICP_GPU_CLOUD_ONLY)
        rc = set_cloud(ctx, role == ICP_GPU_CLOUD_TARGET, (const float*)out, (const float*)(out + t[1]), (const uint8_t*)(out + t[2]), (int64_t)n, true);
    if (xyz_out || nrm_out || rgba_out) CU(cudaStreamSynchronize(ctx->stream));
    return rc;
}

// PointCloud(pcl::PointCloud<pcl::PointXYZ>::Ptr) (PointCloud.h:41-76): k-NN PCA normals (pcl::NormalEstimation, setKSearch(k)) of the
// context's TARGET cloud, computed with the index set_target built.  The normals replace the target's own (used by the next
// registrations) and are returned in the caller's point order.
int icp_gpu_target_normals(icp_gpu_ctx* ctx, int32_t k, const float viewpoint[3], float* nrm_out, float* curvature_out) {
    if (k < 3 || k > 8) return fail(ctx, ICP_GPU_E_ARG, "k %d (3..8)", k);
    if (int rc = enter(ctx)) return rc;
    if (!ctx->grid_built) return fail(ctx, ICP_GPU_E_STATE, "no target cloud set");
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
