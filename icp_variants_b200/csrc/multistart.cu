// multistart.cu -- K registrations of the context's source against the context's indexed target in ONE launch (icp_gpu_estimate_pose_multistart):
// start k runs every iteration of its loop from its own initial pose on a thread-block cluster of C blocks (C = 1 ... 16, chosen from K
// and the SM count so that a handful of starts still fills the GPU), then scores its final pose.  The index (grid.cu) is the context's,
// built once; each start keeps its own remembered neighbour per query.
//
//   search    one thread per query, exact 1-NN under contract D1-D3 (3-D or 6-D colour), as pca_normals_kernel (normals.cu) walks the
//             index with one best instead of k: the leaf of the query's last neighbour for this start (at the first iteration the point
//             key_seed reads off the sorted keys), then that leaf's adjacency list when the ball of the best distance lies inside the
//             leaf's inflated box, otherwise a depth-first walk with a private stack.  Same candidates, same (d2, index) order as the
//             walk of knn.cu, hence the same correspondences.
//   stages    query_active / xform_point / match_weight_and_reject: the device functions every other path uses; the plan (iteration
//             descriptors and selection masks) is make_plan's (registration.cu)
//   rows      accumulate_match (solve.cuh) / lm_accumulate_match (lm.cuh) of the matches of 256 consecutive sorted positions (a tile,
//             one position per thread) -> a tile row (warp reduce-scatter, the 8 warps in order).  Tile t is added to slice t mod 16 in
//             tile order; the 16 slices are summed in slice order through distributed shared memory after a cluster barrier.  A
//             cluster of C blocks (C divides 16) gives block r the tiles t = r mod C, so slice s lives in block s mod C: the sums, and
//             with them every output of a start, are the same bits whatever C and K are.  No floating-point atomics.
//   solve     every block of the cluster holds the same total and runs the finisher (solve.cuh) or the trust-region step (lm.cuh) on
//             it -- identical inputs, identical decisions, so the blocks stay in step without a broadcast; block 0 writes the outputs.
//   scoring   after the last iteration every query matches once more at the final pose (all points, the configuration's threshold,
//             weighting and rejection: icp_gpu_query_matches' matches); the inlier count and the sum of the D1 distances go through
//             the same tile / slice sums.
// Symmetric metric and LM keep a start's matches in its slice of the per-(start, query) scratch between passes, as batch.cu does.
#include "solve.cuh"
#include "lm.cuh"
#include "search.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

#define MS_STACK (32 * ICP_BVH_MAX_LEVELS)   // one top-level subtree at a time: <= 31 * levels + 1 entries
#define MS_MAX_CLUSTER ICP_MS_SLICES

// Every point of the leaf against the best so far, (d2, index) order (better_key: a NaN or infinite distance never wins).
template <bool COLOR, class V>
__device__ __forceinline__ void ms_scan_leaf(const V& a, const Query& q, Best& b, unsigned int leaf) {
    const unsigned int ls = __ldg(&a.leaf_start[leaf]), le = __ldg(&a.leaf_start[leaf + 1]);
    for (unsigned int i = ls; i < le; ++i) {
        const float4 pt = __ldg(&a.tgt_pts[i]);
        const float d = dist2<COLOR>(q, pt, b.d, a.tgt_nrm, i);
        const int idx = __float_as_int(pt.w);
        if (better_key(d, idx, b)) { b.d = d; b.idx = idx; b.pos = (int)i; }
    }
}

// Exact nearest neighbour of q, starting from the leaf of sorted target position `seed` (-1: none).  b.idx == INT_MAX: none within
// the threshold.
template <bool COLOR, class V>
__device__ __noinline__ Best ms_search(const V& a, const BvhDesc& bvh, const Query& q, int seed) {
    Best b; best_init(b, a.max_d2);
    if (bvh.n_leaves <= 0) return b;
    int seed_leaf = -1;
    if (seed >= 0) {
        seed_leaf = (int)(__ldg(&a.leaf_rank[seed + 1]) - 1u);
        ms_scan_leaf<COLOR, V>(a, q, b, (unsigned int)seed_leaf);
        if (b.d < FLT_BIG && seed_leaf < a.adj_capacity) {
            const float4 ilo = __ldg(&a.adj_box[2 * (size_t)seed_leaf]), ihi = __ldg(&a.adj_box[2 * (size_t)seed_leaf + 1]);
            if (ball_inside(q.x, q.y, q.z, search_radius(b.d), ilo, ihi)) {      // never true for the inverted "no list" box
                const int na = __float_as_int(ilo.w);
                for (int j = 0; j < na; ++j) {
                    const unsigned int leaf = __ldg(&a.adj[(size_t)seed_leaf * 32 + j]);
                    const float clb = box_dist2c<COLOR>(q, __ldg(&a.bvh_box[2 * (size_t)leaf]), __ldg(&a.bvh_box[2 * (size_t)leaf + 1]));
                    if (!(clb > b.d)) ms_scan_leaf<COLOR, V>(a, q, b, leaf);
                }
                return b;
            }
        }
    }
    // depth-first walk with a private stack; the seed leaf was scanned already
    unsigned int st[MS_STACK];
    const int top_level = bvh.n_levels - 1;
    for (int c0 = 0; c0 < bvh.count[top_level]; ++c0) {
        st[0] = ((unsigned int)top_level << 27) | (unsigned int)c0;
        int top = 1;
        while (top > 0) {
            const unsigned int e = st[--top];
            const int lvl = (int)(e >> 27); const unsigned int j = e & 0x7FFFFFFu;
            const size_t box = 2 * (size_t)(bvh.offset[lvl] + j);
            const float clb = box_dist2c<COLOR>(q, __ldg(&a.bvh_box[box]), __ldg(&a.bvh_box[box + 1]));
            if (clb > b.d) continue;
            if (lvl == 0) { if ((int)j != seed_leaf) ms_scan_leaf<COLOR, V>(a, q, b, j); continue; }
            const unsigned int first = __ldg(&a.child_start[bvh.coffset[lvl] + j]), last = __ldg(&a.child_start[bvh.coffset[lvl] + j + 1]);
            for (unsigned int c = first; c < last && top < MS_STACK; ++c) st[top++] = ((unsigned int)(lvl - 1) << 27) | c;
        }
    }
    return b;
}

// Stages 2-4 of sorted source position p at pose (P, Nm): the matched sorted target position or -1.  w leaves as
// match_finish_kernel's weight (0 without a neighbour; the weight computed before a rejection), d2 as the neighbour's D1 distance;
// (sx, sy, sz) is the transformed point, sn the source normal record, tp / tn the target point and normal.  nn: this (start, query)'s
// remembered neighbour, updated.  v: the pair (MsArgs itself for multi-start, the shared copy of its MsPair in a batch), a: the
// configuration.
template <bool COLOR, class V>
__device__ __forceinline__ int ms_match(const MsArgs& a, const V& v, const BvhDesc& bvh, const IterDesc& d, const float* P, const float* Nm, int p,
                                        int* nn, float& sx, float& sy, float& sz, float4& sn, float4& tp, float4& tn, float& w, float& d2) {
    w = 0.0f;
    const float4 sp = __ldg(&v.src_pts[p]);
    sn = __ldg(&v.src_nrm[p]);
    if (!query_active(d, v.mask, sp, sn)) return -1;
    xform_point(P, sp.x, sp.y, sp.z, sx, sy, sz);
    if (!finite3(sx, sy, sz)) return -1;
    Query q; q.x = sx; q.y = sy; q.z = sz;
    set_colour(q, __float_as_uint(sn.w));
    int seed = *nn;
    if (seed < 0) seed = key_seed(v.grid, v.keys, v.n_tgt - (int)__ldg(v.nonfinite), v.msd_start, v.msd_shift, sx, sy, sz);
    const Best b = ms_search<COLOR, V>(v, bvh, q, seed);
    if (b.idx == INT_MAX || b.pos < 0) return -1;
    *nn = b.pos;
    tp = __ldg(&v.tgt_pts[b.pos]); tn = __ldg(&v.tgt_nrm[b.pos]);
    float nx, ny, nz;
    xform_normal(Nm, sn.x, sn.y, sn.z, nx, ny, nz);
    w = 1.0f; d2 = b.d;
    if (!match_weight_and_reject(a.weighting, a.rejection, a.weight_max_d2, sx, sy, sz, nx, ny, nz, __float_as_uint(sn.w), tp, tn, w)) return -1;
    return b.pos;
}

struct MsShared {
    double slice[ICP_MS_SLICES][32];        // this block's slices (local index = slice / C)
    double red[ICP_MS_THREADS / 32][32];
    double tot[32];                         // the cluster's summed row
    float P[16], Nm[9], mS[3], mD[3];
    double xs[6];
    LmState lm;
    BvhDesc bvh;
    int done, rc;
};

// The tile row of the block's per-thread rows v, added to its slice.
__device__ __forceinline__ void ms_tile_row(double (&v)[32], MsShared& sm, int t, int C) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    warp_reduce_scatter32(v, lane);
    sm.red[wid][lane] = v[0];
    __syncthreads();
    if (threadIdx.x < 32) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < ICP_MS_THREADS / 32; ++k) s += sm.red[k][threadIdx.x];
        sm.slice[(t % ICP_MS_SLICES) / C][threadIdx.x] += s;
    }
    __syncthreads();
}

// The cluster's total (slices 0 ... 15 in order) into every block's sm.tot; the slices are zeroed for the next row.
__device__ __forceinline__ void ms_cluster_total(MsShared& sm, cg::cluster_group& cl, int C) {
    cl.sync();
    if (threadIdx.x < 32) {
        double s = 0.0;
        for (int k = 0; k < ICP_MS_SLICES; ++k) s += cl.map_shared_rank(&sm, k % C)->slice[k / C][threadIdx.x];
        sm.tot[threadIdx.x] = s;
    }
    cl.sync();                                            // every block has read the slices
    if (threadIdx.x < 32) for (int k = 0; k < ICP_MS_SLICES / C; ++k) sm.slice[k][threadIdx.x] = 0.0;
    __syncthreads();
}

__device__ __forceinline__ void zero32(double (&v)[32]) {
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = 0.0;
}

// Thread 0: the increment inc (rc = its status) applied to the block's pose; block 0 writes row k's history.  Returns "stop".
__device__ __forceinline__ bool ms_apply(const MsArgs& a, MsShared& sm, int k, bool writer, const float* inc, int rc, int& status, int& iters_done) {
    if (rc != 0) { status = rc; return true; }
    float np[16];
    mat4_mul_pinned(inc, sm.P, np);                       // ICPOptimizer.h:614-620
    for (int i = 0; i < 16; ++i) sm.P[i] = np[i];
    inv_transpose3_pinned(np, sm.Nm);
    if (writer && a.history) for (int i = 0; i < 16; ++i) a.history[((size_t)k * a.history_rows + iters_done) * 16 + i] = np[i];
    ++iters_done;
    return increment_is_small(inc, a.stop_rot, a.stop_trans);
}

// LM = 0: the linear minimiser, METRIC 0 point-to-point, 1 point-to-plane, 2 symmetric; LM = 1: the Ceres path (lm.cuh).
// BATCH = false: cluster k runs start k on the MsArgs' own pair; true: cluster k runs pair k = order[cluster] (MsPair in a.pairs).  The
// outputs, the history and the per-query slices of cluster k are row k's.
template <int LM, int METRIC, bool COLOR, bool BATCH>
__global__ void __launch_bounds__(ICP_MS_THREADS, 1) multistart_kernel(const MsArgs a) {
    __shared__ MsShared sm;
    cg::cluster_group cl = cg::this_cluster();
    const int C = (int)cl.num_blocks(), rank = (int)cl.block_rank();
    const int cluster = (int)(blockIdx.x / (unsigned int)C);
    const int k = BATCH ? __ldg(&a.order[cluster]) : cluster;
    __shared__ MsPair pv;                                 // batch: the cluster's pair, copied into shared memory (unused otherwise)
    if (BATCH) {
        if (threadIdx.x < sizeof(MsPair) / 4) reinterpret_cast<int*>(&pv)[threadIdx.x] = reinterpret_cast<const int*>(a.pairs + k)[threadIdx.x];
        __syncthreads();
    }
    // the view: multi-start reads its pair straight from the kernel parameter, as a plain MsArgs
    const auto& v = *[&] { if constexpr (BATCH) return (const MsPair*)&pv; else return &a; }();
    const bool writer = rank == 0;
    const int n = v.n_src, n_tiles = (n + ICP_MS_THREADS - 1) / ICP_MS_THREADS;
    const size_t q_off = BATCH ? (size_t)v.q_off : (size_t)k * n;
    int* nn = a.nn_pos + q_off;
    int2* scr = a.scratch ? a.scratch + q_off : nullptr;
    if (threadIdx.x < 16) sm.P[threadIdx.x] = a.poses_in[16 * (size_t)k + threadIdx.x];
    if (threadIdx.x < sizeof(BvhDesc) / 4) reinterpret_cast<int*>(&sm.bvh)[threadIdx.x] = reinterpret_cast<const int*>(v.bvh)[threadIdx.x];
    if (threadIdx.x < 32) for (int s = 0; s < ICP_MS_SLICES / C; ++s) sm.slice[s][threadIdx.x] = 0.0;
    if (threadIdx.x < 3) { sm.mS[threadIdx.x] = 0.f; sm.mD[threadIdx.x] = 0.f; }
    if (threadIdx.x == 0) sm.done = 0;
    __syncthreads();
    if (threadIdx.x == 0) inv_transpose3_pinned(sm.P, sm.Nm);
    __syncthreads();
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    int status = 0, iters_done = 0;                       // meaningful in thread 0
    for (int it = 0; it < v.n_iters; ++it) {
        const IterDesc d = v.desc[it];
        double row[32];
        if (LM == 0) {
            for (int t = rank; t < n_tiles; t += C) {
                zero32(row);
                const int p = t * ICP_MS_THREADS + threadIdx.x;
                if (p < n) {
                    float sx, sy, sz, w, d2; float4 sn, tp = zero4, tn = zero4;
                    const int j = ms_match<COLOR>(a, v, sm.bvh, d, sm.P, sm.Nm, p, nn + p, sx, sy, sz, sn, tp, tn, w, d2);
                    if (METRIC == 2) scr[p] = make_int2(j, __float_as_int(w));
                    if (j >= 0) accumulate_match<METRIC == 2 ? 3 : METRIC>(row, sx, sy, sz, tp, tn, sn, sm.Nm, sm.mS, sm.mD, (double)w);
                }
                ms_tile_row(row, sm, t, C);
            }
            ms_cluster_total(sm, cl, C);
            if (METRIC == 2) {
                if (threadIdx.x == 0) {                   // unweighted means of the kept matches, rounded to fp32 (finish_sums, solve.cu)
                    const double M = sm.tot[0];
                    for (int c = 0; c < 3; ++c) { sm.mS[c] = M > 0.0 ? (float)(sm.tot[1 + c] / M) : 0.f; sm.mD[c] = M > 0.0 ? (float)(sm.tot[4 + c] / M) : 0.f; }
                }
                __syncthreads();
                for (int t = rank; t < n_tiles; t += C) {
                    zero32(row);
                    const int p = t * ICP_MS_THREADS + threadIdx.x;
                    if (p < n) {
                        const int2 m = scr[p];            // written by this thread in the first pass
                        if (m.x >= 0) {
                            const float4 sp = __ldg(&v.src_pts[p]), sn = __ldg(&v.src_nrm[p]);
                            float sx, sy, sz;
                            xform_point(sm.P, sp.x, sp.y, sp.z, sx, sy, sz);
                            accumulate_match<2>(row, sx, sy, sz, __ldg(&v.tgt_pts[m.x]), __ldg(&v.tgt_nrm[m.x]), sn, sm.Nm, sm.mS, sm.mD, (double)__int_as_float(m.y));
                        }
                    }
                    ms_tile_row(row, sm, t, C);
                }
                ms_cluster_total(sm, cl, C);
            }
            if (threadIdx.x == 0) {
                float inc[16]; int rc;
                if (METRIC == 0) rc = finish_p2p(sm.tot, inc);
                else if (METRIC == 1) rc = finish_p2plane(sm.tot, inc);
                else rc = finish_symmetric(sm.tot, sm.mS, sm.mD, inc);
                if (ms_apply(a, sm, k, writer, inc, rc, status, iters_done)) sm.done = 1;
            }
        } else {
            for (int t = rank; t < n_tiles; t += C) {
                const int p = t * ICP_MS_THREADS + threadIdx.x;
                if (p < n) {
                    float sx, sy, sz, w, d2; float4 sn, tp, tn;
                    const int j = ms_match<COLOR>(a, v, sm.bvh, d, sm.P, sm.Nm, p, nn + p, sx, sy, sz, sn, tp, tn, w, d2);
                    scr[p] = make_int2(j, __float_as_int(w));     // kept matches: both points finite (ICPOptimizer.h:378)
                }
            }
            for (int step = 0; step <= a.lm_max_iterations; ++step) {
                if (threadIdx.x < 6) sm.xs[threadIdx.x] = step == 0 ? 0.0 : sm.lm.cand[threadIdx.x];
                __syncthreads();
                LmJets J;
                lm_jets_init<METRIC>(J, sm.xs);
                for (int t = rank; t < n_tiles; t += C) {
                    zero32(row);
                    const int p = t * ICP_MS_THREADS + threadIdx.x;
                    if (p < n) {
                        const int2 m = scr[p];            // written by this thread above
                        if (m.x >= 0) {
                            const float4 sp = __ldg(&v.src_pts[p]);
                            float sx, sy, sz;
                            xform_point(sm.P, sp.x, sp.y, sp.z, sx, sy, sz);
                            lm_accumulate_match<METRIC>(row, J, sx, sy, sz, __ldg(&v.tgt_pts[m.x]), (double)__int_as_float(m.y), sm.Nm,
                                                        [&] { return __ldg(&v.tgt_nrm[m.x]); }, [&] { return __ldg(&v.src_nrm[p]); });
                        }
                    }
                    ms_tile_row(row, sm, t, C);
                }
                ms_cluster_total(sm, cl, C);
                if (threadIdx.x == 0) sm.rc = lm_advance(&sm.lm, sm.tot, step, a.lm_max_iterations);
                __syncthreads();
                if (sm.rc != LM_NEXT_EVAL) break;
            }
            if (threadIdx.x == 0) {                       // lm_finalize / apply_increment (lm.cu, icp_internal.cuh)
                float inc[16];
                increment_matrix(sm.lm.x, inc);
                if (ms_apply(a, sm, k, writer, inc, sm.rc, status, iters_done)) sm.done = 1;
            }
        }
        __syncthreads();
        if (sm.done) break;
    }
    // scoring pass: every point at the final pose (icp_gpu_query_matches with no selection)
    IterDesc all; all.stride = 1; all.filter_finite = 0; all.mask_word_offset = -1; all.rng_key = 0u; all.proba = -1.0f;
    all.pad0 = all.pad1 = all.pad2 = 0;
    for (int t = rank; t < n_tiles; t += C) {
        double row[32];
        zero32(row);
        const int p = t * ICP_MS_THREADS + threadIdx.x;
        if (p < n) {
            float sx, sy, sz, w, d2 = 0.f; float4 sn, tp = zero4, tn = zero4;
            const int j = ms_match<COLOR>(a, v, sm.bvh, all, sm.P, sm.Nm, p, nn + p, sx, sy, sz, sn, tp, tn, w, d2);
            if (j >= 0) { row[0] = 1.0; row[1] = (double)d2; }
            if (a.match_idx) {
                const size_t o = q_off + (unsigned int)__float_as_int(__ldg(&v.src_pts[p]).w);
                a.match_idx[o] = j >= 0 ? __float_as_int(tp.w) : -1;
                a.match_w[o] = w;
            }
        }
        ms_tile_row(row, sm, t, C);
    }
    ms_cluster_total(sm, cl, C);
    if (writer) {
        if (threadIdx.x < 16) a.poses_out[16 * (size_t)k + threadIdx.x] = sm.P[threadIdx.x];
        if (threadIdx.x == 0) {
            a.n_iter_out[k] = iters_done; a.status_out[k] = status;
            a.inliers_out[k] = (long long)sm.tot[0];
            a.rmse_out[k] = sm.tot[0] > 0.0 ? sqrt(sm.tot[1] / sm.tot[0]) : __longlong_as_double(0x7ff8000000000000ll);
        }
    }
}

template <int LM, int METRIC, bool BATCH>
static void (*pick_color(int color))(const MsArgs) { return color ? multistart_kernel<LM, METRIC, true, BATCH> : multistart_kernel<LM, METRIC, false, BATCH>; }

template <bool BATCH>
static void (*pick_kernel(int lm, int metric, int color))(const MsArgs) {
    if (lm) return metric == ICP_GPU_METRIC_P2P ? pick_color<1, 0, BATCH>(color) : metric == ICP_GPU_METRIC_P2PLANE ? pick_color<1, 1, BATCH>(color) : pick_color<1, 2, BATCH>(color);
    return metric == ICP_GPU_METRIC_P2P ? pick_color<0, 0, BATCH>(color) : metric == ICP_GPU_METRIC_P2PLANE ? pick_color<0, 1, BATCH>(color) : pick_color<0, 2, BATCH>(color);
}

cudaError_t icp_launch_multistart(const MsArgs& a, bool batch, int lm, int metric, int color, int n_clusters, int max_src, int n_sms, cudaStream_t s,
                                  int* cluster) {
    if (n_clusters <= 0) return cudaSuccess;
    void (*k)(const MsArgs) = batch ? pick_kernel<true>(lm, metric, color) : pick_kernel<false>(lm, metric, color);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return e;
    // Cluster size: the largest power of two <= 16 that keeps the clusters within one wave of resident blocks, and no larger than the
    // largest source's tiles need (one launch has one cluster shape); halved while the device cannot hold such a cluster.
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, ICP_MS_THREADS, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    const long long n_tiles = ((long long)max_src + ICP_MS_THREADS - 1) / ICP_MS_THREADS;
    int C = 1;
    while (C < MS_MAX_CLUSTER && (long long)n_clusters * C * 2 <= (long long)per_sm * n_sms && C < n_tiles) C *= 2;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    cfg.blockDim = dim3(ICP_MS_THREADS, 1, 1);
    cfg.dynamicSmemBytes = 0; cfg.stream = s;
    cfg.attrs = attr; cfg.numAttrs = 1;
    for (; C > 1; C /= 2) {
        attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.gridDim = dim3((unsigned int)C, 1, 1);
        int n_clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&n_clusters, k, &cfg) == cudaSuccess && n_clusters > 0) break;
        cudaGetLastError();
    }
    attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3((unsigned int)((long long)n_clusters * C), 1, 1);
    if (cluster) *cluster = C;
    return cudaLaunchKernelEx(&cfg, k, a);
}
