// match.cu -- stages 1-4 of one ICP iteration, one kernel chain per matching method:
//   selection predicate on the sorted source   (selection.h:28-60,88-104, PointCloud.h:325-343)
//   transformPoints / transformNormals        (utils.h:106-133)
//   queryMatches: exact 1-NN (3-D / 6-D) or projective window search
//                                             (NearestNeighbor.h:143-207, :234-303, :333-421)
//   WeightingMethod::applyWeights             (weighting.h:39-99)
//   ICPOptimizer::pruneCorrespondences        (ICPOptimizer.h:157-174)
// The exact 1-NN over the target's index is knn.cu (-> nn_pos, then match_finish_kernel here); the matchers without an index:
//   knn_brute_kernel  small targets: one warp per query over the whole target, warp-shuffle arg-min.
//   projective_kernel one thread per query over its 25 x 25 pixel window, staged in shared memory per block
//                     (32 x 4 pixel tiles of a full-frame source, else 64 or 256 Morton-consecutive points).
#include "search.cuh"

// (d, idx) lexicographic '<' : contract D2
__device__ __forceinline__ bool better(float d, int idx, const Best& b) { return d < b.d || (d == b.d && idx < b.idx); }

// x86-64 gcc semantics of `unsigned = std::round(float)` (NearestNeighbor.h:378-379): cvttss2si to
// 64 bits, low 32 bits kept; NaN / out of range -> 0.
__device__ __forceinline__ unsigned int x86_float_to_u32(float t) {
    if (!(fabsf(t) < 9223372036854775808.0f)) return 0u;
    return (unsigned int)(long long)t;
}

// Stages 3-4 for one query given its match; writes the query's outputs.
__device__ __forceinline__ void finish_match(const MatchArgs& a, int p, bool matched, float w_const, int t_idx, int t_pos,
                                             float sx, float sy, float sz, float snx, float sny, float snz, unsigned int s_rgba,
                                             unsigned int& n_matched) {
    int out_idx = -1, out_pos = -1; float w = 0.0f;
    if (matched) {
        const float4 tn = __ldg(&a.tgt_nrm[t_pos]);
        float4 tp = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.weighting != ICP_GPU_WEIGHT_CONSTANT) tp = __ldg(&a.tgt_pts[t_pos]);
        w = w_const;
        if (match_weight_and_reject(a.weighting, a.rejection, a.weight_max_d2, sx, sy, sz, snx, sny, snz, s_rgba, tp, tn, w)) {
            out_idx = t_idx; out_pos = t_pos; ++n_matched;
        }
    }
    a.match_pos[p] = out_pos;
    a.match_w[p] = w;
    if (a.match_idx) a.match_idx[p] = out_idx;
}

__device__ __forceinline__ void write_no_query(const MatchArgs& a, int p) {
    a.match_pos[p] = -1; a.match_w[p] = 0.0f; if (a.match_idx) a.match_idx[p] = -1;
}

// Loads sorted-source point p, decides whether it is a query of this iteration and transforms it.
__device__ __forceinline__ bool prepare_query(const MatchArgs& a, const IterDesc& d, const PoseSm& sm, int p, Query& q,
                                              float& snx, float& sny, float& snz, unsigned int& s_rgba) {
    const float4 p4 = __ldg(&a.src_pts[p]);
    const float4 n4 = __ldg(&a.src_nrm[p]);
    if (!query_active(d, a.mask, p4, n4)) return false;
    xform_point(sm.P, p4.x, p4.y, p4.z, q.x, q.y, q.z);
    xform_normal(sm.N, n4.x, n4.y, n4.z, snx, sny, snz);
    s_rgba = __float_as_uint(n4.w);
    set_colour(q, s_rgba);
    return true;
}

// Stages 3-4 of the grid search, thread per query: transformNormals, weighting, rejection of the neighbour in nn_pos -> the match records.
__global__ void __launch_bounds__(256) match_finish_kernel(const MatchArgs a) {
    __shared__ PoseSm sm;
    if (registration_stopped(a)) return;
    load_pose(sm, a.state_ro);
    const IterDesc d = a.desc[iter_index(a)];
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int nq = 0, nm = 0;
    if (p < a.n_src) {
        Query q; float snx, sny, snz; unsigned int s_rgba;
        if (prepare_query(a, d, sm, p, q, snx, sny, snz, s_rgba)) {
            ++nq;
            int pos = finite3(q.x, q.y, q.z) ? a.nn_pos[p] : -1;
            if (pos >= a.n_tgt) pos = -1;
            const int idx = pos >= 0 ? __float_as_int(__ldg(&a.tgt_pts[pos].w)) : -1;
            finish_match(a, p, pos >= 0, 1.0f, idx, pos, q.x, q.y, q.z, snx, sny, snz, s_rgba, nm);
        } else {
            write_no_query(a, p);
        }
    }
    flush_stats(a, nq, nm, 0u, 0u);
}

// Small targets: one warp per query, lanes stride over the target (original order, L1-resident),
// warp-shuffle arg-min on (d, idx).
template <bool COLOR, bool NORM>
__global__ void __launch_bounds__(ICP_MATCH_THREADS) knn_brute_kernel(const MatchArgs a) {
    __shared__ PoseSm sm;
    if (registration_stopped(a)) return;
    load_pose(sm, a.state_ro);
    const IterDesc d = a.desc[iter_index(a)];
    const int lane = threadIdx.x & 31;
    const int p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    unsigned int nq = 0, nm = 0, ev = 0, nd = 0;
    if (p < a.n_src) {
        Query q; float snx, sny, snz; unsigned int s_rgba;
        if (prepare_query(a, d, sm, p, q, snx, sny, snz, s_rgba)) {     // warp-uniform
            Best b; b.d = fminf(a.max_d2, FLT_BIG); b.idx = INT_MAX; b.pos = -1;
            if (finite3(q.x, q.y, q.z)) {
                for (int j = lane; j < a.n_tgt; j += 32) {
                    const float4 c = __ldg(&a.tgt_pts[j]);
                    float dd = dist2<COLOR>(q, c, b.d, a.tgt_nrm, (unsigned int)j);
                    if (NORM) dd = __fsqrt_rn(dist3(q.x, q.y, q.z, c));                  // (p - m).norm(), NearestNeighbor.h:86
                    if (better(dd, j, b)) { b.d = dd; b.idx = j; b.pos = j; }
                }
                ev += (unsigned int)((a.n_tgt - lane + 31) / 32);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    Best t; t.d = __shfl_xor_sync(0xFFFFFFFFu, b.d, o); t.idx = __shfl_xor_sync(0xFFFFFFFFu, b.idx, o); t.pos = t.idx;
                    if (better(t.d, t.idx, b)) b = t;
                }
                if (b.idx == INT_MAX) b.pos = -1; else b.pos = b.idx;
            }
            if (lane == 0) { ++nq; finish_match(a, p, b.pos >= 0, 1.0f, b.idx, b.pos, q.x, q.y, q.z, snx, sny, snz, s_rgba, nm); }
        } else if (lane == 0) {
            write_no_query(a, p);
        }
    }
    flush_stats(a, nq, nm, ev, nd);
}

// Projective matching (NearestNeighbor.h:333-421): restatement of the window scan, unsigned wrap-around included
// (a query whose projection is closer than 12 px to the low image border wraps and scans nothing).  One thread per
// query; a block's 256 queries are consecutive in the Morton-sorted source, i.e. a compact patch that projects to a
// compact image region: the block stages the union of its search windows (target points, row by row, coalesced) in
// shared memory and every thread scans its own 25x25 window there.  Blocks whose union does not fit fall back to
// reading the (L2-resident) target map directly.
#define PROJ_TILE_MAX 2800     // float4 entries (44.8 KB static shared memory: five blocks per SM)
// PROJ_THREADS = 256: full frames and large sources.  64: a small source (every 8th valid pixel of a frame, main.cpp:291-298: ~25 k
// queries) -- 256-query blocks would be fewer than the SMs, and the window union of 256 points that lie 8 pixels apart does not fit
// the stage (47 x 47 entries for 64 of them do).
template <int PROJ_THREADS, int TILE_MAX, int MIN_BLOCKS>
__global__ void __launch_bounds__(PROJ_THREADS, MIN_BLOCKS) projective_kernel(const MatchArgs a) {
    __shared__ PoseSm sm;
    __shared__ float4 tile[TILE_MAX];
    __shared__ unsigned int s_box[4][PROJ_THREADS / 32];
    if (registration_stopped(a)) return;
    load_pose(sm, a.state_ro);
    const IterDesc d = a.desc[iter_index(a)];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // Which query this thread answers.  A full-frame source (one point per pixel, original order: a.proj_tiled) is cut
    // into 32 x (PROJ_THREADS / 32) pixel tiles, one per block: the windows of a tile overlap in a (32+24) x (rows+24) region (plus the
    // inter-frame motion), which always fits the shared-memory stage, and the lanes of a warp read consecutive entries
    // of it (no bank conflicts).  Any other source is taken 256 consecutive points of its Morton order at a time.
    int p; bool in;
    if (a.proj_tiled) {
        const unsigned int tiles_x = (a.width + 31u) / 32u;
        const unsigned int u = (blockIdx.x % tiles_x) * 32u + (unsigned int)lane, v = (blockIdx.x / tiles_x) * (PROJ_THREADS / 32) + (unsigned int)wid;
        in = u < a.width && v < a.height;
        p = (int)(v * a.width + u);
    } else {
        p = blockIdx.x * blockDim.x + threadIdx.x;
        in = p < a.n_src;
    }
    const unsigned int searchWindow = 12u;                                 // NearestNeighbor.h:319
    unsigned int nq = 0, nm = 0, ev = 0, nd = 0;
    Query q; float snx = 0.f, sny = 0.f, snz = 0.f; unsigned int s_rgba = 0;
    q.x = q.y = q.z = 0.f; q.cr = q.cg = q.cb = 0.f;
    const bool is_query = in && prepare_query(a, d, sm, p, q, snx, sny, snz, s_rgba);
    const bool scans = is_query && !(q.x == MINF_F);                       // :372-373
    unsigned int uP = 0, vP = 0, u0 = 0xFFFFFFFFu, v0 = 0xFFFFFFFFu, u1 = 0, v1 = 0;
    bool has_window = false;
    if (scans) {
        uP = x86_float_to_u32(roundf(padd(pdiv(pmul(q.x, a.fx), q.z), a.cx)));   // :378-379
        vP = x86_float_to_u32(roundf(padd(pdiv(pmul(q.y, a.fy), q.z), a.cy)));
        // the loops of :385-386 start at vP-12 / uP-12 (unsigned) and stop at the high border or vP+12 / uP+12
        const unsigned int vs = vP - searchWindow, us = uP - searchWindow;
        if (vs < a.height && us < a.width && vs <= vP + searchWindow && us <= uP + searchWindow) {
            has_window = true;
            u0 = us; v0 = vs;
            u1 = min(uP + searchWindow, a.width - 1u); v1 = min(vP + searchWindow, a.height - 1u);
        }
    }
    // union of the block's windows
    unsigned int bu0 = __reduce_min_sync(0xFFFFFFFFu, u0), bv0 = __reduce_min_sync(0xFFFFFFFFu, v0);
    unsigned int bu1 = __reduce_max_sync(0xFFFFFFFFu, has_window ? u1 : 0u), bv1 = __reduce_max_sync(0xFFFFFFFFu, has_window ? v1 : 0u);
    if (lane == 0) { s_box[0][wid] = bu0; s_box[1][wid] = bv0; s_box[2][wid] = bu1; s_box[3][wid] = bv1; }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < PROJ_THREADS / 32; ++w) { bu0 = min(bu0, s_box[0][w]); bv0 = min(bv0, s_box[1][w]); bu1 = max(bu1, s_box[2][w]); bv1 = max(bv1, s_box[3][w]); }
    const bool any_window = bu0 != 0xFFFFFFFFu;
    const unsigned int tw = any_window ? bu1 - bu0 + 1u : 0u, th = any_window ? bv1 - bv0 + 1u : 0u;
    // Row pitch of the staged tile: a MULTIPLE OF 8 entries (128 B).  An LDS.128 is served 8 lanes at a time and is conflict-free
    // when those lanes hit 8 different 16-byte bank groups, i.e. different (row * pitch + column) mod 8: the lanes of a warp scan
    // neighbouring columns of possibly different rows (the frames are rotated against each other), so with pitch = 0 mod 8 the bank
    // group is the column alone.  Round 1 used the raw union width (834 k conflicts per launch); an odd pitch measured 2.4 M.
    const unsigned int tp = (tw + 7u) & ~7u;
    const bool staged = any_window && (unsigned long long)tp * th <= TILE_MAX;           // block-uniform
    if (any_window && !staged && threadIdx.x == 0) ++nd;                                // work counter: blocks that fall back to global reads
    if (staged) {
        for (unsigned int k = threadIdx.x; k < tw * th; k += PROJ_THREADS) {
            const unsigned int ty = k / tw, tx = k - ty * tw;
            tile[ty * tp + tx] = __ldg(&a.tgt_pts[(size_t)a.width * (bv0 + ty) + bu0 + tx]);
        }
    }
    __syncthreads();
    if (in) {
        if (!is_query) write_no_query(a, p);
        else {
            ++nq;
            if (!scans) {
                // :372-373 `continue` leaves the value-initialised Match{0, 0.f} (:353)
                finish_match(a, p, true, 0.0f, 0, 0, q.x, q.y, q.z, snx, sny, snz, s_rgba, nm);
            } else {
                float minDist = FLT_BIG; unsigned int idx = 0xFFFFFFFFu;
                if (has_window) {
                    // Scan order = the reference's (rows, then columns): the strict '>' of :399 keeps the first minimum.  A MINF
                    // target (:392 `continue`) needs no test of its own: its distance is +inf (or NaN), which never passes the
                    // strict comparison against a minDist that starts at FLT_MAX.  The winner is remembered as a running
                    // candidate number and decoded after the loops.
                    const unsigned int n_u = u1 - u0 + 1u;
                    unsigned int cnt = 0u, best = 0xFFFFFFFFu;
                    if (staged) {
                        const float4* row = &tile[(v0 - bv0) * tp + (u0 - bu0)];          // shared-memory pointer: LDS.128
                        for (unsigned int v = v0; v <= v1; ++v, row += tp) {
#pragma unroll 5
                            for (unsigned int k = 0; k < n_u; ++k, ++cnt) {
                                const float dist = dist3(q.x, q.y, q.z, row[k]);
                                if (minDist > dist) { best = cnt; minDist = dist; }
                            }
                        }
                    } else {
                        const float4* row = &a.tgt_pts[(size_t)a.width * v0 + u0];
                        for (unsigned int v = v0; v <= v1; ++v, row += a.width) {
#pragma unroll 5
                            for (unsigned int k = 0; k < n_u; ++k, ++cnt) {
                                const float dist = dist3(q.x, q.y, q.z, __ldg(&row[k]));
                                if (minDist > dist) { best = cnt; minDist = dist; }
                            }
                        }
                    }
                    ev += cnt;                                                            // candidates scanned (MINF ones included)
                    if (best != 0xFFFFFFFFu) idx = a.width * (v0 + best / n_u) + u0 + best % n_u;
                }
                const bool ok = minDist <= a.max_d2 && idx != 0xFFFFFFFFu;               // :407
                finish_match(a, p, ok, 1.0f, (int)idx, (int)idx, q.x, q.y, q.z, snx, sny, snz, s_rgba, nm);
            }
        }
    }
    flush_stats(a, nq, nm, ev, nd);
}

cudaError_t icp_launch_match(const MatchArgs& a, int algorithm, int n_sms, cudaStream_t s, int* n_launches, cudaEvent_t after_prep,
                             const MatchChunks* chunks) {
    if (a.n_src <= 0) return cudaSuccess;
    const int T = ICP_MATCH_THREADS;
    int launches = 0;
    if (algorithm == 2) {
        if (!a.proj_tiled && a.n_src < 2 * 256 * n_sms) {
            projective_kernel<64, PROJ_TILE_MAX, 5><<<(unsigned int)((a.n_src + 63) / 64), 64, 0, s>>>(a);
        } else if (a.proj_tiled) {
            // full frames: 32 x 4 pixel tiles, 2400 blocks of 128 threads at 640 x 480 over 148 x 6 slots -- with 32 x 8 tiles the 1200
            // blocks were 1.6 waves of long blocks (C3: 4.35 -> 4.20 ms per 35 iterations).  The stage holds the (32+24) x (4+24) union
            // plus 8 pixels of inter-frame motion either way.
            const unsigned int nb = ((a.width + 31u) / 32u) * ((a.height + 128 / 32 - 1u) / (128 / 32));
            projective_kernel<128, 2304, 6><<<nb, 128, 0, s>>>(a);
        } else {
            projective_kernel<256, PROJ_TILE_MAX, 5><<<(unsigned int)((a.n_src + 256 - 1) / 256), 256, 0, s>>>(a);
        }
        ++launches;
    } else if (algorithm == 1) {
        const long long threads = (long long)a.n_src * 32;
        const int nb = (int)((threads + T - 1) / T);
        if (a.color_icp) knn_brute_kernel<true, false><<<nb, T, 0, s>>>(a);
        else if (a.brute_norm) knn_brute_kernel<false, true><<<nb, T, 0, s>>>(a);
        else knn_brute_kernel<false, false><<<nb, T, 0, s>>>(a);
        ++launches;
    } else {
        icp_launch_knn(a, n_sms, s, after_prep, chunks, launches);
        if (!a.skip_finish) { match_finish_kernel<<<(a.n_src + 255) / 256, 256, 0, s>>>(a); ++launches; }
    }
    if (n_launches) *n_launches += launches;
    return cudaGetLastError();
}
