// search.cuh -- what the nearest-neighbour searches of knn.cu, match.cu, normals.cu and batch.cu share (device only): the D1 distance,
// its box bound and search radius, the sentinels, the hand-over from the fast path to the group search and the walk, the kernel prologue.
#pragma once
#include "icp_internal.cuh"
#include <limits.h>
#define FLT_BIG 3.4028234e38f      // the largest finite float: the bound of a search with no threshold

struct Query {
    float x, y, z;        // transformed source point
    float cr, cg, cb;     // colour features (6-D search only)
};
struct Best { float d; int idx; int pos; };

// (d, idx) lexicographic '<' (contract D2) as ONE 64-bit unsigned comparison of bits(d) || idx, valid while both distances are >= +0
// (the bit pattern of a non-negative float orders like its value; a NaN distance orders last) and 0 <= idx <= INT_MAX.  best_init
// keeps b.d non-negative: a negative threshold admits nothing, which the smallest key (0, 0) expresses.
__device__ __forceinline__ bool better_key(float d, int idx, const Best& b) {
    return (((unsigned long long)__float_as_uint(d) << 32) | (unsigned int)idx) <
           (((unsigned long long)__float_as_uint(b.d) << 32) | (unsigned int)b.idx);
}
__device__ __forceinline__ void best_init(Best& b, float max_d2) {
    if (max_d2 < 0.f) { b.d = 0.f; b.idx = 0; }
    else { b.d = fminf(max_d2, FLT_BIG); b.idx = INT_MAX; }
    b.pos = -1;
}
__device__ __forceinline__ float color_feature(unsigned int rgba, int k) {
    // NearestNeighbor.h:212-221,245-254: color_scale(1) * color_normalize(1/float(255)) * uchar
    return pmul(1.0f / 255.0f, (float)((rgba >> (8 * k)) & 0xFFu));
}
__device__ __forceinline__ void set_colour(Query& q, unsigned int rgba) { q.cr = color_feature(rgba, 0); q.cg = color_feature(rgba, 1); q.cb = color_feature(rgba, 2); }

__device__ __forceinline__ float dist3(float qx, float qy, float qz, const float4 c) {
    const float dx = psub(qx, c.x), dy = psub(qy, c.y), dz = psub(qz, c.z);
    return padd(padd(pmul(dx, dx), pmul(dy, dy)), pmul(dz, dz));                      // D1 (p* helpers: no FMA, whatever -fmad says)
}
template <bool COLOR>
__device__ __forceinline__ float dist2(const Query& q, const float4 c, float best, const float4* __restrict__ nrm, unsigned int i) {
    float d = dist3(q.x, q.y, q.z, c);
    if (COLOR) {
        if (d > best) return d;                                                // 3-D part already loses; adding squares cannot help
        const unsigned int rgba = __float_as_uint(__ldg(&nrm[i].w));
        const float dr = psub(q.cr, color_feature(rgba, 0)), dg = psub(q.cg, color_feature(rgba, 1)), db = psub(q.cb, color_feature(rgba, 2));
        d = padd(d, pmul(dr, dr)); d = padd(d, pmul(dg, dg)); d = padd(d, pmul(db, db));   // FLANN L2 order for 6 dims
    }
    return d;
}

// fp32 lower bound (under D1's rounding and association, by monotonicity) of the squared distance from q to any point inside the box
__device__ __forceinline__ float box_dist2(float qx, float qy, float qz, const float4 lo, const float4 hi) {
    const float gx = fmaxf(fmaxf(psub(lo.x, qx), psub(qx, hi.x)), 0.0f);
    const float gy = fmaxf(fmaxf(psub(lo.y, qy), psub(qy, hi.y)), 0.0f);
    const float gz = fmaxf(fmaxf(psub(lo.z, qz), psub(qz, hi.z)), 0.0f);
    return padd(padd(pmul(gx, gx), pmul(gy, gy)), pmul(gz, gz));
}
// The same for the 6-D colour search: the node's colour range (packed bytes in lo.w / hi.w, grid.cu) adds the squared gap
// of every colour feature, accumulated in the order of dist2, so the bound stays below the D1 distance of every point
// of the node (the feature map and every rounding involved are monotone).
template <bool COLOR>
__device__ __forceinline__ float box_dist2c(const Query& q, const float4 lo, const float4 hi) {
    float d = box_dist2(q.x, q.y, q.z, lo, hi);
    if (COLOR) {
        const unsigned int cl = __float_as_uint(lo.w), ch = __float_as_uint(hi.w);
        const float gr = fmaxf(fmaxf(psub(color_feature(cl, 0), q.cr), psub(q.cr, color_feature(ch, 0))), 0.0f);
        const float gg = fmaxf(fmaxf(psub(color_feature(cl, 1), q.cg), psub(q.cg, color_feature(ch, 1))), 0.0f);
        const float gb = fmaxf(fmaxf(psub(color_feature(cl, 2), q.cb), psub(q.cb, color_feature(ch, 2))), 0.0f);
        d = padd(d, pmul(gr, gr)); d = padd(d, pmul(gg, gg)); d = padd(d, pmul(gb, gb));
    }
    return d;
}

// Radius of the ball that holds every point whose D1 distance is <= d2 (sqrt rounded up, x 1.00001 for D1's roundings): the "ball
// inside the inflated box" tests of the fast path, the walk's level-1 shortcut and the normals, and GroupBounds (knn.cu) rest on it.
__device__ __forceinline__ float search_radius(float d2) { return __fmul_ru(__fsqrt_ru(d2), 1.00001f); }
// qbuf[p] = the transformed query {x, y, z, rgba}; x = NaN: no search left (not a query, or answered by the fast path / group search)
__device__ __forceinline__ float finished_mark() { return __int_as_float(0x7fc00000); }
__device__ __forceinline__ void mark_finished(float4& q) { q.x = finished_mark(); }
__device__ __forceinline__ bool is_pending(float qx) { return qx == qx; }
// seedbuf[p] (one 128-bit record): knn_prep_kernel's scan of pending query p's seed leaf, the leaf of its last neighbour (`best`: the
// group search and the walk start from it), whose inflated box the query's ball leaves.  node = HANDOVER_NONE: nothing handed over (no
// seed, or a seed leaf beyond the adjacency lists), the walk starts from nn_pos; HANDOVER_NO_NODE: the ball leaves the inflated box of
// the seed leaf's level-1 node too; m >= 0: it lies inside that of the seed leaf's level-1 node m, and the walk starts from m's list.
enum { HANDOVER_NONE = -2, HANDOVER_NO_NODE = -1 };
struct __align__(16) HandOver { Best best; int node; };
static_assert(sizeof(HandOver) == 16, "one 128-bit access");
__device__ __forceinline__ float4 pack_handover(const Best& b, int node) { return make_float4(b.d, __int_as_float(b.idx), __int_as_float(b.pos), __int_as_float(node)); }
__device__ __forceinline__ void store_handover(HandOver* buf, int p, const float4 v) { reinterpret_cast<float4*>(buf)[p] = v; }   // one STG.128
__device__ __forceinline__ bool handed_over(const HandOver& h) { return h.node >= HANDOVER_NO_NODE; }
__device__ __forceinline__ HandOver load_handover(const HandOver* buf, int p) {         // read-only path: written by an earlier launch
    const int4 v = __ldg(reinterpret_cast<const int4*>(buf + p));
    HandOver h; h.best.d = __int_as_float(v.x); h.best.idx = v.y; h.best.pos = v.z; h.node = v.w; return h;
}

// ---------------------------------------------------------------------------- cell codes of the target grid (grid.cu)
__device__ __forceinline__ int cell_index(const GridParams& g, int a, float x) {
    const float u = pmul(psub(x, g.o[a]), g.inv_h[a]);
    int i = (int)floorf(u);
    const int hi = (1 << g.bits[a]) - 1;
    return min(max(i, 0), hi);
}

// The code bits an axis contributes for cell index c: bit j of c lands at bitpos[a][j].
__device__ __forceinline__ unsigned int axis_spread(const GridParams& g, int a, int c) {
    unsigned int code = 0;
#pragma unroll
    for (int j = 0; j < ICP_MAX_BITS_PER_AXIS; ++j)
        if (j < g.bits[a]) code |= (((unsigned int)c >> j) & 1u) << g.bitpos[a][j];
    return code;
}

__device__ __forceinline__ unsigned int cell_code(const GridParams& g, float x, float y, float z) {
    return axis_spread(g, 0, cell_index(g, 0, x)) | axis_spread(g, 1, cell_index(g, 1, y)) | axis_spread(g, 2, cell_index(g, 2, z));
}

// The seed of a query at the transformed position (x, y, z) that remembers no neighbour (seed_from_keys_kernel, grid.cu, and the
// first iteration of the multi-start kernel): the sorted position of a point of the smallest cell-tree node around the position
// that holds any point, or -1 (no finite target point, or a non-finite position).  The keys are sorted, so that point is the lower
// bound of the position's cell code or its predecessor -- whichever shares the longer prefix with the code.  The lower bound is
// searched inside the bucket of the code's most significant digit (msd_start, a by-product of the last sorting pass).
__device__ __forceinline__ int key_seed(const GridParams* __restrict__ gp, const unsigned int* __restrict__ keys, int n_finite,
                                        const unsigned int* __restrict__ msd_start, int msd_shift, float x, float y, float z) {
    if (!(n_finite > 0 && finite3(x, y, z))) return -1;
    const GridParams g = *gp;
    const unsigned int c = cell_code(g, x, y, z);
    int lo = (int)msd_start[c >> msd_shift], hi = (int)msd_start[(c >> msd_shift) + 1];
    if (hi > n_finite) hi = n_finite;
    if (lo > hi) lo = hi;
    while (lo < hi) {                                   // lower bound of c
        const int mid = (lo + hi) >> 1;
        if (keys[mid] < c) lo = mid + 1; else hi = mid;
    }
    int pos = lo;
    if (pos >= n_finite) pos = n_finite - 1;
    else if (pos > 0) {
        const unsigned int xa = keys[pos] ^ c, xb = keys[pos - 1] ^ c;
        if (xb < xa) pos = pos - 1;                     // smaller xor = longer common prefix
    }
    return pos;
}

// Early stop reached: the remaining launches of the registration are no-ops (query_matches, with a fixed descriptor, ignores it).
__device__ __forceinline__ bool registration_stopped(const MatchArgs& a) { return a.desc_index < 0 && a.state_ro->converged; }
__device__ __forceinline__ int iter_index(const MatchArgs& a) { return a.desc_index >= 0 ? a.desc_index : a.state_ro->iter; }   // a.desc[...] of this launch
__device__ __forceinline__ void stage_bvh_desc(BvhDesc& s, const BvhDesc* g) {
    if (threadIdx.x < sizeof(BvhDesc) / 4) reinterpret_cast<int*>(&s)[threadIdx.x] = reinterpret_cast<const int*>(g)[threadIdx.x];
    __syncthreads();
}

// Shared per-block copy of the pose and the normal matrix.
struct PoseSm { float P[16]; float N[9]; };
__device__ __forceinline__ void load_pose(PoseSm& sm, const DevState* st) {
    if (threadIdx.x < 16) sm.P[threadIdx.x] = st->pose[threadIdx.x];
    else if (threadIdx.x < 25) sm.N[threadIdx.x - 16] = st->nrm[threadIdx.x - 16];
    __syncthreads();
}

__device__ __forceinline__ void flush_stats(const MatchArgs& a, unsigned int nq, unsigned int nm, unsigned int ev, unsigned int nd) {
    if (!a.collect_stats) return;     // ~10^5 same-address atomics per launch are not free: off in timed runs
    DevState* st = a.state;
    nq = __reduce_add_sync(0xFFFFFFFFu, nq); nm = __reduce_add_sync(0xFFFFFFFFu, nm);
    // evals / nodes can exceed 32 bits only per launch, not per warp
    ev = __reduce_add_sync(0xFFFFFFFFu, ev); nd = __reduce_add_sync(0xFFFFFFFFu, nd);
    if ((threadIdx.x & 31) == 0) {
        if (nq) atomicAdd(&st->n_queries, (unsigned long long)nq);
        if (nm) atomicAdd(&st->n_matched, (unsigned long long)nm);
        if (ev) atomicAdd(&st->n_evals, (unsigned long long)ev);
        if (nd) atomicAdd(&st->n_nodes, (unsigned long long)nd);
    }
}
