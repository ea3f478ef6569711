// knn.cu -- the grid search: exact 1-NN (3-D / 6-D) over the target's BVH (grid.cu) -> nn_pos; stages 3-4 follow in match.cu.
// The reference's FLANN search (1 randomized kd-tree, 16 checks) is approximate; these kernels return the exact nearest neighbour
// under contract D1-D3 with ties to the lowest target index, i.e. what NearestNeighborSearchBruteForce's scan order
// (NearestNeighbor.h:81-97) yields on squared distances.
//   knn_prep_kernel   one thread per query: selection predicate + transform, and the FAST PATH: a query that remembers a
//                     neighbour scans that neighbour's leaf and, if its search ball stays inside the leaf's inflated box,
//                     the leaves of the leaf's adjacency list -- ~75 % of the queries end here.
//   knn_bvh_kernel    the rest: one warp per query walks a 32-ary bounding-volume hierarchy over the cell-sorted target
//                     (grid.cu) depth-first with an explicit shared-memory stack.  Leaves are the nodes of the
//                     implicit cell tree with <= 32 points (disjoint aligned cells, TIGHT boxes); an internal
//                     node groups 32 consecutive nodes of the level below.  One step tests the 32 children of a
//                     node in parallel (lane = child, one coalesced 1 KB read of boxes); a leaf is scanned by the
//                     32 lanes in parallel (lane = point, one coalesced 512 B read) with a warp arg-min at the end.
//                     Every query starts from an upper bound: the neighbour it had the last time it was matched
//                     (the pose moves little between ICP iterations), else the distance threshold.
//                     In the 6-D colour search every node also carries its colour range, added to the lower bounds.
//   knn_group_kernel  between the two (3-D search, thresholds that admit far matches): one warp per 32 consecutive positions; runs of
//                     deferred neighbours share ONE breadth-first descent, then every member is scanned against the few listed
//                     leaves its own ball meets.  What it finishes the walk skips; what outgrows its stage it leaves to the walk.
#include "search.cuh"

// ---------------------------------------------------------------------------- diagnostic build (-DICP_TIMELINE, profiles/)
// Start and end (%globaltimer, ns) of every warp of the search kernels of ONE iteration (ICP_TL_ITER), plain stores.
#ifdef ICP_TIMELINE
#define ICP_TL_ITER 12
#define ICP_TL_WARPS 40960
__device__ unsigned long long g_timeline[2][2][ICP_TL_WARPS][2];      // [kernel][chunk][warp]{start, end}
__device__ __forceinline__ unsigned long long tl_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
extern "C" int icp_gpu_debug_timeline(unsigned long long* out, int reset) {
    if (reset) { void* p = nullptr; cudaGetSymbolAddress(&p, g_timeline); return (int)cudaMemset(p, 0, sizeof(g_timeline)); }
    return (int)cudaMemcpyFromSymbol(out, g_timeline, sizeof(g_timeline));
}
#define TL_BEGIN(k, it, chunk) const int tl_w = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), tl_c = (chunk); \
    const bool tl_on = (it) == ICP_TL_ITER && (threadIdx.x & 31) == 0 && tl_w < ICP_TL_WARPS; if (tl_on) g_timeline[k][tl_c][tl_w][0] = tl_now()
#define TL_END(k) if (tl_on) g_timeline[k][tl_c][tl_w][1] = tl_now()
#else
#define TL_BEGIN(k, it, chunk)
#define TL_END(k)
#endif

// ---------------------------------------------------------------------------- BVH search, one warp per query
#define BVH_WARPS 4
#define BVH_STACK (32 * ICP_BVH_MAX_LEVELS)   // <= 32 pushed children per level

// Lane l proposes the leaf with points [ls, le) and box distance clb (keep = it can still matter): the proposed leaves are
// scanned nearest first (lane = point) for as long as their box distance does not exceed the shrinking bound.  The callers
// load the point ranges together with the boxes (one dependent memory round trip less per visited node: the walk is
// bound by the length of its chain of dependent loads).
template <bool COLOR>
__device__ __forceinline__ void bvh_scan_leaves(const MatchArgs& a, const Query& q, Best& b, float& bound, unsigned int ls, unsigned int le,
                                                float clb, bool keep, int lane, unsigned int& ev, unsigned int& nd) {
    const unsigned int FULL = 0xFFFFFFFFu;
    unsigned int key = keep ? __float_as_uint(clb) : 0xFFFFFFFFu;
    for (;;) {
        const unsigned int kmin = __reduce_min_sync(FULL, key);
        if (kmin == 0xFFFFFFFFu || __uint_as_float(kmin) > bound) break;
        const int src = __ffs((int)__ballot_sync(FULL, key == kmin)) - 1;
        const unsigned int s0 = __shfl_sync(FULL, ls, src), e0 = __shfl_sync(FULL, le, src);
        if (lane == src) key = 0xFFFFFFFFu;
        const unsigned int i = s0 + lane;
        if (i < e0) {
            const float4 pt = __ldg(&a.tgt_pts[i]);
            const float dd = dist2<COLOR>(q, pt, b.d, a.tgt_nrm, i);
            const int idx = __float_as_int(pt.w);
            if (better_key(dd, idx, b)) { b.d = dd; b.idx = idx; b.pos = (int)i; }
            ++ev;
        }
        if (lane == 0) ++nd;
        bound = __uint_as_float(__reduce_min_sync(FULL, __float_as_uint(b.d)));   // d >= 0: bit order = value order
    }
}

// Tests the nodes [first, last) (last - first <= 32) of level L against the query, lane = node.  Leaves that can still
// matter are scanned at once, nearest first (lane = point); internal nodes are pushed.
template <bool COLOR>
__device__ __forceinline__ void bvh_visit(const MatchArgs& a, const BvhDesc& bvh, const Query& q, Best& b, float& bound, int L,
                                          unsigned int first, unsigned int last, unsigned int* st_node, float* st_lb, int& top, int lane,
                                          unsigned int lt_mask, unsigned int& ev, unsigned int& nd) {
    const unsigned int FULL = 0xFFFFFFFFu;
    const unsigned int c = first + lane;
    float clb = FLT_BIG; bool keep = false;
    unsigned int ls = 0u, le = 0u;
    if (c < last) {
        const float4 lo = __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[L] + c)]), hi = __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[L] + c) + 1]);
        if (L == 0) { ls = __ldg(&a.leaf_start[c]); le = __ldg(&a.leaf_start[c + 1]); }
        clb = box_dist2c<COLOR>(q, lo, hi);
        keep = !(clb > bound);
    }
    if (L == 0) { bvh_scan_leaves<COLOR>(a, q, b, bound, ls, le, clb, keep, lane, ev, nd); return; }
    const unsigned int mk = __ballot_sync(FULL, keep);
    if (keep) { const int s = top + __popc(mk & lt_mask); st_node[s] = ((unsigned int)L << 27) | c; st_lb[s] = clb; }
    top += __popc(mk);
    __syncwarp();
}

// One thread scans one leaf for its own query (fast path of knn_prep_kernel).
template <bool COLOR>
__device__ __forceinline__ void thread_scan_range(const MatchArgs& a, const Query& q, Best& b, int& bleaf, unsigned int leaf, unsigned int ls, unsigned int le, unsigned int& ev) {
    // Contract D2 ((d, idx) lexicographic) without an index comparison per candidate: a leaf's records are stored in ORIGINAL index
    // order (grid.cu: bvh_level_kernel), so the first minimum of the distance in storage order is the lowest original index among
    // equal distances.  The scan accepts d <= the current best (`run` starts one ulp above it; d >= 0, so the bit pattern + 1 is the
    // next float) and the (d, idx) rule is applied once, to the leaf's winner.  This loop is a third of the kernel's instructions.
    if (b.d < 0.f) return;                          // a negative threshold admits nothing
    float run = __uint_as_float(__float_as_uint(b.d) + 1u);
    int pos = -1;
    for (unsigned int i = ls; i < le; ++i) {
        const float4 pt = __ldg(&a.tgt_pts[i]);
        const float dd = dist2<COLOR>(q, pt, run, a.tgt_nrm, i);
        if (dd < run) { run = dd; pos = (int)i; }
    }
    ev += le - ls;
    if (pos >= 0) {
        const int idx = __float_as_int(__ldg(&a.tgt_pts[pos].w));
        if (better_key(run, idx, b)) { b.d = run; b.idx = idx; b.pos = pos; bleaf = (int)leaf; }
    }
}
template <bool COLOR>
__device__ __forceinline__ void thread_scan_leaf(const MatchArgs& a, const Query& q, Best& b, int& bleaf, unsigned int leaf, unsigned int& ev) {
    thread_scan_range<COLOR>(a, q, b, bleaf, leaf, __ldg(&a.leaf_start[leaf]), __ldg(&a.leaf_start[leaf + 1]), ev);
}

// Thread per query: selection predicate + transformPoints -> qbuf, and the FAST PATH of the search.  A query that
// remembers a neighbour scans that neighbour's leaf by itself; if its search ball then lies inside the leaf's inflated box,
// the leaves that can still matter are all in the leaf's adjacency list (grid.cu) and the thread tests and scans them
// itself -- same candidates, same (d, idx) order, hence the same answer as the walk -- and marks the query as done
// (qbuf.x = NaN).  The 32 queries of a warp are spatial neighbours (sorted source), so their leaves coincide and the
// loads are mostly broadcasts.  Everything else (no neighbour yet, ball leaving the box) is left to knn_bvh_kernel.
#define KNN_PREP_THREADS 256
#define PREP_MIN_BLOCKS 5          // measured 5 / 6 / 7 / 8 blocks per SM: 60 / 67 / 78 / 79 us per launch (more blocks = spills)
template <bool COLOR, bool STATS>
__global__ void __launch_bounds__(KNN_PREP_THREADS, PREP_MIN_BLOCKS * 256 / KNN_PREP_THREADS) knn_prep_kernel(const MatchArgs a) {
    __shared__ PoseSm sm;
    const int p = a.q_begin + blockIdx.x * blockDim.x + threadIdx.x;
    // Everything that depends on nothing is requested first, so that the pose, the descriptor and the query's own state
    // arrive together (the kernel is bound by its chain of dependent loads, not by bandwidth).
    float4 p4 = make_float4(0.f, 0.f, 0.f, 0.f), n4 = p4;
    int sp_raw = -1, leaf_raw = -1;
    if (p < a.q_end) {
        p4 = __ldg(&a.src_pts[p]); n4 = __ldg(&a.src_nrm[p]);
        sp_raw = a.nn_pos[p]; leaf_raw = a.nn_leaf[p];          // leaf_raw is meaningless unless sp_raw is a position
    }
    if (registration_stopped(a)) return;
    const int desc_i = iter_index(a);
    TL_BEGIN(0, a.state_ro->iter, a.q_begin > 0 ? 1 : 0);
    load_pose(sm, a.state_ro);
    const IterDesc d = a.desc[desc_i];
    unsigned int ev = 0, nd = 0;
    if (p < a.q_end) {
        float4 o = make_float4(finished_mark(), 0.f, 0.f, n4.w);
        float4 seed = pack_handover(Best{0.f, 0, 0}, HANDOVER_NONE);
        if (query_active(d, a.mask, p4, n4)) {
            float x, y, z;
            xform_point(sm.P, p4.x, p4.y, p4.z, x, y, z);
            if (finite3(x, y, z)) {
                o.x = x; o.y = y; o.z = z;
                const int seed_leaf = (sp_raw >= 0 && sp_raw < a.n_tgt) ? leaf_raw : -1;
                if (seed_leaf >= 0 && seed_leaf < a.adj_capacity) {
                    Query q; q.x = x; q.y = y; q.z = z;
                    set_colour(q, __float_as_uint(n4.w));
                    Best b; best_init(b, a.max_d2);
                    int bleaf = -1;
                    thread_scan_leaf<COLOR>(a, q, b, bleaf, (unsigned int)seed_leaf, ev); ++nd;
                    seed = pack_handover(b, HANDOVER_NO_NODE);
                    if (b.d < FLT_BIG) {
                        const float r = search_radius(b.d);
                        const float4 ilo = __ldg(&a.adj_box[2 * (size_t)seed_leaf]), ihi = __ldg(&a.adj_box[2 * (size_t)seed_leaf + 1]);
                        if (ball_inside(x, y, z, r, ilo, ihi)) {                // never true for the inverted "no list" box
                            const int na = __float_as_int(ilo.w);
                            const unsigned int* list = a.adj + (size_t)seed_leaf * 32;
                            // two phases, so that the lanes of a warp scan their leaves side by side instead of one
                            // list position at a time: first the box tests, then the scans of the leaves that passed
                            unsigned int todo = 0;
                            // the list is in the order of the entries' gaps to the seed leaf's box: with the best candidate inside that
                            // box, an entry whose gap exceeds twice the search radius (4 x in squares, rounded up) cannot hold a nearer
                            // point, nor can any entry after it
                            const float* gap = a.adj_gap + (size_t)seed_leaf * 32;
                            const float lim = bleaf == seed_leaf ? __fmul_ru(__fmul_ru(4.0f, b.d), 1.00001f) : FLT_BIG;
                            for (int j = 0; j < na; ++j) {
                                if (__ldg(&gap[j]) > lim) break;
                                const unsigned int leaf = __ldg(&list[j]);
                                const float clb = box_dist2c<COLOR>(q, __ldg(&a.bvh_box[2 * (size_t)leaf]), __ldg(&a.bvh_box[2 * (size_t)leaf + 1]));
                                if (!(clb > b.d)) todo |= 1u << j;
                            }
                            while (todo) {
                                const int j = __ffs((int)todo) - 1; todo &= todo - 1u;
                                const unsigned int leaf = __ldg(&list[j]);
                                const float clb = box_dist2c<COLOR>(q, __ldg(&a.bvh_box[2 * (size_t)leaf]), __ldg(&a.bvh_box[2 * (size_t)leaf + 1]));
                                if (!(clb > b.d)) { thread_scan_leaf<COLOR>(a, q, b, bleaf, leaf, ev); ++nd; }
                            }
                            ++nd;
                            a.nn_pos[p] = b.idx == INT_MAX ? -1 : b.pos;
                            a.nn_leaf[p] = b.idx == INT_MAX ? -1 : bleaf;
                            mark_finished(o);                                   // searched: nothing left for the walk
                        } else if (a.adj1_capacity > 0 && a.bvh->n_levels >= 2) {
                            // left to the walk: does the ball at least stay inside the inflated box of the seed leaf's level-1 node?
                            // Then the walk starts from that node's list (lanes of deferred queries are otherwise idle here).
                            const int m = (int)(__ldg(&a.node_rank[a.bvh->coffset[1] + seed_leaf + 1]) - 1u);
                            if (m < a.adj1_capacity) {
                                const float4 jlo = __ldg(&a.adj1_box[2 * (size_t)m]), jhi = __ldg(&a.adj1_box[2 * (size_t)m + 1]);
                                if (ball_inside(x, y, z, r, jlo, jhi)) seed = pack_handover(b, m);
                            }
                        }
                    }
                }
            }
        }
        a.qbuf[p] = o;
        if (is_pending(o.x)) store_handover(a.seedbuf, p, seed);
    }
    TL_END(0);
    if (STATS) flush_stats(a, 0u, 0u, ev, nd);     // STATS = false: the counters are dead code (2.6 % of the walk's instructions)
}

// ---------------------------------------------------------------------------- group search: 32 neighbouring queries, ONE descent
// The queries the fast path defers come in runs: a scan region the target does not cover (an occlusion shadow, the far side of the
// sensor's field of view) is a run of Morton-consecutive source points whose search balls -- 0.2 ... 3 m wide -- all touch the same
// few target leaves at the edge of the covered region.  For such a query the walk's time goes into FINDING those leaves (about
// 11 node visits of 32 box tests each for 2-5 leaf scans), and its 31 neighbours repeat the same descent.  Here one warp takes 32
// consecutive positions of the sorted source (lane = query) and, if at least `group_min` of them were handed over with a bound,
// descends ONCE for all of them: a node is kept when its box meets the bounding box of the members' search balls AND lies within
// the largest member radius of the bounding box of the member points.  These bounds do not shrink during the descent, so it needs
// no order: it runs breadth-first, level by level (lane = child; the frontier's child ranges are fetched in one round, the next
// boxes of several nodes are requested together) -- a handful of dependent memory round trips instead of one per node.  The
// surviving leaves (boxes and point ranges staged in shared memory) are a superset of every member's candidates; each member then
// tests them against its own ball, and the few it still wants are scanned for it by the warp (lane = point) -- same candidates,
// same (d, idx) rule, hence the same answer as the walk.  A group whose frontier or list outgrows its stage (a run
// that jumps across the scene, a member without a neighbour inside the threshold) is left to the walk untouched.  A finished query
// is marked like one the fast path finished (qbuf.x = NaN), so the walk skips it.
#define GROUP_CAP 48           // candidate leaves per group   (the kernel ends with its longest group: 128 / 128 / unlimited measured
                               //                               4.39 -> 5.3 ms on the bench pair against 4.25 with 48 / 64 / 160)
#define GROUP_FRONT 64         // frontier nodes per level
#define GROUP_WARPS 4
#define GROUP_UNROLL 3
#define GROUP_STEP_LIMIT 160   // (member, leaf) scans per group
#define GROUP_SIZE 32          // consecutive positions per group (the members sit in the warp's first GROUP_SIZE lanes)
static_assert(GROUP_CAP <= GROUP_FRONT, "pass A keeps the want masks of the listed leaves in cfirst[]");
struct GroupStage {
    unsigned int front[2][GROUP_FRONT];                       // frontier of the level being expanded / of the next level
    unsigned int cfirst[GROUP_FRONT], clast[GROUP_FRONT];     // child ranges of the frontier's nodes
    float4 lo[GROUP_CAP], hi[GROUP_CAP];                      // candidate leaves: box, id, point range
    unsigned int leaf[GROUP_CAP], ls[GROUP_CAP], le[GROUP_CAP];
};
#ifdef ICP_GROUP_PROBE   // diagnostic build (make groupprobe, profiles/probe_group.py): per launch with collect_stats -- windows seen, groups
// started, finished, members finished, leaves listed, (member, leaf) scans, -, cycles of the descent, of the scans, longest group, box rounds
__device__ unsigned long long g_group_stats[12];
extern "C" int icp_gpu_debug_group_stats(unsigned long long* out12, int reset) {
    if (reset) { void* p = nullptr; cudaGetSymbolAddress(&p, g_group_stats); return (int)cudaMemset(p, 0, sizeof(g_group_stats)); }
    return (int)cudaMemcpyFromSymbol(out12, g_group_stats, sizeof(g_group_stats));
}
#define GROUP_PROBE(x) x
#else
#define GROUP_PROBE(x)
#endif
__device__ __forceinline__ unsigned int f2ord(float f) { const unsigned int u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float ord2f(unsigned int u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u); }
__device__ __forceinline__ float warp_min_f(float v) { return ord2f(__reduce_min_sync(0xFFFFFFFFu, f2ord(v))); }
__device__ __forceinline__ float warp_max_f(float v) { return ord2f(__reduce_max_sync(0xFFFFFFFFu, f2ord(v))); }

// Why no candidate is lost.  Let p be a target point that can change member m's answer: its D1 distance d(q_m, p) (fp32, rounded as
// contract D1 says) is <= the member's bound bd_m, the distance of a real point.  (1) |q_m.x - p.x| <= sqrt(bd_m) up to D1's rounding,
// which the factor 1.00001 of search_radius covers (the fast path's "inside" test makes the same step), so p lies in the box of m's
// ball [q_m - r_m, q_m + r_m] (bounds rounded outwards), hence in the union box [bl, bh]; every box of the hierarchy is the exact
// min / max of its points, so each ancestor box of p meets [bl, bh] -- comparisons only, nothing rounds.  (2) The gap between an
// ancestor box and the box [ql, qh] of the member points is, per axis, at most |q_m - p| on that axis, so its exact squared norm
// is <= the exact squared distance <= bd_m (1 + 4 ulp) <= the largest bound; the fp32 evaluation below (any association, FMA or not)
// is off by a few ulp, the margin 1.0001 by a thousand, and 1e-36 covers products that underflow.  Ties (equal distance, lower
// index) satisfy d <= bd_m as well.  So every leaf holding such a point survives both tests at every level.
struct GroupBounds { float blx, bly, blz, bhx, bhy, bhz, qlx, qly, qlz, qhx, qhy, qhz, dlim; };
__device__ __forceinline__ bool group_keeps(const GroupBounds& g, const float4 lo, const float4 hi) {
    const bool meets = lo.x <= g.bhx && hi.x >= g.blx && lo.y <= g.bhy && hi.y >= g.bly && lo.z <= g.bhz && hi.z >= g.blz;
    const float gx = fmaxf(fmaxf(lo.x - g.qhx, g.qlx - hi.x), 0.0f), gy = fmaxf(fmaxf(lo.y - g.qhy, g.qly - hi.y), 0.0f), gz = fmaxf(fmaxf(lo.z - g.qhz, g.qlz - hi.z), 0.0f);
    return meets && !(gx * gx + gy * gy + gz * gz > g.dlim);
}

// One warp: the group's bounds, the breadth-first descent and pass A (which members want which listed leaf).  Returns the number
// of wanted leaves, compacted to the front of the stage {leaf, ls, le, cfirst = mask of the wanting members} (0: the seed scans'
// results are final), or GROUP_LEFT: the group is too wide (frontier, list or number of scans beyond the stage) and is left to the walk.
#define GROUP_LEFT 0xFFFFFFFFu
__device__ __forceinline__ unsigned int group_collect(const MatchArgs& a, const BvhDesc& bvh, GroupStage& sm, const Query& q, bool member, float bd, int own,
                                                      int lane, unsigned int& nd, unsigned int& n_list_out, unsigned int& scans_out) {
    const unsigned int FULL = 0xFFFFFFFFu;
    // box of the members' balls (search_radius, as the fast path's "inside" test), box of the member points, largest squared
    // radius (with a margin that covers D1's roundings against the box-to-box gap of group_keeps)
    GroupBounds g;
    {
        const float INF = __int_as_float(0x7f800000);
        const float r = member ? search_radius(bd) : 0.f;
        g.blx = warp_min_f(member ? __fsub_rd(q.x, r) : INF); g.bhx = warp_max_f(member ? __fadd_ru(q.x, r) : -INF);
        g.bly = warp_min_f(member ? __fsub_rd(q.y, r) : INF); g.bhy = warp_max_f(member ? __fadd_ru(q.y, r) : -INF);
        g.blz = warp_min_f(member ? __fsub_rd(q.z, r) : INF); g.bhz = warp_max_f(member ? __fadd_ru(q.z, r) : -INF);
        g.qlx = warp_min_f(member ? q.x : INF); g.qhx = warp_max_f(member ? q.x : -INF);
        g.qly = warp_min_f(member ? q.y : INF); g.qhy = warp_max_f(member ? q.y : -INF);
        g.qlz = warp_min_f(member ? q.z : INF); g.qhz = warp_max_f(member ? q.z : -INF);
        g.dlim = __fadd_ru(__fmul_ru(warp_max_f(member ? bd : 0.f), 1.0001f), 1e-36f);
    }
    const unsigned int lt_mask = (1u << lane) - 1u;
    const int top_level = bvh.n_levels - 1;
    const unsigned int n_top = (unsigned int)bvh.count[top_level];
    unsigned int n_list = 0u, n_cur = 0u;
    int cur = 0;
    // top level: its nodes are tested directly (<= 32 of them unless the level cap was hit)
    for (unsigned int base = 0; base < n_top; base += 32) {
        const unsigned int c = base + lane;
        bool keep = false; float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo; unsigned int ls = 0u, le = 0u;
        if (c < n_top) {
            lo = __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[top_level] + c)]); hi = __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[top_level] + c) + 1]);
            if (top_level == 0) { ls = __ldg(&a.leaf_start[c]); le = __ldg(&a.leaf_start[c + 1]); }
            keep = group_keeps(g, lo, hi);
        }
        const unsigned int mk = __ballot_sync(FULL, keep);
        if (top_level == 0) {
            if (n_list + __popc(mk) > GROUP_CAP) return GROUP_LEFT;
            if (keep) { const unsigned int k = n_list + __popc(mk & lt_mask); sm.leaf[k] = c; sm.lo[k] = lo; sm.hi[k] = hi; sm.ls[k] = ls; sm.le[k] = le; }
            n_list += __popc(mk);
        } else {
            if (n_cur + __popc(mk) > GROUP_FRONT) return GROUP_LEFT;
            if (keep) sm.front[cur][n_cur + __popc(mk & lt_mask)] = c;
            n_cur += __popc(mk);
        }
        if (lane == 0) ++nd;
    }
    __syncwarp();
    // breadth-first: the frontier holds the kept nodes of level L; their children (level L - 1) are tested, lane = child
    for (int L = top_level; L >= 1 && n_cur > 0u; --L) {
        for (unsigned int j = lane; j < n_cur; j += 32) {
            const unsigned int node = sm.front[cur][j];
            sm.cfirst[j] = __ldg(&a.child_start[bvh.coffset[L] + node]); sm.clast[j] = __ldg(&a.child_start[bvh.coffset[L] + node + 1]);
        }
        __syncwarp();
        const bool to_leaves = L == 1;
        const size_t box0 = (size_t)bvh.offset[L - 1];
        unsigned int n_nxt = 0u;
        // the frontier in rounds of GROUP_UNROLL nodes: all their boxes are requested before the first is tested (one memory round
        // trip per round instead of one per node)
        for (unsigned int j0 = 0; j0 < n_cur; j0 += GROUP_UNROLL) {
            unsigned int c[GROUP_UNROLL], ls[GROUP_UNROLL], le[GROUP_UNROLL]; bool v[GROUP_UNROLL]; float4 lo[GROUP_UNROLL], hi[GROUP_UNROLL];
#pragma unroll
            for (int u = 0; u < GROUP_UNROLL; ++u) {
                v[u] = false; c[u] = 0u; ls[u] = 0u; le[u] = 0u; lo[u] = make_float4(0.f, 0.f, 0.f, 0.f); hi[u] = lo[u];
                if (j0 + u < n_cur) {
                    c[u] = sm.cfirst[j0 + u] + lane; v[u] = c[u] < sm.clast[j0 + u];
                    if (v[u]) {
                        lo[u] = __ldg(&a.bvh_box[2 * (box0 + c[u])]); hi[u] = __ldg(&a.bvh_box[2 * (box0 + c[u]) + 1]);
                        if (to_leaves) { ls[u] = __ldg(&a.leaf_start[c[u]]); le[u] = __ldg(&a.leaf_start[c[u] + 1]); }
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < GROUP_UNROLL; ++u) {
                if (j0 + u >= n_cur) break;
                const bool keep = v[u] && group_keeps(g, lo[u], hi[u]);
                const unsigned int mk = __ballot_sync(FULL, keep);
                if (to_leaves) {
                    if (n_list + __popc(mk) > GROUP_CAP) return GROUP_LEFT;             // too wide a group: left to the walk
                    if (keep) { const unsigned int k = n_list + __popc(mk & lt_mask); sm.leaf[k] = c[u]; sm.lo[k] = lo[u]; sm.hi[k] = hi[u]; sm.ls[k] = ls[u]; sm.le[k] = le[u]; }
                    n_list += __popc(mk);
                } else {
                    if (n_nxt + __popc(mk) > GROUP_FRONT) return GROUP_LEFT;
                    if (keep) sm.front[cur ^ 1][n_nxt + __popc(mk & lt_mask)] = c[u];
                    n_nxt += __popc(mk);
                }
                if (lane == 0) ++nd;
            }
        }
        __syncwarp();
        cur ^= 1; n_cur = n_nxt;
    }
    // pass A (shared memory only): which members' own balls does each listed leaf's box meet -- three of the 32 on average, none
    // for a quarter of the leaves; the list is compacted to the wanted leaves
    unsigned int scans = 0u, n_w = 0u;
    for (unsigned int j = 0; j < n_list; ++j) {
        const unsigned int leaf = sm.leaf[j];
        const bool want = member && (int)leaf != own && !(box_dist2(q.x, q.y, q.z, sm.lo[j], sm.hi[j]) > bd);
        const unsigned int wm = __ballot_sync(FULL, want);
        if (wm != 0u) {
            const unsigned int ls = sm.ls[j], le = sm.le[j];
            __syncwarp();
            if (lane == 0) { sm.leaf[n_w] = leaf; sm.ls[n_w] = ls; sm.le[n_w] = le; sm.cfirst[n_w] = wm; }   // n_w <= j: in place
            ++n_w; scans += __popc(wm);
        }
    }
    __syncwarp();
    n_list_out = n_list; scans_out = scans;
    // a group with too many (member, leaf) scans ahead is a long chain of dependent steps on few warps: left to the walk's many
    return scans > GROUP_STEP_LIMIT ? GROUP_LEFT : n_w;
}

// One warp per group.  (Measured and dropped: one block per group whose warps share the wanted leaves and merge their candidates
// by the (d, idx) order -- the descent is the latency-bound part and then runs on a quarter of the resident warps: 4.98 against 4.39 ms.)
template <bool STATS>
__global__ void __launch_bounds__(GROUP_WARPS * 32, 6) knn_group_kernel(const MatchArgs a) {
    __shared__ GroupStage s_stage[GROUP_WARPS];
    __shared__ BvhDesc s_bvh;
    if (registration_stopped(a)) return;
    stage_bvh_desc(s_bvh, a.bvh);
    const unsigned int FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const BvhDesc& bvh = s_bvh;
    if (bvh.n_leaves <= 0) return;
    GroupStage& sm = s_stage[wid];
    const long long pl = (long long)a.q_begin + (long long)(blockIdx.x * GROUP_WARPS + wid) * GROUP_SIZE + lane;
    const int p = (int)pl;
    float4 q4 = make_float4(finished_mark(), 0.f, 0.f, 0.f); HandOver sb = {{0.f, 0, 0}, HANDOVER_NONE};
    int own = -1;
    if (lane < GROUP_SIZE && pl < (long long)a.q_end) {
        q4 = a.qbuf[p];                                                          // plain loads: written by the launch before
        if (is_pending(q4.x)) { sb = a.seedbuf[p]; own = a.nn_leaf[p]; }         // own = the seed leaf (scanned by the fast path already)
    }
    // member: deferred by the fast path after its seed-leaf scan, with a neighbour inside the threshold (a query whose bound is the
    // threshold itself wants every leaf its threshold ball meets: such groups outgrow the stage, their descent would be wasted).
    // (Measured: members restricted to the queries whose ball leaves even the level-1 node's inflated box, HANDOVER_NO_NODE: 4.54
    // against 4.25 ms on the bench pair -- the nearer deferred queries are the ones that share their leaves best.)
    const bool member = is_pending(q4.x) && handed_over(sb) && sb.best.idx != INT_MAX;
    const int n_members = __popc(__ballot_sync(FULL, member));
    GROUP_PROBE(if (STATS && lane == 0) { atomicAdd(&g_group_stats[0], 1ull); if (n_members >= a.group_min) atomicAdd(&g_group_stats[1], 1ull); })
    if (n_members < a.group_min) return;                                         // (whole warp)
    GROUP_PROBE(long long t_0 = 0; long long t_2 = 0; if (STATS) t_0 = clock64();)
    Query q; q.x = q4.x; q.y = q4.y; q.z = q4.z;
    q.cr = q.cg = q.cb = 0.f;                                                   // 3-D search only (icp_launch_match)
    unsigned int ev = 0, nd = 0, n_list = 0u, scans = 0u;
    const unsigned int n_w = group_collect(a, bvh, sm, q, member, sb.best.d, own, lane, nd, n_list, scans);
    if (n_w == GROUP_LEFT) return;                                               // (whole warp) left to the walk
    GROUP_PROBE(if (STATS) t_2 = clock64();)
    // Pass B: the scan is transposed -- the leaf's points sit in the lanes (lane = point, one coalesced read, three leaves in flight),
    // the wanting members take turns, two at a time (independent chains), each broadcasting its query and receiving the leaf's
    // (d, idx) minimum by a warp arg-min: the walk's leaf scan (bvh_scan_leaves) without the walk.
    Best b = sb.best;
    int bleaf = -1;
    float4 pf[3];
#pragma unroll
    for (int u = 0; u < 3; ++u) {
        pf[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        const unsigned int j = (unsigned int)u;
        if (j < n_w) {
            const unsigned int i = sm.ls[j] + lane;
            if (i < sm.le[j]) pf[u] = __ldg(&a.tgt_pts[i]);
        }
    }
    for (unsigned int j0 = 0; j0 < n_w; j0 += 3) {
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const unsigned int j = j0 + u;
            if (j >= n_w) break;
            const float4 pt = pf[u];
            if (j + 3 < n_w) {
                const unsigned int i = sm.ls[j + 3] + lane;
                if (i < sm.le[j + 3]) pf[u] = __ldg(&a.tgt_pts[i]);
            }
            const unsigned int leaf = sm.leaf[j], ls = sm.ls[j], cnt = sm.le[j] - ls;
            unsigned int wm = sm.cfirst[j];
            const bool has = (unsigned int)lane < cnt;
            const int pidx = __float_as_int(pt.w);
            while (wm) {
                const int m0 = __ffs((int)wm) - 1; wm &= wm - 1u;
                const bool two = wm != 0u;
                const int m1 = two ? __ffs((int)wm) - 1 : m0; wm &= wm - 1u;      // (0 & anything = 0)
                Query q0, q1; Best b0, b1;
                q0.x = __shfl_sync(FULL, q.x, m0); q0.y = __shfl_sync(FULL, q.y, m0); q0.z = __shfl_sync(FULL, q.z, m0);
                q1.x = __shfl_sync(FULL, q.x, m1); q1.y = __shfl_sync(FULL, q.y, m1); q1.z = __shfl_sync(FULL, q.z, m1);
                b0.d = __shfl_sync(FULL, b.d, m0); b0.idx = __shfl_sync(FULL, b.idx, m0); b0.pos = -1;
                b1.d = __shfl_sync(FULL, b.d, m1); b1.idx = __shfl_sync(FULL, b.idx, m1); b1.pos = -1;
                unsigned int key0 = 0xFFFFFFFFu, key1 = 0xFFFFFFFFu;
                if (has) {
                    key0 = __float_as_uint(dist3(q0.x, q0.y, q0.z, pt)); key1 = __float_as_uint(dist3(q1.x, q1.y, q1.z, pt));
                }
                ev += has ? (two ? 2u : 1u) : 0u;
                const unsigned int dmin0 = __reduce_min_sync(FULL, key0), dmin1 = __reduce_min_sync(FULL, key1);
                const int cand0 = (has && key0 == dmin0) ? pidx : INT_MAX, cand1 = (has && key1 == dmin1) ? pidx : INT_MAX;
                const int imin0 = __reduce_min_sync(FULL, cand0), imin1 = __reduce_min_sync(FULL, cand1);
                if (imin0 != INT_MAX && better_key(__uint_as_float(dmin0), imin0, b0)) {
                    const int src = __ffs((int)__ballot_sync(FULL, cand0 == imin0)) - 1;
                    if (lane == m0) { b.d = __uint_as_float(dmin0); b.idx = imin0; b.pos = (int)(ls + src); bleaf = (int)leaf; }
                }
                if (two && imin1 != INT_MAX && better_key(__uint_as_float(dmin1), imin1, b1)) {
                    const int src = __ffs((int)__ballot_sync(FULL, cand1 == imin1)) - 1;
                    if (lane == m1) { b.d = __uint_as_float(dmin1); b.idx = imin1; b.pos = (int)(ls + src); bleaf = (int)leaf; }
                }
            }
        }
    }
    if (member) {
        const int pos = b.idx == INT_MAX ? -1 : b.pos;
        a.nn_pos[p] = pos;
        a.nn_leaf[p] = pos >= 0 ? (bleaf >= 0 ? bleaf : own) : -1;                // no better point than the seed scan's: it lies in the seed leaf
        mark_finished(a.qbuf[p]);                                                // searched: nothing left for the walk
    }
    if (STATS) {
#ifdef ICP_GROUP_PROBE
        const long long t_3 = clock64();
        if (lane == 0) {
            atomicAdd(&g_group_stats[7], (unsigned long long)(t_2 - t_0)); atomicAdd(&g_group_stats[8], (unsigned long long)(t_3 - t_2));
            atomicMax(&g_group_stats[9], (unsigned long long)(t_3 - t_0)); atomicAdd(&g_group_stats[10], (unsigned long long)nd);
            atomicAdd(&g_group_stats[2], 1ull); atomicAdd(&g_group_stats[3], (unsigned long long)n_members);
            atomicAdd(&g_group_stats[4], (unsigned long long)n_list); atomicAdd(&g_group_stats[5], (unsigned long long)scans);
        }
#endif
        flush_stats(a, 0u, 0u, ev, nd);
    }
}

#define WALK_MIN_BLOCKS 16         // 32 registers: all 64 warp slots of an SM (the walk is latency-bound: 11 / 8 / 5 resident blocks
                                   // measured 150 / 196 / 241 us per launch against 118 at 16)
#define WALK_GRID_PER_SM 64        // blocks of 4 warps per SM in the walk's grid: 128 / 192 / 256 measured 4.65 / 4.88 / 4.86 ms per
                                   // registration against 4.53 (DESIGN §4)

// The warp scans one leaf, lane = point; every lane keeps its own best.
template <bool COLOR>
__device__ __forceinline__ void warp_scan_leaf(const MatchArgs& a, const Query& q, Best& b, unsigned int leaf, int lane, unsigned int& ev) {
    const unsigned int i = __ldg(&a.leaf_start[leaf]) + lane;
    if (i < __ldg(&a.leaf_start[leaf + 1])) {
        const float4 c = __ldg(&a.tgt_pts[i]);
        const float dd = dist2<COLOR>(q, c, b.d, a.tgt_nrm, i);
        const int idx = __float_as_int(c.w);
        if (better_key(dd, idx, b)) { b.d = dd; b.idx = idx; b.pos = (int)i; }
        ++ev;
    }
}

template <bool COLOR, bool STATS>
__global__ void __launch_bounds__(BVH_WARPS * 32, WALK_MIN_BLOCKS) knn_bvh_kernel(const MatchArgs a) {
    __shared__ unsigned int s_node[BVH_WARPS][BVH_STACK];
    __shared__ float s_lb[BVH_WARPS][BVH_STACK];
    __shared__ BvhDesc s_bvh;
    if (registration_stopped(a)) return;
    stage_bvh_desc(s_bvh, a.bvh);
    const unsigned int FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const BvhDesc& bvh = s_bvh;
    const int top_level = bvh.n_levels - 1;
    const unsigned int n_top = (unsigned int)bvh.count[top_level];
    unsigned int ev = 0, nd = 0;
    unsigned int* st_node = s_node[wid]; float* st_lb = s_lb[wid];
    const unsigned int lt_mask = (1u << lane) - 1u;
    if (bvh.n_leaves <= 0) return;                 // empty target: match_finish_kernel sees nn_pos = -1 (set_target reset it)
    TL_BEGIN(1, a.state_ro->iter, a.q_begin > 0 ? 1 : 0);
    // The warp's positions are p0, p0 + warps, p0 + 2 warps, ...; three quarters of them were answered by the fast path.
    // Lane k fetches the transformed query of position p0 + k * warps, so that one round of loads (instead of one
    // dependent load per position) tells the warp which positions it has to search.
    const int p0 = a.q_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    for (int pb = p0; pb < a.q_end; pb += 32 * warps) {
      const long long pl = (long long)pb + (long long)lane * warps;
      float qx = finished_mark();
      if (pl < (long long)a.q_end) qx = __ldg(&a.qbuf[pl].x);
      unsigned int todo = __ballot_sync(FULL, is_pending(qx));
      while (todo) {
        const int k = __ffs((int)todo) - 1; todo &= todo - 1u;
        const int p = pb + k * warps;
        const float4 q4 = __ldg(&a.qbuf[p]);                                    // its sector was fetched a moment ago
        Query q; q.x = q4.x; q.y = q4.y; q.z = q4.z;
        set_colour(q, __float_as_uint(q4.w));
        Best b; best_init(b, a.max_d2);
        // Start from the neighbour this query had before: scan that neighbour's whole leaf (lane = point).  After a
        // small pose change the new neighbour is almost always in it, so the search starts with a (nearly) final bound.
        int seed_leaf = -1;
        const HandOver sb = load_handover(a.seedbuf, p);
        const bool handed = handed_over(sb);
        if (handed) {
            if (lane == 0) b = sb.best;
        } else {
            const int sp = a.nn_pos[p];
            if (sp >= 0 && sp < a.n_tgt) {
                seed_leaf = a.nn_leaf[p];
                warp_scan_leaf<COLOR>(a, q, b, (unsigned int)seed_leaf, lane, ev);
                if (lane == 0) ++nd;
            }
        }
        bool done = false;
        if ((handed ? sb.node >= 0 : seed_leaf >= 0) && bvh.n_levels >= 2 && a.adj1_capacity > 0) {
            // Shortcut without the whole tree: the ball inside the inflated box of the seed leaf's level-1 node => every level-1
            // node that meets the ball is in that node's list (grid.cu); their leaves are tested 32 at a time.  For a query handed
            // over with a node (sb.node = m) the fast path made the containment test.
            const int m = handed ? sb.node : (int)(__ldg(&a.node_rank[bvh.coffset[1] + seed_leaf + 1]) - 1u);
            float bnd = __uint_as_float(__reduce_min_sync(FULL, __float_as_uint(b.d)));
            if (m < a.adj1_capacity && bnd < FLT_BIG) {
                const float4 ilo = __ldg(&a.adj1_box[2 * (size_t)m]);
                if (handed || ball_inside(q.x, q.y, q.z, search_radius(bnd), ilo, __ldg(&a.adj1_box[2 * (size_t)m + 1]))) {
                    const int na = __float_as_int(ilo.w);
                    unsigned int node = 0; unsigned int key = 0xFFFFFFFFu;
                    unsigned int cfirst = 0u, clast = 0u;                        // the node's children, loaded with the boxes (not after the pick)
                    if (lane < na) {
                        node = __ldg(&a.adj1[(size_t)m * 32 + lane]);
                        cfirst = __ldg(&a.child_start[bvh.coffset[1] + node]); clast = __ldg(&a.child_start[bvh.coffset[1] + node + 1]);
                        const float clb = box_dist2c<COLOR>(q, __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[1] + node)]), __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[1] + node) + 1]));
                        if (!(clb > bnd)) key = __float_as_uint(clb);
                    }
                    if (lane == 0) ++nd;
                    int top = 0;
                    for (;;) {                                                   // the level-1 nodes that can matter, nearest first
                        const unsigned int kmin = __reduce_min_sync(FULL, key);
                        if (kmin == 0xFFFFFFFFu || __uint_as_float(kmin) > bnd) break;
                        const int src = __ffs((int)__ballot_sync(FULL, key == kmin)) - 1;
                        const unsigned int first = __shfl_sync(FULL, cfirst, src), last = __shfl_sync(FULL, clast, src);
                        if (lane == src) key = 0xFFFFFFFFu;
                        if (lane == 0) ++nd;
                        bvh_visit<COLOR>(a, bvh, q, b, bnd, 0, first, last, st_node, st_lb, top, lane, lt_mask, ev, nd);
                    }
                    done = true;
                }
            }
        }
        if (!done && !__any_sync(FULL, b.pos >= 0) && bvh.n_levels > 1) {
            // No neighbour remembered (first iteration): follow the nearest node down to one leaf and take its best
            // point as the starting bound, so that the walk below prunes from its first step on.
            int L = top_level; unsigned int first = 0, last = n_top;
            unsigned int best_node = 0;
            for (;;) {
                unsigned int kbest = 0xFFFFFFFFu; best_node = first;
                for (unsigned int base = first; base < last; base += 32) {
                    const unsigned int c = base + lane;
                    unsigned int key = 0xFFFFFFFFu;
                    if (c < last) {
                        const float4 lo = __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[L] + c)]), hi = __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[L] + c) + 1]);
                        key = __float_as_uint(box_dist2c<COLOR>(q, lo, hi));
                    }
                    const unsigned int kmin = __reduce_min_sync(FULL, key);
                    if (kmin < kbest) { kbest = kmin; best_node = base + (unsigned int)(__ffs((int)__ballot_sync(FULL, key == kmin)) - 1); }
                }
                if (L == 0) break;
                first = __ldg(&a.child_start[bvh.coffset[L] + best_node]); last = __ldg(&a.child_start[bvh.coffset[L] + best_node + 1]);
                --L;
            }
            warp_scan_leaf<COLOR>(a, q, b, best_node, lane, ev);
        }
        float bound = __uint_as_float(__reduce_min_sync(FULL, __float_as_uint(b.d)));
        int top = 0;
        // the nodes of the top level (<= 32 unless the level cap was hit), 32 at a time, each batch followed depth-first
        for (unsigned int base = 0; base < n_top && !done; base += 32) {
            bvh_visit<COLOR>(a, bvh, q, b, bound, top_level, base, min(base + 32u, n_top), st_node, st_lb, top, lane, lt_mask, ev, nd);
            if (lane == 0) ++nd;
            while (top > 0) {
                --top;
                const unsigned int nd_id = st_node[top]; const float nlb = st_lb[top];
                __syncwarp();
                if (nlb > bound) continue;
                const int lvl = (int)(nd_id >> 27); const unsigned int j = nd_id & 0x7FFFFFFu;
                if (lane == 0) ++nd;
                const unsigned int first = __ldg(&a.child_start[bvh.coffset[lvl] + j]), last = __ldg(&a.child_start[bvh.coffset[lvl] + j + 1]);
                bvh_visit<COLOR>(a, bvh, q, b, bound, lvl - 1, first, last, st_node, st_lb, top, lane, lt_mask, ev, nd);
            }
        }
        // warp arg-min on (d, idx)
        const unsigned int dmin = __reduce_min_sync(FULL, __float_as_uint(b.d));
        const int cand = (__float_as_uint(b.d) == dmin) ? b.idx : INT_MAX;
        const int imin = __reduce_min_sync(FULL, cand);
        const int src_lane = __ffs((int)__ballot_sync(FULL, cand == imin)) - 1;
        const int pos = imin == INT_MAX ? -1 : __shfl_sync(FULL, b.pos, src_lane);
        if (lane == 0) {
            a.nn_pos[p] = pos;
            a.nn_leaf[p] = pos >= 0 ? (int)(__ldg(&a.leaf_rank[pos + 1]) - 1u) : -1;      // off the critical path: nothing waits for it
        }
      }
    }
    TL_END(1);
    if (STATS) flush_stats(a, 0u, 0u, ev, nd);     // STATS = false: the counters are dead code (2.6 % of the walk's instructions)
}

void icp_launch_knn(const MatchArgs& a, int n_sms, cudaStream_t s, cudaEvent_t after_prep, const MatchChunks* chunks, int& launches) {
    // One chunk of queries = one {prep, walk} chain; the chains run side by side on their own streams between a fork and a
    // join (MatchChunks): the block scheduler fills the ramps and tails of one chain's kernels with the other's blocks.
    int K = (chunks && !after_prep) ? chunks->n : 1;
    if (K < 1) K = 1;
    long long per = ((long long)a.n_src + K - 1) / K;
    per = (per + KNN_PREP_THREADS - 1) / KNN_PREP_THREADS * KNN_PREP_THREADS;    // whole prep blocks
    if (K > 1) cudaEventRecord(chunks->fork, s);
    for (int c = 0; c < K; ++c) {
        MatchArgs ac = a;
        ac.q_begin = (int)std::min<long long>((long long)c * per, a.n_src);
        ac.q_end = (int)std::min<long long>((long long)(c + 1) * per, a.n_src);
        const int nq = ac.q_end - ac.q_begin;
        if (nq <= 0) continue;
        cudaStream_t cs = c == 0 ? s : chunks->stream[c - 1];
        if (c > 0) cudaStreamWaitEvent(cs, chunks->fork, 0);
        const int np = (nq + KNN_PREP_THREADS - 1) / KNN_PREP_THREADS;
        if (a.collect_stats) { if (a.color_icp) knn_prep_kernel<true, true><<<np, KNN_PREP_THREADS, 0, cs>>>(ac); else knn_prep_kernel<false, true><<<np, KNN_PREP_THREADS, 0, cs>>>(ac); }
        else { if (a.color_icp) knn_prep_kernel<true, false><<<np, KNN_PREP_THREADS, 0, cs>>>(ac); else knn_prep_kernel<false, false><<<np, KNN_PREP_THREADS, 0, cs>>>(ac); }
        ++launches;
        if (after_prep) cudaEventRecord(after_prep, s);
        // runs of deferred neighbours share one descent (knn_group_kernel); what it leaves goes to the walk
        // Policy: on when the matcher's threshold admits far matches (max distance^2 >= 1: the reference's ETH driver uses 10,
        // main.cpp:361) -- runs of far queries with a neighbour are what the group search is for (3 M-point pair 61.7 -> 47.8 ms,
        // 44-pair queue 291 -> 324 pairs/s, far-heavy pairs -18 %; the bench pair +0.5 %); with a tight threshold (0.1 in the
        // experiment runner) the far queries have no neighbour, the groups that remain cost more than they save (4.0 -> 4.75 ms).
        const int group_min = getenv("ICP_GPU_GROUP_MIN") ? atoi(getenv("ICP_GPU_GROUP_MIN")) : (a.max_d2 >= 1.0f ? 8 : 0);   // test hook; 0 = off
        // (3-D search only: a 6-D bound holds colour differences too, as a radius in space it makes every group too wide)
        if (group_min > 0 && !a.color_icp) {
            ac.group_min = group_min;
            const int ng = (nq + GROUP_SIZE * GROUP_WARPS - 1) / (GROUP_SIZE * GROUP_WARPS);
            if (a.collect_stats) knn_group_kernel<true><<<ng, GROUP_WARPS * 32, 0, cs>>>(ac); else knn_group_kernel<false><<<ng, GROUP_WARPS * 32, 0, cs>>>(ac);
            ++launches;
        }
        // every chunk's walk gets the full grid (its warps then take fewer positions each): a heavy chunk left alone at the end
        // of the iteration still fills the machine
        int nb = (nq + BVH_WARPS - 1) / BVH_WARPS;
        const int cap = std::max(1, WALK_GRID_PER_SM * n_sms * 4 / BVH_WARPS);
        if (nb > cap) nb = cap;
        if (a.collect_stats) { if (a.color_icp) knn_bvh_kernel<true, true><<<nb, BVH_WARPS * 32, 0, cs>>>(ac); else knn_bvh_kernel<false, true><<<nb, BVH_WARPS * 32, 0, cs>>>(ac); }
        else { if (a.color_icp) knn_bvh_kernel<true, false><<<nb, BVH_WARPS * 32, 0, cs>>>(ac); else knn_bvh_kernel<false, false><<<nb, BVH_WARPS * 32, 0, cs>>>(ac); }
        ++launches;
        if (c > 0) { cudaEventRecord(chunks->done[c - 1], cs); cudaStreamWaitEvent(s, chunks->done[c - 1], 0); }
    }
}
