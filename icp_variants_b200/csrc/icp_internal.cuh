// icp_internal.cuh -- shared device/host declarations of libicp_gpu (sm_100a).
//
// Numerics contract (DESIGN.md "Numerics contract"; the oracle follows the same one):
//   D1 squared distance: fp32, dx=q-p.., ((dx*dx+dy*dy)+dz*dz) [+dr^2, +dg^2, +db^2], no FMA
//   D2 ties -> lowest original target index;  D3 valid iff d2 <= max (fp32)
//   D4 transform ((r0*x+r1*y)+r2*z)+t in fp32, no FMA; normals with the cofactor inverse-transpose
//   D5 normal equations in fp64 from fp32 inputs; solve in fp64; increment rounded to fp32;
//      pose product in fp32, no FMA
//   D6 rejection: acos(c) > 60 deg  <=>  -1 <= c <= 0.5f
// Everything that must be bit-exact goes through the p* helpers below (explicit round-to-nearest
// intrinsics are never contracted into FMAs by nvcc).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/icp_gpu.h"

#define ICP_MAX_ITERS 256          // upper bound on iterations per estimate_pose call
#define ICP_NRED 32                // doubles per partial-sum row (27..30 used)
#define ICP_REDUCE_THREADS 256
#define ICP_MAX_PEERS 8            // ranks of one point-sharded registration (one B200 box); <= ICP_REDUCE_THREADS / 32
#define ICP_MATCH_THREADS 128
#define ICP_LEAF_MAX 8             // a grid node with <= this many points is scanned, not split
#define ICP_CELLS_PER_POINT 32      // target grid: cells per point (2^T >= this x N); the finer, the more compact the BVH leaves
#define ICP_SOURCE_CELLS_PER_POINT 4 // source grid (sort order + voxel pyramid only); oracle/icp_oracle.c:orc_pick_T restates it
#define ICP_MAX_BITS_PER_AXIS 10   // keeps the cell-index rounding error << the bound margin

__device__ __forceinline__ float pmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float padd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float psub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float pdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ bool finite3(float x, float y, float z) { return isfinite(x) && isfinite(y) && isfinite(z); }
// The ball of radius r around (x, y, z) lies inside the box [lo, hi].  The ball's bounds are rounded outwards by the explicit _rd / _ru
// operations, so the answer does not depend on FMA contraction (-fmad) and holds for the exact ball.
__device__ __forceinline__ bool ball_inside(float x, float y, float z, float r, const float4 lo, const float4 hi) {
    return __fsub_rd(x, r) >= lo.x && __fadd_ru(x, r) <= hi.x && __fsub_rd(y, r) >= lo.y &&
           __fadd_ru(y, r) <= hi.y && __fsub_rd(z, r) >= lo.z && __fadd_ru(z, r) <= hi.z;
}

// Implicit binary tree over a dense table of 2^T Morton-ordered cells (see grid.cu).
struct GridParams {
    float o[3];       // origin = min finite coordinate per axis
    float h[3];       // cell size per axis at full depth
    float inv_h[3];
    float delta[3];   // bound margin: every point of cell k lies in [o+k*h-delta, o+(k+1)*h+delta]
    int bits[3];      // bits per axis, sum = T
    int T;            // depth of the implicit tree, 2^T cells
    unsigned long long axis_seq;  // 2 bits per level, level 0 (root split) in the low bits
    int n_finite;     // unused (the sort counts the non-finite points instead)
    int pad;
    unsigned char bitpos[3][ICP_MAX_BITS_PER_AXIS];   // bit j of axis a's cell index is bit bitpos[a][j] of the cell code
    unsigned char pad2[2];
};

// Bounding-volume hierarchy over the cell-sorted target (grid.cu), fan-out <= 32.  Every node of every level is
// a node of the implicit cell tree (an aligned box of the grid), so the nodes of one level are pairwise disjoint
// in space: level 0 = leaves = cell-tree nodes with <= 32 points (leaf j = sorted points [leaf_start[j],
// leaf_start[j+1])); a level-l node = a cell-tree node with <= 32 nodes of level l-1 (its children are the
// consecutive nodes [child_start[coffset[l]+j], child_start[coffset[l]+j+1]) of level l-1).  Every node stores the
// TIGHT axis-aligned box of its points as two float4 {lo.xyz,_} {hi.xyz,_} at box[2*(offset[l]+j)].  The top level
// is the first one with <= 32 nodes (a search tests all of them in one step).  Node counts are only known on the
// device, so the descriptor lives in device memory.
#define ICP_BVH_MAX_LEVELS 7
struct BvhDesc {
    int n_levels;                      // levels 0 .. n_levels-1
    int n_leaves;
    int count[ICP_BVH_MAX_LEVELS];     // nodes per level
    int offset[ICP_BVH_MAX_LEVELS];    // first node of the level in the box array and in pstart[]
    int coffset[ICP_BVH_MAX_LEVELS];   // first entry of the level in child_start[] (count+1 entries per level >= 1)
};

// One ICP iteration's query set.  Queries are addressed by p = position in the Morton-sorted source
// (grid.cu); the sorted source keeps the original index in pts.w.  Query p is active iff
//   orig % stride == 0                           (PointCloud.h:325-343 level stride; 1 = all)
//   and (filter_finite == 0 or point and normal finite)          (PointCloud.h:335)
//   and (mask_word_offset < 0 or bit `orig` of the mask is set)  (selection.h:88-104, drawn on the host)
//   and (proba < 0 or hash(rng_key, orig) < proba)               (device selection stream)
struct IterDesc {
    int stride;
    int filter_finite;
    int mask_word_offset;   // offset (32-bit words) into the selection mask array, or -1
    unsigned int rng_key;
    float proba;
    int pad0, pad1, pad2;
};

// The multi-resolution schedule of estimatePose (ICPOptimizer.h:503-525, :634-655) for a source of n points: the level strides
// coarsest, coarsest / 2, ..., 1, one iteration at every stride above 1, the remaining iterations at stride 1.  make_plan,
// icp_gpu_iterations_bound and the batch kernels all read it from here.
struct IcpSchedule {
    int coarsest;   // stride of iteration 0 (a power of two; 1 without multires)
    int levels;     // log2(coarsest) + 1
    int n_iters;    // iterations run at most: n_iterations, or max(n_iterations, levels) with multires
};
__host__ __device__ inline IcpSchedule icp_schedule(int n_iterations, int multires, long long n) {
    IcpSchedule s; s.coarsest = 1; s.levels = 1; s.n_iters = n_iterations;
    if (!multires) return s;
    float res = 1.0f; int sz = (int)n;                                    // ICPOptimizer.h:503-516
    for (;;) { sz = (int)(sz / 2.0); if (sz < 100) break; res *= 2.0f; }
    s.coarsest = (int)res;
    for (int c = s.coarsest; c > 1; c /= 2) ++s.levels;
    if (s.levels > s.n_iters) s.n_iters = s.levels;
    return s;
}
// stride and pyramid level (0 = coarsest) of iteration i
__host__ __device__ inline int icp_schedule_stride(const IcpSchedule& s, int i) { return i < s.levels ? s.coarsest >> i : 1; }
__host__ __device__ inline int icp_schedule_level(const IcpSchedule& s, int i) { return i < s.levels ? i : s.levels - 1; }

// Levenberg-Marquardt trust-region state of one outer iteration (lm.cuh); lives in DevState (lm.cu) or in a batch block's shared
// memory (batch.cu)
struct LmState {
    double x[6], cand[6], cost, H[36], g[6], scale[6], diag[6];
    double radius, decrease, model_change;
    int iter, done, reuse_diag, invalid, step_ok, have_cand;
};

// Device-resident loop state; one per context.
struct DevState {
    float pose[16];      // current estimate, column-major
    float nrm[9];        // (R^-1)^T row-major, rebuilt whenever pose changes
    int iter;            // iterations launched so far in this call (indexes the descriptors)
    int iters_done;      // iterations whose increment was applied
    int status;          // 0 or first ICP_GPU_E_* raised on the device
    unsigned int ticket; // last-block ticket of the reduction
    unsigned int ticket2;
    float mean_s[3];     // unweighted means of the kept matches (symmetric metric), rounded to fp32
    float mean_d[3];
    double mean_s64[3], mean_d64[3];
    unsigned long long n_queries, n_matched, n_evals, n_nodes;
    LmState lm;          // Levenberg-Marquardt state (lm.cu)
    double shard_partials[ICP_NRED];
    unsigned int xchg_seq;   // peer exchanges completed since the mailboxes were attached (never reset by pose_init)
    int pad_xchg;
    // early stop (icp_gpu_config.early_stop_*; 0 = off): set once an applied increment is smaller than both thresholds; every
    // later launch of the registration then returns at once
    float stop_rot, stop_trans; int converged; int pad_stop;
    unsigned long long prof[6];   // ReduceArgs::profile: %globaltimer marks of the last reduction launch (icp_gpu_stats)
};

// Point-sharded registration over peer memory (NVLink): every rank owns one mailbox; the last block of a reduction
// STORES its summed row straight into every peer's mailbox and waits for the peers' rows in its own -- the all-reduce of
// the <= 32 doubles is part of the reduction kernel, nothing returns to the host between iterations.
// Two slots (exchange number & 1): a rank can be at most one exchange ahead of a peer, because finishing exchange k
// needs every peer's row k, which a peer only sends after it has read all rows of exchange k-1.
struct PeerBox {
    double row[2][ICP_MAX_PEERS][ICP_NRED];
    unsigned int flag[2][ICP_MAX_PEERS];       // exchange number whose row is complete
};

struct PeerXchg {
    int world, rank;                   // world <= 1: no exchange
    unsigned long long timeout_ns;     // a peer that does not show up raises ICP_GPU_E_PEER instead of hanging the GPU
    int plan_check;                    // iterations + metric / minimiser this rank planned: element 31 of every row carries it, ranks that disagree raise ICP_GPU_E_PEER
    int pad_;
    PeerBox* box[ICP_MAX_PEERS];       // box[j] = rank j's mailbox as mapped into this process (box[rank] = own)
};

struct MatchArgs {
    // source, Morton-sorted (grid.cu): pts {x,y,z,orig idx bits}, nrm {nx,ny,nz,rgba bits}
    const float4* src_pts;
    const float4* src_nrm;
    int n_src;
    const unsigned int* mask; // selection masks (bit per original source index), all iterations concatenated
    const IterDesc* desc;    // [ICP_MAX_ITERS + 2]
    const DevState* state_ro;
    DevState* state;
    // target
    const float4* tgt_pts;   // grid order {x,y,z,orig idx bits}; brute / projective: original order
    const float4* tgt_nrm;   // same order {nx,ny,nz,rgba bits}
    int n_tgt;
    const float4* bvh_box;   // tight boxes of the BVH nodes (grid order only)
    const BvhDesc* bvh;      // device-resident
    const unsigned int* leaf_start;
    const unsigned int* child_start; // children ranges of the levels >= 1
    const unsigned int* leaf_rank;   // [n_tgt + 2] number of leaf starts before sorted position i: leaf of point i = leaf_rank[i + 1] - 1
    // Leaf adjacency (grid.cu): adj[32*l .. 32*l + n) = every other leaf whose box meets box(l) inflated by R;
    // adj_box[2*l] = {lo - R, n as int bits}, adj_box[2*l+1] = {hi + R, _}; an inverted box (lo > hi) means "no list".
    // A query whose search ball lies inside the inflated box needs no tree walk.
    const unsigned int* adj; const float4* adj_box; int adj_capacity;
    const float* adj_gap;    // squared box-to-box gap of every list entry to its leaf, ascending along the list (rounded down); never null
    // the same one level up: adj1[32*m ..] = the level-1 nodes (m itself included) whose box meets box(m) inflated; node_rank
    // maps a leaf to its level-1 node (node_rank[coffset[1] + leaf + 1] - 1)
    const unsigned int* adj1; const float4* adj1_box; int adj1_capacity; const unsigned int* node_rank;
    int* nn_leaf;            // leaf of nn_pos (or -1): saves the position -> leaf lookup at the start of the next search
    // projective
    float fx, fy, cx, cy; unsigned int width, height;
    // config
    int weighting, rejection, color_icp;
    float max_d2;            // the matcher's threshold
    float weight_max_d2;     // WeightingMethod's maxDistance (the reference keeps the two apart, ICPOptimizer.h:41-44,71-78)
    // per-query state, indexed by p
    int* match_pos;          // position in tgt_pts order, -1 = none
    float* match_w;
    int* match_idx;          // original target index (API output), may be null
    int* nn_pos;             // nearest neighbour found the last time p was a query (-1 none): seeds the next search
    float4* seedbuf;         // knn_prep_kernel -> knn_bvh_kernel, per deferred query: {best d2, best idx, best pos, seed leaf} of the seed-leaf
                             // scan the fast path already made (w = -2: not scanned, the walk starts from nn_pos itself)
    float4* qbuf;            // transformed query points of the current iteration {x,y,z,rgba}; x = NaN: not searched
    int desc_index;          // >= 0: fixed descriptor (query_matches); -1: use state->iter
    int brute_norm;          // brute force on rounded Euclidean norms, max_d2 = a plain distance (NearestNeighborSearchBruteForce, NearestNeighbor.h:81-97)
    int proj_tiled;          // projective matching of a full-frame source: src arrays are in ORIGINAL (pixel) order, one 32x4 tile per block
    int collect_stats;       // work counters in DevState (atomics); off in timed runs
    int skip_finish;         // BVH path: the reduction evaluates stages 3-4 itself (ReduceArgs::fused), no match records
    int q_begin, q_end;      // BVH path: the sorted-source positions [q_begin, q_end) this launch searches (a chunk; the whole cloud by default)
    int group_min;           // knn_group_kernel: fewest handed-over queries among 32 consecutive positions that share one descent
};

// Concurrency inside one iteration (registration.cu, match.cu): the queries are cut into chunks, each chunk's {prep, walk} chain runs on its own
// stream between a fork and a join event; the per-query results do not depend on the cut.
#define ICP_MAX_MATCH_CHUNKS 8
struct MatchChunks {
    int n = 1;                                         // 1 = everything on the caller's stream
    cudaStream_t stream[ICP_MAX_MATCH_CHUNKS - 1] = {};
    cudaEvent_t done[ICP_MAX_MATCH_CHUNKS - 1] = {};
    cudaEvent_t fork = nullptr;
};

struct ReduceArgs {
    const float4* src_pts; const float4* src_nrm; int n_src;
    DevState* state;
    const float4* tgt_pts; const float4* tgt_nrm;
    const int* match_pos; const float* match_w;
    double* partials;        // [grid][ICP_NRED]
    float* pose_history;     // [ICP_MAX_ITERS][16] or null
    int metric; int solve;   // solve=0: leave the summed row in state->shard_partials
    // fused = 1: stages 3-4 (selection predicate, weighting, rejection) are evaluated here from the search result nn_pos
    // instead of being read back from the match records (saves the match_finish launch); linear minimiser only
    int fused; const int* nn_pos; int n_tgt; const unsigned int* mask; const IterDesc* desc; int desc_index;
    int weighting, rejection; float max_d2, weight_max_d2;
    int profile;             // write DevState::prof (diagnostic, ICP_GPU_REDUCE_PROFILE=1)
    PeerXchg peer;           // world > 1: the summed row is all-reduced over the peers' mailboxes before the solve
};

// batch.cu: B independent small registrations, one thread block per pair running every iteration of its loop
#define ICP_BATCH_MAX_TARGET ICP_GPU_BATCH_MAX_TARGET    // target points staged in shared memory per pair (float4: 128 KB of the 227 KB a block may use)
#define ICP_BATCH_THREADS 512
#define ICP_BATCH_LM_THREADS 256                         // batch_lm_kernel: the fp64 jets need up to 255 registers a thread
// What the batch kernels read of a pair's configuration (one table entry per configuration of the call).
struct BatchCfg {
    int n_iterations, multires, weighting, rejection, lm_max_iterations;
    int mt_mask;             // 1: mt19937 selection, the pair's masks at BatchArgs::mask + mask_off[pair]
    float max_d2, weight_max_d2;
    float proba;             // device selection stream: keep a query iff hash < proba; < 0 = off
    unsigned int seed;
    float stop_rot, stop_trans;
};
struct BatchArgs {
    const float* src_xyz; const float* src_nrm; const long long* src_off;   // packed float[3n]; nrm nullable (= zero normals)
    const float* tgt_xyz; const float* tgt_nrm; const long long* tgt_off;
    const float* poses_in;   // [B][16] column-major
    float* poses_out; int* n_iter_out; int* status_out;
    float* history;          // [B][history_rows][16] or null
    int history_rows;
    int2* scratch;           // symmetric metric and LM: one {target index or -1, weight bits} per source point, kept between the passes
    const BatchCfg* cfgs; const int* cfg_index;   // pair b runs with cfgs[cfg_index[b]]
    const int* pairs;        // block k of the launch registers pair pairs[k]
    // mt19937 selection: iteration i's mask of pair b (one bit per pair-local source index) is the ceil(max(n_s, 1) / 32) words at
    // mask + mask_off[b] + i * that many; pairs with the same masks share one copy
    const unsigned int* mask; const long long* mask_off;
};
// metric: ICP_GPU_METRIC_*, lm: the minimiser; pairs: n_pairs block indices in device memory (BatchArgs::pairs)
cudaError_t icp_launch_batch(const BatchArgs& a, int metric, int lm, int n_pairs, int max_tgt, cudaStream_t s);

// standalone.cu: the reference API's value-level operations outside the loop
cudaError_t icp_launch_transform(const float* in, long long n, const float pose16[16], int normals, float* out, cudaStream_t s);
cudaError_t icp_launch_apply_weights(int method, float max_d2, const float* sp, const float* sn, const unsigned int* sc, const float* tp, const float* tn,
                                     const unsigned int* tc, long long n_tgt, const int* idx, float* w, long long n, cudaStream_t s);
cudaError_t icp_launch_pack_pairs(const float* s, const float* sn, const float* t, const float* tn, const float* w, int n, float4* sp4, float4* sn4,
                                  float4* tp4, float4* tn4, int* pos, float* wo, cudaStream_t st);
// peak.cu: measured FP32 throughput of the device (mode 0 FFMA, 1 FMUL+FADD), TFLOP/s
cudaError_t icp_measure_fp32_peak(int mode, int n_sms, cudaStream_t s, double* tflops);
// ---- launchers (defined in grid.cu / match.cu / solve.cu / lm.cu) ----
// AoS3 -> float4 records, the bounding box of the finite points and from it the grid parameters; clears the sort's histograms
// (scratch: 8 words, [7] = number of points with a non-finite coordinate afterwards)
cudaError_t icp_launch_pack_cloud(const float* xyz, const float* nrm, const uint8_t* rgba, int n, float4* pts, float4* nrmo,
                                  unsigned int* scratch, int T, GridParams* grid, unsigned int* hist, long long hist_words, int with_normals, cudaStream_t s);
// Stable LSD radix sort of a packed cloud into (cell code, original index) order; points with a non-finite coordinate end up
// after the last cell.  T + 1 key bits in passes of <= 8 bits.
// normal / colour records packed late (before the last pass of the sort), once `ready` has happened: host uploads
struct IcpLatePack { const float* nrm; const uint8_t* rgba; float4* nrmo; cudaEvent_t ready; };
struct IcpRadixPlan { int n_pass; int shift[4]; int bits[4]; int ipt; int tile_items; int n_tiles; int tiles_pad; };
void icp_radix_plan(int n, int T, IcpRadixPlan* p);
size_t icp_radix_hist_words(int n, int T);
#define ICP_MSD_WORDS 257
cudaError_t icp_launch_cloud_sort(const float4* pts_in, const float4* nrm_in, int n, int T, const GridParams* grid,
                                  unsigned int* keys_a, unsigned int* keys_b, unsigned int* idx_a, unsigned int* idx_b,
                                  unsigned int* hist, float4* pts_sorted, float4* nrm_sorted, unsigned int* msd_start,
                                  unsigned int** keys_sorted_out, int* msd_shift_out, const IcpLatePack* late, cudaStream_t s, int* n_launches);
// Tight-box BVH over the sorted cloud, read off the common-prefix lengths of neighbouring sorted keys.
size_t icp_bvh_max_nodes(int n);
cudaError_t icp_launch_bvh_build(float4* pts_sorted, float4* nrm_sorted, int n, int T, const unsigned int* keys,
                                 const unsigned int* nonfinite, unsigned char* flags, unsigned int* tile_count,
                                 int* delta_a, int* delta_b, unsigned int* leaf_rank, unsigned int* leaf_start, unsigned int* node_rank,
                                 unsigned int* child_start, BvhDesc* bvh_dev, float4* box, int n_sms, cudaStream_t s, int* n_launches);
// One voxel pyramid level (depth D of the source grid) as a selection mask; table: scratch of 2^D entries.
cudaError_t icp_launch_voxel_level(const float4* pts_sorted, const float4* nrm_sorted, int n, const GridParams* grid, int T, int D,
                                   unsigned int* table, unsigned int* mask, size_t mask_words, cudaStream_t s, int* n_launches);
// Adjacency lists of the nodes [0, min(count[level], capacity)) of `level` (0 leaves, 1 their parents).  The level-0 call takes the
// level-1 lists (node_rank, adj1, adj1_box); the level-1 call passes null there.  adj_gap (non-null: the level-0 call): sort the
// entries by their gap to the node and store the gaps.
cudaError_t icp_launch_leaf_adjacency(const BvhDesc* bvh_dev, const float4* box, const unsigned int* child_start, unsigned int* adj,
                                      float4* adj_box, int capacity, int level, const unsigned int* node_rank, const unsigned int* adj1,
                                      const float4* adj1_box, int adj1_capacity, int n_sms, cudaStream_t s, int* n_launches, float* adj_gap);
cudaError_t icp_launch_extract_order(const float4* pts_sorted, int n, int* order, cudaStream_t s);
cudaError_t icp_launch_fill_int(int* p, int n, int v, cudaStream_t s);
// Seeds (nn_pos / nn_leaf) for the queries that have none (reset: for every query), from the target's sorted keys at the pose in `st`.
cudaError_t icp_launch_seed_from_keys(const float4* src_pts, int n_src, const DevState* st, const GridParams* grid, const unsigned int* keys, int n_tgt,
                                      const unsigned int* nonfinite, const unsigned int* msd_start, int msd_shift, const unsigned int* leaf_rank,
                                      int* nn_pos, int* nn_leaf, int reset, cudaStream_t s);
// algorithm: 0 BVH search (one warp per query), 1 brute force, 2 projective
// prep.cu: depth map -> cloud (PointCloud.h:78-165) and convergence metrics (ConvergenceMeasure.h:50-66,104-151)
struct DepthArgs {
    unsigned int width, height, downsample; int keep_original_size;
    long long n_candidates;            // ceil(width*height / downsample)
    float fovX, fovY, cX, cY, half_max_distance;
    float Einv[16];                    // inverse depth extrinsics, column-major
};
cudaError_t icp_launch_depth_cloud(const float* depth, const unsigned char* color, const DepthArgs& a, float* pts_tmp, float* nrm_tmp,
                                   unsigned char* rgba_tmp, unsigned int* flag, unsigned int* block_count, unsigned int* total,
                                   float* pts_out, float* nrm_out, unsigned char* rgba_out, cudaStream_t s, int* n_launches);
cudaError_t icp_launch_gt_from_source(const float4* src_raw, long long n, const float* pose16_dev, float* gt_src, float* gt_ref, cudaStream_t s);
int icp_metrics_blocks(long long m, int n_sms);
cudaError_t icp_launch_metrics(const float* src, const float* ref, long long m, const float* history, int n_iters, int n_blocks, double* partial,
                               float* rmse, float* centroid, double* bench, cudaStream_t s, int* n_launches);
// normals.cu: k-NN PCA normals of the indexed cloud (PointCloud.h:41-76)
struct NormalArgs {
    const float4* pts; int n;                // cell-sorted cloud {x,y,z,orig idx}
    const float4* bvh_box; const BvhDesc* bvh; const unsigned int* leaf_start; const unsigned int* leaf_rank; const unsigned int* child_start;
    const unsigned int* adj; const float4* adj_box; int adj_capacity;
    int k; float vp[3];
    float* out_nrm; float* out_curv;         // original order: 3n, n
    float4* nrm_sorted; float4* nrm_orig;    // the cloud's own normal arrays {nx,ny,nz,rgba}: x,y,z overwritten
};
cudaError_t icp_launch_pca_normals(const NormalArgs& a, cudaStream_t s);
cudaError_t icp_launch_match(const MatchArgs& a, int algorithm, int n_sms, cudaStream_t s, int* n_launches, cudaEvent_t after_prep = nullptr,
                             const MatchChunks* chunks = nullptr);
cudaError_t icp_launch_pose_init(DevState* st, const float* pose_dev16, cudaStream_t s, float stop_rot = 0.f, float stop_trans = 0.f);
cudaError_t icp_launch_reduce(const ReduceArgs& a, int n_blocks, cudaStream_t s, int* n_launches);
// one phase of the point-sharded iteration: the summed row is left in state->shard_partials
cudaError_t icp_launch_reduce_phase(const ReduceArgs& a, int n_blocks, int phase, cudaStream_t s, int* n_launches);
int icp_reduce_blocks(int n_src, int n_sms);
cudaError_t icp_launch_shard_apply(DevState* st, int mode, float* history, cudaStream_t s);
cudaError_t icp_launch_lm(const ReduceArgs& a, int n_blocks, int lm_max_iterations, cudaStream_t s, int* n_launches);

// pinned 4x4 product, column-major: C = A * B  (ICPOptimizer.h:614-620)
__device__ __forceinline__ void mat4_mul_pinned(const float* A, const float* B, float* C) {
    float T[16];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i)
            T[i + 4 * j] = padd(padd(padd(pmul(A[i], B[4 * j]), pmul(A[i + 4], B[1 + 4 * j])), pmul(A[i + 8], B[2 + 4 * j])),
                                pmul(A[i + 12], B[3 + 4 * j]));
#pragma unroll
    for (int k = 0; k < 16; ++k) C[k] = T[k];
}

// (R^-1)^T by cofactors (utils.h:129, Eigen's 3x3 inverse), row-major out.
__device__ __forceinline__ void inv_transpose3_pinned(const float* P, float* N) {
    const float r00 = P[0], r10 = P[1], r20 = P[2], r01 = P[4], r11 = P[5], r21 = P[6], r02 = P[8], r12 = P[9], r22 = P[10];
    const float c00 = psub(pmul(r11, r22), pmul(r12, r21)), c01 = psub(pmul(r12, r20), pmul(r10, r22)), c02 = psub(pmul(r10, r21), pmul(r11, r20));
    const float c10 = psub(pmul(r02, r21), pmul(r01, r22)), c11 = psub(pmul(r00, r22), pmul(r02, r20)), c12 = psub(pmul(r01, r20), pmul(r00, r21));
    const float c20 = psub(pmul(r01, r12), pmul(r02, r11)), c21 = psub(pmul(r02, r10), pmul(r00, r12)), c22 = psub(pmul(r00, r11), pmul(r01, r10));
    const float det = padd(padd(pmul(r00, c00), pmul(r01, c01)), pmul(r02, c02));
    const float id = pdiv(1.0f, det);
    N[0] = pmul(c00, id); N[1] = pmul(c01, id); N[2] = pmul(c02, id);
    N[3] = pmul(c10, id); N[4] = pmul(c11, id); N[5] = pmul(c12, id);
    N[6] = pmul(c20, id); N[7] = pmul(c21, id); N[8] = pmul(c22, id);
}

// transformPoints (utils.h:106-118), contract D4
__device__ __forceinline__ void xform_point(const float* P, float x, float y, float z, float& ox, float& oy, float& oz) {
    ox = padd(padd(padd(pmul(P[0], x), pmul(P[4], y)), pmul(P[8], z)), P[12]);
    oy = padd(padd(padd(pmul(P[1], x), pmul(P[5], y)), pmul(P[9], z)), P[13]);
    oz = padd(padd(padd(pmul(P[2], x), pmul(P[6], y)), pmul(P[10], z)), P[14]);
}
// transformNormals (utils.h:122-133)
__device__ __forceinline__ void xform_normal(const float* N, float x, float y, float z, float& ox, float& oy, float& oz) {
    ox = padd(padd(pmul(N[0], x), pmul(N[1], y)), pmul(N[2], z));
    oy = padd(padd(pmul(N[3], x), pmul(N[4], y)), pmul(N[5], z));
    oz = padd(padd(pmul(N[6], x), pmul(N[7], y)), pmul(N[8], z));
}

__device__ __forceinline__ float unit_hash(unsigned int key, unsigned int k) {
    // counter-based stream for ICP_GPU_RNG_DEVICE (two rounds of a 32-bit mix)
    unsigned int x = k * 0x9E3779B9u + key;
    x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
    x += key * 0x85EBCA6Bu; x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
    return (float)(x >> 8) * (1.0f / 16777216.0f);
}

// Is the sorted-source point (p4 = point, n4 = normal) a query of the iteration described by d?
__device__ __forceinline__ bool query_active(const IterDesc& d, const unsigned int* __restrict__ mask, const float4& p4, const float4& n4) {
    const unsigned int orig = (unsigned int)__float_as_int(p4.w);
    if (d.stride > 1 && (orig % (unsigned int)d.stride) != 0u) return false;
    if (d.filter_finite && !(finite3(p4.x, p4.y, p4.z) && finite3(n4.x, n4.y, n4.z))) return false;
    if (d.mask_word_offset >= 0 && !((__ldg(&mask[d.mask_word_offset + (orig >> 5)]) >> (orig & 31u)) & 1u)) return false;
    if (d.proba >= 0.0f && !(unit_hash(d.rng_key, orig) < d.proba)) return false;
    return true;
}

// Stages 3-4 for one matched pair: WeightingMethod::applyWeights (weighting.h:39-99) and
// ICPOptimizer::pruneCorrespondences (ICPOptimizer.h:157-174).  w comes in as the matcher's weight (1, or 0 for the
// projective matcher's skipped queries) and leaves as the match weight; returns false when the pair is rejected.  max_d2 is
// WeightingMethod's maxDistance (weighting.h:33-37), not the matcher's threshold.
// (sx,sy,sz) / (snx,sny,snz): transformed source point / normal; tp / tn: target point {x,y,z,_} / normal {x,y,z,rgba}.
__device__ __forceinline__ bool match_weight_and_reject(int weighting, int rejection, float max_d2, float sx, float sy, float sz,
                                                        float snx, float sny, float snz, unsigned int s_rgba, const float4 tp,
                                                        const float4 tn, float& w) {
    if (weighting != ICP_GPU_WEIGHT_CONSTANT) {                               // weighting.h:44 early return
        w = 0.0f;
        if (weighting == ICP_GPU_WEIGHT_DISTANCES || weighting == ICP_GPU_WEIGHT_COLORS) {
            if (finite3(sx, sy, sz) && finite3(tp.x, tp.y, tp.z)) {            // weighting.h:58-59
                const float d0 = psub(sx, tp.x), d1 = psub(sy, tp.y), d2 = psub(sz, tp.z);
                const float q = pdiv(padd(padd(pmul(d0, d0), pmul(d1, d1)), pmul(d2, d2)), max_d2);
                w = (float)(1.0 - (double)q);                                  // weighting.h:16-20
            }
        }
        if (weighting == ICP_GPU_WEIGHT_NORMALS) {
            if (finite3(snx, sny, snz) && finite3(tn.x, tn.y, tn.z))           // weighting.h:72-73
                w = padd(padd(pmul(snx, tn.x), pmul(sny, tn.y)), pmul(snz, tn.z));   // weighting.h:22-25 (unclamped)
        }
        if (weighting == ICP_GPU_WEIGHT_COLORS) {
            // weighting.h:27-30: Vector4uc difference wraps modulo 256 before squaring
            const unsigned int t_rgba = __float_as_uint(tn.w);
            int s = 0;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int e = (int)((((s_rgba >> (8 * k)) & 0xFFu) - ((t_rgba >> (8 * k)) & 0xFFu)) & 0xFFu);
                s += e * e;
            }
            const float cw = (float)(1.0 - (double)pdiv((float)s, 195075.0f));
            w = pmul(w, cw);
        }
    }
    if (rejection == 1) {                                                      // ICPOptimizer.h:157-174
        const float dot = padd(padd(pmul(snx, tn.x), pmul(sny, tn.y)), pmul(snz, tn.z));
        const float na = __fsqrt_rn(padd(padd(pmul(snx, snx), pmul(sny, sny)), pmul(snz, snz)));
        const float nb = __fsqrt_rn(padd(padd(pmul(tn.x, tn.x), pmul(tn.y, tn.y)), pmul(tn.z, tn.z)));
        const float c = pdiv(dot, pmul(na, nb));
        if (c <= 0.5f && c >= -1.0f) return false;                             // D6; NaN and |c|>1 are kept like acos()'s NaN
    }
    return true;
}

// ---------------------------------------------------------------------------- reductions
template <int H>
__device__ __forceinline__ void halve_step(double (&v)[32], int lane) {
    const bool upper = (lane & H) != 0;
#pragma unroll
    for (int k = 0; k < H; ++k) {
        const double send = upper ? v[k] : v[k + H];
        const double keep = upper ? v[k + H] : v[k];
        v[k] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, H);
    }
}
// After the call, lane L holds in v[0] the warp-wide sum of element L.
__device__ __forceinline__ void warp_reduce_scatter32(double (&v)[32], int lane) {
    halve_step<16>(v, lane); halve_step<8>(v, lane); halve_step<4>(v, lane); halve_step<2>(v, lane); halve_step<1>(v, lane);
}

// ---------------------------------------------------------------------------- small dense algebra (fp64, one thread)
static __device__ int solve6_dev(double* A /*row-major 6x6, destroyed*/, double* b, double* x) {
    for (int k = 0; k < 6; ++k) {
        int p = k; double mx = fabs(A[k * 6 + k]);
        for (int i = k + 1; i < 6; ++i) if (fabs(A[i * 6 + k]) > mx) { mx = fabs(A[i * 6 + k]); p = i; }
        if (!(mx > 0.0)) return -1;
        if (p != k) {
            for (int j = 0; j < 6; ++j) { const double t = A[k * 6 + j]; A[k * 6 + j] = A[p * 6 + j]; A[p * 6 + j] = t; }
            const double t = b[k]; b[k] = b[p]; b[p] = t;
        }
        for (int i = k + 1; i < 6; ++i) {
            const double f = A[i * 6 + k] / A[k * 6 + k];
            for (int j = k; j < 6; ++j) A[i * 6 + j] -= f * A[k * 6 + j];
            b[i] -= f * b[k];
        }
    }
    for (int i = 5; i >= 0; --i) {
        double s = b[i];
        for (int j = i + 1; j < 6; ++j) s -= A[i * 6 + j] * x[j];
        x[i] = s / A[i * 6 + i];
    }
    for (int i = 0; i < 6; ++i) if (!isfinite(x[i])) return -1;
    return 0;
}


__device__ __forceinline__ void mat4_identity_dev(float* M) {
    for (int i = 0; i < 16; ++i) M[i] = (i % 5 == 0) ? 1.f : 0.f;
}


// Early-stop criterion (SURVEY.md 8f rank 2; the reference always runs all iterations): the increment just applied rotates by no
// more than stop_rot radians and translates by no more than stop_trans metres.  Off unless both thresholds are positive.
__device__ __forceinline__ bool increment_is_small(const float* inc, float stop_rot, float stop_trans) {
    if (!(stop_rot > 0.f) || !(stop_trans > 0.f)) return false;
    double f = 0.0;     // |R - I|_F = 2 sqrt(2) sin(theta / 2)
    for (int c = 0; c < 3; ++c) for (int r = 0; r < 3; ++r) { const double d = (double)inc[r + 4 * c] - (r == c ? 1.0 : 0.0); f += d * d; }
    const double theta = 2.0 * asin(fmin(sqrt(f) / (2.0 * sqrt(2.0)), 1.0));
    const double t = sqrt((double)inc[12] * inc[12] + (double)inc[13] * inc[13] + (double)inc[14] * inc[14]);
    return theta <= (double)stop_rot && t <= (double)stop_trans;
}

// estimatedPose = increment * estimatedPose (ICPOptimizer.h:614-620); history as handed to
// ConvergenceMeasure::recordAlignmentError (:629-631).
static __device__ void apply_increment(DevState* st, const float* inc, int rc, float* history) {
    if (st->status == 0) {
        if (rc != 0) st->status = rc;
        else {
            float np[16];
            mat4_mul_pinned(inc, st->pose, np);
            for (int i = 0; i < 16; ++i) st->pose[i] = np[i];
            inv_transpose3_pinned(st->pose, st->nrm);
            if (history) for (int i = 0; i < 16; ++i) history[16 * st->iters_done + i] = np[i];
            st->iters_done += 1;
            if (increment_is_small(inc, st->stop_rot, st->stop_trans)) st->converged = 1;
        }
    }
    st->iter += 1;
}


// Block + grid reduction of one 32-double row per thread.  Every block writes its row to
// partials[block][32]; the block that draws the last ticket sums all rows in a fixed order
// (deterministic, no floating-point atomics).  Returns true in every thread of that last block,
// with the total in fin[0][0..31].  red: [THREADS/32][32], fin: [THREADS/32][32] shared scratch.
// ---- all-reduce of the summed row over the peers' mailboxes (NVLink peer memory), run by the last block ----
__device__ __forceinline__ void st_release_sys_u32(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Called by every thread of the last block with the local total in fin[0][0..31]; returns with the sum over all ranks
// there, added in rank order on every rank (=> bit-identical rows, identical solves, identical poses: no broadcast).
// Warp j (j < world, j != rank) serves peer j: it pushes the local row into rank j's mailbox (remote stores, then a
// system-scope fence and a release store of the exchange number) and then polls its own mailbox for rank j's row.
// A rank whose peer did not show up in time (ICP_GPU_E_PEER) POISONS the exchange: it stores ICP_PEER_POISON into its flag
// words of every peer's mailbox (both slots), so that the peers fail in their current or next exchange instead of finishing
// with sums built from a stale row, and it skips every later exchange of the registration -- a lost peer costs one time-out
// per registration, not one per launch.  The mailboxes stay poisoned until they are exported and attached again.
#define ICP_PEER_POISON 0xFFFFFFFFu
template <int THREADS>
__device__ __forceinline__ void peer_exchange_row(const PeerXchg& px, DevState* st, double (*red)[32], double (*fin)[32]) {
    static_assert(THREADS / 32 >= ICP_MAX_PEERS, "one warp per peer");
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __shared__ int s_failed;
    if (threadIdx.x == 0) s_failed = (*reinterpret_cast<volatile int*>(&st->status) == ICP_GPU_E_PEER) ? 1 : 0;
    __syncthreads();
    const bool failed_before = s_failed != 0;
    const unsigned int seq = st->xchg_seq + 1u;     // written back by thread 0 after the last read below
    const int slot = (int)(seq & 1u);
    bool lost = false;
    if (!failed_before && w < px.world) {
        if (w != px.rank) {
            PeerBox* theirs = px.box[w];
            theirs->row[slot][px.rank][lane] = lane == 31 ? (double)px.plan_check : fin[0][lane];   // element 31 is no sum: the plan check
            __threadfence_system();
            __syncwarp();
            if (lane == 0) st_release_sys_u32(&theirs->flag[slot][px.rank], seq);
            const PeerBox* mine = px.box[px.rank];
            const unsigned long long t0 = global_timer_ns();
            for (;;) {
                const unsigned int f = ld_acquire_sys_u32(&mine->flag[slot][w]);
                if (f == seq) break;
                if (f == ICP_PEER_POISON || global_timer_ns() - t0 > px.timeout_ns) { lost = true; break; }
                __nanosleep(64);
            }
            red[w][lane] = ld_relaxed_sys_f64(&mine->row[slot][w][lane]);
        } else {
            red[w][lane] = lane == 31 ? (double)px.plan_check : fin[0][lane];
        }
    }
    // every rank must have planned the same registration (iterations, metric, minimiser): a rank with another plan would leave
    // the others waiting for exchanges that never come
    if (!failed_before && !lost && w < px.world && lane == 31 && red[w][31] != (double)px.plan_check) lost = true;
    if (lost && (lane == 0 || lane == 31)) { atomicCAS(&st->status, 0, ICP_GPU_E_PEER); s_failed = 1; }
    __syncthreads();
    if (s_failed) {
        // tell every peer (whatever exchange it is in, or enters next); the totals of this exchange are not used: the status is set
        if (w < px.world && w != px.rank && lane < 2) st_release_sys_u32(&px.box[w]->flag[lane][px.rank], ICP_PEER_POISON);
        if (failed_before) return;
    }
    if (threadIdx.x < 32) {
        double s = 0.0;
        for (int j = 0; j < px.world; ++j) s += red[j][threadIdx.x];
        fin[0][threadIdx.x] = s;
    }
    if (threadIdx.x == 0) st->xchg_seq = seq;
    __syncthreads();
}

template <int THREADS>
__device__ __forceinline__ bool grid_reduce_row(double (&v)[32], double* __restrict__ partials, unsigned int* ticket,
                                                double (*red)[32], double (*fin)[32], bool* is_last,
                                                const PeerXchg* px = nullptr, DevState* px_state = nullptr) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    warp_reduce_scatter32(v, lane);
    red[wid][lane] = v[0];
    __syncthreads();
    if (threadIdx.x < 32) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) s += red[w][threadIdx.x];
        partials[(size_t)blockIdx.x * ICP_NRED + threadIdx.x] = s;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(ticket, 1u);
        *is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!*is_last) return false;
    __threadfence();
    {
        const int c = threadIdx.x & 31, g = threadIdx.x >> 5;
        // fixed order (deterministic); eight independent chains so that the loads of a whole pass are in flight at
        // once -- the last block is alone on the critical path of every iteration, each pass costs one L2 round trip
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0, s4 = 0.0, s5 = 0.0, s6 = 0.0, s7 = 0.0;
        const int step = THREADS / 32, nb = (int)gridDim.x;
        int b = g;
        for (; b + 7 * step < nb; b += 8 * step) {
            const double x0 = __ldcg(&partials[(size_t)b * ICP_NRED + c]);
            const double x1 = __ldcg(&partials[(size_t)(b + step) * ICP_NRED + c]);
            const double x2 = __ldcg(&partials[(size_t)(b + 2 * step) * ICP_NRED + c]);
            const double x3 = __ldcg(&partials[(size_t)(b + 3 * step) * ICP_NRED + c]);
            const double x4 = __ldcg(&partials[(size_t)(b + 4 * step) * ICP_NRED + c]);
            const double x5 = __ldcg(&partials[(size_t)(b + 5 * step) * ICP_NRED + c]);
            const double x6 = __ldcg(&partials[(size_t)(b + 6 * step) * ICP_NRED + c]);
            const double x7 = __ldcg(&partials[(size_t)(b + 7 * step) * ICP_NRED + c]);
            s0 += x0; s1 += x1; s2 += x2; s3 += x3; s4 += x4; s5 += x5; s6 += x6; s7 += x7;
        }
        for (; b < nb; b += step) s0 += __ldcg(&partials[(size_t)b * ICP_NRED + c]);
        fin[g][c] = ((s0 + s1) + (s2 + s3)) + ((s4 + s5) + (s6 + s7));
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        double s = 0.0;
#pragma unroll
        for (int g = 0; g < THREADS / 32; ++g) s += fin[g][threadIdx.x];
        fin[0][threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) *ticket = 0;
    if (px && px->world > 1) peer_exchange_row<THREADS>(*px, px_state, red, fin);
    return true;
}
