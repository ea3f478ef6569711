/*
 * icp_gpu.h -- C ABI of the B200 (sm_100a) registration inner loop.
 *
 * This is the drop-in boundary for the path BASELINE.json names: the body of
 * ICPOptimizer::estimatePose's iteration loop plus NearestNeighborSearch::buildIndex /
 * queryMatches of the reference (icp-variants/ICPOptimizer.h:185-349, :493-663;
 * icp-variants/NearestNeighbor.h:12-36).  The reference has no FFI layer -- its seam is the C++
 * virtual interface -- so the entry points below are what the C++14 drop-in classes in
 * include/icp_b200/ (same names and signatures as the reference's) bind, and what any other
 * host (ctypes, cgo, JNI) would bind.  See INTEGRATION.md for the reference-side stubs.
 *
 * Conventions
 *   - plain C, no exceptions, no torch / Eigen types: pointers and sizes only;
 *   - points / normals: packed float[3*n]  (std::vector<Eigen::Vector3f>::data());
 *     colours: uint8_t[4*n]                (std::vector<Vector4uc>::data());
 *     poses: float[16] column-major        (Eigen::Matrix4f::data());
 *     camera matrix: float[9] column-major (Eigen::Matrix3f::data());
 *   - every call returns ICP_GPU_OK (0) or a negative ICP_GPU_E_* code; the message is
 *     available from icp_gpu_last_error().  Nothing hangs (the reference's ASSERT is
 *     `while(1);`, Eigen.h:9) and nothing throws across the ABI;
 *   - the caller owns every host array (borrowed for the duration of the call); the context
 *     owns device memory, its stream and its CUDA graphs;
 *   - one context = one device + one stream; calls on one context must be serialised by the
 *     caller, different contexts may be driven concurrently from different threads/processes;
 *   - there is NO CPU fallback: every entry point fails with ICP_GPU_E_CUDA when no sm_100-class
 *     device is usable.
 */
#ifndef ICP_GPU_H
#define ICP_GPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ICP_GPU_ABI_VERSION 4

enum {
    ICP_GPU_OK = 0,
    ICP_GPU_E_CUDA = -1,       /* CUDA runtime / driver error, or no usable device                  */
    ICP_GPU_E_ARG = -2,        /* bad argument (null pointer, negative size, unknown enum value)    */
    ICP_GPU_E_STATE = -3,      /* call order: no target / source / camera set for what was asked    */
    ICP_GPU_E_NO_MATCHES = -4, /* an iteration had no surviving correspondence (reference: hangs in
                                  ASSERT, ICPOptimizer.h:668,680,788); pose is the last good one    */
    ICP_GPU_E_NUMERIC = -5,    /* singular normal equations                                         */
    ICP_GPU_E_PEER = -6        /* point-sharded registration: a peer's row did not arrive in time   */
};

/* ICPOptimizer::setMetric (ICPOptimizer.h:46): 0 point-to-point, 1 point-to-plane, 2 symmetric   */
enum { ICP_GPU_METRIC_P2P = 0, ICP_GPU_METRIC_P2PLANE = 1, ICP_GPU_METRIC_SYMMETRIC = 2 };
/* LinearICPOptimizer (ICPOptimizer.h:489) / CeresICPOptimizer (:181)                              */
enum { ICP_GPU_MIN_LINEAR = 0, ICP_GPU_MIN_LM = 1 };
/* ICPOptimizer::setMatchingMethod (ICPOptimizer.h:71): 0 k-NN, 1 projective                       */
enum { ICP_GPU_MATCH_KNN = 0, ICP_GPU_MATCH_PROJECTIVE = 1 };
/* selection.h:8                                                                                  */
enum { ICP_GPU_SELECT_ALL = 0, ICP_GPU_SELECT_RANDOM = 1 };
/* weighting.h:8                                                                                  */
enum { ICP_GPU_WEIGHT_CONSTANT = 0, ICP_GPU_WEIGHT_DISTANCES = 1, ICP_GPU_WEIGHT_NORMALS = 2, ICP_GPU_WEIGHT_COLORS = 3 };
/* Nearest-neighbour kernel choice (both exact, same answers): AUTO = by target size; BRUTE = one warp per
 * query over the whole target; GRID = one warp per query over a tight-box 32-ary BVH built on the target
 * sorted into the cell (Morton) order of a uniform grid                                               */
enum { ICP_GPU_NN_AUTO = 0, ICP_GPU_NN_BRUTE = 1, ICP_GPU_NN_GRID = 2,
       /* NearestNeighborSearchBruteForce's own rule (NearestNeighbor.h:81-97; 3-D only): candidates are compared on the
        * Euclidean NORM (p - m).norm() = sqrt of the D1 squared distance, rounded to fp32 -- ties are ties of the rounded
        * norms, lowest index first -- and max_distance_sq is taken as a plain distance (the reference compares the norm with
        * m_maxDistance, :93).  The optimizers never use this class; it exists for the reference's matcher API. */
       ICP_GPU_NN_BRUTE_NORM = 3 };
/* Random selection stream: 0 = std::mt19937 + uniform_real_distribution<double> drawn on the host
 * exactly as selection.h:88-104 does (reference-compatible for a given seed); 1 = counter-based
 * hash drawn on the device (fast, not reference-compatible).                                      */
enum { ICP_GPU_RNG_MT19937 = 0, ICP_GPU_RNG_DEVICE = 1 };
/* Multi-resolution level construction.  STRIDE: every f-th point of the scan order with finite point and
 * normal, the reference's PointCloud::getCoarseResolution (PointCloud.h:325-343).  VOXEL: one point per occupied
 * cell of a uniform grid over the source (the valid point with the lowest index; cell depth = grid depth -
 * ceil(1.5 * log2 f)) -- spatially uniform levels; NOT what the reference computes, results differ.  Level count
 * and iteration schedule are the reference's in both modes (ICPOptimizer.h:503-525,634-655).                  */
enum { ICP_GPU_PYRAMID_STRIDE = 0, ICP_GPU_PYRAMID_VOXEL = 1 };

typedef struct icp_gpu_config {
    int32_t  metric;            /* setMetric                 default 0      (ICPOptimizer.h:29)      */
    int32_t  minimizer;         /* Linear / Ceres-LM class   default linear                          */
    int32_t  matching;          /* setMatchingMethod         default k-NN   (ICPOptimizer.h:31)      */
    int32_t  selection;         /* setSelectionMethod        default all    (ICPOptimizer.h:29)      */
    double   proba;             /* setSelectionMethod proba  default 1.0                             */
    uint32_t seed;              /* reference seeds from std::random_device (selection.h:76-79)       */
    int32_t  selection_rng;     /* ICP_GPU_RNG_*                                                    */
    int32_t  weighting;         /* setWeightingMethod        default constant                        */
    int32_t  rejection;         /* setRejectionMethod        default 1 = on (ICPOptimizer.h:30)      */
    float    max_distance_sq;   /* the matcher's threshold NearestNeighborSearch::m_maxDistance, SQUARED metres
                                   (NearestNeighbor.h:17-19,35; valid iff d2 <= it, :182).  Default 0.0003 = what
                                   setMatchingMaxDistance(0.0003f) leaves in both members (ICPOptimizer.h:41-44)   */
    int32_t  color_icp;         /* enableColorICP            default off                             */
    int32_t  multires;          /* enableMultiResolution     default off                             */
    int32_t  pyramid_mode;      /* ICP_GPU_PYRAMID_*                                                */
    int32_t  n_iterations;      /* setNbOfIterations         default 20                              */
    int32_t  lm_max_iterations; /* Ceres max_num_iterations  default 10     (ICPOptimizer.h:358)     */
    int32_t  nn_algorithm;      /* ICP_GPU_NN_*                                                     */
    int32_t  use_graph;         /* 1 (default): replay the iteration loop as one CUDA graph          */
    int32_t  collect_stats;     /* 1 (default): fill icp_gpu_stats' work counters (device atomics);
                                   0: fastest, icp_gpu_get_stats then only reports kernel launches   */
    float    weight_max_distance_sq; /* ICPOptimizer::maxDistance as handed to WeightingMethod (ICPOptimizer.h:220,528;
                                   weighting.h:16-20,33-37): the divisor of the distance / colour weights.  The reference keeps
                                   it apart from the matcher's threshold: setMatchingMethod re-creates the matcher with
                                   MAX_DISTANCE = 0.005 (ICPOptimizer.h:71-78, NearestNeighbor.h:5) and leaves this one alone;
                                   only setMatchingMaxDistance sets both.  0 (default) = max_distance_sq               */
    float    early_stop_rotation;    /* extension (SURVEY.md 8f rank 2): stop once an applied increment rotates by <= this (radians) AND   */
    float    early_stop_translation; /* translates by <= this (metres); the remaining iterations are skipped on the device and
                                   n_iterations_out reports the executed ones.  0 (default, either one) = run every iteration,
                                   as the reference does                                                                 */
    int32_t  reserved_;
} icp_gpu_config;

/* Per-stage device times of the last icp_gpu_estimate_pose call made with timings != NULL
 * (the fields TimeMeasure accumulates, TimeMeasure.h:7-62), in milliseconds, CUDA-event timed
 * on the context's stream.  Requesting timings runs the loop launch-by-launch (no graph). */
typedef struct icp_gpu_timings {
    double selection_ms;   /* TimeMeasure::selectionTime   */
    double matching_ms;    /* TimeMeasure::matchingTime    (transform + search + weighting + rejection kernel) */
    double weighting_ms;   /* TimeMeasure::weighingTime    (0: fused into matching)                */
    double rejection_ms;   /* TimeMeasure::rejectionTime   (0: fused into matching)                */
    double solver_ms;      /* TimeMeasure::solverTime      (residual/Jacobian reduction + solve + pose update) */
    double index_ms;       /* buildIndex (grid build), once per registration                       */
    double total_ms;       /* TimeMeasure::convergenceTime                                         */
    int32_t n_iterations;  /* iterations executed                                                   */
    int32_t n_match_launches, n_solver_launches;
    int32_t reserved_;
    double search_prep_ms; /* part of matching_ms spent in the thread-per-query kernel (transform + fast-path search);
                              the rest is the warp-per-query tree walk                              */
} icp_gpu_timings;

/* Work counters of the last estimate_pose / query_matches (for roofline accounting). */
typedef struct icp_gpu_stats {
    uint64_t n_queries;        /* source points submitted to matching, summed over iterations      */
    uint64_t n_matched;        /* correspondences that survived threshold + rejection              */
    uint64_t n_distance_evals; /* point-to-point squared distances evaluated by the search         */
    uint64_t n_nodes_visited;  /* BVH nodes entered (internal nodes and leaves)                    */
    uint64_t n_kernel_launches;/* kernels launched by this library in the call                     */
    uint64_t reduce_profile_ns[6]; /* ICP_GPU_REDUCE_PROFILE=1 (environment): device timestamps (%globaltimer, ns) of the LAST
                                      reduction launch -- [0] first block starts, [1] the block that ends up last starts,
                                      [2] its point loop is done, [3] all rows summed (and exchanged with the peers),
                                      [4] system solved and pose written; else 0                        */
} icp_gpu_stats;

typedef struct icp_gpu_ctx icp_gpu_ctx;

int icp_gpu_abi_version(void);
/* Number of CUDA devices visible (0 when there is none or no driver). */
int icp_gpu_device_count(void);

int icp_gpu_create(icp_gpu_ctx** out, int device);
int icp_gpu_destroy(icp_gpu_ctx* ctx);
const char* icp_gpu_last_error(const icp_gpu_ctx* ctx);
/* Run on a caller-owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream); NULL restores
 * the context's own stream. */
int icp_gpu_set_stream(icp_gpu_ctx* ctx, void* cuda_stream);
int icp_gpu_synchronize(icp_gpu_ctx* ctx);

/* ICPOptimizer constructor defaults (ICPOptimizer.h:29-37). */
void icp_gpu_default_config(icp_gpu_config* cfg);
/* The ICPOptimizer setters (ICPOptimizer.h:41-95) in one call. */
int icp_gpu_set_config(icp_gpu_ctx* ctx, const icp_gpu_config* cfg);
int icp_gpu_get_config(const icp_gpu_ctx* ctx, icp_gpu_config* cfg);
/* ICPOptimizer::setCameraParamsMatchingMethod / NearestNeighborSearch::setCameraParams
 * (ICPOptimizer.h:80, NearestNeighbor.h:26-30). */
int icp_gpu_set_camera(icp_gpu_ctx* ctx, const float K_colmajor[9], uint32_t width, uint32_t height);

/* NearestNeighborSearch::buildIndex(points[, colours]) (NearestNeighbor.h:122-141, :209-232,
 * :324-331) plus the target normals the later stages read.  nrm / rgba may be NULL when the
 * configured variant does not read them.  Copies to device and builds the search grid. */
int icp_gpu_set_target(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n);
/* The source cloud estimatePose iterates over (ICPOptimizer.h:493). */
int icp_gpu_set_source(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n);
/* Same, from device pointers (same packed layouts) already resident on the context's device. */
int icp_gpu_set_target_dev(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n);
int icp_gpu_set_source_dev(icp_gpu_ctx* ctx, const float* xyz, const float* nrm, const uint8_t* rgba, int64_t n);

/* Stages 2-4 of one iteration at a given pose: transformPoints/transformNormals (utils.h:106-133),
 * queryMatches (NearestNeighbor.h:143-207, :234-303, :333-421), applyWeights (weighting.h:39-99)
 * and pruneCorrespondences (ICPOptimizer.h:157-174).  sel_idx (nullable) = ascending source
 * indices of the selected subset; NULL = all points.  idx_out / weight_out have n_sel (or n_source)
 * entries: Match{idx, weight}; idx is an index into the target as passed to set_target. */
int icp_gpu_query_matches(icp_gpu_ctx* ctx, const float pose[16], const int32_t* sel_idx, int64_t n_sel,
                          int32_t* idx_out, float* weight_out);

/* ICPOptimizer::estimatePose (ICPOptimizer.h:140): the whole iteration loop on the device.
 * pose_history (nullable) receives 16 floats per executed iteration (what the reference hands to
 * ConvergenceMeasure::recordAlignmentError, ICPOptimizer.h:629-631); it must hold
 * icp_gpu_max_iterations() entries.  n_iterations_out (nullable) = iterations executed. */
int icp_gpu_estimate_pose(icp_gpu_ctx* ctx, float pose_inout[16], float* pose_history, int32_t* n_iterations_out,
                          icp_gpu_timings* timings);
/* Upper bound of the iterations estimate_pose will run for the current config and source
 * (max(nIter, pyramid levels) in multi-resolution mode, ICPOptimizer.h:540,634-655). */
int icp_gpu_max_iterations(const icp_gpu_ctx* ctx);
/* Asynchronous form for queues of pairs: enqueue the registration on the context's stream without
 * waiting; the result is fetched (and waited for) by icp_gpu_estimate_pose_finish. */
int icp_gpu_estimate_pose_async(icp_gpu_ctx* ctx, const float pose_in[16]);
int icp_gpu_estimate_pose_finish(icp_gpu_ctx* ctx, float pose_out[16], float* pose_history, int32_t* n_iterations_out);

/* B independent registrations with the context's configuration, one thread block per pair, one launch: for many small
 * pairs (bunny-sized trials, multi-start registration), where the per-pair index build and launch chain of
 * icp_gpu_estimate_pose cost more than the work.  Clouds are concatenated; pair b owns source points
 * [src_off[b], src_off[b+1]) and target points [tgt_off[b], tgt_off[b+1]) (B+1 offsets each, starting at 0, monotone).
 * Indices are local to the pair (the device selection stream hashes the pair-local source index).  src_nrm / tgt_nrm
 * nullable (= zero normals); no colours (the colour weighting sees equal colours).  poses_in / poses_out: B x 16 floats;
 * n_iterations_out[b] = iterations applied; status_out[b] = ICP_GPU_OK / ICP_GPU_E_NO_MATCHES / ICP_GPU_E_NUMERIC per pair,
 * a failed pair keeping its last good pose (the call itself returns OK once the batch ran).  pose_history (nullable) =
 * B x n_iterations x 16 floats, rows past a pair's last iteration 0.
 * Supported: k-NN matching (exact, the brute-force scan's correspondences), the linear minimiser, every metric, weighting
 * and rejection, select-all or ICP_GPU_RNG_DEVICE random selection, early stop.  Refused with ICP_GPU_E_ARG: LM,
 * multi-resolution, projective, colour ICP, ICP_GPU_NN_BRUTE_NORM, mt19937 selection (LM, multi-resolution and mt19937
 * selection run through icp_gpu_estimate_pose_batch_configs), a pair with more than
 * ICP_GPU_BATCH_MAX_TARGET target points (register it with icp_gpu_estimate_pose), bad offsets.  ICP_GPU_E_STATE while a
 * registration is pending.  The context's own clouds, index and graphs are left as they are; the call runs on the
 * context's stream and returns when the batch is done.
 * _dev: every array (offsets included) is a device pointer on the context's device; the offsets are read back to check them. */
#define ICP_GPU_BATCH_MAX_TARGET 8192
int icp_gpu_estimate_pose_batch(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                                const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in, float* poses_out,
                                int32_t* n_iterations_out, int32_t* status_out, float* pose_history);
int icp_gpu_estimate_pose_batch_dev(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                                    const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in, float* poses_out,
                                    int32_t* n_iterations_out, int32_t* status_out, float* pose_history);

/* The number of iterations estimate_pose runs at most for configuration cfg and a source of n_source points: n_iterations, or
 * max(n_iterations, pyramid levels) with multires (ICPOptimizer.h:503-525, :634-655).  A pure function of its arguments, no
 * context or device needed; ICP_GPU_E_ARG for a null cfg or n_source outside [0, INT32_MAX]. */
int icp_gpu_iterations_bound(const icp_gpu_config* cfg, int64_t n_source);

/* B registrations with one configuration per pair: pair b runs with configs[config_index[b]] (n_configs >= 1 entries; the
 * context's own configuration is not used).  Cloud, offset, pose and status layout as icp_gpu_estimate_pose_batch.
 * pose_history (nullable) = B x history_rows x 16 floats, history_rows >= the largest icp_gpu_iterations_bound of the batch's
 * pairs; rows past a pair's last iteration 0.  n_iterations_out[b] = iterations applied.
 * Accepted per configuration: both minimisers (one block per pair either way), every metric and weighting, rejection on or off,
 * select-all, random selection with mt19937 (reference-compatible, masks drawn on the host and shared by every pair with the
 * same configuration, source size and, with multires, the same finite points) or with the device stream, the STRIDE
 * multi-resolution schedule, early stop, lm_max_iterations.  Every field is checked as icp_gpu_set_config checks it.
 * Refused with ICP_GPU_E_ARG, the message naming the pair or configuration: projective matching, colour ICP,
 * ICP_GPU_NN_BRUTE_NORM, the VOXEL pyramid, a target above ICP_GPU_BATCH_MAX_TARGET points, a config_index out of range,
 * n_configs < 1, history_rows below the bound when a history is asked for, bad offsets.
 * Pairs are grouped by (minimiser, metric); the groups run concurrently, one launch each, and the call returns when all are done.
 * _dev: every per-pair array (offsets and config_index included) is a device pointer on the context's device; configs stays a
 * host array.  The offsets and config_index are read back to check them and plan the groups; with multires and mt19937
 * selection the sources' points and normals are read back too (once per call), for the finite flags the masks depend on. */
int icp_gpu_estimate_pose_batch_configs(icp_gpu_ctx* ctx, int32_t n_configs, const icp_gpu_config* configs, int32_t n_pairs,
                                        const int32_t* config_index, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                                        const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in,
                                        float* poses_out, int32_t* n_iterations_out, int32_t* status_out, float* pose_history,
                                        int32_t history_rows);
int icp_gpu_estimate_pose_batch_configs_dev(icp_gpu_ctx* ctx, int32_t n_configs, const icp_gpu_config* configs, int32_t n_pairs,
                                            const int32_t* config_index, const float* src_xyz, const float* src_nrm, const int64_t* src_off,
                                            const float* tgt_xyz, const float* tgt_nrm, const int64_t* tgt_off, const float* poses_in,
                                            float* poses_out, int32_t* n_iterations_out, int32_t* status_out, float* pose_history,
                                            int32_t history_rows);

/* Multi-start registration: n_starts (K) registrations of the context's source against the context's target, with the context's
 * configuration, in one launch; start k begins at poses_in[k] (K x 16 floats, column-major).  The target's index is the one
 * set_target built; every start keeps its own neighbours, so the context's pose, remembered neighbours and graphs are left as they are.
 * Per start: poses_out[k], n_iterations_out[k] and pose_history (nullable: K x icp_gpu_max_iterations() x 16 floats, rows past a
 * start's last iteration 0) as icp_gpu_estimate_pose gives them from that start, and status_out[k] = ICP_GPU_OK /
 * ICP_GPU_E_NO_MATCHES / ICP_GPU_E_NUMERIC, a failed start keeping its last good pose (the call returns OK once the launch ran).
 * Scoring: after its last iteration each start matches once more at its final pose, every source point (no selection, no stride),
 * with the configuration's threshold, weighting and rejection -- icp_gpu_query_matches(poses_out[k], NULL).  inliers_out[k] = the
 * surviving matches; rmse_out[k] = sqrt of the fp64 mean of their D1 squared distances (the 6-D distance with colour ICP; NaN without
 * an inlier); match_idx_out / match_w_out (nullable, together: K x n_source, original source order) = that call's idx / weight.
 * n_iterations = 0 makes the call a pose scorer.  Accepted: everything icp_gpu_estimate_pose runs with k-NN matching -- both
 * minimisers, every metric and weighting, rejection, 3-D or colour 6-D search, select-all / mt19937 / device-stream selection, the
 * STRIDE and VOXEL pyramids, early stop; nn_algorithm AUTO, BRUTE and GRID all search the index (the same correspondences).
 * Refused with ICP_GPU_E_ARG: projective matching, ICP_GPU_NN_BRUTE_NORM, attached peers, a null required array, n_starts < 0,
 * n_starts x n_source above INT32_MAX.  ICP_GPU_E_STATE: no source or target, a pending registration.  n_starts = 0: OK, nothing runs.
 * Each start runs on a cluster of up to 16 thread blocks (more blocks per start when K is small); its outputs are the same bits
 * whatever K is.  Where it pays (measured on one B200 at 1000 W, DESIGN.md section 6): subsampled sources of ~10k points, 1.5x a loop
 * of icp_gpu_estimate_pose at K = 24 and 3x from K = 148 on.  Where it loses: K = 1 (8x slower) and K = 8 (0.76x), and full-size
 * sources at any K (a loop of icp_gpu_estimate_pose is 1.4x to 18x faster there).
 * _dev: every array is a device pointer on the context's device.  The call waits for the launch either way. */
int icp_gpu_estimate_pose_multistart(icp_gpu_ctx* ctx, int32_t n_starts, const float* poses_in, float* poses_out, int32_t* n_iterations_out,
                                     int32_t* status_out, int64_t* inliers_out, double* rmse_out, float* pose_history, int32_t* match_idx_out,
                                     float* match_w_out);
int icp_gpu_estimate_pose_multistart_dev(icp_gpu_ctx* ctx, int32_t n_starts, const float* poses_in, float* poses_out, int32_t* n_iterations_out,
                                         int32_t* status_out, int64_t* inliers_out, double* rmse_out, float* pose_history, int32_t* match_idx_out,
                                         float* match_w_out);

/* ---- many pairs of any size, each against its own index, in one launch --------------------------------------------------
 * icp_gpu_estimate_pose_batch_indexed: B = n_pairs independent registrations with the context's configuration.  The clouds are
 * concatenated as in icp_gpu_estimate_pose_batch: pair b owns source points [src_off[b], src_off[b+1]) and target points
 * [tgt_off[b], tgt_off[b+1]) (B+1 offsets each, starting at 0); normals and colours (RGBA, 4 bytes a point) are nullable with the
 * meaning icp_gpu_set_source / icp_gpu_set_target give to NULL.  The call builds an index of every pair's target (the one set_target
 * builds), then runs every pair on its own thread-block cluster in one launch.  Per pair the outputs are exactly those of
 * icp_gpu_estimate_pose_multistart with one start on a context holding that pair: poses_out[b] (B x 16 floats, column-major; pair b
 * starts at poses_in[b]), n_iterations_out[b], status_out[b] (a failed pair keeps its last good pose), the scoring pass's
 * inliers_out[b] and rmse_out[b], and with match_idx_out / match_w_out (nullable, together) sum(n_src) entries in each pair's original
 * source order, pair b's at src_off[b].  pose_history (nullable): B x history_rows x 16 floats, history_rows at least the largest
 * icp_gpu_iterations_bound over the batch's sources; rows past a pair's last iteration 0.  Accepted: what multistart accepts, pairs of
 * any size, empty sources and targets included.  Refused with ICP_GPU_E_ARG: projective matching, ICP_GPU_NN_BRUTE_NORM, attached
 * peers, a null required array or only one of the two match arrays, n_pairs < 0, offsets that do not start at 0 or are not monotone,
 * a pair above set_target's size limit, sum(n_src) above INT32_MAX, history_rows below the bound when a history is asked for.
 * ICP_GPU_E_STATE while a registration is pending.  n_pairs = 0: OK, nothing runs.  The context's clouds, index, pose, remembered
 * neighbours and graphs are left as they are.  _dev: every array is a device pointer on the context's device.  The call waits for
 * its work either way.  Measured on one B200 at 1000 W, point-to-plane, from host arrays, every arm on warmed contexts (DESIGN.md
 * section 6): against a loop of set_target + set_source + icp_gpu_estimate_pose on one context it pays 2.2x to 2.7x for 64 to 4096
 * small or ~12.9k-point pairs, only 1.2x to 1.3x for ~45k-point pairs, and it LOSES for a single pair (0.48x).  Against the same
 * registrations spread over three contexts (alignPairs) it is 0.93x to 1.02x for ~12.9k-point, 8192-point and bunny-sized pairs and
 * 0.5x for ~45k-point pairs and for a single pair.  Against icp_gpu_estimate_pose_batch it is 35x faster on 8192-point pairs and
 * 0.19x on bunny-sized pairs.  The pairs' index builds run one after another and take 0.5 to 0.97 of the call. */
int icp_gpu_estimate_pose_batch_indexed(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const uint8_t* src_rgba,
                                        const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm, const uint8_t* tgt_rgba, const int64_t* tgt_off,
                                        const float* poses_in, float* poses_out, int32_t* n_iterations_out, int32_t* status_out, int64_t* inliers_out,
                                        double* rmse_out, float* pose_history, int32_t history_rows, int32_t* match_idx_out, float* match_w_out);
int icp_gpu_estimate_pose_batch_indexed_dev(icp_gpu_ctx* ctx, int32_t n_pairs, const float* src_xyz, const float* src_nrm, const uint8_t* src_rgba,
                                            const int64_t* src_off, const float* tgt_xyz, const float* tgt_nrm, const uint8_t* tgt_rgba,
                                            const int64_t* tgt_off, const float* poses_in, float* poses_out, int32_t* n_iterations_out,
                                            int32_t* status_out, int64_t* inliers_out, double* rmse_out, float* pose_history, int32_t history_rows,
                                            int32_t* match_idx_out, float* match_w_out);

int icp_gpu_get_stats(icp_gpu_ctx* ctx, icp_gpu_stats* out);
/* The FP32 (non-tensor) roofline denominator of the context's device, measured with a register-resident microbenchmark on
 * the context's stream (SURVEY.md 8d; the reference has no counterpart): mode 0 = FFMA (2 flop / instruction), mode 1 =
 * FMUL + FADD pairs (the un-fused arithmetic contract D1 prescribes for squared distances).  TFLOP/s. */
int icp_gpu_measure_fp32_peak(icp_gpu_ctx* ctx, int32_t mode, double* tflops_out);

/* ---- either side of the loop (SURVEY.md 8f) -------------------------------------------------------
 * icp_gpu_cloud_from_depth = PointCloud(float* depthMap, BYTE* colorFrame, const Matrix3f& depthIntrinsics,
 *   const Matrix4f& depthExtrinsics, width, height, keepOriginalSize, downsampleFactor, maxDistance)
 *   (PointCloud.h:78-165): back-projection, central-difference normals (MINF where invalid), the
 *   "point and normal finite" filter, every downsample-th pixel.  depth: width*height floats (MINF =
 *   invalid, VirtualSensor.h:119-124); rgbx: the RGBX frame (4*width*height bytes, nullable) -- the colour
 *   of kept pixel i is bytes rgbx[i .. i+3], exactly as PointCloud.h:151-152 indexes it; K: column-major
 *   3x3 intrinsics; E: column-major 4x4 depth extrinsics (nullable = identity).  role: the cloud becomes the
 *   context's target (= buildIndex), its source, or is only returned.  xyz_out / nrm_out / rgba_out
 *   (nullable, host) need room for ceil(width*height / downsample) points; *n_out = points produced. */
enum { ICP_GPU_CLOUD_TARGET = 0, ICP_GPU_CLOUD_SOURCE = 1, ICP_GPU_CLOUD_ONLY = 2 };
int icp_gpu_cloud_from_depth(icp_gpu_ctx* ctx, const float* depth, const uint8_t* rgbx, const float K_colmajor[9],
                             const float E_colmajor[16], uint32_t width, uint32_t height, int keep_original_size,
                             uint32_t downsample, float max_distance, int role,
                             float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* n_out);
/* PointCloud(pcl::PointCloud<pcl::PointXYZ>::Ptr) (PointCloud.h:41-76): pcl::NormalEstimation with setKSearch(k) (the
 * reference uses k = 5) and viewpoint (nullable = the origin) on the context's TARGET cloud, with the index
 * icp_gpu_set_target built: the k nearest neighbours of every point (itself included), the eigenvector of the smallest
 * eigenvalue of their covariance, flipped towards the viewpoint; NaN for non-finite points.  The normals replace the
 * target's own for the following registrations and are returned in the caller's point order (nrm_out: 3*n floats,
 * curvature_out: n floats, both nullable).  3 <= k <= 8. */
int icp_gpu_target_normals(icp_gpu_ctx* ctx, int32_t k, const float viewpoint[3], float* nrm_out, float* curvature_out);
/* icp_gpu_voxel_downsample: a voxel-grid filter (pcl::VoxelGrid, Open3D's voxel_down_sample) of n_clouds clouds in one pass: one
 * point per occupied voxel of edge voxel_size, the centroid of the voxel's points.  Cloud b is points [off[b], off[b+1]) (n_clouds+1
 * offsets, starting at 0, monotone, as icp_gpu_estimate_pose_batch_indexed takes them); nrm and rgba are nullable.  Cloud b's voxels
 * come back at [off_out[b], off_out[b+1]) of xyz_out / nrm_out / rgba_out, each of which needs room for off[n_clouds] points.
 * Arithmetic (DESIGN.md section 4, V1-V5): only points with three finite coordinates are used; a point's voxel is
 * floorf(x * (1.0f / voxel_size)) per axis (PCL's world-anchored grid: clouds filtered at one size share it); a cloud's voxels come in
 * ascending (iz, iy, ix); a coordinate is the fp64 sum of the voxel's points in ascending input order over their count, rounded once
 * to fp32; a normal the same sum over the points whose normal is finite, over its fp64 norm (MINF when there is none or the norm is
 * 0); a colour channel (2 sum + k) / 2k in integers.  The result is a fixed function of the input, bit for bit.  nrm_out / rgba_out
 * are written only when nrm / rgba are given.  role (the values of icp_gpu_cloud_from_depth): with TARGET or SOURCE (n_clouds must
 * be 1) the result becomes the context's target, indexed, or source, as set_target / set_source of the returned arrays would make
 * it, and every output is nullable; with ONLY the context's clouds, index, pose, remembered neighbours and graphs stay as they are,
 * and xyz_out and off_out are required.  Refused with ICP_GPU_E_ARG: n_clouds < 0, a null required array, a non-null nrm_out /
 * rgba_out without its input, offsets that do not start at 0 or are not monotone, voxel_size not finite and > 0, a role out of range
 * or TARGET / SOURCE with n_clouds != 1, more than set_target's limit of points in all, a cloud whose finite points span more than
 * 2^21 voxels on an axis or whose voxel index does not fit int32 (the message names the cloud).  ICP_GPU_E_STATE while a
 * registration is pending.  n_clouds = 0: OK, nothing runs.  The kernels launched do not depend on n_clouds.  _dev: every array is
 * a device pointer on the context's device.  The call waits for its work either way.  Measured on one B200 at 1000 W (DESIGN.md
 * section 6): a 370k-point lidar scan takes 0.64 ms (_dev) at 2 cm and 5.9 ms at 20 cm -- one thread sums each voxel, so the largest
 * voxel bounds the call -- 85x to 7.6x the host round trip (download, filter on one core, upload); a 3 M-point scan at 5 cm 15.7 ms
 * (27x); batches of 44 to 512 scans in one call 17x to 24x a loop of single-cloud calls.  Where it loses: tiny clouds (the 1k-point
 * bunny: 0.18 ms, 0.72x a host filter on one core). */
int icp_gpu_voxel_downsample(icp_gpu_ctx* ctx, int32_t n_clouds, const float* xyz, const float* nrm, const uint8_t* rgba, const int64_t* off,
                             float voxel_size, int role, float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* off_out);
int icp_gpu_voxel_downsample_dev(icp_gpu_ctx* ctx, int32_t n_clouds, const float* xyz, const float* nrm, const uint8_t* rgba, const int64_t* off,
                                 float voxel_size, int role, float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* off_out);
/* ConvergenceMeasure(sourcePoints, unchangedPoints) (ConvergenceMeasure.h:32-41): m known correspondences
 * (source point i of the UNTRANSFORMED source <-> reference point i). */
int icp_gpu_set_correspondences(icp_gpu_ctx* ctx, const float* src_xyz, const float* ref_xyz, int64_t m);
/* The correspondences of reconstructRoom (main.cpp:300-307): every point of the current source against itself under a
 * ground-truth pose, unchangedPoints = transformPoints(source.getPoints(), gt_pose); built on the device. */
int icp_gpu_set_correspondences_pose(icp_gpu_ctx* ctx, const float gt_pose[16]);
/* recordAlignmentError after every iteration of the last finished registration (ICPOptimizer.h:629-631):
 * rmse_out[k] = rmseAlignmentError(pose after iteration k) (ConvergenceMeasure.h:50-66); benchmark_out[k]
 * (nullable) = benchmarkError (ConvergenceMeasure.h:104-151).  Evaluated on the device from the pose history. */
int icp_gpu_convergence_errors(icp_gpu_ctx* ctx, float* rmse_out, double* benchmark_out, int32_t capacity, int32_t* n_out);
/* rmseAlignmentError(pose) and (nullable) benchmarkError(pose) of one pose the caller supplies (ConvergenceMeasure.h:50-66, :104-151),
 * over the correspondences set before. */
int icp_gpu_alignment_error(icp_gpu_ctx* ctx, const float pose[16], float* rmse_out, double* benchmark_out);

/* ---- the reference API's value-level operations, for callers that use them outside estimatePose (the loop runs the same device
 * functions fused).  Host arrays in and out; each call synchronises the context's stream.
 *   icp_gpu_transform_points / _normals   transformPoints / transformNormals (utils.h:106-118, :122-133): q = R p + t;
 *                                         n' = (R^-1)^T n with the 3x3 inverse by cofactors.
 *   icp_gpu_apply_weights                 WeightingMethod(weighting, max_distance_sq).applyWeights (weighting.h:39-99): per source
 *                                         point i with idx[i] >= 0 the weight of the pair (i, idx[i]) replaces weight_inout[i];
 *                                         CONSTANT leaves everything as it is.  The source arrays are the TRANSFORMED ones.
 *   icp_gpu_solve_linear                  the closed-form minimisers on n matched pairs (source point i <-> target point i, both in
 *                                         the target's frame): metric 0 ProcrustesAligner::estimatePose (ProcrustesAligner.h:6-29),
 *                                         1 estimatePosePointToPlane (ICPOptimizer.h:676-782), 2 estimatePoseSymmetricICP (:784-898);
 *                                         weights nullable (= 1).  pose_out = the increment, column-major.  ICP_GPU_E_NO_MATCHES /
 *                                         ICP_GPU_E_NUMERIC instead of the reference's ASSERT / NaN pose. */
int icp_gpu_transform_points(icp_gpu_ctx* ctx, const float pose[16], const float* xyz_in, int64_t n, float* xyz_out);
int icp_gpu_transform_normals(icp_gpu_ctx* ctx, const float pose[16], const float* nrm_in, int64_t n, float* nrm_out);
int icp_gpu_apply_weights(icp_gpu_ctx* ctx, int32_t weighting, float max_distance_sq, const float* src_xyz, const float* src_nrm,
                          const uint8_t* src_rgba, int64_t n_src, const float* tgt_xyz, const float* tgt_nrm, const uint8_t* tgt_rgba,
                          int64_t n_tgt, const int32_t* idx, float* weight_inout);
int icp_gpu_solve_linear(icp_gpu_ctx* ctx, int32_t metric, const float* src_xyz, const float* src_nrm, const float* tgt_xyz, const float* tgt_nrm,
                         const float* weights, int64_t n, float pose_out[16]);

/* Point-sharded registration of one very large pair across ranks (one context per rank, each
 * holding the whole target and its shard of the source).  Per iteration:
 *   icp_gpu_iteration_local   -> this rank's partial sums (linear metrics: the normal equations,
 *                                <= ICP_GPU_MAX_PARTIALS doubles; the count is written to *n_values);
 *   (the caller all-reduces them, e.g. one NCCL ncclAllReduce(ncclDouble, ncclSum));
 *   icp_gpu_iteration_apply   -> every rank solves the identical system and updates its pose.
 * Symmetric / point-to-point need the matched-set means first: phase 0 yields 7 sums, phase 1 the
 * system.  n_phases = icp_gpu_iteration_phases(). */
#define ICP_GPU_MAX_PARTIALS 32
int icp_gpu_iteration_phases(const icp_gpu_ctx* ctx);
int icp_gpu_iteration_begin(icp_gpu_ctx* ctx, const float pose_in[16]);
int icp_gpu_iteration_local(icp_gpu_ctx* ctx, int phase, double* partials_out, int32_t* n_values);
int icp_gpu_iteration_apply(icp_gpu_ctx* ctx, int phase, const double* reduced_in, int32_t n_values);
int icp_gpu_iteration_end(icp_gpu_ctx* ctx, float pose_out[16]);
/* Device-pointer forms of the two above for collectives that run on the stream (NCCL):
 * returns the device address of the context's partial-sum buffer (ICP_GPU_MAX_PARTIALS doubles). */
int icp_gpu_iteration_local_dev(icp_gpu_ctx* ctx, int phase, double** partials_dev, int32_t* n_values);
int icp_gpu_iteration_apply_dev(icp_gpu_ctx* ctx, int phase);


/* The same registration with the exchange INSIDE the reduction kernel (no NCCL call, no host round trip per
 * iteration): every rank owns a small mailbox in device memory; the last block of each reduction stores its summed
 * row into every peer's mailbox over NVLink peer memory, waits for the peers' rows in its own, adds the rows in
 * rank order (bit-identical totals, hence identical poses on every rank) and solves.  Once the peers are attached,
 * icp_gpu_estimate_pose[_async] IS the point-sharded registration: a collective call -- every rank makes it with
 * the same configuration, the whole target and its own shard of the source -- whose loop is one CUDA graph.
 *   icp_gpu_peer_export       allocates (or resets) this context's mailbox and returns a 64-byte handle
 *                             (cudaIpcMemHandle_t) the caller hands to the other ranks (MPI / torch.distributed);
 *   icp_gpu_peer_attach       handles = world x 64 bytes in rank order; opens the peers' mailboxes;
 *   icp_gpu_peer_address / icp_gpu_peer_attach_ptrs
 *                             the same for contexts of ONE process (device addresses instead of handles; devices
 *                             other than the context's own need peer access enabled by the caller);
 *   icp_gpu_peer_detach       back to a single-context registration.
 * Every rank must export before any rank attaches, and all ranks attach before the first registration (the handle
 * exchange is that barrier).  A rank whose peer does not arrive within ICP_GPU_PEER_TIMEOUT_MS (environment,
 * default 2000) finishes with ICP_GPU_E_PEER instead of hanging; the ranks' exchange counters are then out of step, so
 * every rank has to export and attach again before the next registration.  world <= ICP_GPU_MAX_PEERS. */
#define ICP_GPU_MAX_PEERS 8
#define ICP_GPU_PEER_HANDLE_BYTES 64
int icp_gpu_peer_export(icp_gpu_ctx* ctx, void* handle_out);
int icp_gpu_peer_attach(icp_gpu_ctx* ctx, int32_t rank, int32_t world, const void* handles);
int icp_gpu_peer_address(icp_gpu_ctx* ctx, void** mailbox_dev);
int icp_gpu_peer_attach_ptrs(icp_gpu_ctx* ctx, int32_t rank, int32_t world, void* const* mailboxes_dev);
int icp_gpu_peer_detach(icp_gpu_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* ICP_GPU_H */
