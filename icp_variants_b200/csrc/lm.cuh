// lm.cuh -- the Levenberg-Marquardt pieces shared by lm_eval_kernel (lm.cu, one registration over the whole grid) and
// batch_lm_kernel (batch.cu, one registration per block), each compiled into its own translation unit: the fp64 jets and
// ceres::AngleAxisRotatePoint, one match's residual blocks, and the trust-region state machine on an LmState.
//
// Reference: CeresICPOptimizer::estimatePose inner solve (ICPOptimizer.h:283-310), configureSolver
// (:352-360: LEVENBERG_MARQUARDT, monotonic steps, DENSE_QR, max_num_iterations 10, Ceres defaults
// otherwise), prepareConstraints* (:362-482), the functors of constraints.h and PoseIncrement
// (utils.h:25-102).  Ceres itself is an un-vendored dependency; its trust-region loop is restated from
// the published algorithm exactly as oracle/icp_oracle.c:orc_solve_lm does (same order of tests).
// Jacobians are forward-mode dual numbers in fp64 (what Ceres' autodiff computes), with the rotation jets
// shared by all residuals of a thread.
#pragma once
#include "icp_internal.cuh"
#include <float.h>

struct Jet { double v; double d[6]; };

__device__ __forceinline__ Jet jconst(double v) { Jet r; r.v = v; for (int i = 0; i < 6; ++i) r.d[i] = 0.0; return r; }
__device__ __forceinline__ Jet jadd(const Jet& a, const Jet& b) { Jet r; r.v = a.v + b.v; for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] + b.d[i]; return r; }
__device__ __forceinline__ Jet jsub(const Jet& a, const Jet& b) { Jet r; r.v = a.v - b.v; for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] - b.d[i]; return r; }
__device__ __forceinline__ Jet jmul(const Jet& a, const Jet& b) { Jet r; r.v = a.v * b.v; for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] * b.v + a.v * b.d[i]; return r; }
__device__ __forceinline__ Jet jscale(const Jet& a, double c) { Jet r; r.v = a.v * c; for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] * c; return r; }
__device__ __forceinline__ Jet jaddc(const Jet& a, double c) { Jet r = a; r.v += c; return r; }
__device__ __forceinline__ Jet jneg(const Jet& a) { Jet r; r.v = -a.v; for (int i = 0; i < 6; ++i) r.d[i] = -a.d[i]; return r; }
__device__ __forceinline__ Jet jdiv(const Jet& a, const Jet& b) { Jet r; const double inv = 1.0 / b.v; r.v = a.v * inv; for (int i = 0; i < 6; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) * inv; return r; }
__device__ __forceinline__ Jet jsqrt(const Jet& a) { Jet r; r.v = sqrt(a.v); const double k = 1.0 / (2.0 * r.v); for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] * k; return r; }
__device__ __forceinline__ Jet jcos(const Jet& a) { Jet r; r.v = cos(a.v); const double k = -sin(a.v); for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] * k; return r; }
__device__ __forceinline__ Jet jsin(const Jet& a) { Jet r; r.v = sin(a.v); const double k = cos(a.v); for (int i = 0; i < 6; ++i) r.d[i] = a.d[i] * k; return r; }

// ceres::AngleAxisRotatePoint for a fixed angle-axis jet triple, applied to constant points.
struct Rotator {
    bool big;          // theta^2 > DBL_EPSILON: Rodrigues; else first-order p + aa x p
    Jet aa[3], w[3], c, s, omc;
};

static __device__ void rotator_init(Rotator& R, const Jet aa[3]) {
    for (int k = 0; k < 3; ++k) R.aa[k] = aa[k];
    const Jet theta2 = jadd(jadd(jmul(aa[0], aa[0]), jmul(aa[1], aa[1])), jmul(aa[2], aa[2]));
    R.big = theta2.v > DBL_EPSILON;
    if (R.big) {
        const Jet theta = jsqrt(theta2);
        R.c = jcos(theta); R.s = jsin(theta);
        const Jet ti = jdiv(jconst(1.0), theta);
        for (int k = 0; k < 3; ++k) R.w[k] = jmul(aa[k], ti);
        R.omc = jsub(jconst(1.0), R.c);
    }
}

static __device__ void rotate_const(const Rotator& R, const double p[3], Jet out[3]) {
    if (R.big) {
        const Jet wxp[3] = {jsub(jscale(R.w[1], p[2]), jscale(R.w[2], p[1])), jsub(jscale(R.w[2], p[0]), jscale(R.w[0], p[2])),
                            jsub(jscale(R.w[0], p[1]), jscale(R.w[1], p[0]))};
        const Jet tmp = jmul(jadd(jadd(jscale(R.w[0], p[0]), jscale(R.w[1], p[1])), jscale(R.w[2], p[2])), R.omc);
        for (int i = 0; i < 3; ++i) out[i] = jadd(jadd(jscale(R.c, p[i]), jmul(wxp[i], R.s)), jmul(R.w[i], tmp));
    } else {
        const Jet wxp[3] = {jsub(jscale(R.aa[1], p[2]), jscale(R.aa[2], p[1])), jsub(jscale(R.aa[2], p[0]), jscale(R.aa[0], p[2])),
                            jsub(jscale(R.aa[0], p[1]), jscale(R.aa[1], p[0]))};
        for (int i = 0; i < 3; ++i) out[i] = jaddc(wxp[i], p[i]);
    }
}

// Row layout: [0..20] J^T J upper triangle row-major, [21..26] J^T r, [27] sum r^2, [28] residual count.
__device__ __forceinline__ void accumulate(double (&v)[32], const Jet& r) {
    int k = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = a; b < 6; ++b) v[k++] += r.d[a] * r.d[b];
#pragma unroll
    for (int a = 0; a < 6; ++a) v[21 + a] += r.d[a] * r.v;
    v[27] += r.v * r.v;
    v[28] += 1.0;
}

// The residual jets of one evaluation at x: the pose increment (with unit derivatives) and its rotations (PoseIncrement::apply,
// utils.h:44-56; the symmetric metric's inverse rotation, utils.h:60-72).
struct LmJets { Jet pose[6]; Rotator rot, rinv; };

template <int METRIC>
__device__ __forceinline__ void lm_jets_init(LmJets& J, const double* x) {
    for (int i = 0; i < 6; ++i) { J.pose[i] = jconst(x[i]); J.pose[i].d[i] = 1.0; }
    rotator_init(J.rot, J.pose);
    if (METRIC == ICP_GPU_METRIC_SYMMETRIC) { const Jet ninv[3] = {jneg(J.pose[0]), jneg(J.pose[1]), jneg(J.pose[2])}; rotator_init(J.rinv, ninv); }
}

// One match's residual blocks into the row above.  (sxf, syf, szf): the source point transformed by the current pose, tp: the
// matched target point (both finite: ICPOptimizer.h:378 skips the others), w: the match weight; tn() / sn() fetch the target normal and the source normal, called only by the
// metrics that read them; Nm: the current pose's inverse-transpose.
template <int METRIC, class TN, class SN>
__device__ __forceinline__ void lm_accumulate_match(double (&v)[32], const LmJets& J, float sxf, float syf, float szf, const float4 tp,
                                                    const double w, const float* Nm, TN&& tn_of, SN&& sn_of) {
    const double s[3] = {sxf, syf, szf}, t[3] = {tp.x, tp.y, tp.z};
    Jet y[3];
    rotate_const(J.rot, s, y);
    for (int k = 0; k < 3; ++k) y[k] = jadd(y[k], J.pose[3 + k]);
    const double lw_pt = (double)0.1f * w;                                        // PointToPointConstraint LAMBDA (constraints.h)
    for (int k = 0; k < 3; ++k) accumulate(v, jscale(jaddc(y[k], -t[k]), lw_pt));
    if (METRIC == ICP_GPU_METRIC_P2PLANE) {
        const float4 tn = tn_of();
        if (finite3(tn.x, tn.y, tn.z)) {                                          // ICPOptimizer.h:420-423
            const Jet acc = jadd(jadd(jscale(jaddc(y[0], -t[0]), (double)tn.x), jscale(jaddc(y[1], -t[1]), (double)tn.y)),
                                 jscale(jaddc(y[2], -t[2]), (double)tn.z));
            accumulate(v, jscale(acc, (double)1.0f * w));
        }
    } else if (METRIC == ICP_GPU_METRIC_SYMMETRIC) {
        const float4 tn = tn_of();
        const float4 sn4 = sn_of();
        float nx, ny, nz;
        xform_normal(Nm, sn4.x, sn4.y, sn4.z, nx, ny, nz);
        if (finite3(tn.x, tn.y, tn.z) && finite3(nx, ny, nz)) {                   // ICPOptimizer.h:465-469
            Jet z[3];
            rotate_const(J.rinv, t, z);
            const double m[3] = {(double)tn.x + (double)nx, (double)tn.y + (double)ny, (double)tn.z + (double)nz};
            const Jet acc = jadd(jadd(jscale(jsub(y[0], z[0]), m[0]), jscale(jsub(y[1], z[1]), m[1])), jscale(jsub(y[2], z[2]), m[2]));
            accumulate(v, jscale(acc, (double)1.0f * w));
        }
    }
}

// PoseIncrement<double>::convertToMatrix (utils.h:79-98) via ceres::AngleAxisToRotationMatrix
static __device__ void increment_matrix(const double* x, float* inc) {
    double R[9];
    const double theta2 = x[0] * x[0] + x[1] * x[1] + x[2] * x[2];
    if (theta2 > DBL_EPSILON) {
        const double theta = sqrt(theta2);
        const double wx = x[0] / theta, wy = x[1] / theta, wz = x[2] / theta;
        const double ct = cos(theta), st = sin(theta);
        R[0] = ct + wx * wx * (1.0 - ct);      R[1] = wz * st + wx * wy * (1.0 - ct);  R[2] = -wy * st + wx * wz * (1.0 - ct);
        R[3] = wx * wy * (1.0 - ct) - wz * st; R[4] = ct + wy * wy * (1.0 - ct);       R[5] = wx * st + wy * wz * (1.0 - ct);
        R[6] = wy * st + wx * wz * (1.0 - ct); R[7] = -wx * st + wy * wz * (1.0 - ct); R[8] = ct + wz * wz * (1.0 - ct);
    } else {
        R[0] = 1; R[1] = x[2]; R[2] = -x[1]; R[3] = -x[2]; R[4] = 1; R[5] = x[0]; R[6] = x[1]; R[7] = -x[0]; R[8] = 1;
    }
    mat4_identity_dev(inc);
    for (int c = 0; c < 3; ++c) for (int r = 0; r < 3; ++r) inc[r + 4 * c] = (float)R[r + 3 * c];   // column-major both sides
    inc[12] = (float)x[3]; inc[13] = (float)x[4]; inc[14] = (float)x[5];
}

static __device__ void unpack_system(const double* row, double* H, double* g, double* cost) {
    int k = 0;
    for (int i = 0; i < 6; ++i) for (int j = i; j < 6; ++j) { H[i * 6 + j] = row[k]; H[j * 6 + i] = row[k]; ++k; }
    for (int i = 0; i < 6; ++i) g[i] = row[21 + i];
    *cost = 0.5 * row[27];
}

// The state machine returns LM_NEXT_EVAL when a candidate waits in st->cand for its evaluation; otherwise the solve is over
// (st->done = 1) and the return value is the status of the outer iteration (0, or ICP_GPU_E_NO_MATCHES): the caller then applies
// increment_matrix(st->x).
#define LM_NEXT_EVAL (-1)

// Top of TrustRegionMinimizer's loop: termination tests, then LevenbergMarquardtStrategy::ComputeStep
// in the Jacobi-scaled space; loops over invalid steps (they need no evaluation).
static __device__ int lm_next_step(LmState* st, int max_iterations) {
    const double min_radius = 1e-32, min_diag = 1e-6, max_diag = 1e32, gradient_tolerance = 1e-10;
    for (;;) {
        double gmax = 0.0;
        for (int i = 0; i < 6; ++i) gmax = fmax(gmax, fabs(st->g[i]));
        if (st->iter >= max_iterations || (st->step_ok && gmax <= gradient_tolerance) || st->radius <= min_radius) { st->done = 1; return 0; }
        st->iter += 1;
        double Hs[36], gs[6], A[36], b[6], ds[6];
        for (int a = 0; a < 6; ++a) {
            gs[a] = st->g[a] * st->scale[a];
            for (int c = 0; c < 6; ++c) Hs[a * 6 + c] = st->H[a * 6 + c] * st->scale[a] * st->scale[c];
        }
        if (!st->reuse_diag)
            for (int a = 0; a < 6; ++a) { const double v = Hs[a * 6 + a]; st->diag[a] = v < min_diag ? min_diag : (v > max_diag ? max_diag : v); }
        for (int i = 0; i < 36; ++i) A[i] = Hs[i];
        for (int a = 0; a < 6; ++a) { A[a * 6 + a] += st->diag[a] / st->radius; b[a] = -gs[a]; }
        const bool lin_ok = solve6_dev(A, b, ds) == 0;
        double model_cost_change = 0.0;
        if (lin_ok)
            for (int a = 0; a < 6; ++a) {
                double hd = 0.0;
                for (int c = 0; c < 6; ++c) hd += Hs[a * 6 + c] * ds[c];
                model_cost_change -= ds[a] * (gs[a] + 0.5 * hd);
            }
        if (!lin_ok || !(model_cost_change > 0.0)) {            // HandleInvalidStep
            st->invalid += 1;
            if (st->invalid >= 5) { st->done = 1; return 0; }
            st->radius *= 0.5; st->reuse_diag = 1; st->step_ok = 0;
            continue;
        }
        st->invalid = 0;
        st->model_change = model_cost_change;
        for (int a = 0; a < 6; ++a) st->cand[a] = st->x[a] + ds[a] * st->scale[a];
        st->have_cand = 1;
        return LM_NEXT_EVAL;
    }
}

// One evaluation's summed row: step_index 0 = the evaluation at x = 0, else the evaluation at st->cand.
static __device__ int lm_advance(LmState* st, const double* row, int step_index, int max_iterations) {
    const double min_relative_decrease = 1e-3, function_tolerance = 1e-6, parameter_tolerance = 1e-8, max_radius = 1e16;
    if (step_index == 0) {
        // initial evaluation at x = 0 (poseIncrement.setZero(), ICPOptimizer.h:236,310)
        for (int i = 0; i < 6; ++i) st->x[i] = 0.0;
        st->iter = 0; st->done = 0; st->reuse_diag = 0; st->invalid = 0; st->step_ok = 1; st->have_cand = 0;
        st->radius = 1e4; st->decrease = 2.0;
        if (!(row[28] > 0.0)) { st->done = 1; return ICP_GPU_E_NO_MATCHES; }
        unpack_system(row, st->H, st->g, &st->cost);
        for (int i = 0; i < 6; ++i) st->scale[i] = 1.0 / (1.0 + sqrt(st->H[i * 6 + i]));   // jacobi_scaling
        return lm_next_step(st, max_iterations);
    }
    // evaluation at the candidate
    double Hc[36], gc[6], cand_cost;
    unpack_system(row, Hc, gc, &cand_cost);
    double step_norm = 0.0, x_norm = 0.0;
    for (int a = 0; a < 6; ++a) { const double d = st->x[a] - st->cand[a]; step_norm += d * d; x_norm += st->x[a] * st->x[a]; }
    step_norm = sqrt(step_norm); x_norm = sqrt(x_norm);
    if (step_norm <= parameter_tolerance * (x_norm + parameter_tolerance)) { st->done = 1; return 0; }   // ParameterToleranceReached
    const double cost_change = st->cost - cand_cost;
    if (fabs(cost_change) <= function_tolerance * st->cost) { st->done = 1; return 0; }                // FunctionToleranceReached
    const double rho = cost_change / st->model_change;
    if (rho > min_relative_decrease) {                                                                  // HandleSuccessfulStep
        for (int a = 0; a < 6; ++a) { st->x[a] = st->cand[a]; st->g[a] = gc[a]; }
        for (int i = 0; i < 36; ++i) st->H[i] = Hc[i];
        st->cost = cand_cost;
        const double t = 2.0 * rho - 1.0;
        double denom = 1.0 - t * t * t; if (denom < 1.0 / 3.0) denom = 1.0 / 3.0;
        st->radius = st->radius / denom; if (st->radius > max_radius) st->radius = max_radius;
        st->decrease = 2.0; st->reuse_diag = 0; st->step_ok = 1;
    } else {                                                                                            // HandleUnsuccessfulStep
        st->radius = st->radius / st->decrease; st->decrease *= 2.0; st->reuse_diag = 1; st->step_ok = 0;
    }
    return lm_next_step(st, max_iterations);
}
