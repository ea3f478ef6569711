// solve.cuh -- the per-match accumulation of the normal equations and the one-thread solvers that turn a summed row into a
// pose increment.  Shared by reduce_kernel (solve.cu) and batch_icp_kernel (batch.cu), each compiled into its own translation unit.
//
// Reference: gather (ICPOptimizer.h:583-610), estimatePosePointToPoint -> ProcrustesAligner
// (ICPOptimizer.h:666-674, ProcrustesAligner.h:6-70), estimatePosePointToPlane (:676-782),
// estimatePoseSymmetricICP (:784-898).
#pragma once
#include "icp_internal.cuh"

// One-sided Jacobi SVD of a 3x3 (row-major), singular values descending, A = U diag(S) V^T.
static __device__ void svd3_dev(const double* A, double* U, double* S, double* V) {
    double W[9];
    for (int i = 0; i < 9; ++i) { W[i] = A[i]; V[i] = (i % 4 == 0) ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < 2; ++p) for (int q = p + 1; q < 3; ++q) {
            double a = 0, b = 0, c = 0;
            for (int k = 0; k < 3; ++k) { a += W[k * 3 + p] * W[k * 3 + p]; b += W[k * 3 + q] * W[k * 3 + q]; c += W[k * 3 + p] * W[k * 3 + q]; }
            if (fabs(c) <= 1e-300 || fabs(c) <= 1e-17 * sqrt(a * b)) continue;
            off += fabs(c);
            const double zeta = (b - a) / (2.0 * c);
            const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
            const double cs = 1.0 / sqrt(1.0 + t * t), sn = cs * t;
            for (int k = 0; k < 3; ++k) {
                const double wp = W[k * 3 + p], wq = W[k * 3 + q];
                W[k * 3 + p] = cs * wp - sn * wq; W[k * 3 + q] = sn * wp + cs * wq;
                const double vp = V[k * 3 + p], vq = V[k * 3 + q];
                V[k * 3 + p] = cs * vp - sn * vq; V[k * 3 + q] = sn * vp + cs * vq;
            }
        }
        if (off == 0.0) break;
    }
    for (int j = 0; j < 3; ++j) S[j] = sqrt(W[j] * W[j] + W[3 + j] * W[3 + j] + W[6 + j] * W[6 + j]);
    int ord[3] = {0, 1, 2};
    for (int i = 0; i < 2; ++i) for (int j = i + 1; j < 3; ++j) if (S[ord[j]] > S[ord[i]]) { const int t = ord[i]; ord[i] = ord[j]; ord[j] = t; }
    double Ws[9], Vs[9], Ss[3];
    for (int j = 0; j < 3; ++j) { Ss[j] = S[ord[j]]; for (int k = 0; k < 3; ++k) { Ws[k * 3 + j] = W[k * 3 + ord[j]]; Vs[k * 3 + j] = V[k * 3 + ord[j]]; } }
    for (int j = 0; j < 3; ++j) S[j] = Ss[j];
    for (int i = 0; i < 9; ++i) V[i] = Vs[i];
    const double tiny = 1e-14 * (S[0] > 0 ? S[0] : 1.0);
    for (int j = 0; j < 3; ++j)
        for (int k = 0; k < 3; ++k) U[k * 3 + j] = S[j] > tiny ? Ws[k * 3 + j] / S[j] : 0.0;
    if (!(S[0] > tiny)) { for (int i = 0; i < 9; ++i) U[i] = (i % 4 == 0) ? 1.0 : 0.0; return; }
    if (!(S[1] > tiny)) {   // complete a rank-1 U
        const double u0[3] = {U[0], U[3], U[6]};
        const int m = fabs(u0[0]) < fabs(u0[1]) ? (fabs(u0[0]) < fabs(u0[2]) ? 0 : 2) : (fabs(u0[1]) < fabs(u0[2]) ? 1 : 2);
        double e[3] = {0, 0, 0}; e[m] = 1.0;
        const double u1[3] = {u0[1] * e[2] - u0[2] * e[1], u0[2] * e[0] - u0[0] * e[2], u0[0] * e[1] - u0[1] * e[0]};
        const double n1 = sqrt(u1[0] * u1[0] + u1[1] * u1[1] + u1[2] * u1[2]);
        for (int k = 0; k < 3; ++k) U[k * 3 + 1] = u1[k] / n1;
    }
    if (!(S[2] > tiny)) {
        const double u0[3] = {U[0], U[3], U[6]}, u1[3] = {U[1], U[4], U[7]};
        U[2] = u0[1] * u1[2] - u0[2] * u1[1]; U[5] = u0[2] * u1[0] - u0[0] * u1[2]; U[8] = u0[0] * u1[1] - u0[1] * u1[0];
    }
}

// ---------------------------------------------------------------------------- finishers: summed row -> increment
// Row layouts.  PLANE / SYMMETRIC: [0..20] A^T A upper triangle row-major, [21..26] A^T b, [27] count.
//               P2P: [0] count, [1..3] sum s, [4..6] sum d, [7] sum w, [8..10] sum w s, [11..13] sum w d, [14..22] sum w d s^T.
//               SUMS: [0] count, [1..3] sum s, [4..6] sum d.
// 6x6 Cholesky solve of the normal equations (symmetric positive definite by construction), every loop fully
// unrolled so that the factor lives in registers -- one thread runs this on the critical path of every iteration,
// and a local-memory (dynamically indexed) elimination costs ~10 us there.  A non-positive pivot (degenerate
// geometry) falls back to Gaussian elimination with partial pivoting, the solver the oracle uses.
static __device__ __forceinline__ bool chol6_solve(const double* row, double lambda2, double* x) {
    double L[6][6];
    int k = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = i; j < 6; ++j) { L[j][i] = row[k]; ++k; }        // lower triangle
#pragma unroll
    for (int i = 0; i < 6; ++i) L[i][i] += lambda2;
    bool ok = true;
    double Linv[6];          // 1 / L[j][j]: one rsqrt per column instead of a sqrt and 3 divisions (this is the serial tail
                             // of every iteration: one thread, every dependent fp64 division costs ~100 cycles)
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        double d = L[j][j];
#pragma unroll
        for (int m = 0; m < j; ++m) d -= L[j][m] * L[j][m];
        if (!(d > 0.0)) ok = false;
        const double inv = rsqrt(d);
        Linv[j] = inv;
        L[j][j] = d * inv;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            double v = L[i][j];
#pragma unroll
            for (int m = 0; m < j; ++m) v -= L[i][m] * L[j][m];
            L[i][j] = v * inv;
        }
    }
    double y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double v = row[21 + i];
#pragma unroll
        for (int m = 0; m < i; ++m) v -= L[i][m] * y[m];
        y[i] = v * Linv[i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        double v = y[i];
#pragma unroll
        for (int m = i + 1; m < 6; ++m) v -= L[m][i] * x[m];
        x[i] = v * Linv[i];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) if (!isfinite(x[i])) ok = false;
    return ok;
}

static __device__ __noinline__ int expand_and_solve_pivoted(const double* row, double lambda2, double* x) {
    double A[36], b[6];
    int k = 0;
    for (int i = 0; i < 6; ++i) for (int j = i; j < 6; ++j) { A[i * 6 + j] = row[k]; A[j * 6 + i] = row[k]; ++k; }
    for (int i = 0; i < 6; ++i) { A[i * 6 + i] += lambda2; b[i] = row[21 + i]; }
    return solve6_dev(A, b, x);
}

static __device__ int expand_and_solve(const double* row, double lambda2, double* x) {
    if (chol6_solve(row, lambda2, x)) return 0;
    return expand_and_solve_pivoted(row, lambda2, x);
}

static __device__ int finish_p2plane(const double* row, float* inc) {
    mat4_identity_dev(inc);
    if (!(row[27] > 0.0)) return ICP_GPU_E_NO_MATCHES;
    double x[6];
    if (expand_and_solve(row, 0.0, x) != 0) return ICP_GPU_E_NUMERIC;
    // ICPOptimizer.h:768-779: R = Rx(alpha) * Ry(beta) * Rz(gamma) in fp32, t = x[3..5]
    const float al = (float)x[0], be = (float)x[1], ga = (float)x[2];
    double sd, cd;
    sincos((double)al, &sd, &cd); const float ca = (float)cd, sa = (float)sd;
    sincos((double)be, &sd, &cd); const float cb = (float)cd, sb = (float)sd;
    sincos((double)ga, &sd, &cd); const float cg = (float)cd, sg = (float)sd;
    float Rx[16], Ry[16], Rz[16], T[16];
    mat4_identity_dev(Rx); mat4_identity_dev(Ry); mat4_identity_dev(Rz);
    Rx[5] = ca; Rx[9] = -sa; Rx[6] = sa; Rx[10] = ca;
    Ry[0] = cb; Ry[8] = sb; Ry[2] = -sb; Ry[10] = cb;
    Rz[0] = cg; Rz[4] = -sg; Rz[1] = sg; Rz[5] = cg;
    mat4_mul_pinned(Rx, Ry, T); mat4_mul_pinned(T, Rz, inc);
    inc[12] = (float)x[3]; inc[13] = (float)x[4]; inc[14] = (float)x[5];
    return 0;
}

static __device__ int finish_symmetric(const double* row, const float* meanS, const float* meanT, float* inc) {
    mat4_identity_dev(inc);
    if (!(row[27] > 0.0)) return ICP_GPU_E_NO_MATCHES;
    const float lambda = 0.0001f;                                   // ICPOptimizer.h:858-864
    double x[6];
    if (expand_and_solve(row, (double)pmul(lambda, lambda), x) != 0) return ICP_GPU_E_NUMERIC;
    // ICPOptimizer.h:876-895
    const float at0 = (float)x[0], at1 = (float)x[1], at2 = (float)x[2];
    const float tt[3] = {(float)x[3], (float)x[4], (float)x[5]};
    const float tan_theta = __fsqrt_rn(padd(padd(pmul(at0, at0), pmul(at1, at1)), pmul(at2, at2)));
    float R4[16]; mat4_identity_dev(R4);
    float cos_theta = 1.0f;
    if (tan_theta > 0.f) {       // the reference divides 0/0 here; guarded (documented deviation)
        const float a[3] = {pdiv(at0, tan_theta), pdiv(at1, tan_theta), pdiv(at2, tan_theta)};
        const float sin_theta = (float)((double)tan_theta / sqrt(1.0 + (double)pmul(tan_theta, tan_theta)));
        cos_theta = pdiv(sin_theta, tan_theta);
        const float K[9] = {0.f, -a[2], a[1], a[2], 0.f, -a[0], -a[1], a[0], 0.f};   // row-major [a]x
        const float omc = psub(1.0f, cos_theta);
        float K1[9], KK[9];
        for (int i = 0; i < 9; ++i) K1[i] = pmul(omc, K[i]);
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c)
            KK[r * 3 + c] = padd(padd(pmul(K1[r * 3], K[c]), pmul(K1[r * 3 + 1], K[3 + c])), pmul(K1[r * 3 + 2], K[6 + c]));
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c)
            R4[r + 4 * c] = padd((r == c) ? 1.0f : 0.0f, padd(pmul(sin_theta, K[r * 3 + c]), KK[r * 3 + c]));   // getRodriguesMatrix, utils.h:171-176
    }
    float Td[16], Tt[16], Ts[16], M1[16], M2[16], M3[16];
    mat4_identity_dev(Td); mat4_identity_dev(Tt); mat4_identity_dev(Ts);
    for (int k = 0; k < 3; ++k) { Td[12 + k] = meanT[k]; Tt[12 + k] = pmul(tt[k], cos_theta); Ts[12 + k] = -meanS[k]; }
    mat4_mul_pinned(Td, R4, M1); mat4_mul_pinned(M1, Tt, M2); mat4_mul_pinned(M2, R4, M3); mat4_mul_pinned(M3, Ts, inc);
    return 0;
}

static __device__ int finish_p2p(const double* row, float* inc) {
    mat4_identity_dev(inc);
    const double M = row[0];
    if (!(M > 0.0)) return ICP_GPU_E_NO_MATCHES;
    double sm[3], dm[3];
    for (int k = 0; k < 3; ++k) { sm[k] = row[1 + k] / M; dm[k] = row[4 + k] / M; }
    // ProcrustesAligner.h:50-54 with unweighted means: sum w (d - dm)(s - sm)^T expanded in raw moments
    double A[9];
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c)
        A[r * 3 + c] = row[14 + r * 3 + c] - dm[r] * row[8 + c] - row[11 + r] * sm[c] + row[7] * dm[r] * sm[c];
    double U[9], S[3], V[9];
    svd3_dev(A, U, S, V);
    double UVt[9];
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) UVt[r * 3 + c] = U[r * 3] * V[c * 3] + U[r * 3 + 1] * V[c * 3 + 1] + U[r * 3 + 2] * V[c * 3 + 2];
    const double dd = UVt[0] * (UVt[4] * UVt[8] - UVt[5] * UVt[7]) - UVt[1] * (UVt[3] * UVt[8] - UVt[5] * UVt[6]) + UVt[2] * (UVt[3] * UVt[7] - UVt[4] * UVt[6]);
    double R[9];
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) R[r * 3 + c] = U[r * 3] * V[c * 3] + U[r * 3 + 1] * V[c * 3 + 1] + dd * U[r * 3 + 2] * V[c * 3 + 2];
    for (int r = 0; r < 3; ++r) {
        double rt = 0, rd = 0;
        for (int c = 0; c < 3; ++c) { rt += R[r * 3 + c] * (dm[c] - sm[c]); rd += R[r * 3 + c] * dm[c]; }
        inc[r + 12] = (float)(rt - rd + dm[r]);                       // ProcrustesAligner.h:26
        for (int c = 0; c < 3; ++c) inc[r + 4 * c] = (float)R[r * 3 + c];
    }
    for (int i = 0; i < 16; ++i) if (!isfinite(inc[i])) return ICP_GPU_E_NUMERIC;
    return 0;
}

// One match's contribution to the rows above: MODE 0 point-to-point moments, 1 point-to-plane, 2 symmetric (source and target
// centred on the matched means mS / mD; the source normal sn4 goes through Nm, the current pose's inverse-transpose), 3 the
// sums the symmetric means come from.  (sxf, syf, szf): transformed source point, tp / tn: matched target point / normal,
// w: the match weight.  reduce_kernel and batch_icp_kernel (batch.cu) both accumulate through this.
template <int MODE>
__device__ __forceinline__ void accumulate_match(double (&v)[32], float sxf, float syf, float szf, const float4 tp, const float4 tn,
                                                 const float4 sn4, const float* Nm, const float* mS, const float* mD, const double w) {
    const double LP = (double)0.1f, LQ = (double)1.0f;   // LAMBDA_POINT / LAMBDA_PLANE|SYMMETRIC (ICPOptimizer.h:737-738, :840-841)
    if (MODE == 3) {
        v[0] += 1.0; v[1] += sxf; v[2] += syf; v[3] += szf; v[4] += tp.x; v[5] += tp.y; v[6] += tp.z;
    } else if (MODE == 0) {
        const double s[3] = {sxf, syf, szf}, t[3] = {tp.x, tp.y, tp.z};
        v[0] += 1.0; v[7] += w;
#pragma unroll
        for (int k = 0; k < 3; ++k) { v[1 + k] += s[k]; v[4 + k] += t[k]; v[8 + k] += w * s[k]; v[11 + k] += w * t[k]; }
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c) v[14 + r * 3 + c] += w * t[r] * s[c];
    } else {
        double s[3] = {sxf, syf, szf}, t[3] = {tp.x, tp.y, tp.z};
        double n[3] = {tn.x, tn.y, tn.z};
        bool use_row = finite3(tn.x, tn.y, tn.z);
        double u[3] = {s[0], s[1], s[2]};
        if (MODE == 2) {
            // the source normal is transformed by the current pose's inverse-transpose (ICPOptimizer.h:554)
            float nx, ny, nz;
            xform_normal(Nm, sn4.x, sn4.y, sn4.z, nx, ny, nz);
            use_row = use_row && finite3(nx, ny, nz);
#pragma unroll
            for (int k = 0; k < 3; ++k) { s[k] -= (double)mS[k]; t[k] -= (double)mD[k]; }   // :797-806
            n[0] += (double)nx; n[1] += (double)ny; n[2] += (double)nz;                      // n_t + n_s
#pragma unroll
            for (int k = 0; k < 3; ++k) u[k] = s[k] + t[k];
        }
        const double e[3] = {t[0] - s[0], t[1] - s[1], t[2] - s[2]};
        const double b2 = (LP * w) * (LP * w);
        // three point rows [-[s]x | I], rhs e  (:716-733 / :817-835):  P^T P = [[|s|^2 I - s s^T, [s]x], [-[s]x, I]]
        const double ss = s[0] * s[0] + s[1] * s[1] + s[2] * s[2];
        double c[6] = {0, 0, 0, 0, 0, 0}; double r = 0.0, a2 = 0.0;
        if (use_row) {
            // plane row [u x n | n], rhs n.e  (:698-710 ; symmetric :809-815 with u = s~ + d~, n = n_t + n_s)
            c[0] = u[1] * n[2] - u[2] * n[1]; c[1] = u[2] * n[0] - u[0] * n[2]; c[2] = u[0] * n[1] - u[1] * n[0];
            c[3] = n[0]; c[4] = n[1]; c[5] = n[2];
            r = n[0] * e[0] + n[1] * e[1] + n[2] * e[2];
            a2 = (LQ * w) * (LQ * w);
        }
        // upper triangle, row-major
        v[0] += a2 * c[0] * c[0] + b2 * (ss - s[0] * s[0]);
        v[1] += a2 * c[0] * c[1] - b2 * s[0] * s[1];
        v[2] += a2 * c[0] * c[2] - b2 * s[0] * s[2];
        v[3] += a2 * c[0] * c[3];
        v[4] += a2 * c[0] * c[4] - b2 * s[2];
        v[5] += a2 * c[0] * c[5] + b2 * s[1];
        v[6] += a2 * c[1] * c[1] + b2 * (ss - s[1] * s[1]);
        v[7] += a2 * c[1] * c[2] - b2 * s[1] * s[2];
        v[8] += a2 * c[1] * c[3] + b2 * s[2];
        v[9] += a2 * c[1] * c[4];
        v[10] += a2 * c[1] * c[5] - b2 * s[0];
        v[11] += a2 * c[2] * c[2] + b2 * (ss - s[2] * s[2]);
        v[12] += a2 * c[2] * c[3] - b2 * s[1];
        v[13] += a2 * c[2] * c[4] + b2 * s[0];
        v[14] += a2 * c[2] * c[5];
        v[15] += a2 * c[3] * c[3] + b2;
        v[16] += a2 * c[3] * c[4];
        v[17] += a2 * c[3] * c[5];
        v[18] += a2 * c[4] * c[4] + b2;
        v[19] += a2 * c[4] * c[5];
        v[20] += a2 * c[5] * c[5] + b2;
        // rhs: a^2 r c + b^2 [s x d ; e]   (s x e == s x d)
        v[21] += a2 * r * c[0] + b2 * (s[1] * e[2] - s[2] * e[1]);
        v[22] += a2 * r * c[1] + b2 * (s[2] * e[0] - s[0] * e[2]);
        v[23] += a2 * r * c[2] + b2 * (s[0] * e[1] - s[1] * e[0]);
        v[24] += a2 * r * c[3] + b2 * e[0];
        v[25] += a2 * r * c[4] + b2 * e[1];
        v[26] += a2 * r * c[5] + b2 * e[2];
        v[27] += 1.0;
    }
}
