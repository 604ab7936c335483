// so_internal.cuh -- shared device structs + FP64 device math for the sm_100a ICP kernels.
// Not part of the public ABI (include/superodom_b200.h is).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <float.h>

#include "../../include/superodom_b200.h"

namespace so {

// LocalMap.h:131-138
constexpr int kW = 21, kH = 21, kD = 11, kNumBlocks = kW * kH * kD;
constexpr double kBlock = 50.0, kHalfBlock = 25.0;
constexpr int kAcc = 28;            // 21 (upper triangle of H) + 6 (g) + 1 (cost)
constexpr int kThreads = 256;       // threads per CTA for the per-point kernels

// ICP / LM phases (device-side state machine, see so_icp.cu)
enum { PH_CORR = 0, PH_EVAL = 1, PH_DONE = 2 };

// Read-only view of the map index, passed by value to kernels.
struct MapView {
    const float4* pts;          // sorted by (block slot, cell); w = bitcast(uint32 point id)
    const int32_t* block_slot;  // [4851] slot of a grid block, -1 if it holds no surf points
    const int32_t* block_count; // [4851] points per grid block
    const uint32_t* cell_start; // [n_slots * nb^3 + 1] first sorted point of every cell (x fastest)
    int32_t origin[3];          // LocalMap::origin_
    int32_t nb;                 // cells per block axis
    double inv_cs;              // nb / 50  (cells per metre)
    float cs;                   // cell edge (m)
    float bound_d2;             // float(3 * planeRes_)  -- the NEIGHBORS_TOO_FAR gate doubles as search radius^2
    double inv_bound_d2;        // 1 / double(bound_d2)
    float plane_res;
    int32_t R;                  // search rings: R * cs >= sqrt(bound_d2)
};

// Per-scan device state: the Ceres trust-region minimiser + the outer ICP loop, advanced by the last CTA of every
// per-point kernel (no host round trip inside a scan).
struct IcpState {
    // --- inputs
    double x0[7];          // T_w_initial_guess
    int32_t n_points;      // points the ICP kernels run over (after scan preparation: those shouldProcessPoint keeps)
    int32_t n_input;       // points of the scan as uploaded
    int32_t n_edge;        // edge points of this scan (0: edge branch idle, as upstream)
    int32_t max_icp_iters, lm_max_iterations;
    double sampling_rate;  // calculateSamplingRate(): <0 = keep all
    int32_t use_prior;     // addAbsolutePoseConstraints rows active (LidarSlam.cpp:281-298)
    float prior_vcf, prior_unc[3];   // Visual_confidence_factor, lidarOdomUncer.uncertainty_{x,y,z}
    double prior_sqrt_info[6];       // set when a solve begins (depends on the number of accepted correspondences)
    // --- minimiser state (one ceres::Solve)
    double x[7];           // last accepted iterate (parameters_)
    double cand[7];        // candidate being evaluated
    double H[21], g[6], cost;      // at x
    double scale[6];       // Jacobi scaling, fixed at iteration 0 of the solve
    double diag[6];        // LM diagonal (on the scaled system), reused after rejected steps
    double radius, decrease_factor, x_norm, gmax, model_cost_change;
    int32_t phase, icp_iter, lm_iter, num_successful, num_unsuccessful, reuse_diagonal, consecutive_invalid, termination;
    // --- per-ICP-iteration bookkeeping
    double x_iter_start[7];
    int32_t n_ok;          // accepted correspondences, edges + planes (features_corres.size())
    int32_t n_ok_edge;
    // --- outputs
    int32_t status, n_iterations;
    int32_t iter_n_surf[SO_MAX_ICP_ITERS], iter_n_edge[SO_MAX_ICP_ITERS];
    double iter_dtrans[SO_MAX_ICP_ITERS], iter_drot[SO_MAX_ICP_ITERS], iter_cost[SO_MAX_ICP_ITERS];
    int32_t iter_lm_steps[SO_MAX_ICP_ITERS], iter_lm_successful[SO_MAX_ICP_ITERS], iter_lm_termination[SO_MAX_ICP_ITERS];
    int32_t hist_obs[9], hist_rej[7], hist_rej_line[7];
    int32_t knn_searched, knn_verified;      // over the whole registration: queries that ran the grid walk / whose stored neighbours were proven still exact
    int32_t need_cov;                        // set by the serial step that ends the registration: the CTA's first warp then runs the covariance
    double cov[36];
    double pos_err, pos_dir[3], pos_inv_cond, ori_err_deg, ori_dir[3], ori_inv_cond;
};

// ------------------------------------------------------------------------------------------------ quaternion / pose
// pose7 = tx,ty,tz,qx,qy,qz,qw (LidarSlam.cpp:7-9)
__host__ __device__ inline void qmul(const double a[4], const double b[4], double o[4]) {   // xyzw, Hamilton
    o[0] = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1];
    o[1] = a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2];
    o[2] = a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0];
    o[3] = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
}
// v + 2w (q x v) + 2 q x (q x v)   (what Eigen's quaternion * vector evaluates; Twist.h:187)
__host__ __device__ inline void qrot(const double q[4], const double v[3], double o[3]) {
    double ux = q[1] * v[2] - q[2] * v[1], uy = q[2] * v[0] - q[0] * v[2], uz = q[0] * v[1] - q[1] * v[0];
    ux += ux; uy += uy; uz += uz;
    o[0] = v[0] + q[3] * ux + (q[1] * uz - q[2] * uy);
    o[1] = v[1] + q[3] * uy + (q[2] * ux - q[0] * uz);
    o[2] = v[2] + q[3] * uz + (q[0] * uy - q[1] * ux);
}
__host__ __device__ inline void qtoR(const double q[4], double R[9]) {
    const double tx = 2 * q[0], ty = 2 * q[1], tz = 2 * q[2];
    const double twx = tx * q[3], twy = ty * q[3], twz = tz * q[3];
    const double txx = tx * q[0], txy = ty * q[0], txz = tz * q[0], tyy = ty * q[1], tyz = tz * q[1], tzz = tz * q[2];
    R[0] = 1 - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
    R[3] = txy + twz; R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1 - (txx + tyy);
}
// PoseLocalParameterization::Plus (pose_local_parameterization.cpp:7-22): p += dp; q <- (q * [1, dth/2]).normalized()
__host__ __device__ inline void pose_plus(const double x[7], const double d[6], double o[7]) {
    o[0] = x[0] + d[0]; o[1] = x[1] + d[1]; o[2] = x[2] + d[2];
    const double dq[4] = {d[3] / 2.0, d[4] / 2.0, d[5] / 2.0, 1.0};
    double r[4]; qmul(x + 3, dq, r);
    const double n2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2] + r[3] * r[3];
    const double s = n2 > 0 ? 1.0 / sqrt(n2) : 1.0;
    o[3] = r[0] * s; o[4] = r[1] * s; o[5] = r[2] * s; o[6] = r[3] * s;
}
// |t| and angle of a^-1 * b  (recordIterationStats, LidarSlam.cpp:242-251)
__host__ __device__ inline void rel_motion(const double a[7], const double b[7], double* trans, double* rot) {
    const double qi[4] = {-a[3], -a[4], -a[5], a[6]};
    const double dt[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
    double t[3], r[4];
    qrot(qi, dt, t); qmul(qi, b + 3, r);
    *trans = sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
    *rot = 2.0 * atan2(sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]), r[3]);
}

// ------------------------------------------------------------------------------------------------ small dense algebra
// Cyclic Jacobi for a symmetric NxN (row-major full storage).  On return a's diagonal holds the eigenvalues and
// v (row-major) the eigenvectors in columns; then sorted ascending.  With N a compile-time constant and full
// unrolling every index is static, so for N=3 the whole thing lives in registers.
// WITH_V = false: eigenvalues only (v is not touched and may be null).
// Convergence test of the sweeps: sum of squared off-diagonals <= SO_JACOBI_OFF_TOL * sum of squared diagonals.  1e-33 drives the
// off-diagonals to full double precision (4 sweeps for the 3x3 scatter matrices of k_fit); 1e-30 would usually stop a sweep
// earlier at an eigenvalue error far below an ulp -- left for a measured change.
#ifndef SO_JACOBI_OFF_TOL
#define SO_JACOBI_OFF_TOL 1e-33
#endif
// The 2x2 block [app apq; apq aqq] after one rotation J = [c s; -s c]: the exact similarity J^T A J of the (c, s) actually used.
// The angle comes from an FP32 tangent, so the classic shortcut app -= t apq, aqq += t apq, apq = 0 -- exact only for the exact
// root t -- would perturb the matrix by ~1e-7 |apq| per rotation (eigenvalue error ~1e-8 cond, direction error up to 5e-8).  With
// the exact update the inexact angle only leaves a ~1e-7 |apq| off-diagonal for the next sweep to remove.  Explicit roundings:
// the serial and warp covariance routines produce the same bits from it.
__device__ __forceinline__ void jacobi_rot2(double app, double aqq, double apq, double c, double s, double& npp, double& nqq, double& npq) {
    const double cc = __dmul_rn(c, c), ss = __dmul_rn(s, s), cs = __dmul_rn(c, s);
    const double x = __dmul_rn(2.0 * cs, apq);
    npp = __fma_rn(ss, aqq, __fma_rn(cc, app, -x));
    nqq = __fma_rn(ss, app, __fma_rn(cc, aqq, x));
    npq = __fma_rn(cs, __dsub_rn(app, aqq), __dmul_rn(__dsub_rn(cc, ss), apq));
}

template <int N, int SWEEPS, bool WITH_V = true>
__device__ inline void jacobi_eig(double* a, double* v, double* w) {
    if (WITH_V) {
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
            for (int j = 0; j < N; ++j) v[i * N + j] = (i == j) ? 1.0 : 0.0;
    }
#pragma unroll 1
    for (int sweep = 0; sweep < SWEEPS; ++sweep) {
        double off = 0.0, dia = 0.0;
#pragma unroll
        for (int p = 0; p < N; ++p) {
            dia += a[p * N + p] * a[p * N + p];
#pragma unroll
            for (int q = p + 1; q < N; ++q) off += a[p * N + q] * a[p * N + q];
        }
        if (off <= SO_JACOBI_OFF_TOL * dia || off == 0.0) break;
#pragma unroll
        for (int p = 0; p < N - 1; ++p) {
#pragma unroll
            for (int q = p + 1; q < N; ++q) {
                const double apq = a[p * N + q];
                if (apq != 0.0) {
                    // tan of the rotation angle, t = sgn(theta) / (|theta| + sqrt(theta^2 + 1)), theta = (aqq - app) / (2 apq),
                    // evaluated in FP32 (one MUFU sqrt + one MUFU rcp instead of an FP64 sqrt and divide).  The rotation
                    // itself stays exactly orthogonal in FP64 because c = rsqrt(1 + t^2), s = t c are formed in FP64 from
                    // whatever t is, and jacobi_rot2 applies exactly that rotation to the 2x2 block, so a 1e-7-accurate t
                    // only leaves a 1e-7-times-smaller apq for the next sweep.
                    const float dlt = float(a[q * N + q] - a[p * N + p]), b2 = float(2.0 * apq);
                    float tf = __fdividef(b2, fabsf(dlt) + sqrtf(fmaf(dlt, dlt, b2 * b2)));
                    if (!(fabsf(tf) <= 1.0f)) tf = 0.0f;             // b2 == 0 after the cast (or inf/nan): no rotation
                    const double t = double(dlt < 0.0f ? -tf : tf);
                    const double c = rsqrt(t * t + 1.0), s = t * c;
                    double npp, nqq, npq;
                    jacobi_rot2(a[p * N + p], a[q * N + q], apq, c, s, npp, nqq, npq);
                    a[p * N + p] = npp; a[q * N + q] = nqq; a[p * N + q] = npq; a[q * N + p] = npq;
#pragma unroll
                    for (int r = 0; r < N; ++r) {
                        if (r != p && r != q) {
                            const double arp = a[r * N + p], arq = a[r * N + q];
                            a[r * N + p] = a[p * N + r] = c * arp - s * arq;
                            a[r * N + q] = a[q * N + r] = s * arp + c * arq;
                        }
                        if (WITH_V) {
                            const double vrp = v[r * N + p], vrq = v[r * N + q];
                            v[r * N + p] = c * vrp - s * vrq;
                            v[r * N + q] = s * vrp + c * vrq;
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) w[i] = a[i * N + i];
    // ascending selection sort (swaps columns of v)
#pragma unroll
    for (int i = 0; i < N - 1; ++i) {
#pragma unroll
        for (int j = i + 1; j < N; ++j) {
            if (w[j] < w[i]) {
                const double t = w[i]; w[i] = w[j]; w[j] = t;
                if (WITH_V) {
#pragma unroll
                    for (int r = 0; r < N; ++r) { const double u = v[r * N + i]; v[r * N + i] = v[r * N + j]; v[r * N + j] = u; }
                }
            }
        }
    }
}

// Cyclic Jacobi for the symmetric 6x6 of the covariance step, rotations taken in ROUND-ROBIN order: five rounds of three pairs
// with disjoint indices -- (0,5)(1,4)(2,3) / (0,4)(3,5)(1,2) / (0,3)(2,4)(1,5) / (0,2)(1,3)(4,5) / (0,1)(2,5)(3,4).  The angle of a
// pair depends only on its own 2x2 block, which the other two rotations of the round do not touch, so the three angle
// computations (the latency-bound part: reciprocal, square roots) are independent instruction streams for the one thread that
// runs them; the row-cyclic order chained all fifteen.  Same convergence test and ascending output as jacobi_eig<6>.
template <int SWEEPS>
__device__ inline void jacobi_eig6_rr(double* a, double* v, double* w) {
    constexpr int N = 6;
    constexpr int PP[15] = {0, 1, 2, 0, 3, 1, 0, 2, 1, 0, 1, 4, 0, 2, 3};
    constexpr int QQ[15] = {5, 4, 3, 4, 5, 2, 3, 4, 5, 2, 3, 5, 1, 5, 4};
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) v[i * N + j] = (i == j) ? 1.0 : 0.0;
#pragma unroll 1
    for (int sweep = 0; sweep < SWEEPS; ++sweep) {
        double off = 0.0, dia = 0.0;
#pragma unroll
        for (int p = 0; p < N; ++p) {
            dia += a[p * N + p] * a[p * N + p];
#pragma unroll
            for (int q = p + 1; q < N; ++q) off += a[p * N + q] * a[p * N + q];
        }
        if (off <= SO_JACOBI_OFF_TOL * dia || off == 0.0) break;
#pragma unroll
        for (int round = 0; round < 5; ++round) {
            double tt[3], cc[3], ss[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {                    // three independent angles
                const int p = PP[round * 3 + k], q = QQ[round * 3 + k];
                const double apq = a[p * N + q];
                const float dlt = float(a[q * N + q] - a[p * N + p]), b2 = float(2.0 * apq);
                float tf = __fdividef(b2, fabsf(dlt) + sqrtf(fmaf(dlt, dlt, b2 * b2)));
                if (!(fabsf(tf) <= 1.0f)) tf = 0.0f;         // apq == 0 after the cast (or inf / nan): no rotation
                const double t = apq != 0.0 ? double(dlt < 0.0f ? -tf : tf) : 0.0;
                const double c = rsqrt(t * t + 1.0);
                tt[k] = t; cc[k] = c; ss[k] = t * c;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int p = PP[round * 3 + k], q = QQ[round * 3 + k];
                const double t = tt[k], c = cc[k], sn = ss[k], apq = a[p * N + q];
                if (t != 0.0) {
                    double npp, nqq, npq;
                    jacobi_rot2(a[p * N + p], a[q * N + q], apq, c, sn, npp, nqq, npq);
                    a[p * N + p] = npp; a[q * N + q] = nqq; a[p * N + q] = npq; a[q * N + p] = npq;
#pragma unroll
                    for (int r = 0; r < N; ++r) {
                        if (r != p && r != q) {
                            const double arp = a[r * N + p], arq = a[r * N + q];
                            a[r * N + p] = a[p * N + r] = c * arp - sn * arq;
                            a[r * N + q] = a[q * N + r] = sn * arp + c * arq;
                        }
                        const double vrp = v[r * N + p], vrq = v[r * N + q];
                        v[r * N + p] = c * vrp - sn * vrq;
                        v[r * N + q] = sn * vrp + c * vrq;
                    }
                }
            }
        }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) w[i] = a[i * N + i];
#pragma unroll
    for (int i = 0; i < N - 1; ++i) {
#pragma unroll
        for (int j = i + 1; j < N; ++j) {
            if (w[j] < w[i]) {
                const double t = w[i]; w[i] = w[j]; w[j] = t;
#pragma unroll
                for (int r = 0; r < N; ++r) { const double u = v[r * N + i]; v[r * N + i] = v[r * N + j]; v[r * N + j] = u; }
            }
        }
    }
}

// Eigenvalues (ascending) of the symmetric 3x3 [a00 a01 a02; . a11 a12; . . a22] by the trigonometric solution of its
// characteristic cubic: with q = tr/3, p^2 = |A - qI|_F^2 / 6 and r = det((A - qI)/p)/2 in [-1, 1], the roots are
// q + 2p cos(phi + 2k pi/3), phi = acos(r)/3 in [0, pi/3] -- one FP64 acos and one sincos instead of the ~12 Jacobi rotations an
// iterative solver needs.  Absolute accuracy ~1e-13 |A| (measured against LAPACK on 800 k five-point scatter matrices); the
// smallest eigenvalue, which a hard gate reads (lambda0 < 1e-6, LidarSlam.cpp:772), is therefore polished by the caller with the
// Rayleigh quotient of its eigenvector (error ~1e-16 |A|, the class of an iterative solver).
__device__ __forceinline__ void sym3_eigenvalues(double a00, double a01, double a02, double a11, double a12, double a22, double ev[3]) {
    const double tr = a00 + a11 + a22, q = tr * (1.0 / 3.0);
    const double b00 = a00 - q, b11 = a11 - q, b22 = a22 - q;
    const double p2 = b00 * b00 + b11 * b11 + b22 * b22 + 2.0 * (a01 * a01 + a02 * a02 + a12 * a12);
    if (!(p2 > 0.0)) { ev[0] = ev[1] = ev[2] = q; return; }          // a multiple of the identity (or NaN, which then propagates)
    const double ip = rsqrt(p2 * (1.0 / 6.0)), p = p2 * (1.0 / 6.0) * ip;
    const double detb = b00 * (b11 * b22 - a12 * a12) - a01 * (a01 * b22 - a12 * a02) + a02 * (a01 * a12 - b11 * a02);
    double r = 0.5 * detb * ip * ip * ip;
    r = fmin(fmax(r, -1.0), 1.0);
    double sn, cs;
    sincos(acos(r) * (1.0 / 3.0), &sn, &cs);
    ev[2] = q + 2.0 * p * cs;
    ev[0] = q - p * (cs + 1.7320508075688772 * sn);                   // q + 2p cos(phi + 2pi/3)
    ev[1] = tr - ev[0] - ev[2];
}

// Unit eigenvector of the symmetric 3x3 S = [xx xy xz; xy yy yz; xz yz zz] for its (simple) eigenvalue lam: S - lam I has rank
// two, so the cross product of any two independent rows spans its null space; the pair with the longest product is the
// best conditioned.  Direction error ~ eps * |S| / gap, the same as an iterative solver's; the sign is arbitrary (the caller
// orients it).
__device__ __forceinline__ void eigvec3_from_value(double xx, double xy, double xz, double yy, double yz, double zz, double lam, double n[3]) {
    const double a = xx - lam, d = yy - lam, f = zz - lam, b = xy, c = xz, e = yz;
    const double c01[3] = {b * e - c * d, c * b - a * e, a * d - b * b};
    const double c02[3] = {b * f - c * e, c * c - a * f, a * e - b * c};
    const double c12[3] = {d * f - e * e, e * c - b * f, b * e - d * c};
    const double n01 = c01[0] * c01[0] + c01[1] * c01[1] + c01[2] * c01[2];
    const double n02 = c02[0] * c02[0] + c02[1] * c02[1] + c02[2] * c02[2];
    const double n12 = c12[0] * c12[0] + c12[1] * c12[1] + c12[2] * c12[2];
    double m = n01;
    n[0] = c01[0]; n[1] = c01[1]; n[2] = c01[2];
    if (n02 > m) { m = n02; n[0] = c02[0]; n[1] = c02[1]; n[2] = c02[2]; }
    if (n12 > m) { m = n12; n[0] = c12[0]; n[1] = c12[1]; n[2] = c12[2]; }
    const double inv = 1.0 / sqrt(m);
    n[0] *= inv; n[1] *= inv; n[2] *= inv;
}

// Least-squares solve of the 5x3 system A n = b by column-pivoted Householder QR -- the operation
// `matA0.colPivHouseholderQr().solve(matB0)` of computePlaneQualityMetrics (LidarSlam.cpp:798-806), including
// Eigen's rank rule (|R_ii| > maxpivot * eps * 3).  A is [5][3] (destroyed), b [5] (destroyed).
__host__ __device__ inline void colpiv_qr_solve_5x3(double A[5][3], double b[5], double x[3]) {
    const double eps = 2.220446049250313e-16;
    int perm0 = 0, perm1 = 1, perm2 = 2;
    double rdiag[3], rinv[3] = {0.0, 0.0, 0.0};      // rinv[k] = 1 / R_kk
    double maxpivot = 0.0;
    int nonzero = 3;
    double n0 = 0, n1 = 0, n2 = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i) { n0 += A[i][0] * A[i][0]; n1 += A[i][1] * A[i][1]; n2 += A[i][2] * A[i][2]; }
    const double th = fmax(n0, fmax(n1, n2)) * eps * eps / 5.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int piv = k; double best = -1.0;
#pragma unroll
        for (int j = k; j < 3; ++j) {
            double s = 0;
#pragma unroll
            for (int i = k; i < 5; ++i) s += A[i][j] * A[i][j];
            if (s > best) { best = s; piv = j; }
        }
        if (nonzero == 3 && best < th * double(5 - k)) nonzero = k;
#pragma unroll
        for (int j = k + 1; j < 3; ++j) {
            if (piv == j) {
#pragma unroll
                for (int i = 0; i < 5; ++i) { const double t = A[i][k]; A[i][k] = A[i][j]; A[i][j] = t; }
                // swap perm[k], perm[j]
                int pk = (k == 0 ? perm0 : (k == 1 ? perm1 : perm2));
                int pj = (j == 1 ? perm1 : perm2);
                if (k == 0) perm0 = pj; else if (k == 1) perm1 = pj; else perm2 = pj;
                if (j == 1) perm1 = pk; else perm2 = pk;
            }
        }
        const double c0 = A[k][k];
        double tail2 = 0;
#pragma unroll
        for (int i = k + 1; i < 5; ++i) tail2 += A[i][k] * A[i][k];
        double beta, tau;
        double ess[5];
        if (tail2 <= DBL_MIN) {
            tau = 0.0; beta = c0;
            rinv[k] = 1.0 / c0;
#pragma unroll
            for (int i = 0; i < 5; ++i) ess[i] = 0.0;
        } else {
            // beta = -sign(c0) |col|, 1/beta from one reciprocal square root: the divisions Eigen writes ((beta - c0) / beta,
            // s / R_kk in the back-substitution) become multiplications by it -- same values to an ulp, a third of the
            // instructions (FP64 divide and square root are ~25-instruction software sequences on the GPU)
            const double nrm2 = c0 * c0 + tail2;
#ifdef __CUDA_ARCH__
            double rb = rsqrt(nrm2);
#else
            double rb = 1.0 / sqrt(nrm2);
#endif
            beta = nrm2 * rb;
            if (c0 >= 0.0) { beta = -beta; rb = -rb; }
            rinv[k] = rb;
            const double inv = 1.0 / (c0 - beta);
#pragma unroll
            for (int i = 0; i < 5; ++i) ess[i] = (i > k) ? A[i][k] * inv : 0.0;
            tau = (beta - c0) * rb;
        }
#pragma unroll
        for (int j = k + 1; j < 3; ++j) {
            double s = A[k][j];
#pragma unroll
            for (int i = k + 1; i < 5; ++i) s += ess[i] * A[i][j];
            s *= tau;
            A[k][j] -= s;
#pragma unroll
            for (int i = k + 1; i < 5; ++i) A[i][j] -= s * ess[i];
        }
        {
            double s = b[k];
#pragma unroll
            for (int i = k + 1; i < 5; ++i) s += ess[i] * b[i];
            s *= tau;
            b[k] -= s;
#pragma unroll
            for (int i = k + 1; i < 5; ++i) b[i] -= s * ess[i];
        }
        A[k][k] = beta;
        rdiag[k] = beta;
        maxpivot = fmax(maxpivot, fabs(beta));
    }
    const double premult = maxpivot * eps * 3.0;
    int rank = 0;
#pragma unroll
    for (int i = 0; i < 3; ++i) if (i < nonzero && fabs(rdiag[i]) > premult) rank++;
    double y[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int i = 2; i >= 0; --i) {
        if (i < rank) {
            double s = b[i];
#pragma unroll
            for (int j = i + 1; j < 3; ++j) if (j < rank) s -= A[i][j] * y[j];
            y[i] = s * rinv[i];
        }
    }
    x[0] = x[1] = x[2] = 0.0;
    const int perm[3] = {perm0, perm1, perm2};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double yi = (i < rank) ? y[i] : 0.0;
        if (perm[i] == 0) x[0] = yi; else if (perm[i] == 1) x[1] = yi; else x[2] = yi;
    }
}

// Solve the SPD 6x6 system M y = r by Cholesky (M full row-major, destroyed).  Returns false on a non-positive pivot.
// Fully unrolled: every index is a compile-time constant, so on the device the 36 + 18 values live in registers instead of a
// dynamically indexed local-memory array (the optimiser step is ONE thread's dependent FP64 chain; local-memory round trips
// were most of its 10-20 us).
__host__ __device__ inline bool chol6_solve(double* M, const double* r, double* y) {
    bool ok = true;
    double inv[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        double s = M[j * 6 + j];
#pragma unroll
        for (int k = 0; k < j; ++k) s -= M[j * 6 + k] * M[j * 6 + k];
        if (!(s > 0.0)) ok = false;
        // one reciprocal square root per column; every division by the pivot becomes a multiplication (the step this solves is
        // compared with Ceres' QR-based one to ~1e-12 in any case: another algorithm, not another rounding)
#ifdef __CUDA_ARCH__
        const double il = rsqrt(s);
#else
        const double il = 1.0 / sqrt(s);
#endif
        inv[j] = il;
        M[j * 6 + j] = s * il;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            double t = M[i * 6 + j];
#pragma unroll
            for (int k = 0; k < j; ++k) t -= M[i * 6 + k] * M[j * 6 + k];
            M[i * 6 + j] = t * il;
        }
    }
    if (!ok) return false;
    double z[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double t = r[i];
#pragma unroll
        for (int k = 0; k < i; ++k) t -= M[i * 6 + k] * z[k];
        z[i] = t * inv[i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        double t = z[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) t -= M[k * 6 + i] * y[k];
        y[i] = t * inv[i];
    }
    return true;
}

// upper-triangle packing of the 6x6: index of (i,j), i<=j
__host__ __device__ inline int tri(int i, int j) { return i * 6 - (i * (i - 1)) / 2 + (j - i); }

}  // namespace so
