// so_icp.cu -- sm_100a kernels of the per-scan ICP registration path.
//
//   k_scan_keys / k_scan_gather : order the scan by map cell once per registration (warp-coherent cell walks).
//   k_knn_scan   : per scan point -- pose transform, block lookup, radius-bounded 5-NN in the sorted hash grid
//                  (three-round select: bound, gather, refine); hands the five neighbours to k_fit.         [a5-a7]
//   k_fit        : 3x3 PCA + 5x3 column-pivoted QR plane fit with the reference's accept/reject gates, observability
//                  labels + histograms, fit weight; writes the correspondence record.                     [a8-a11]
//   k_knn_fit    : optional fusion of the two (SO_FUSE_KNN_FIT; measured slower, see so_icp.cuh).
//   k_evaluate   : per correspondence -- residual, 1x6 Jacobian, Tukey/Scaled robust weight at the matched pose (first
//                  evaluation of a solve) or at the LM candidate, warp/CTA-reduced in FP64 (21+6+1 accumulators). [a12-a13]
//   k_edge_fit / k_edge_evaluate : the edge / line branch (10-NN in the edge map, best-line selection, line factor).   [a19]
//   k_lm_step    : fixed-order cross-CTA reduction, then ONE thread per scan advances the device-resident state
//                  machine: Ceres' trust-region LM (step solve by 6x6 Cholesky, accept/reject, tolerances), the SE3 prior
//                  rows, the outer ICP convergence rule, and at the end the covariance pseudo-inverse + 3x3 eigen
//                  analysis.                                                                        [a3, a14-a16, a20]
//   k_loop_cond  : CUDA-graph WHILE condition of a chunk (any scan still iterating).
//   k_knn        : stand-alone k-NN (so_knn*), radius-bounded or exact with ring expansion.
//
// Reference citations are relative to /root/reference/super_odometry/.
#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>

#include "so_icp.cuh"
#include "so_knn.cuh"

namespace so {

// ------------------------------------------------------------------------------------------------------------------
// CTA reduction of kAcc doubles per thread into partials[scan][cta][kAcc].  Fixed thread->point mapping and fixed
// reduction trees => run-to-run deterministic sums.  The cross-CTA sum and the optimiser step run in k_lm_step
// (keeping that scalar FP64 code out of the per-point kernels saves ~70 registers per thread in them).
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void reduce_to_partials(double acc[kAcc], const BatchView& bv, int s, uint32_t slot_offset = 0) {
    static_assert(kAcc <= 32, "one component per lane");
    __shared__ double s_red[kThreads / 32][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // Warp stage: a halving butterfly.  At distance o each lane keeps the half of its (padded to 32) components that matches
    // its lane bit, hands the other half to its partner and adds what it receives, so lane l ends up with the warp total of
    // component l after 16+8+4+2+1 = 31 FP64 shuffles -- the SHFL pipe (one warp-wide shuffle per clock per SM) was the
    // cost of the plain 28 x 5 butterfly.
    double v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = k < kAcc ? acc[k] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int k = 0; k < o; ++k) {
            const double send = up ? v[k] : v[k + o];
            const double keep = up ? v[k + o] : v[k];
            v[k] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    s_red[warp][lane] = v[0];
    __syncthreads();
    if (threadIdx.x < kAcc) {
        double t = 0.0;
#pragma unroll
        for (int wv = 0; wv < kThreads / 32; ++wv) t += s_red[wv][threadIdx.x];
        bv.partials[(size_t(s) * bv.partial_stride + slot_offset + blockIdx.x) * kAcc + threadIdx.x] = t;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Device-resident optimiser state machine (runs on one thread of the last CTA).
// Restates ceres::Solve {max_num_iterations=4, DENSE_QR, defaults} of Ceres 2.0.0 as called at LidarSlam.cpp:230-240:
// TrustRegionMinimizer::Minimize, LevenbergMarquardtStrategy::ComputeStep/StepAccepted/StepRejected and the monotonic
// TrustRegionStepEvaluator, expressed on the robustified normal equations H = sum rho' J^T J, g = sum rho' J^T r
// (the QR of [J;D] that DENSE_QR performs solves exactly (H + D^2) y = g).
// ------------------------------------------------------------------------------------------------------------------
__device__ __noinline__ double grad_max_norm(const double x[7], const double g[6]) {
    // ||x - Plus(x, -g)||_inf  (TrustRegionMinimizer::EvaluateGradientAndJacobian)
    double neg[6], xp[7];
    _Pragma("unroll") for (int j = 0; j < 6; ++j) neg[j] = -g[j];
    pose_plus(x, neg, xp);
    double m = 0.0;
    _Pragma("unroll") for (int i = 0; i < 7; ++i) m = fmax(m, fabs(x[i] - xp[i]));
    return m;
}

__device__ __noinline__ void covariance_and_errors(IcpState& st) {
    // ceres::Covariance{apply_loss_function, DENSE_SVD, null_space_rank=-1} in tangent space (LidarSlam.cpp:854-871):
    // pseudo-inverse of J^T J dropping singular directions with s_i/s_max < sqrt(1e-14) (covariance_impl.cc).
    double A[36], V[36], w[6];
    _Pragma("unroll") for (int i = 0; i < 6; ++i) _Pragma("unroll") for (int j = 0; j < 6; ++j) A[i * 6 + j] = st.H[i <= j ? tri(i, j) : tri(j, i)];
    jacobi_eig6_rr<30>(A, V, w);
    const double lmax = w[5];
    double inv[6];
    bool cut = false;
    _Pragma("unroll") for (int k = 5; k >= 0; --k) {          // descending singular values = descending eigenvalues
        const double ratio = (w[k] > 0.0 && lmax > 0.0) ? sqrt(w[k] / lmax) : 0.0;
        if (cut || ratio < 1e-7) { cut = true; inv[k] = 0.0; } else inv[k] = 1.0 / w[k];
    }
    _Pragma("unroll") for (int i = 0; i < 6; ++i) _Pragma("unroll") for (int j = 0; j < 6; ++j) {
        double t = 0.0;
        _Pragma("unroll") for (int k = 0; k < 6; ++k) t += V[i * 6 + k] * inv[k] * V[j * 6 + k];
        st.cov[i * 6 + j] = t;
    }
    // EstimateRegistrationError (LidarSlam.cpp:873-884): 3x3 eigen of the position / orientation blocks
    double P[9], O[9], E[9], e[3];
    _Pragma("unroll") for (int i = 0; i < 3; ++i) _Pragma("unroll") for (int j = 0; j < 3; ++j) { P[i * 3 + j] = st.cov[i * 6 + j]; O[i * 3 + j] = st.cov[(i + 3) * 6 + (j + 3)]; }
    jacobi_eig<3, 20>(P, E, e);
    st.pos_err = sqrt(e[2]); st.pos_dir[0] = E[2]; st.pos_dir[1] = E[5]; st.pos_dir[2] = E[8];
    st.pos_inv_cond = sqrt(e[0]) / sqrt(e[2]);
    jacobi_eig<3, 20>(O, E, e);
    st.ori_err_deg = sqrt(e[2]) / M_PI * 180.0; st.ori_dir[0] = E[2]; st.ori_dir[1] = E[5]; st.ori_dir[2] = E[8];
    st.ori_inv_cond = sqrt(e[0]) / sqrt(e[2]);
}

#ifndef SO_COV_SERIAL
#define SO_COV_SERIAL 0           // 1: the covariance step on the one thread that runs the optimiser (A/B aid)
#endif
// The same computation spread over the 32 lanes of one warp (S and sc in shared memory).  The 6x6 Jacobi takes its rotations in the
// round-robin order of jacobi_eig6_rr: the three angles of a round are computed by three lanes at once, and each rotation updates
// its 8 off-diagonal entries, 12 eigenvector entries and 2x2 block on 15 lanes in one step instead of ~110 dependent FP64
// instructions on one thread (the covariance was 38 of the ~50 us the last optimiser step of a registration took).  Per element
// the arithmetic and its order are those of the serial routine; the 2x2 block goes through the same jacobi_rot2.
__constant__ int c_rr_p[15] = {0, 1, 2, 0, 3, 1, 0, 2, 1, 0, 1, 4, 0, 2, 3};
__constant__ int c_rr_q[15] = {5, 4, 3, 4, 5, 2, 3, 4, 5, 2, 3, 5, 1, 5, 4};
struct CovScratch { double a[36], v[36], w[6], inv[6], t[3], c[3], s[3]; int perm[6]; };

__device__ __noinline__ void covariance_and_errors_warp(IcpState& S, CovScratch& sc) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    for (int e = lane; e < 36; e += 32) {
        const int i = e / 6, j = e % 6;
        sc.a[e] = S.H[i <= j ? tri(i, j) : tri(j, i)];
        sc.v[e] = i == j ? 1.0 : 0.0;
    }
    __syncwarp();
#pragma unroll 1
    for (int sweep = 0; sweep < 30; ++sweep) {
        int stop = 0;
        if (lane == 0) {
            double off = 0.0, dia = 0.0;
#pragma unroll
            for (int p = 0; p < 6; ++p) {
                dia += sc.a[p * 6 + p] * sc.a[p * 6 + p];
#pragma unroll
                for (int q = p + 1; q < 6; ++q) off += sc.a[p * 6 + q] * sc.a[p * 6 + q];
            }
            stop = (off <= SO_JACOBI_OFF_TOL * dia || off == 0.0) ? 1 : 0;
        }
        if (__shfl_sync(full, stop, 0)) break;
#pragma unroll 1
        for (int round = 0; round < 5; ++round) {
            if (lane < 3) {                                  // the three angles of the round (disjoint 2x2 blocks)
                const int p = c_rr_p[round * 3 + lane], q = c_rr_q[round * 3 + lane];
                const double apq = sc.a[p * 6 + q];
                const float dlt = float(sc.a[q * 6 + q] - sc.a[p * 6 + p]), b2 = float(2.0 * apq);
                float tf = __fdividef(b2, fabsf(dlt) + sqrtf(fmaf(dlt, dlt, b2 * b2)));
                if (!(fabsf(tf) <= 1.0f)) tf = 0.0f;         // apq == 0 after the cast (or inf / nan): no rotation
                const double t = apq != 0.0 ? double(dlt < 0.0f ? -tf : tf) : 0.0;
                const double c = rsqrt(t * t + 1.0);
                sc.t[lane] = t; sc.c[lane] = c; sc.s[lane] = t * c;
            }
            __syncwarp();
#pragma unroll 1
            for (int k = 0; k < 3; ++k) {
                const int p = c_rr_p[round * 3 + k], q = c_rr_q[round * 3 + k];
                const double t = sc.t[k], c = sc.c[k], sn = sc.s[k];
                if (t != 0.0) {                              // warp-uniform
                    // lanes 0..5: row r of a (r outside the pair); lanes 8..13: row r of v; lane 16: the 2x2 block
                    const int r = lane < 8 ? lane : lane - 8;
                    const bool do_a = lane < 6 && r != p && r != q, do_v = lane >= 8 && lane < 14, do_d = lane == 16;
                    double n0 = 0.0, n1 = 0.0, n2 = 0.0;
                    if (do_a) { const double arp = sc.a[r * 6 + p], arq = sc.a[r * 6 + q]; n0 = c * arp - sn * arq; n1 = sn * arp + c * arq; }
                    if (do_v) { const double vrp = sc.v[r * 6 + p], vrq = sc.v[r * 6 + q]; n0 = c * vrp - sn * vrq; n1 = sn * vrp + c * vrq; }
                    if (do_d) jacobi_rot2(sc.a[p * 6 + p], sc.a[q * 6 + q], sc.a[p * 6 + q], c, sn, n0, n1, n2);
                    __syncwarp();
                    if (do_a) { sc.a[r * 6 + p] = sc.a[p * 6 + r] = n0; sc.a[r * 6 + q] = sc.a[q * 6 + r] = n1; }
                    if (do_v) { sc.v[r * 6 + p] = n0; sc.v[r * 6 + q] = n1; }
                    if (do_d) { sc.a[p * 6 + p] = n0; sc.a[q * 6 + q] = n1; sc.a[p * 6 + q] = n2; sc.a[q * 6 + p] = n2; }
                    __syncwarp();
                }
            }
        }
    }
    if (lane == 0) {                                         // ascending order, as a column permutation
        double w[6];
        int pm[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) { w[i] = sc.a[i * 6 + i]; pm[i] = i; }
#pragma unroll
        for (int i = 0; i < 5; ++i)
#pragma unroll
            for (int j = i + 1; j < 6; ++j)
                if (w[j] < w[i]) { const double tw = w[i]; w[i] = w[j]; w[j] = tw; const int tp = pm[i]; pm[i] = pm[j]; pm[j] = tp; }
#pragma unroll
        for (int i = 0; i < 6; ++i) { sc.w[i] = w[i]; sc.perm[i] = pm[i]; }
    }
    __syncwarp();
    {
        const int e0 = lane, e1 = lane + 32;
        const double v0 = sc.v[(e0 / 6) * 6 + sc.perm[e0 % 6]];
        const double v1 = e1 < 36 ? sc.v[(e1 / 6) * 6 + sc.perm[e1 % 6]] : 0.0;
        __syncwarp();
        sc.v[e0] = v0;
        if (e1 < 36) sc.v[e1] = v1;
    }
    __syncwarp();
    // ceres::Covariance{apply_loss_function, DENSE_SVD, null_space_rank=-1} in tangent space (LidarSlam.cpp:854-871):
    // pseudo-inverse of J^T J dropping singular directions with s_i/s_max < sqrt(1e-14) (covariance_impl.cc).
    {
        const double lmax = sc.w[5];
        const double wk = lane < 6 ? sc.w[lane] : 1.0;
        const double ratio = (wk > 0.0 && lmax > 0.0) ? sqrt(wk / lmax) : 0.0;
        const unsigned bad = __ballot_sync(full, lane < 6 && ratio < 1e-7);
        if (lane < 6) sc.inv[lane] = (bad >> lane) ? 0.0 : 1.0 / wk;     // a cut direction cuts every smaller one (descending singular values)
    }
    __syncwarp();
    for (int e = lane; e < 36; e += 32) {
        const int i = e / 6, j = e % 6;
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) t += sc.v[i * 6 + k] * sc.inv[k] * sc.v[j * 6 + k];
        S.cov[e] = t;
    }
    __syncwarp();
    // EstimateRegistrationError (LidarSlam.cpp:873-884): 3x3 eigen of the position (lane 0) / orientation (lane 1) blocks
    if (lane < 2) {
        double M[9], E[9], e[3];
        const int o = lane * 3;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) M[i * 3 + j] = S.cov[(i + o) * 6 + (j + o)];
        jacobi_eig<3, 20>(M, E, e);
        const double err = sqrt(e[2]), inv_cond = sqrt(e[0]) / sqrt(e[2]);
        if (lane == 0) { S.pos_err = err; S.pos_dir[0] = E[2]; S.pos_dir[1] = E[5]; S.pos_dir[2] = E[8]; S.pos_inv_cond = inv_cond; }
        else { S.ori_err_deg = err / M_PI * 180.0; S.ori_dir[0] = E[2]; S.ori_dir[1] = E[5]; S.ori_dir[2] = E[8]; S.ori_inv_cond = inv_cond; }
    }
    __syncwarp();
}

// End of one ceres::Solve == end of one ICP iteration (LidarSlam.cpp:134-146).
__device__ __noinline__ void end_solve(IcpState& st) {
    const int it = st.icp_iter;
    st.iter_n_surf[it] = st.n_ok - st.n_ok_edge;
    st.iter_n_edge[it] = st.n_ok_edge;
    rel_motion(st.x_iter_start, st.x, &st.iter_dtrans[it], &st.iter_drot[it]);      // recordIterationStats (:242-251)
    st.iter_lm_steps[it] = st.lm_iter;
    st.iter_lm_successful[it] = st.num_successful;
    st.iter_lm_termination[it] = st.termination;
    st.iter_cost[it] = st.cost;
    st.n_iterations = it + 1;
    if (st.n_ok == 0 && !st.use_prior) {          // reference: ceres::Covariance CHECK-fails on an empty problem; we stop with a status
        st.status = SO_STATUS_NO_CORRESPONDENCES; st.phase = PH_DONE; return;
    }
    if (st.num_successful == 1 || it == st.max_icp_iters - 1) {      // (:141)
#if SO_COV_SERIAL
        covariance_and_errors(st);
#else
        st.need_cov = 1;                          // lm_step_body: first warp of the CTA, right after this serial step
#endif
        st.phase = PH_DONE;
    } else {
        st.icp_iter = it + 1;
        st.phase = PH_CORR;
    }
}

// TrustRegionMinimizer loop from FinalizeIterationAndCheckIfMinimizerCanContinue up to the next cost evaluation.
__device__ __noinline__ void lm_continue(IcpState& st, bool step_successful) {
    for (;;) {
        if (step_successful) st.num_successful++; else st.num_unsuccessful++;
        if (st.lm_iter >= st.lm_max_iterations) { st.termination = 0; end_solve(st); return; }
        if (st.gmax <= 1e-10) { st.termination = 1; end_solve(st); return; }
        if (st.radius <= 1e-32) { st.termination = 4; end_solve(st); return; }
        st.lm_iter++;
        step_successful = false;
        // LevenbergMarquardtStrategy::ComputeStep on the Jacobi-scaled system
        double Hs[36], gs[6];
        _Pragma("unroll") for (int i = 0; i < 6; ++i) {
            gs[i] = st.g[i] * st.scale[i];
            _Pragma("unroll") for (int j = 0; j < 6; ++j) Hs[i * 6 + j] = st.H[i <= j ? tri(i, j) : tri(j, i)] * st.scale[i] * st.scale[j];
        }
        if (!st.reuse_diagonal)
            _Pragma("unroll") for (int j = 0; j < 6; ++j) st.diag[j] = fmin(fmax(Hs[j * 6 + j], 1e-6), 1e32);
        st.reuse_diagonal = 1;
        double M[36], y[6];
        _Pragma("unroll") for (int i = 0; i < 36; ++i) M[i] = Hs[i];
        _Pragma("unroll") for (int j = 0; j < 6; ++j) M[j * 6 + j] += st.diag[j] / st.radius;       // lm_diagonal^2 = diagonal / radius
        bool valid = chol6_solve(M, gs, y);
        double step[6], mcc = 0.0;
        if (valid) {
            _Pragma("unroll") for (int j = 0; j < 6; ++j) { step[j] = -y[j]; valid = valid && isfinite(step[j]); }
            // model_cost_change = -(J step)'(f + J step / 2) = -step'gs - step'Hs step / 2
            double sg = 0.0, sHs = 0.0;
            _Pragma("unroll") for (int i = 0; i < 6; ++i) { sg += step[i] * gs[i]; double t = 0.0; _Pragma("unroll") for (int j = 0; j < 6; ++j) t += Hs[i * 6 + j] * step[j]; sHs += step[i] * t; }
            mcc = -sg - 0.5 * sHs;
        }
        if (!valid || !(mcc > 0.0)) {           // HandleInvalidStep
            if (++st.consecutive_invalid >= 5) { st.termination = 5; end_solve(st); return; }
            st.radius *= 0.5; st.reuse_diagonal = 1;
            continue;
        }
        st.consecutive_invalid = 0;
        st.model_cost_change = mcc;
        double delta[6];
        _Pragma("unroll") for (int j = 0; j < 6; ++j) delta[j] = step[j] * st.scale[j];
        pose_plus(st.x, delta, st.cand);
        st.phase = PH_EVAL;
        return;
    }
}

// SE3AbsolutatePoseFactor (factor/SE3AbsolutatePoseFactor.cpp:9-51) added by addAbsolutePoseConstraints (LidarSlam.cpp:285-298):
// residual [p - p_meas ; 2 vec(q_meas^* q)] times sqrt_information (diagonal here), no loss function; local Jacobian
// [I 0; 0 (w I + [v]x)] of q_e = q_meas^* q (Utility::Qleft bottom-right block), T_meas = T_w_initial_guess.
// Adds its J^T J, J^T r and 1/2 r^T r to the 28 reduced sums at pose x.
__device__ __noinline__ void add_pose_prior(const IcpState& st, const double x[7], double a[kAcc]) {
    const double qm[4] = {-st.x0[3], -st.x0[4], -st.x0[5], st.x0[6]};
    double e[4];
    qmul(qm, x + 3, e);
    double r[6] = {x[0] - st.x0[0], x[1] - st.x0[1], x[2] - st.x0[2], 2.0 * e[0], 2.0 * e[1], 2.0 * e[2]};
    double J[36];
    _Pragma("unroll") for (int i = 0; i < 36; ++i) J[i] = 0.0;
    J[0] = J[7] = J[14] = 1.0;
    J[3 * 6 + 3] = e[3];  J[3 * 6 + 4] = -e[2]; J[3 * 6 + 5] = e[1];
    J[4 * 6 + 3] = e[2];  J[4 * 6 + 4] = e[3];  J[4 * 6 + 5] = -e[0];
    J[5 * 6 + 3] = -e[1]; J[5 * 6 + 4] = e[0];  J[5 * 6 + 5] = e[3];
    _Pragma("unroll") for (int i = 0; i < 6; ++i) { r[i] *= st.prior_sqrt_info[i]; _Pragma("unroll") for (int j = 0; j < 6; ++j) J[i * 6 + j] *= st.prior_sqrt_info[i]; }
    _Pragma("unroll") for (int i = 0; i < 6; ++i) {
        _Pragma("unroll") for (int j = i; j < 6; ++j) { double t = 0.0; _Pragma("unroll") for (int k = 0; k < 6; ++k) t += J[k * 6 + i] * J[k * 6 + j]; a[tri(i, j)] += t; }
        double t = 0.0; _Pragma("unroll") for (int k = 0; k < 6; ++k) t += J[k * 6 + i] * r[k];
        a[21 + i] += t;
    }
    double sq = 0.0; _Pragma("unroll") for (int k = 0; k < 6; ++k) sq += r[k] * r[k];
    a[27] += 0.5 * sq;
}

// IterationZero of a new solve, fed by k_fit's reduction.
__device__ __noinline__ void lm_begin_solve(IcpState& st, const double* acc_in, int n_ok) {
    double acc[kAcc];
    _Pragma("unroll") for (int k = 0; k < kAcc; ++k) acc[k] = acc_in[k];
    if (st.use_prior) {
        // information diagonal (LidarSlam.cpp:287-294); sqrt by Eigen's unblocked LLT: the first non-positive pivot and
        // everything after it stay un-square-rooted
        const double vcf = double(st.prior_vcf);
        double info[6];
        const int m1 = max(50, int(n_ok * 0.1)), m2 = max(10, int(n_ok * 0.01));
        _Pragma("unroll") for (int a = 0; a < 3; ++a) info[a] = (1 - double(st.prior_unc[a])) * m1 * vcf;
        info[3] = info[4] = m2 * vcf;
        info[5] = max(5, int(n_ok * 0.001)) * 0;
        bool failed = false;
        _Pragma("unroll") for (int k = 0; k < 6; ++k) { if (!failed && info[k] <= 0.0) failed = true; st.prior_sqrt_info[k] = failed ? info[k] : sqrt(info[k]); }
        add_pose_prior(st, st.x, acc);
    }
    _Pragma("unroll") for (int k = 0; k < 21; ++k) st.H[k] = acc[k];
    _Pragma("unroll") for (int k = 0; k < 6; ++k) st.g[k] = acc[21 + k];
    st.cost = acc[27];
    st.n_ok = n_ok;
    _Pragma("unroll") for (int i = 0; i < 7; ++i) st.x_iter_start[i] = st.x[i];
    st.lm_iter = 0; st.num_successful = 0; st.num_unsuccessful = 0; st.consecutive_invalid = 0; st.termination = 0;
    if (n_ok == 0 && !st.use_prior) { st.termination = 6; end_solve(st); return; }
    _Pragma("unroll") for (int j = 0; j < 6; ++j) st.scale[j] = 1.0 / (1.0 + sqrt(st.H[tri(j, j)]));      // jacobi_scaling at iteration 0
    double xn = 0.0; _Pragma("unroll") for (int i = 0; i < 7; ++i) xn += st.x[i] * st.x[i];
    st.x_norm = sqrt(xn);
    st.gmax = grad_max_norm(st.x, st.g);
    st.radius = 1e4; st.decrease_factor = 2.0; st.reuse_diagonal = 0;
    lm_continue(st, false);
}

// After the cost (and H, g) at the candidate are known.
__device__ __noinline__ void lm_after_eval(IcpState& st, const double* acc_in) {
    double acc[kAcc];
    _Pragma("unroll") for (int k = 0; k < kAcc; ++k) acc[k] = acc_in[k];
    if (st.use_prior) add_pose_prior(st, st.cand, acc);
    const double cand_cost = acc[27];
    // ParameterToleranceReached
    double sn = 0.0; _Pragma("unroll") for (int i = 0; i < 7; ++i) { const double d = st.x[i] - st.cand[i]; sn += d * d; }
    sn = sqrt(sn);
    if (sn <= 1e-8 * (st.x_norm + 1e-8)) { st.termination = 2; end_solve(st); return; }
    // FunctionToleranceReached
    const double cost_change = st.cost - cand_cost;
    if (fabs(cost_change) <= 1e-6 * st.cost) { st.termination = 3; end_solve(st); return; }
    const double rd = cost_change / st.model_cost_change;
    if (rd > 1e-3) {        // HandleSuccessfulStep
        _Pragma("unroll") for (int i = 0; i < 7; ++i) st.x[i] = st.cand[i];
        double xn = 0.0; _Pragma("unroll") for (int i = 0; i < 7; ++i) xn += st.x[i] * st.x[i];
        st.x_norm = sqrt(xn);
        _Pragma("unroll") for (int k = 0; k < 21; ++k) st.H[k] = acc[k];
        _Pragma("unroll") for (int k = 0; k < 6; ++k) st.g[k] = acc[21 + k];
        st.cost = cand_cost;
        st.gmax = grad_max_norm(st.x, st.g);
        const double t = 2.0 * rd - 1.0;
        st.radius = st.radius / fmax(1.0 / 3.0, 1.0 - t * t * t);
        st.radius = fmin(1e16, st.radius);
        st.decrease_factor = 2.0; st.reuse_diagonal = 0;
        lm_continue(st, true);
    } else {                // StepRejected
        st.radius = st.radius / st.decrease_factor; st.decrease_factor *= 2.0; st.reuse_diagonal = 1;
        lm_continue(st, false);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// residual + Jacobian + robust weight accumulation for one correspondence at pose (q, t) with rotation matrix R.
// SurfNormAnalyticCostFunction::Evaluate (lidarOptimization.cpp:55-80); ScaledLoss(TukeyLoss(a), w) through Ceres'
// Corrector: Tukey has rho'' <= 0, so residual and Jacobian are both scaled by sqrt(rho') (corrector.cc);
// TukeyLoss of Ceres 2.0.0: rho = a^2/6 (1-(1-s/a^2)^3), rho' = (1-s/a^2)^2 / 2 for s <= a^2.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void accumulate(double acc[kAcc], const double n[3], double d, double w, const double p[3],
                                           const double pw[3], const double R[9], double a2) {
    const double r = n[0] * pw[0] + n[1] * pw[1] + n[2] * pw[2] + d;
    const double s = r * r;
    double rho0, rho1;
    if (s <= a2) { const double v = 1.0 - s / a2, v2 = v * v; rho0 = a2 / 6.0 * (1.0 - v2 * v); rho1 = 0.5 * v2; }      // TukeyLoss::Evaluate divides (loss_function.cc)
    else { rho0 = a2 / 6.0; rho1 = 0.0; }
    rho0 *= w; rho1 *= w;
    // J = [ n^T , -n^T R [p]x ] ;  -a^T [p]x = p x a  with a = R^T n
    const double a0 = R[0] * n[0] + R[3] * n[1] + R[6] * n[2];
    const double a1 = R[1] * n[0] + R[4] * n[1] + R[7] * n[2];
    const double a2v = R[2] * n[0] + R[5] * n[1] + R[8] * n[2];
    const double J[6] = {n[0], n[1], n[2], p[1] * a2v - p[2] * a1, p[2] * a0 - p[0] * a2v, p[0] * a1 - p[1] * a0};
    int k = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const double wi = rho1 * J[i];
#pragma unroll
        for (int j = i; j < 6; ++j) acc[k++] += wi * J[j];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) acc[21 + i] += rho1 * J[i] * r;
    acc[27] += 0.5 * rho0;
}

#ifndef SO_KNN_VERIFY
#define SO_KNN_VERIFY 0           // 1: try to PROVE the previous five neighbours still exact before searching again.  Off: measured slower
                                  // on every BASELINE workload (3.6 % of the queries verify on cfg2; DESIGN.md section 4, tried-and-measured)
#endif
// ICP iterations after the first, before any walk: the record of the query's last FULL search (nb.vq: where the query was, q0, and a
// lower bound D on the squared distance from q0 to every point of the block outside the five found) proves the five still ARE the
// 5-NN at the new position q1 whenever   max_i |q1 - s_i| < sqrt(D) - |q1 - q0|   -- any other point x has
// |q1 - x| >= |q0 - x| - |q1 - q0| >= sqrt(D) - |q1 - q0| (triangle inequality), strictly beyond all five, so neither membership nor
// ties with outsiders can differ from what a fresh search returns.  Then only their distances (the reference's rounding) and their
// (d2, id) order are renewed -- ~150 instructions instead of the ~3 700 of a walk.  Margins cover the float evaluation of the norms.
// Requires the five to lie in the block the query is in NOW (the search is block-local, LocalMap.h:488-507).  On success tk holds
// the five in order (tk.pos = positions in the sorted map) and true is returned.
__device__ __forceinline__ bool verify_neighbours(const MapView& m, const QueryCell& qc, const NnBuf& nb, size_t gi, float qx, float qy, float qz,
                                                  TopK<5>& tk) {
    const float4 rec = nb.vq[gi];
    if (!(rec.w > 0.f)) return false;
    const uint32_t cells = uint32_t(m.nb) * uint32_t(m.nb) * uint32_t(m.nb);
    const uint32_t lo = __ldg(&m.cell_start[uint32_t(qc.slot) * cells]), hi = __ldg(&m.cell_start[uint32_t(qc.slot) * cells + cells]);
    const float mx = qx - rec.x, my = qy - rec.y, mz = qz - rec.z;
    const float moved = sqrtf(fmaf(mx, mx, fmaf(my, my, mz * mz))) * 1.000002f + 1e-6f;
    const float reach = sqrtf(rec.w) * 0.999998f - moved - 1e-6f;           // every outsider is at least this far from q1
    if (!(reach > 0.f)) return false;
    bool ok = true;
    float4 c[5]; uint32_t pos[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        pos[j] = nb.pos[size_t(j) * nb.cap + gi];
        ok = ok && pos[j] >= lo && pos[j] < hi;
        c[j] = __ldg(&m.pts[ok ? pos[j] : lo]);
    }
    if (!ok) return false;
    float far2 = 0.f;
#pragma unroll
    for (int j = 0; j < 5; ++j) far2 = fmaxf(far2, exact_d2(c[j], qx, qy, qz));
    if (!(sqrtf(far2) * 1.000002f < reach)) return false;
    tk.init(FLT_MAX);
#pragma unroll
    for (int j = 0; j < 5; ++j) tk.offer(exact_d2(c[j], qx, qy, qz), __float_as_uint(c[j].w), pos[j]);
    return true;
}

// ICP iterations after the first: the previous iteration's five neighbours still exist, so the largest of their (exact)
// distances to the moved query bounds the new 5th-neighbour distance -- provided they lie in the block the query is in NOW
// (the search is block-local, LocalMap.h:488-507: after a pose update that carries the point across a 50 m block face the old
// neighbours belong to another block and bound nothing).  Returns the bound or -1 (no usable seed).
__device__ __forceinline__ float seed_bound(const MapView& m, const QueryCell& qc, const NnBuf& nb, size_t gi, float qx, float qy, float qz) {
    const uint32_t cells = uint32_t(m.nb) * uint32_t(m.nb) * uint32_t(m.nb);
    const uint32_t lo = __ldg(&m.cell_start[uint32_t(qc.slot) * cells]), hi = __ldg(&m.cell_start[uint32_t(qc.slot) * cells + cells]);
    float u = 0.f;
    bool same_block = true;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const uint32_t pos = nb.pos[size_t(j) * nb.cap + gi];
        same_block = same_block && pos >= lo && pos < hi;
        const float4 c = __ldg(&m.pts[same_block ? pos : lo]);
        const float dx = qx - c.x, dy = qy - c.y, dz = qz - c.z;
        u = fmaxf(u, float(double(dx) * double(dx) + double(dy) * double(dy) + double(dz) * double(dz)));
    }
    // use it only while it is about as tight as a freshly estimated bound would be (small pose update); after a large update
    // the cell-neighbourhood estimate of round 1 prunes better than a loose seed
    return (same_block && u <= 1.3f * nb.d5[gi]) ? u : -1.f;
}

// shouldProcessPoint (LidarSlam.cpp:353-359)
__device__ __forceinline__ bool should_process(uint32_t i, double rate) {
    if (rate < 0.0) return true;
    // explicit round-to-nearest operations: no FMA contraction, so that the host twin (so_api.cu: should_process_h, the decimated
    // upload of so_register) and the reference's x86 arithmetic select exactly the same points
    const double x = __dmul_rn(double(i), rate);
    const double rem = __dsub_rn(x, floor(x));            // == std::fmod(x, 1.0) for x >= 0: both are exact
    return !(__dadd_rn(rem, 0.001) > rate);
}

// ------------------------------------------------------------------------------------------------------------------
// Scan preparation (once per registration): order the scan points by the map cell they fall into at the PRIOR pose, cells
// grouped into 8x8x8 bricks (scan_order_key), so that the 128 queries of a CTA sit in a compact box of cells (one shared,
// bulk-copied candidate tile) and the 32 lanes of a warp walk the same cell rows.  Pose updates inside one registration are a
// few cm against 0.39 m cells, so the order stays coherent for all ICP iterations.  The sorted copy carries the point's original index in .w (the reference's
// shouldProcessPoint() decimation is defined on the original index, LidarSlam.cpp:353-359).
// ------------------------------------------------------------------------------------------------------------------
// Key = (scan index inside the chunk) << cell_bits | cell; cells beyond the mask and off-map points sort last inside their scan.
// KeyT = uint32_t when cell_bits + scan bits fit (the usual case: 4 radix passes over 8-byte pairs instead of 5 over 12-byte ones).
// COMPACT: points that shouldProcessPoint (LidarSlam.cpp:353-359) drops get one more key bit above the cell and sort behind every
// survivor of their scan; k_scan_finish then shrinks the scan to its survivors (the decimation depends on the original index only,
// so it is decided once per registration and the ICP kernels run over max_surface_features points instead of the whole scan).
template <class KeyT, bool COMPACT>
__global__ void __launch_bounds__(kThreads) k_scan_keys(MapView m, BatchView bv, KeyT* __restrict__ keys, uint32_t* __restrict__ vals, int cell_bits) {
    const int s = blockIdx.y;
    const IcpState* st = bv.st + s;
    const uint32_t n = uint32_t(st->n_points);
    const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const size_t gi = size_t(bv.offset[s]) + i;
    if (COMPACT && !should_process(i, st->sampling_rate)) {
        keys[gi] = KeyT((KeyT(s) << (cell_bits + 1)) | (KeyT(1) << cell_bits));
        vals[gi] = uint32_t(gi);
        return;
    }
    const float4 sp = __ldg(&bv.scan[gi]);
    const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
    double pf[3];
    qrot(st->x + 3, pin, pf);
    QueryCell qc;
    locate(m, float(pf[0] + st->x[0]), float(pf[1] + st->x[1]), float(pf[2] + st->x[2]), qc);
    const uint32_t cell = qc.slot >= 0 ? scan_order_key(m, qc) : 0xFFFFFFFFu;      // brick order (so_knn.cuh)
    const uint32_t mask = cell_bits >= 32 ? 0xFFFFFFFFu : ((1u << cell_bits) - 1u);
    keys[gi] = KeyT((KeyT(s) << (cell_bits + (COMPACT ? 1 : 0))) | KeyT(cell < mask ? cell : mask));
    vals[gi] = uint32_t(gi);
}

// After the sort of a COMPACT chunk: survivors of scan s = sorted keys of its range without the dropped bit (binary search);
// the scan shrinks to them and its decimation is switched off.
template <class KeyT>
__global__ void k_scan_finish(BatchView bv, const KeyT* __restrict__ sorted_keys, uint32_t pt_first, int cell_bits, uint32_t n_scans) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_scans) return;
    IcpState* st = bv.st + s;
    if (st->phase != PH_CORR) return;
    const KeyT* k = sorted_keys + (bv.offset[s] - pt_first);
    uint32_t lo = 0, hi = uint32_t(st->n_points);
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if ((k[mid] >> cell_bits) & 1) hi = mid; else lo = mid + 1; }
    st->n_points = int32_t(lo);
    st->sampling_rate = -1.0;
}

template <class KeyT>
__global__ void __launch_bounds__(kThreads) k_scan_gather(const float4* __restrict__ in, const uint32_t* __restrict__ vals, const KeyT* __restrict__ keys,
                                                          const uint32_t* __restrict__ offset, size_t total, float4* __restrict__ out, int cell_bits) {
    const size_t j = size_t(blockIdx.x) * kThreads + threadIdx.x;
    if (j >= total) return;
    const uint32_t g = vals[j];
    const uint32_t s = uint32_t(keys[j] >> cell_bits);                 // cell_bits here = all key bits below the scan index
    const float4 p = __ldg(&in[g]);
    out[j] = make_float4(p.x, p.y, p.z, __uint_as_float(g - offset[s]));
}

// ------------------------------------------------------------------------------------------------------------------
// k_prepare_small: the whole scan preparation of a SMALL registration in one CTA per scan -- what k_scan_keys + a device-wide
// radix sort (4-5 launches whose fixed cost, ~35 us, is most of a latency-bound so_register) + k_scan_gather do for batches.
// Points that shouldProcessPoint (LidarSlam.cpp:353-359) drops are removed HERE, once (the decimation is a function of the
// original index only): the ICP kernels then run over the <= max_surface_features + 1 surviving points with sampling off.
// Deterministic: the survivors are compacted in index order (block scans), sorted by cell key with a stable block radix sort.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kSmallThreads = 1024, kSmallCap = kPrepareSmallCap;
static_assert(kSmallCap == kSmallThreads * 4, "k_prepare_small<4> covers kPrepareSmallCap survivors");
// ITEMS: survivors per thread in the sort (2 when they fit 2048 -- the shipped max_surface_features of 2000 -- else 4)
template <int ITEMS>
__global__ void __launch_bounds__(kSmallThreads) k_prepare_small(MapView m, BatchView bv, float4* __restrict__ out, int key_bits) {
    constexpr int kCap = kSmallThreads * ITEMS;
    using Sort = cub::BlockRadixSort<uint32_t, kSmallThreads, ITEMS, uint32_t>;
    using Scan = cub::BlockScan<uint32_t, kSmallThreads>;
    struct Compact { typename Scan::TempStorage scan; uint32_t idx[kCap]; };
    __shared__ union { typename Sort::TempStorage sort; Compact c; } s_tmp;      // the index list is consumed (into registers) before the sort starts
    uint32_t* s_idx = s_tmp.c.idx;
    __shared__ double s_pose[7];
    const int s = blockIdx.x;
    IcpState* st = bv.st + s;
    if (st->phase != PH_CORR) return;
    if (threadIdx.x < 7) s_pose[threadIdx.x] = st->x[threadIdx.x];
    const uint32_t n = uint32_t(st->n_points);
    const double rate = st->sampling_rate;
    const size_t base = size_t(bv.offset[s]);
    // survivors, in index order: every thread owns a contiguous run of indices, ONE block scan places the runs
    const uint32_t per = (n + kSmallThreads - 1) / kSmallThreads, lo = min(n, threadIdx.x * per), hi = min(n, lo + per);
    uint32_t mine = 0;
    for (uint32_t i = lo; i < hi; ++i) mine += should_process(i, rate) ? 1u : 0u;
    uint32_t pos, total;
    Scan(s_tmp.c.scan).ExclusiveSum(mine, pos, total);
    for (uint32_t i = lo; i < hi && pos < uint32_t(kCap); ++i) if (should_process(i, rate)) s_idx[pos++] = i;
    __syncthreads();
    const uint32_t n_act = min(total, uint32_t(kCap));                  // the host chose this path only when the survivors fit
    uint32_t key[ITEMS], val[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t j = threadIdx.x * ITEMS + k;                     // blocked arrangement
        key[k] = 0xFFFFFFFFu; val[k] = 0xFFFFFFFFu;
        if (j < n_act) {
            const uint32_t i = s_idx[j];
            const float4 sp = __ldg(&bv.scan[base + i]);
            const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
            double pf[3];
            qrot(s_pose + 3, pin, pf);
            QueryCell qc;
            locate(m, float(pf[0] + s_pose[0]), float(pf[1] + s_pose[1]), float(pf[2] + s_pose[2]), qc);
            const uint32_t mask = key_bits >= 32 ? 0xFFFFFFFFu : ((1u << key_bits) - 1u);
            const uint32_t cell = qc.slot >= 0 ? scan_order_key(m, qc) : 0xFFFFFFFFu;
            key[k] = cell < mask ? cell : mask;                          // off-map points sort last among the survivors, as in the batch path
            val[k] = i;
        }
    }
    __syncthreads();
    Sort(s_tmp.sort).Sort(key, val, 0, key_bits < 32 ? key_bits + 1 : 32);      // + 1: the padding keys (all ones) sort behind the mask
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t j = threadIdx.x * ITEMS + k;
        if (j < n_act) {
            const float4 p = __ldg(&bv.scan[base + val[k]]);
            out[base + j] = make_float4(p.x, p.y, p.z, __uint_as_float(val[k]));
        }
    }
    if (threadIdx.x == 0) { st->n_points = int32_t(n_act); st->sampling_rate = -1.0; }
}

// ------------------------------------------------------------------------------------------------------------------
// k_knn_scan: findNearestNeighbors (LidarSlam.cpp:720-747) for every processed scan point at the current pose: the select k-NN of
// so_knn.cuh, one query per thread, queries consecutive in scan order.  Light on registers (FP32 search, FP64 only for the pose
// transform and the exact d2 of real contenders) so that many warps per SM hide the latency of the cell walks.
// SO_KNN_TILE build: 128 queries per CTA in brick order; the CTA stages the candidate tile of its queries' cell box (build_tile:
// one cp.async.bulk per map row onto an mbarrier, a 16-bit local cell table) and searches shared memory; CTAs whose box does not
// fit search global memory.  Measured slower than the global search (so_knn.cuh), so it is not the default.
// ------------------------------------------------------------------------------------------------------------------
#ifndef SO_KNN_MINB
#define SO_KNN_MINB (SO_KNN_TILE ? 6 : 1024 / SO_KNN_THREADS)      // 64 registers per thread either way
#endif
__global__ void __launch_bounds__(kTileThreads, SO_KNN_MINB) k_knn_scan(MapView m, BatchView bv, NnBuf nb) {
    const int s = blockIdx.y;
    IcpState* st = bv.st + s;
    if (st->phase != PH_CORR) return;
    __shared__ double s_pose[7];
    __shared__ uint32_t s_buf[kBufCap * kTileThreads];
#if SO_KNN_TILE
    __shared__ TileSmem s_tile;
#endif
    if (threadIdx.x < 7) s_pose[threadIdx.x] = st->x[threadIdx.x];
    __syncthreads();
    const uint32_t n = uint32_t(st->n_points);
    const uint32_t i = blockIdx.x * kTileThreads + threadIdx.x;
    if (blockIdx.x * kTileThreads >= n) return;           // whole CTA past the end; partial CTAs stay together for the tile build
    const bool in_range = i < n;
    const size_t gi = size_t(bv.offset[s]) + (in_range ? i : 0);
    const float4 sp = __ldg(&bv.scan[gi]);
    int pre = SO_MATCH_SKIPPED;
    TopK<5> tk;
    tk.init(m.bound_d2);
    bool searchable = false, verified = false;
    float qx = 0.f, qy = 0.f, qz = 0.f, u_seed = -1.f;
    QueryCell qc;
    qc.slot = -1; qc.nblock = 0; qc.c[0] = qc.c[1] = qc.c[2] = 0; qc.f[0] = qc.f[1] = qc.f[2] = 0.f;
    if (in_range && should_process(__float_as_uint(sp.w), st->sampling_rate)) {
        const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
        double pf[3];
        qrot(s_pose + 3, pin, pf);
        qx = float(pf[0] + s_pose[0]); qy = float(pf[1] + s_pose[1]); qz = float(pf[2] + s_pose[2]);
        locate(m, qx, qy, qz, qc);
        if (qc.slot < 0 || qc.nblock < 5) pre = SO_MATCH_NOT_ENOUGH_NEIGHBORS;
        else {
            searchable = true;
            if (st->icp_iter > 0) {
                verified = SO_KNN_VERIFY && verify_neighbours(m, qc, nb, gi, qx, qy, qz, tk);
                if (!verified && nb.pre[gi] == SO_MATCH_SUCCESS) u_seed = seed_bound(m, qc, nb, gi, qx, qy, qz);
            }
        }
    }
    if (verified) {                                       // the stored five are still the 5-NN: distances and order renewed, no walk
        searchable = false;
        pre = tk.d2[4] > m.bound_d2 ? SO_MATCH_NEIGHBORS_TOO_FAR : SO_MATCH_SUCCESS;       // d2[4] > 3*planeRes_ (:741-744)
    }
    if (SO_KNN_VERIFY) {                                  // telemetry: one atomic pair per warp
        const unsigned ms = __ballot_sync(0xffffffffu, searchable), mv = __ballot_sync(0xffffffffu, verified);
        if ((threadIdx.x & 31) == 0) { if (ms) atomicAdd(&st->knn_searched, __popc(ms)); if (mv) atomicAdd(&st->knn_verified, __popc(mv)); }
    }
#if SO_KNN_TILE
    TileGrid tg;
    const bool tiled = build_tile(m, s_tile, searchable, qc, tg);
#else
    const bool tiled = false;
#endif
    float next_lb = -1.f;
    if (searchable) {
#if SO_KNN_TILE
        if (tiled) {
            knn_select<5, SO_R1_OCTANT != 0>(tg, m, qc, qx, qy, qz, u_seed, m.bound_d2, s_buf, tk, SO_KNN_VERIFY ? &next_lb : nullptr);
#pragma unroll
            for (int j = 0; j < 5; ++j) if (tk.id[j] != 0xFFFFFFFFu) tk.pos[j] = tg.pos_of(tk.pos[j]);
        } else
#endif
        {
            const GlobalGrid gg(m, qc.slot);
            knn_select<5, SO_R1_OCTANT != 0>(gg, m, qc, qx, qy, qz, u_seed, m.bound_d2, s_buf, tk, SO_KNN_VERIFY ? &next_lb : nullptr);
        }
        pre = tk.count() < 5 ? SO_MATCH_NEIGHBORS_TOO_FAR : SO_MATCH_SUCCESS;       // d2[4] > 3*planeRes_ (:741-744)
        if (pre != SO_MATCH_SUCCESS) next_lb = -1.f;
    }
    if (!in_range) return;
    if (SO_KNN_VERIFY && !verified) nb.vq[gi] = make_float4(qx, qy, qz, next_lb);       // a verified query keeps the record of its last full search
    if (verified && pre != SO_MATCH_SUCCESS) {             // the fifth of the stored neighbours moved beyond the gate: the set stays on record
        nb.pre[gi] = (unsigned char)pre;
        nb.d5[gi] = m.bound_d2;
        return;
    }
    nb.pre[gi] = (unsigned char)pre;
    nb.d5[gi] = tk.d2[4];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const bool ok = tk.id[j] != 0xFFFFFFFFu;
        nb.pos[size_t(j) * nb.cap + gi] = ok ? tk.pos[j] : 0xFFFFFFFFu;
        // the five points are L1-hot here; handing them on as coalesced 16-byte stores saves k_fit five scattered gathers
        if (pre == SO_MATCH_SUCCESS) nb.pts[size_t(j) * nb.cap + gi] = __ldg(&m.pts[tk.pos[j]]);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// k_knn_scan_coop: the same search for SMALL registrations (a live scan after the shouldProcessPoint decimation: ~2 000 queries),
// one WARP per query.  With one query per thread such a launch is eight CTAs whose threads each walk ~3 800 dependent instructions
// (~20 us); here lane l < 25 takes row l of the 5 x 5 rows of the two-ring cube (the same pruning against the gate 3 * planeRes_
// as walk_cube), a warp scan flattens the rows' candidate spans, the lanes take the candidates 32 at a time -- FP32 filter, the
// reference's exact d2, a private top-5 -- and five warp arg-min rounds over (d2, id) merge the private lists.  The result is
// the exact block-local 5-NN in (d2, id) order with the same distances, i.e. bit-identical to k_knn_scan's, in ~700 instructions
// per warp spread over every SM.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kCoopWarps = kThreads / 32;
__global__ void __launch_bounds__(kThreads) k_knn_scan_coop(MapView m, BatchView bv, NnBuf nb) {
    const int s = blockIdx.y;
    const IcpState* st = bv.st + s;
    if (st->phase != PH_CORR) return;
    __shared__ double s_pose[7];
    __shared__ uint32_t s_scan[kCoopWarps][33], s_t[kCoopWarps][32];
    if (threadIdx.x < 7) s_pose[threadIdx.x] = st->x[threadIdx.x];
    __syncthreads();
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t n = uint32_t(st->n_points);
    const uint32_t i = blockIdx.x * kCoopWarps + warp;     // the warp's query
    if (i >= n) return;
    const size_t gi = size_t(bv.offset[s]) + i;
    const float4 sp = __ldg(&bv.scan[gi]);
    int pre = SO_MATCH_SKIPPED;
    TopK<5> tk;
    tk.init(m.bound_d2);
    if (should_process(__float_as_uint(sp.w), st->sampling_rate)) {
        const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
        double pf[3];
        qrot(s_pose + 3, pin, pf);
        const float qx = float(pf[0] + s_pose[0]), qy = float(pf[1] + s_pose[1]), qz = float(pf[2] + s_pose[2]);
        QueryCell qc;
        locate(m, qx, qy, qz, qc);
        if (qc.slot < 0 || qc.nblock < 5) pre = SO_MATCH_NOT_ENOUGH_NEIGHBORS;
        else {
            const GlobalGrid g(m, qc.slot);
            const int nbc = m.nb, R = m.R;
            const float cs = m.cs, U = m.bound_d2 * 1.000004f, Um = U * 1.0001f;
            // ---- lane l: row (oz, oy) of the cube, its candidate span
            uint32_t t = 0, len = 0;
            const int side = 2 * R + 1;
            if (lane < side * side) {                      // R <= 2 by construction of the grid (cells >= half the search radius)
                const int oz = lane / side - R, oy = lane % side - R;
                const int zz = qc.c[2] + oz, yy = qc.c[1] + oy, cx = qc.c[0];
                const float fx = qc.f[0], gx = cs - fx;
                const float lz = axis_gap(oz, qc.f[2], cs - qc.f[2], cs), ly = axis_gap(oy, qc.f[1], cs - qc.f[1], cs);
                const float lb = fmaf(ly, ly, lz * lz);
                if (zz >= 0 && zz < nbc && yy >= 0 && yy < nbc && lb <= Um) {
                    const bool l1 = cx >= 1 && fmaf(fx, fx, lb) <= Um;
                    const bool l2 = l1 && R >= 2 && cx >= 2 && fmaf(fx + cs, fx + cs, lb) <= Um;
                    const bool r1 = cx + 1 < nbc && fmaf(gx, gx, lb) <= Um;
                    const bool r2 = r1 && R >= 2 && cx + 2 < nbc && fmaf(gx + cs, gx + cs, lb) <= Um;
                    uint32_t end, tag;
                    g.row(zz, yy, cx - int(l1) - int(l2), cx + int(r1) + int(r2), t, end, tag);
                    len = end - t;
                }
            }
            // ---- exclusive scan of the span lengths: candidate c of the flattened list sits in the row whose prefix interval holds c
            uint32_t incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(full, incl, o); if (lane >= o) incl += v; }
            const uint32_t total = __shfl_sync(full, incl, 31);
            s_scan[warp][lane] = incl - len;
            s_t[warp][lane] = t;
            if (lane == 0) s_scan[warp][32] = total;
            __syncwarp();
            for (uint32_t c = lane; c < total; c += 32) {
                int lo = 0;                                // largest row with prefix <= c (empty rows share a prefix: the search lands past them)
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) if (s_scan[warp][lo + o] <= c) lo += o;
                const uint32_t e = s_t[warp][lo] + (c - s_scan[warp][lo]);
                const float4 cand = g.load(e);
                if (approx_d2(cand, qx, qy, qz) <= U) tk.offer(exact_d2(cand, qx, qy, qz), __float_as_uint(cand.w), e);
            }
            // ---- merge: five rounds of warp arg-min over the heads of the private lists
            TopK<5> out;
            out.init(m.bound_d2);
            int head = 0;
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                float hd = m.bound_d2; uint32_t hi = 0xFFFFFFFFu, hp = 0;
#pragma unroll
                for (int k = 0; k < 5; ++k) if (k == head) { hd = tk.d2[k]; hi = tk.id[k]; hp = tk.pos[k]; }
                if (head >= 5) { hd = FLT_MAX; hi = 0xFFFFFFFFu; }
                const uint32_t dbits = hi != 0xFFFFFFFFu ? __float_as_uint(hd) : 0xFFFFFFFFu;      // d2 >= 0: the bit pattern orders like the value
                const uint32_t dmin = __reduce_min_sync(full, dbits);
                if (dmin == 0xFFFFFFFFu) break;            // fewer than five within the gate (warp-uniform)
                const uint32_t imin = __reduce_min_sync(full, dbits == dmin ? hi : 0xFFFFFFFFu);
                const bool win = dbits == dmin && hi == imin;      // ids are unique: exactly one lane
                const int src = __ffs(__ballot_sync(full, win)) - 1;
                out.d2[j] = __uint_as_float(dmin); out.id[j] = imin; out.pos[j] = __shfl_sync(full, hp, src);
                if (win) ++head;
            }
            tk = out;
            pre = tk.count() < 5 ? SO_MATCH_NEIGHBORS_TOO_FAR : SO_MATCH_SUCCESS;       // d2[4] > 3*planeRes_ (:741-744)
        }
    }
    if (lane == 0) { nb.pre[gi] = (unsigned char)pre; nb.d5[gi] = tk.d2[4]; }
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        if (lane == j) {
            const bool ok = tk.id[j] != 0xFFFFFFFFu;
            nb.pos[size_t(j) * nb.cap + gi] = ok ? tk.pos[j] : 0xFFFFFFFFu;
            if (pre == SO_MATCH_SUCCESS) nb.pts[size_t(j) * nb.cap + gi] = __ldg(&m.pts[tk.pos[j]]);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// k_knn_inject: test hook behind so_register_injected -- the neighbour SEARCH of k_knn_scan replaced by caller-supplied
// neighbour ids (ids[it][original point index][5], map point ids in so_map_set_points order, 0xFFFFFFFF = no result), everything
// after it (the NEIGHBORS_TOO_FAR gate on the 5th distance, LidarSlam.cpp:741-744, the hand-off to k_fit) unchanged.  Feeding it
// the neighbour sets of the reference's own octree (oracle knn_mode 2) isolates the one known deviation of this library from the
// reference path: exact in-block k-NN instead of the octree's data-dependent misses (flann/octree.h:383-385,984-1001).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_knn_inject(MapView m, const float4* __restrict__ by_id, uint32_t n_map, BatchView bv, NnBuf nb,
                                                         const uint32_t* __restrict__ ids, int n_trace_iters) {
    const int s = blockIdx.y;
    const IcpState* st = bv.st + s;
    if (st->phase != PH_CORR) return;
    __shared__ double s_pose[7];
    if (threadIdx.x < 7) s_pose[threadIdx.x] = st->x[threadIdx.x];
    __syncthreads();
    const uint32_t n = uint32_t(st->n_points);
    const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const size_t gi = size_t(bv.offset[s]) + i;
    const float4 sp = __ldg(&bv.scan[gi]);
    const uint32_t orig = __float_as_uint(sp.w);
    int pre = SO_MATCH_SKIPPED;
    float d5 = m.bound_d2;
    if (should_process(orig, st->sampling_rate)) {
        pre = SO_MATCH_NOT_ENOUGH_NEIGHBORS;
        const int it = st->icp_iter;
        if (it < n_trace_iters) {
            const uint32_t* p = ids + (size_t(it) * uint32_t(st->n_input) + orig) * 5;      // the trace is laid out over the scan as uploaded
            bool ok = true;
#pragma unroll
            for (int j = 0; j < 5; ++j) ok = ok && p[j] < n_map;
            if (ok) {
                const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
                double pf[3];
                qrot(s_pose + 3, pin, pf);
                const float qx = float(pf[0] + s_pose[0]), qy = float(pf[1] + s_pose[1]), qz = float(pf[2] + s_pose[2]);
#pragma unroll
                for (int j = 0; j < 5; ++j) {
                    const float4 c = __ldg(&by_id[p[j]]);
                    const float dx = qx - c.x, dy = qy - c.y, dz = qz - c.z;
                    d5 = float(double(dx) * double(dx) + double(dy) * double(dy) + double(dz) * double(dz));
                    nb.pts[size_t(j) * nb.cap + gi] = make_float4(c.x, c.y, c.z, __uint_as_float(p[j]));
                }
                pre = double(d5) > double(m.bound_d2) ? SO_MATCH_NEIGHBORS_TOO_FAR : SO_MATCH_SUCCESS;      // pointSearchSqDis[4] > 3*planeRes_ (:741-744)
            }
        }
    }
    nb.pre[gi] = (unsigned char)pre;
    nb.d5[gi] = d5;
#pragma unroll
    for (int j = 0; j < 5; ++j) nb.pos[size_t(j) * nb.cap + gi] = 0xFFFFFFFFu;
}

// A 16-byte global load the compiler may neither merge with an earlier load of the same address nor hoist: k_fit re-reads
// its neighbours (L1 hits) rather than keeping them live in registers.
__device__ __forceinline__ float4 ld_f4_again(const float4* p) {
    float4 v;
    asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// ------------------------------------------------------------------------------------------------------------------
// k_fit: the rest of LidarSLAM::ComputePlaneDistanceParameters (LidarSlam.cpp:536-572) for every scan point, from the
// neighbours k_knn_scan handed over: fit_point() below + the per-scan histograms.  The first residual/Jacobian evaluation of
// the following ceres::Solve is a separate k_evaluate<PH_CORR> launch, which keeps this kernel at 64 registers.
// ------------------------------------------------------------------------------------------------------------------
// The rest of LidarSLAM::ComputePlaneDistanceParameters (LidarSlam.cpp:536-572) for one scan point whose k-NN outcome is
// `status`: PCA, plane fit, gates, observability labels, fit weight; writes the correspondence record and counts the
// histograms.  nbr(j) re-reads neighbour j (a volatile, L1-hit load: the neighbours are read three times rather than held in
// 30 FP64 registers across the eigen-solve).  FP64 throughout.
template <class NbrLoad>
__device__ __forceinline__ void fit_point(const MapView& m, const CorrBuf& cb, const NnBuf& nb, size_t gi, const float4 sp, const double* s_pose,
                                          int status, NbrLoad nbr, int* s_hist) {
    int o0 = 0, o1 = 0, o2 = 0;
    double nrm[3] = {0, 0, 0}, dpl = 0.0, wq = 0.0;
    if (status == SO_MATCH_SUCCESS) {
                    // ComputePointInitAndFinalPose (:382-400): pInit = double(p), pFinal = T_w_lidar * pInit
        const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
        double pf[3];
        qrot(s_pose + 3, pin, pf);
        pf[0] += s_pose[0]; pf[1] += s_pose[1]; pf[2] += s_pose[2];
        const float qx = float(pf[0]), qy = float(pf[1]), qz = float(pf[2]);
        // computePCAForFeature (:749-790) + utils::ComputePCA (superodom_utils.h:143-151).  The five neighbours are read
        // three times (here, for the QR, for the distances) through nbr() instead of being held in 30 FP64 registers across
        // the eigen-solve: the re-reads hit L1 and the kernel fits 4 CTAs per SM.
        double mean[3] = {0, 0, 0};
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const float4 c = nbr(j);
            mean[0] += double(c.x); mean[1] += double(c.y); mean[2] += double(c.z);
            if (cb.nn) {
                const float dx = qx - c.x, dy = qy - c.y, dz = qz - c.z;
                cb.nn[gi * 5 + j] = __float_as_uint(c.w);
                cb.nn_d2[gi * 5 + j] = float(double(dx) * double(dx) + double(dy) * double(dy) + double(dz) * double(dz));
            }
        }
        mean[0] /= 5.0; mean[1] /= 5.0; mean[2] /= 5.0;        // utils::ComputePCA divides (superodom_utils.h:146): the eigenvalue gates below read this
        double S[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const float4 c = nbr(j);
            const double c0 = double(c.x) - mean[0], c1 = double(c.y) - mean[1], c2 = double(c.z) - mean[2];
            S[0] += c0 * c0; S[1] += c0 * c1; S[2] += c0 * c2; S[4] += c1 * c1; S[5] += c1 * c2; S[8] += c2 * c2;
        }
        S[3] = S[1]; S[6] = S[2]; S[7] = S[5];
        const double sxx = S[0], sxy = S[1], sxz = S[2], syy = S[4], syz = S[5], szz = S[8];
        // SelfAdjointEigenSolver<Matrix3d> (utils::ComputePCA, superodom_utils.h:150): eigenvalues by the closed form, the smallest
        // eigenvector from its eigenvalue, then the smallest eigenvalue once more as the Rayleigh quotient of that vector (full
        // double precision where the lambda0 < 1e-6 gate reads it)
        double ev[3], no[3];
#if SO_FIT_JACOBI
        jacobi_eig<3, 12, false>(S, nullptr, ev);
        eigvec3_from_value(sxx, sxy, sxz, syy, syz, szz, ev[0], no);
#else
        sym3_eigenvalues(sxx, sxy, sxz, syy, syz, szz, ev);
        eigvec3_from_value(sxx, sxy, sxz, syy, syz, szz, ev[0], no);
        ev[0] = no[0] * (sxx * no[0] + sxy * no[1] + sxz * no[2]) + no[1] * (sxy * no[0] + syy * no[1] + syz * no[2]) +
                no[2] * (sxz * no[0] + syz * no[1] + szz * no[2]);
        ev[1] = (sxx + syy + szz) - ev[0] - ev[2];
#endif
        if (ev[0] < 1e-6 || ev[1] / ev[2] < 0.1) status = SO_MATCH_BAD_PCA_STRUCTURE;      // the reference's quotient, literally (:772)
        else {
            // What FeatureObservabilityAnalysis (:574-693) needs from the PCA -- the oriented normal (:553-561) and the
            // planarity -- is reduced to four floats here, ahead of the register-hungry QR.
            float nf[3], cr[3], planar_sq;
            {
                if (pf[0] * no[0] + pf[1] * no[1] + pf[2] * no[2] < 0) { no[0] = -no[0]; no[1] = -no[1]; no[2] = -no[2]; }
                const double l1 = sqrt(ev[2]), l2 = sqrt(ev[1]), l3 = sqrt(ev[0]);
                const double planar_2 = (l2 - l3) / l1;
                planar_sq = float(planar_2 * planar_2);
                nf[0] = float(no[0]); nf[1] = float(no[1]); nf[2] = float(no[2]);
                cr[0] = __fmul_rn(qy, nf[2]) - __fmul_rn(qz, nf[1]);
                cr[1] = __fmul_rn(qz, nf[0]) - __fmul_rn(qx, nf[2]);
                cr[2] = __fmul_rn(qx, nf[1]) - __fmul_rn(qy, nf[0]);
            }
            // computePlaneQualityMetrics (:792-844)
            double x[3];
            {
                double A[5][3], b[5];
#pragma unroll
                for (int j = 0; j < 5; ++j) {
                    const float4 c = nbr(j);
                    A[j][0] = double(c.x); A[j][1] = double(c.y); A[j][2] = double(c.z); b[j] = -1.0;
                }
                colpiv_qr_solve_5x3(A, b, x);
            }
            if (!(isfinite(x[0]) && isfinite(x[1]) && isfinite(x[2]))) status = SO_MATCH_INVALID_NUMERICAL;
            else {
                // negative_OA_dot_norm = 1 / norm.norm(); norm.normalize()  (:812-816): square root and divisions as written there,
                // because the planeRes/2 gate below reads both
                const double nn = sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
                const double dd = 1.0 / nn;
                x[0] /= nn; x[1] /= nn; x[2] /= nn;
                const double maxd = double(m.plane_res) / 2.0;
                double msum = 0.0;
                bool ok = true;
#pragma unroll
                for (int j = 0; j < 5; ++j) {
                    const float4 c = nbr(j);
                    const double dist = fabs(x[0] * double(c.x) + x[1] * double(c.y) + x[2] * double(c.z) + dd);
                    if (ok && dist > maxd) ok = false;
                    msum += dist;
                }
                if (!ok) status = SO_MATCH_MSE_TOO_LARGE;
                else {
                    const double mean_dist = msum / 5.0;
                    const float fq[4] = {float(s_pose[3]), float(s_pose[4]), float(s_pose[5]), float(s_pose[6])};
                    float rotq[6], trq[3];
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
                        // computeRotatedAxes (:624-638): float quaternion * e_a, no FMA contraction (host code is plain IEEE)
                        const float v0 = a == 0 ? 1.f : 0.f, v1 = a == 1 ? 1.f : 0.f, v2 = a == 2 ? 1.f : 0.f;
                        float ux = __fsub_rn(__fmul_rn(fq[1], v2), __fmul_rn(fq[2], v1));
                        float uy = __fsub_rn(__fmul_rn(fq[2], v0), __fmul_rn(fq[0], v2));
                        float uz = __fsub_rn(__fmul_rn(fq[0], v1), __fmul_rn(fq[1], v0));
                        ux = __fadd_rn(ux, ux); uy = __fadd_rn(uy, uy); uz = __fadd_rn(uz, uz);
                        const float ax = __fadd_rn(__fadd_rn(v0, __fmul_rn(fq[3], ux)), __fsub_rn(__fmul_rn(fq[1], uz), __fmul_rn(fq[2], uy)));
                        const float ay = __fadd_rn(__fadd_rn(v1, __fmul_rn(fq[3], uy)), __fsub_rn(__fmul_rn(fq[2], ux), __fmul_rn(fq[0], uz)));
                        const float az = __fadd_rn(__fadd_rn(v2, __fmul_rn(fq[3], uz)), __fsub_rn(__fmul_rn(fq[0], uy), __fmul_rn(fq[1], ux)));
                        // Eigen's unrolled 3-vector dot associates as a0*b0 + (a1*b1 + a2*b2)
                        const float rc = __fadd_rn(__fmul_rn(cr[0], ax), __fadd_rn(__fmul_rn(cr[1], ay), __fmul_rn(cr[2], az)));
                        rotq[2 * a] = rc; rotq[2 * a + 1] = -rc;
                        const float dn = __fadd_rn(__fmul_rn(nf[0], ax), __fadd_rn(__fmul_rn(nf[1], ay), __fmul_rn(nf[2], az)));
                        trq[a] = __fmul_rn(planar_sq, fabsf(dn));
                    }
                    // top-2 rotation labels and top-1 translation label of a stable descending sort (:654-679).  The six rotation
                    // scores are {+rc_a, -rc_a}, a = 0..2, so the largest is +|rc_a| of the axis with the largest magnitude (first axis
                    // on ties, as the stable sort keeps index order; index 2a for rc_a >= 0, 2a+1 below) and the runner-up the same
                    // among the other two axes -- unless every score is zero (or the winner's is NaN), when index order decides: 0, 1.
                    const float m0 = fabsf(rotq[0]), m1 = fabsf(rotq[2]), m2 = fabsf(rotq[4]);
                    int a0 = 0; float mb = m0;
                    if (m1 > mb) { a0 = 1; mb = m1; }
                    if (m2 > mb) { a0 = 2; mb = m2; }
                    const int b0 = a0 == 0 ? 1 : 0, b1 = a0 == 2 ? 1 : 2;             // the other two axes, ascending
                    const float mb0 = a0 == 0 ? m1 : m0, mb1 = a0 == 2 ? m1 : m2;
                    const int a1 = mb1 > mb0 ? b1 : b0;
                    const int r0 = 2 * a0 + (rotq[2 * a0] < 0.f ? 1 : 0);
                    const int r1 = (mb > 0.f) ? 2 * a1 + (rotq[2 * a1] < 0.f ? 1 : 0) : 1;
                    int t0 = 0;
#pragma unroll
                    for (int q = 1; q < 3; ++q) if (trq[q] > trq[t0]) t0 = q;
                    o0 = r0; o1 = r1; o2 = 6 + t0;
                    nrm[0] = x[0]; nrm[1] = x[1]; nrm[2] = x[2]; dpl = dd;
                    wq = 1.0 - sqrt(mean_dist / double(m.bound_d2));     // fitQualityCoeff = 1 - sqrt(meanDist / (3*planeRes_)) (:568)
                    status = SO_MATCH_SUCCESS;
                }
            }
        }
    } else if (cb.nn) {
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const uint32_t pos = nb.pos[size_t(j) * nb.cap + gi];
            cb.nn[gi * 5 + j] = pos != 0xFFFFFFFFu ? __float_as_uint(__ldg(&m.pts[pos]).w) : 0xFFFFFFFFu;
            cb.nn_d2[gi * 5 + j] = 0.f;
        }
    }
    if (status != SO_MATCH_SKIPPED) {
        if (status == SO_MATCH_SUCCESS) { atomicAdd(&s_hist[o0], 1); atomicAdd(&s_hist[o1], 1); atomicAdd(&s_hist[o2], 1); }
        atomicAdd(&s_hist[9 + status], 1);
    }
    cb.nd[gi] = make_double4(nrm[0], nrm[1], nrm[2], dpl);
    cb.w[gi] = wq;
    cb.flags[gi] = make_uchar4((unsigned char)status, (unsigned char)o0, (unsigned char)o1, (unsigned char)o2);
}

__global__ void __launch_bounds__(kFitThreads, SO_FIT_MINB) k_fit(MapView m, BatchView bv, CorrBuf cb, NnBuf nb) {
    const int s = blockIdx.y;
    IcpState* st = bv.st + s;
    if (st->phase != PH_CORR) return;
    __shared__ double s_pose[7];
    __shared__ int s_hist[16];
    if (threadIdx.x < 7) s_pose[threadIdx.x] = st->x[threadIdx.x];
    if (threadIdx.x < 16) s_hist[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t n = uint32_t(st->n_points);
#pragma unroll 1
    for (int rr = 0; rr < kFitPts; ++rr) {          // kFitPts points per thread
        const uint32_t i = (blockIdx.x * kFitPts + rr) * kFitThreads + threadIdx.x;
        const size_t gi = size_t(bv.offset[s]) + i;
        if (i < n) {
            const float4* npts = nb.pts + gi;
            fit_point(m, cb, nb, gi, __ldg(&bv.scan[gi]), s_pose, int(nb.pre[gi]), [&](int j) { return ld_f4_again(npts + size_t(j) * nb.cap); }, s_hist);
        }
    }
    __syncthreads();
    if (threadIdx.x < 16 && s_hist[threadIdx.x]) atomicAdd(&bv.hist[s * kHistStride + threadIdx.x], s_hist[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------------------------
// k_knn_fit: k_knn_scan and k_fit for the same point in one thread.  Both halves fit 64 registers, so fusing costs no
// occupancy, and it (a) drops the 80 B/point neighbour hand-over through HBM (write + read back) and the second read of the
// scan, (b) removes a kernel boundary per ICP iteration, and (c) lets warps that are in the integer-heavy search and warps
// that are in the FP64-heavy fit share an SM, so both pipes stay busy.  The fit reads its neighbours straight from the
// search-ordered map at the positions the search just visited (L1/L2 hits).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 4) k_knn_fit(MapView m, BatchView bv, CorrBuf cb, NnBuf nb) {
    const int s = blockIdx.y;
    const IcpState* st = bv.st + s;
    if (st->phase != PH_CORR) return;
    __shared__ double s_pose[7];
    __shared__ int s_hist[16];
    __shared__ uint32_t s_buf[kBufCap * kThreads];
    if (threadIdx.x < 7) s_pose[threadIdx.x] = st->x[threadIdx.x];
    if (threadIdx.x < 16) s_hist[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t n = uint32_t(st->n_points);
    const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
    if (i < n) {
        const size_t gi = size_t(bv.offset[s]) + i;
        const float4 sp = __ldg(&bv.scan[gi]);
        int pre = SO_MATCH_SKIPPED;
        TopK<5> tk;
        tk.init(m.bound_d2);
        if (should_process(__float_as_uint(sp.w), st->sampling_rate)) {
            const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
            double pf[3];
            qrot(s_pose + 3, pin, pf);
            const float qx = float(pf[0] + s_pose[0]), qy = float(pf[1] + s_pose[1]), qz = float(pf[2] + s_pose[2]);
            QueryCell qc;
            locate(m, qx, qy, qz, qc);
            if (qc.slot < 0 || qc.nblock < 5) pre = SO_MATCH_NOT_ENOUGH_NEIGHBORS;
            else {
                float u_seed = -1.f;
                if (st->icp_iter > 0 && nb.pre[gi] == SO_MATCH_SUCCESS) u_seed = seed_bound(m, qc, nb, gi, qx, qy, qz);        // see k_knn_scan
                const GlobalGrid gg(m, qc.slot);
                knn_select<5, SO_R1_OCTANT != 0>(gg, m, qc, qx, qy, qz, u_seed, m.bound_d2, s_buf, tk);
                pre = tk.count() < 5 ? SO_MATCH_NEIGHBORS_TOO_FAR : SO_MATCH_SUCCESS;       // d2[4] > 3*planeRes_ (:741-744)
            }
        }
        nb.pre[gi] = (unsigned char)pre;
        nb.d5[gi] = tk.d2[4];
        uint32_t pos[5];
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            pos[j] = tk.id[j] != 0xFFFFFFFFu ? tk.pos[j] : 0xFFFFFFFFu;
            nb.pos[size_t(j) * nb.cap + gi] = pos[j];
        }
        fit_point(m, cb, nb, gi, sp, s_pose, pre, [&](int j) { return ld_f4_again(m.pts + pos[j]); }, s_hist);
    }
    __syncthreads();
    if (threadIdx.x < 16 && s_hist[threadIdx.x]) atomicAdd(&bv.hist[s * kHistStride + threadIdx.x], s_hist[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------------------------
// k_evaluate: robustified normal equations at the candidate pose over the stored correspondences.
// kEvalPts points per thread (strided by the CTA width, so loads stay coalesced) before the one warp/CTA reduction.
// ------------------------------------------------------------------------------------------------------------------
template <int PHASE>
__device__ __forceinline__ void evaluate_body(const BatchView& bv, const CorrBuf& cb, int s) {
    IcpState* st = bv.st + s;
    __shared__ double s_pose[7];
    __shared__ double s_R[9];
    // PH_EVAL: the LM candidate; PH_CORR: the first evaluation of a new solve, at the pose k_fit just matched at
    if (threadIdx.x < 7) s_pose[threadIdx.x] = PHASE == PH_EVAL ? st->cand[threadIdx.x] : st->x[threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) qtoR(s_pose + 3, s_R);
    __syncthreads();
    const uint32_t n = uint32_t(st->n_points);
    const size_t base = size_t(bv.offset[s]);
    double acc[kAcc];
#pragma unroll
    for (int k = 0; k < kAcc; ++k) acc[k] = 0.0;
    // Software-pipelined: the three loads of point r+1 are issued (unconditionally, so they do not chain behind the weight)
    // before the FP64 work of point r, which keeps two points' worth of the 56 B/pt stream in flight per thread.
    const int pts = eval_pts(n);
    if (blockIdx.x >= eval_ctas(n)) return;                // the grid covers the largest scan of the chunk
    const uint32_t i0 = blockIdx.x * uint32_t(pts) * kThreads + threadIdx.x;
    double w_n = 0.0;
    double4 nd_n = make_double4(0.0, 0.0, 0.0, 0.0);
    float4 sp_n = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i0 < n) {
        w_n = cb.w[base + i0];
        nd_n = cb.nd[base + i0];
        sp_n = __ldg(&bv.scan[base + i0]);
    }
#pragma unroll 1
    for (int r = 0; r < pts; ++r) {
        const double w = w_n;
        const double4 nd = nd_n;
        const float4 sp = sp_n;
        const uint32_t inext = i0 + (r + 1) * kThreads;
        w_n = 0.0;
        if (r + 1 < pts && inext < n) {
            w_n = cb.w[base + inext];
            nd_n = cb.nd[base + inext];
            sp_n = __ldg(&bv.scan[base + inext]);
        }
        if (w != 0.0) {
            const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
            double pw[3];
            qrot(s_pose + 3, pin, pw);
            pw[0] += s_pose[0]; pw[1] += s_pose[1]; pw[2] += s_pose[2];
            const double nn[3] = {nd.x, nd.y, nd.z};
            accumulate(acc, nn, nd.w, w, pin, pw, s_R, bv.tukey_a2);
        }
    }
    reduce_to_partials(acc, bv, s);
}

#ifndef SO_EVAL_TMA
#define SO_EVAL_TMA 1             // 0: k_evaluate streams its correspondences with per-thread loads (evaluate_body)
#endif
// The same evaluation with the 56 B/point stream staged by the TMA engine.  A CTA's points are eval_pts(n) consecutive tiles of
// kThreads points, and a tile is three contiguous spans (normals+offset 32 B/pt, scan point 16 B/pt, weight 8 B/pt): one elected
// thread enqueues three cp.async.bulk copies per tile into a kEvalStages-deep shared-memory ring, each stage completing on its
// own mbarrier; every thread then takes its own point from the stage (thread -> point mapping, arithmetic and reduction are
// those of evaluate_body: results are bit-identical).  kEvalStages tiles (42 KB) are in flight per CTA whatever the threads are
// doing, instead of the one software-prefetched point per thread that 124 registers x 2 CTAs per SM leave room for.
// Falls back to generic loads for the ragged last tile of a scan and for scans whose first point is at an odd offset (the 8 B
// weights of a tile must start 16 B-aligned for the bulk copy).
constexpr int kEvalStages = 3;
struct __align__(128) EvalStage { double4 nd[kThreads]; float4 sp[kThreads]; double w[kThreads]; };
constexpr uint32_t kEvalStageBytes = uint32_t(sizeof(double4) + sizeof(float4) + sizeof(double)) * kThreads;

template <int PHASE>
__device__ __forceinline__ void evaluate_body_tma(const BatchView& bv, const CorrBuf& cb, int s) {
    IcpState* st = bv.st + s;
    __shared__ double s_pose[7];
    __shared__ double s_R[9];
    __shared__ EvalStage s_stage[kEvalStages];
    __shared__ unsigned long long s_bar[kEvalStages];
    const uint32_t n = uint32_t(st->n_points);
    const int pts = eval_pts(n);
    if (blockIdx.x >= eval_ctas(n)) return;                // the grid covers the largest scan of the chunk
    if (threadIdx.x < 7) s_pose[threadIdx.x] = PHASE == PH_EVAL ? st->cand[threadIdx.x] : st->x[threadIdx.x];
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < kEvalStages; ++k) mbar_init(&s_bar[k], 1);
    }
    __syncthreads();
    const size_t base = size_t(bv.offset[s]);
    const uint32_t cta0 = blockIdx.x * uint32_t(pts) * kThreads;
    // tiles [0, full) of this CTA are complete (kThreads points each); tile `full` may be ragged, later ones are empty
    const int full = (base & 1) ? 0 : int(min(uint32_t(pts), (n - min(n, cta0)) / kThreads));
    auto issue = [&](int r) {                              // thread 0 only
        EvalStage& sg = s_stage[r % kEvalStages];
        unsigned long long* bar = &s_bar[r % kEvalStages];
        const size_t g = base + cta0 + size_t(r) * kThreads;
        mbar_arrive_expect_tx(bar, kEvalStageBytes);
        bulk_copy_g2s(sg.nd, cb.nd + g, uint32_t(sizeof(double4)) * kThreads, bar);
        bulk_copy_g2s(sg.sp, bv.scan + g, uint32_t(sizeof(float4)) * kThreads, bar);
        bulk_copy_g2s(sg.w, cb.w + g, uint32_t(sizeof(double)) * kThreads, bar);
    };
    if (threadIdx.x == 0) {
        for (int r = 0; r < kEvalStages && r < full; ++r) issue(r);
        qtoR(s_pose + 3, s_R);
    }
    __syncthreads();
    double acc[kAcc];
#pragma unroll
    for (int k = 0; k < kAcc; ++k) acc[k] = 0.0;
#pragma unroll 1
    for (int r = 0; r < pts; ++r) {
        const uint32_t i = cta0 + uint32_t(r) * kThreads + threadIdx.x;
        double w = 0.0;
        double4 nd = make_double4(0.0, 0.0, 0.0, 0.0);
        float4 sp = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < full) {                                    // CTA-uniform
            const EvalStage& sg = s_stage[r % kEvalStages];
            mbar_wait(&s_bar[r % kEvalStages], uint32_t(r / kEvalStages) & 1u);
            w = sg.w[threadIdx.x];
            nd = sg.nd[threadIdx.x];
            sp = sg.sp[threadIdx.x];
            __syncthreads();                               // every thread holds its point: the stage may be refilled
            if (threadIdx.x == 0 && r + kEvalStages < full) issue(r + kEvalStages);
        } else {
            if (cta0 + uint32_t(r) * kThreads >= n) break;
            if (i < n) {
                w = cb.w[base + i];
                nd = cb.nd[base + i];
                sp = __ldg(&bv.scan[base + i]);
            }
        }
        if (w != 0.0) {
            const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
            double pw[3];
            qrot(s_pose + 3, pin, pw);
            pw[0] += s_pose[0]; pw[1] += s_pose[1]; pw[2] += s_pose[2];
            const double nn[3] = {nd.x, nd.y, nd.z};
            accumulate(acc, nn, nd.w, w, pin, pw, s_R, bv.tukey_a2);
        }
    }
    reduce_to_partials(acc, bv, s);
}

template <int PHASE>
__global__ void __launch_bounds__(kThreads, 2) k_evaluate(BatchView bv, CorrBuf cb) {
    const int s = blockIdx.y;
    if (bv.st[s].phase != PHASE) return;
#if SO_EVAL_TMA
    evaluate_body_tma<PHASE>(bv, cb, s);
#else
    evaluate_body<PHASE>(bv, cb, s);
#endif
}

// ------------------------------------------------------------------------------------------------------------------
// Edge / line branch (a19; dormant upstream because featureExtraction emits an empty edge cloud, featureExtraction.cpp:429-436).
// k_edge_fit: LidarSLAM::ComputeLineDistanceParameters (LidarSlam.cpp:402-435) for every edge point -- exact 10-NN in the
// point's block of the EDGE map, LocalMap::nearestKSearchSpecificEdgePoint's best-line-by-inliers selection in float
// (LocalMap.h:377-474), PCA of the selected points, the line gates and processLineResults (:438-493) -- plus the first
// evaluation of EdgeAnalyticCostFunction (lidarOptimization.cpp:12-47) for the following solve.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void accumulate_edge(double acc[kAcc], const double a[3], const double b[3], double w, const double p[3],
                                                const double lp[3], const double R[9], double a2_line) {
    const double u[3] = {lp[0] - a[0], lp[1] - a[1], lp[2] - a[2]}, v[3] = {lp[0] - b[0], lp[1] - b[1], lp[2] - b[2]};
    const double de[3] = {a[0] - b[0], a[1] - b[1], a[2] - b[2]};
    const double den = sqrt(de[0] * de[0] + de[1] * de[1] + de[2] * de[2]);
    const double r[3] = {(u[1] * v[2] - u[2] * v[1]) / den, (u[2] * v[0] - u[0] * v[2]) / den, (u[0] * v[1] - u[1] * v[0]) / den};
    const double s = r[0] * r[0] + r[1] * r[1] + r[2] * r[2];
    double rho0, rho1;
    if (s <= a2_line) { const double t = 1.0 - s / a2_line, t2 = t * t; rho0 = a2_line / 6.0 * (1.0 - t2 * t); rho1 = 0.5 * t2; }
    else { rho0 = a2_line / 6.0; rho1 = 0.0; }
    rho0 *= w; rho1 *= w;
    // J = skew(b - a) [I, -R [p]x] / |a - b|
    const double re[3] = {-de[0], -de[1], -de[2]};
    const double K[9] = {0, -re[2], re[1], re[2], 0, -re[0], -re[1], re[0], 0};
    const double Sp[9] = {0, -p[2], p[1], p[2], 0, -p[0], -p[1], p[0], 0};
    double J[18];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) {
        J[i * 6 + j] = K[i * 3 + j] / den;
        double t = 0.0;
        for (int k = 0; k < 3; ++k) { double rs = 0.0; for (int l = 0; l < 3; ++l) rs += R[k * 3 + l] * Sp[l * 3 + j]; t += K[i * 3 + k] * (-rs); }
        J[i * 6 + 3 + j] = t / den;
    }
    int kk = 0;
    for (int i = 0; i < 6; ++i) for (int j = i; j < 6; ++j) { acc[kk++] += rho1 * (J[i] * J[j] + J[6 + i] * J[6 + j] + J[12 + i] * J[12 + j]); }
    for (int i = 0; i < 6; ++i) acc[21 + i] += rho1 * (J[i] * r[0] + J[6 + i] * r[1] + J[12 + i] * r[2]);
    acc[27] += 0.5 * rho0;
}

__global__ void __launch_bounds__(kThreads) k_edge_fit(MapView m, BatchView bv, EdgeBuf eb, uint32_t partial_offset) {
    const int s = blockIdx.y;
    IcpState* st = bv.st + s;
    if (st->phase != PH_CORR || st->n_edge == 0) return;
    __shared__ double s_pose[7];
    __shared__ double s_R[9];
    __shared__ int s_hist[8];
    __shared__ uint32_t s_buf[kBufCap * kThreads];
    if (threadIdx.x < 7) s_pose[threadIdx.x] = st->x[threadIdx.x];
    if (threadIdx.x < 8) s_hist[threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x == 0) qtoR(s_pose + 3, s_R);
    __syncthreads();
    const uint32_t n = uint32_t(st->n_edge);
    const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
    double acc[kAcc];
#pragma unroll
    for (int k = 0; k < kAcc; ++k) acc[k] = 0.0;
    if (i < n) {
        const size_t gi = size_t(eb.offset[s]) + i;
        const float4 sp = __ldg(&eb.scan[gi]);
        const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
        double pf[3];
        qrot(s_pose + 3, pin, pf);
        pf[0] += s_pose[0]; pf[1] += s_pose[1]; pf[2] += s_pose[2];
        const float qx = float(pf[0]), qy = float(pf[1]), qz = float(pf[2]);
        int status = SO_MATCH_NOT_ENOUGH_NEIGHBORS;
        double ea[3] = {0, 0, 0}, ebb[3] = {0, 0, 0}, wq = 0.0;
        int nsel = 0;
        uint32_t selmask = 0;
        TopK<10> tk;
        tk.init(FLT_MAX);
        QueryCell qc;
        locate(m, qx, qy, qz, qc);
        // "<10 points in the block": the reference indexes with size_t(-1) (LocalMap.h:404-419); treated as NOT_ENOUGH_NEIGHBORS
        if (qc.slot >= 0 && qc.nblock >= 10) {
            knn_search<10>(GlobalGrid(m, qc.slot), m, qc, qx, qy, qz, 0.f, s_buf, tk);
            float P[10][3];
#pragma unroll
            for (int j = 0; j < 10; ++j) { const float4 c = __ldg(&m.pts[tk.pos[j]]); P[j][0] = c.x; P[j][1] = c.y; P[j][2] = c.z; }
            // best line through the closest point by inlier count: float arithmetic in Eigen's evaluation order, no FMA contraction
            const float thr = __fmul_rn(0.2f, 0.2f);
            int best_n = 0;
            for (int pi = 1; pi < 10; ++pi) {
                float dx = __fsub_rn(P[pi][0], P[0][0]), dy = __fsub_rn(P[pi][1], P[0][1]), dz = __fsub_rn(P[pi][2], P[0][2]);
                const float z2 = __fadd_rn(__fmul_rn(dx, dx), __fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dz, dz)));
                if (z2 > 0.f) { const float sq = __fsqrt_rn(z2); dx = __fdiv_rn(dx, sq); dy = __fdiv_rn(dy, sq); dz = __fdiv_rn(dz, sq); }
                uint32_t mask = 0; int cnt = 0;
                for (int ci = 1; ci < 10; ++ci) {
                    bool ok;
                    if (ci == pi) ok = true;
                    else {
                        const float vx = __fsub_rn(P[ci][0], P[0][0]), vy = __fsub_rn(P[ci][1], P[0][1]), vz = __fsub_rn(P[ci][2], P[0][2]);
                        const float cx = __fsub_rn(__fmul_rn(vy, dz), __fmul_rn(vz, dy)), cy = __fsub_rn(__fmul_rn(vz, dx), __fmul_rn(vx, dz)),
                                    cz = __fsub_rn(__fmul_rn(vx, dy), __fmul_rn(vy, dx));
                        ok = __fadd_rn(__fmul_rn(cx, cx), __fadd_rn(__fmul_rn(cy, cy), __fmul_rn(cz, cz))) < thr;
                    }
                    if (ok) { mask |= 1u << ci; ++cnt; }
                }
                if (cnt > best_n) { best_n = cnt; selmask = mask; }
            }
            selmask |= 1u;                                               // the closest point is always kept, first
            nsel = __popc(selmask);
            const int last = 31 - __clz(selmask);
            if (nsel < 4) status = SO_MATCH_NOT_ENOUGH_NEIGHBORS;                                 // validateNeighborSearch (:495-512)
            else if (tk.d2[last] > __fmul_rn(3.f, m.plane_res)) status = SO_MATCH_NEIGHBORS_TOO_FAR;   // MapView::plane_res holds lineRes_ for the edge map
            else {
                // PCA of the selected points (computePCAForFeature, EdgeFeature branch, :749-790)
                double mean[3] = {0, 0, 0};
                for (int j = 0; j < 10; ++j) if (selmask >> j & 1) { mean[0] += double(P[j][0]); mean[1] += double(P[j][1]); mean[2] += double(P[j][2]); }
                mean[0] /= double(nsel); mean[1] /= double(nsel); mean[2] /= double(nsel);
                double S[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
                for (int j = 0; j < 10; ++j) if (selmask >> j & 1) {
                    const double c0 = double(P[j][0]) - mean[0], c1 = double(P[j][1]) - mean[1], c2 = double(P[j][2]) - mean[2];
                    S[0] += c0 * c0; S[1] += c0 * c1; S[2] += c0 * c2; S[4] += c1 * c1; S[5] += c1 * c2; S[8] += c2 * c2;
                }
                S[3] = S[1]; S[6] = S[2]; S[7] = S[5];
                double V[9], ev[3];
                jacobi_eig<3, 12>(S, V, ev);
                if (!(isfinite(ev[0]) && isfinite(ev[1]) && isfinite(ev[2]))) status = SO_MATCH_INVALID_NUMERICAL;
                else if (ev[2] < 4.0 * ev[1]) status = SO_MATCH_BAD_PCA_STRUCTURE;
                else {
                    double dir[3] = {V[2], V[5], V[8]};                     // processLineResults (:438-493)
                    const double dn = sqrt(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
                    dir[0] /= dn; dir[1] /= dn; dir[2] /= dn;
                    const double lim = double(__fmul_rn(3.f, m.plane_res));
                    double msd = 0.0;
                    bool ok = isfinite(dir[0]) && isfinite(dir[1]) && isfinite(dir[2]);
                    if (!ok) status = SO_MATCH_INVALID_NUMERICAL;
                    else {
                        for (int j = 0; j < 10; ++j) if (selmask >> j & 1) {
                            const double c[3] = {double(P[j][0]) - mean[0], double(P[j][1]) - mean[1], double(P[j][2]) - mean[2]};
                            double sd = 0.0;
                            for (int a2 = 0; a2 < 3; ++a2) {
                                double Ac = 0.0;
                                for (int b2 = 0; b2 < 3; ++b2) Ac += ((a2 == b2 ? 1.0 : 0.0) - dir[a2] * dir[b2]) * c[b2];
                                sd += c[a2] * Ac;
                            }
                            if (ok && sd > lim) ok = false;
                            msd += sd;
                        }
                        if (!ok) status = SO_MATCH_MSE_TOO_LARGE;
                        else {
                            msd /= double(nsel);
                            wq = 1.0 - sqrt(msd / lim);
                            for (int a2 = 0; a2 < 3; ++a2) { ea[a2] = 0.1 * dir[a2] + mean[a2]; ebb[a2] = -0.1 * dir[a2] + mean[a2]; }
                            status = SO_MATCH_SUCCESS;
                            accumulate_edge(acc, ea, ebb, wq, pin, pf, s_R, bv.tukey_a2_line);
                        }
                    }
                }
            }
        }
        atomicAdd(&s_hist[status], 1);
        eb.a[gi] = make_double4(ea[0], ea[1], ea[2], wq);
        eb.b[gi] = make_double4(ebb[0], ebb[1], ebb[2], 0.0);
        eb.flags[gi] = make_uchar4((unsigned char)status, (unsigned char)nsel, 0, 0);
        if (eb.nn) {
#pragma unroll
            for (int j = 0; j < 10; ++j) eb.nn[gi * 10 + j] = tk.id[j];
            eb.selmask[gi] = selmask;
        }
    }
    __syncthreads();
    if (threadIdx.x < 7 && s_hist[threadIdx.x]) atomicAdd(&bv.hist[s * kHistStride + 16 + threadIdx.x], s_hist[threadIdx.x]);
    reduce_to_partials(acc, bv, s, partial_offset);
}

__global__ void __launch_bounds__(kThreads) k_edge_evaluate(BatchView bv, EdgeBuf eb, uint32_t partial_offset) {
    const int s = blockIdx.y;
    IcpState* st = bv.st + s;
    if (st->phase != PH_EVAL || st->n_edge == 0) return;
    __shared__ double s_pose[7];
    __shared__ double s_R[9];
    if (threadIdx.x < 7) s_pose[threadIdx.x] = st->cand[threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) qtoR(s_pose + 3, s_R);
    __syncthreads();
    const uint32_t n = uint32_t(st->n_edge);
    const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
    double acc[kAcc];
#pragma unroll
    for (int k = 0; k < kAcc; ++k) acc[k] = 0.0;
    if (i < n) {
        const size_t gi = size_t(eb.offset[s]) + i;
        const double4 a = eb.a[gi];
        if (a.w != 0.0) {
            const double4 b = eb.b[gi];
            const float4 sp = __ldg(&eb.scan[gi]);
            const double pin[3] = {double(sp.x), double(sp.y), double(sp.z)};
            double lp[3];
            qrot(s_pose + 3, pin, lp);
            lp[0] += s_pose[0]; lp[1] += s_pose[1]; lp[2] += s_pose[2];
            const double aa[3] = {a.x, a.y, a.z}, bb[3] = {b.x, b.y, b.z};
            accumulate_edge(acc, aa, bb, a.w, pin, lp, s_R, bv.tukey_a2_line);
        }
    }
    reduce_to_partials(acc, bv, s, partial_offset);
}

// ------------------------------------------------------------------------------------------------------------------
// k_lm_step: one CTA per scan.  Sums the per-CTA partials of the preceding k_fit (AFTER == PH_CORR) or k_evaluate
// (AFTER == PH_EVAL) in a fixed order, then one thread advances the optimiser / ICP state machine.
// ------------------------------------------------------------------------------------------------------------------
// Called by >= 128 threads of one CTA (all of them: it synchronises the CTA); the first 128 do the work.
template <int AFTER>
__device__ __forceinline__ void lm_step_body(const BatchView& bv, int s, uint32_t n_partials, uint32_t edge_partial_offset) {
    IcpState* st = bv.st + s;
    __shared__ double s_red[4][kAcc];
    __shared__ double s_sum[kAcc];
    const int comp = threadIdx.x & 31, sub = threadIdx.x >> 5;
    double v = 0.0;
    if (comp < kAcc && sub < 4) {
        const double* base = bv.partials + size_t(s) * bv.partial_stride * kAcc;
        const uint32_t np = eval_ctas(uint32_t(st->n_points));
        // __ldcg: straight from L2 -- in k_evaluate_lm the rows were written by other CTAs of the same launch
        for (uint32_t b = sub; b < np && b < n_partials; b += 4) v += __ldcg(&base[size_t(b) * kAcc + comp]);
        const uint32_t ne = (uint32_t(st->n_edge) + kThreads - 1) / kThreads;          // edge branch partials (0 when no edge cloud)
        for (uint32_t b = sub; b < ne; b += 4) v += __ldcg(&base[size_t(edge_partial_offset + b) * kAcc + comp]);
        s_red[sub][comp] = v;
    }
    // The serial step works on a SHARED-MEMORY copy of the scan's state: through the global pointer every field access of the
    // one working thread was a dependent L2 round trip (the step took 5-12 us, the covariance 40 us); the copy in and out is two
    // coalesced passes of the CTA.
    __shared__ IcpState s_st;
    static_assert(sizeof(IcpState) % 8 == 0, "copied as 8-byte words");
    {
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(st);
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(&s_st);
        for (uint32_t k = threadIdx.x; k < sizeof(IcpState) / 8; k += blockDim.x) dst[k] = src[k];
    }
    __syncthreads();
    if (threadIdx.x < kAcc) s_sum[threadIdx.x] = (s_red[0][threadIdx.x] + s_red[1][threadIdx.x]) + (s_red[2][threadIdx.x] + s_red[3][threadIdx.x]);
    __syncthreads();
    if (threadIdx.x == 0) {
        IcpState& S = s_st;
        if (AFTER == PH_CORR) {
            // histograms of this ICP iteration (ResetDistanceParameters + processPlannerFeatures, :847-852,:336-341)
            for (int k = 0; k < 9; ++k) S.hist_obs[k] = bv.hist[s * kHistStride + k];
            for (int k = 0; k < 7; ++k) S.hist_rej[k] = bv.hist[s * kHistStride + 9 + k];
            for (int k = 0; k < 7; ++k) S.hist_rej_line[k] = bv.hist[s * kHistStride + 16 + k];
            S.n_ok_edge = S.hist_rej_line[0];
            const int n_ok = S.hist_rej[0] + S.n_ok_edge;       // features_corres.size(): edges + planes
            for (int k = 0; k < kHistStride; ++k) bv.hist[s * kHistStride + k] = 0;
            if (S.max_icp_iters < 0) {          // stage mode (so_correspond): stop here
                for (int k = 0; k < 21; ++k) S.H[k] = s_sum[k];
                for (int k = 0; k < 6; ++k) S.g[k] = s_sum[21 + k];
                S.cost = s_sum[27]; S.n_ok = n_ok; S.phase = PH_DONE;
            } else lm_begin_solve(S, s_sum, n_ok);
        } else {
            if (S.max_icp_iters < 0) {          // stage mode (so_evaluate): report and stop
                for (int k = 0; k < 21; ++k) S.H[k] = s_sum[k];
                for (int k = 0; k < 6; ++k) S.g[k] = s_sum[21 + k];
                S.cost = s_sum[27]; S.phase = PH_DONE;
            } else lm_after_eval(S, s_sum);
        }
    }
    __syncthreads();
    if (s_st.need_cov) {                                   // the registration just ended (CTA-uniform)
        __shared__ CovScratch s_cov;
        if (threadIdx.x < 32) covariance_and_errors_warp(s_st, s_cov);      // need_cov stays set: the state is re-initialised per registration
        __syncthreads();
    }
    {
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&s_st);
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(st);
        for (uint32_t k = threadIdx.x; k < sizeof(IcpState) / 8; k += blockDim.x) dst[k] = src[k];
    }
}

template <int AFTER>
__global__ void __launch_bounds__(128) k_lm_step(BatchView bv, uint32_t n_partials, uint32_t edge_partial_offset) {
    const int s = blockIdx.x;
    if (bv.st[s].phase != AFTER) return;
    lm_step_body<AFTER>(bv, s, n_partials, edge_partial_offset);
}


// ------------------------------------------------------------------------------------------------------------------
// k_evaluate_lm: k_evaluate with the optimiser step of k_lm_step folded in -- the CTA that finishes LAST (ticket counter, after a
// device-scope fence) sums the partial rows in their fixed order and advances the state machine.  Same arithmetic in the same
// order as the two-kernel form, one launch less per cost evaluation: used when a registration is launch-latency bound (one or
// two scans in flight, no edge cloud), where the ~190 registers of the serial step cost no occupancy that matters.
// ------------------------------------------------------------------------------------------------------------------
template <int PHASE>
__global__ void __launch_bounds__(kThreads, 1) k_evaluate_lm(BatchView bv, CorrBuf cb, uint32_t* __restrict__ counters) {
    const int s = blockIdx.y;
    if (bv.st[s].phase != PHASE) return;
    evaluate_body<PHASE>(bv, cb, s);
    __shared__ uint32_t s_ticket;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(&counters[s], 1u);
    __syncthreads();
    if (s_ticket != gridDim.x - 1) return;
    if (threadIdx.x == 0) counters[s] = 0;               // ready for the next launch
    __threadfence();
    lm_step_body<PHASE>(bv, s, gridDim.x, bv.edge_partial_offset);
}

// Loop condition of the CUDA-graph WHILE node that wraps one ICP iteration: keep iterating while any scan of the
// batch is still registering (LidarSlam.cpp:119-148 runs this loop on the host, one scan at a time).
__global__ void k_loop_cond(const IcpState* __restrict__ st, uint32_t n_scans, cudaGraphConditionalHandle handle) {
    int active = 0;
    for (uint32_t s = threadIdx.x; s < n_scans; s += 32) active |= (st[s].phase != PH_DONE);
    active = __any_sync(0xffffffffu, active);
    if (threadIdx.x == 0) cudaGraphSetConditional(handle, active ? 1u : 0u);
}

// ------------------------------------------------------------------------------------------------------------------
// k_knn: LocalMap::nearestKSearchSurf for a batch of world-frame queries (so_knn / so_knn_device)
// ------------------------------------------------------------------------------------------------------------------
// brick-order key of every query (so_knn* orders large query sets first, for the same reason scans are ordered)
__global__ void __launch_bounds__(kThreads) k_query_keys(MapView m, const float4* __restrict__ q, size_t nq, uint32_t* __restrict__ keys,
                                                         uint32_t* __restrict__ vals) {
    const size_t i = size_t(blockIdx.x) * kThreads + threadIdx.x;
    if (i >= nq) return;
    const float4 p = __ldg(&q[i]);
    QueryCell qc;
    locate(m, p.x, p.y, p.z, qc);
    keys[i] = qc.slot >= 0 ? scan_order_key(m, qc) : 0xFFFFFFFFu;
    vals[i] = uint32_t(i);
}

// 128 queries per CTA.  ORDERED: the queries arrive in brick order (`order`), so the CTA first tries the shared candidate tile.
template <int K, bool ORDERED>
__global__ void __launch_bounds__(kTileThreads) k_knn(MapView m, const float4* __restrict__ q, const uint32_t* __restrict__ order, size_t nq,
                                                      float max_d2, uint32_t* __restrict__ idx, float* __restrict__ d2) {
    __shared__ uint32_t s_buf[kBufCap * kTileThreads];
#if SO_KNN_TILE
    __shared__ TileSmem s_tile;
#endif
    const size_t j0 = size_t(blockIdx.x) * kTileThreads;
    if (j0 >= nq) return;
    const size_t j = j0 + threadIdx.x;
    const bool in_range = j < nq;
    const size_t i = in_range ? (order ? size_t(order[j]) : j) : 0;        // thread j handles the j-th query in brick order, answers in caller order
    const float4 p = __ldg(&q[i]);
    TopK<K> tk;
    tk.init(max_d2 > 0.f ? max_d2 : FLT_MAX);
    QueryCell qc;
    qc.slot = -1; qc.nblock = 0; qc.c[0] = qc.c[1] = qc.c[2] = 0; qc.f[0] = qc.f[1] = qc.f[2] = 0.f;
    if (in_range) locate(m, p.x, p.y, p.z, qc);
    const bool searchable = in_range && qc.slot >= 0;
#if SO_KNN_TILE
    TileGrid tg;
    const bool tiled = ORDERED && build_tile(m, s_tile, searchable, qc, tg);        // every thread takes part in the build
#endif
    if (searchable) {
#if SO_KNN_TILE
        if (tiled) knn_search<K>(tg, m, qc, p.x, p.y, p.z, max_d2, s_buf, tk);
        else
#endif
            knn_search<K>(GlobalGrid(m, qc.slot), m, qc, p.x, p.y, p.z, max_d2, s_buf, tk);
    }
    if (!in_range) return;
#pragma unroll
    for (int jj = 0; jj < K; ++jj) {
        const bool ok = tk.id[jj] != 0xFFFFFFFFu;
        idx[i * K + jj] = tk.id[jj];
        d2[i * K + jj] = ok ? tk.d2[jj] : 0.f;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Replay plumbing (SURVEY 8e, K8): one row of 8 doubles per scan -- the optimiser's pose {tx,ty,tz,qx,qy,qz,qw} (so_icp_result.pose_opt)
// and status + 256 * n_iterations -- into a caller-owned device buffer, so that the NCCL gather of a sharded replay reads device
// memory on the compute stream instead of waiting for a host round trip.
__global__ void k_pack_poses(const IcpState* __restrict__ st, uint32_t n_scans, double* __restrict__ rows) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_scans) return;
#pragma unroll
    for (int k = 0; k < 7; ++k) rows[size_t(s) * 8 + k] = st[s].x[k];
    rows[size_t(s) * 8 + 7] = double(st[s].status + 256 * st[s].n_iterations);
}

// ------------------------------------------------------------------------------------------------------------------
// host-side launchers
// ------------------------------------------------------------------------------------------------------------------
// keys: the 64-bit key buffer; with key32 it is used as an array of uint32_t (same point indexing)
void launch_scan_keys(const MapView& m, const BatchView& bv, uint64_t* keys, uint32_t* vals, uint32_t grid_x, uint32_t n_scans, int cell_bits, bool key32,
                      bool compact, cudaStream_t st) {
    const dim3 g(grid_x, n_scans);
    uint32_t* k32 = reinterpret_cast<uint32_t*>(keys);
    if (key32) { if (compact) k_scan_keys<uint32_t, true><<<g, kThreads, 0, st>>>(m, bv, k32, vals, cell_bits); else k_scan_keys<uint32_t, false><<<g, kThreads, 0, st>>>(m, bv, k32, vals, cell_bits); }
    else { if (compact) k_scan_keys<uint64_t, true><<<g, kThreads, 0, st>>>(m, bv, keys, vals, cell_bits); else k_scan_keys<uint64_t, false><<<g, kThreads, 0, st>>>(m, bv, keys, vals, cell_bits); }
}
void launch_scan_finish(const BatchView& bv, const uint64_t* sorted_keys, size_t first, uint32_t pt_first, int cell_bits, bool key32, uint32_t n_scans, cudaStream_t st) {
    if (key32) k_scan_finish<uint32_t><<<(n_scans + 63) / 64, 64, 0, st>>>(bv, reinterpret_cast<const uint32_t*>(sorted_keys) + first, pt_first, cell_bits, n_scans);
    else k_scan_finish<uint64_t><<<(n_scans + 63) / 64, 64, 0, st>>>(bv, sorted_keys + first, pt_first, cell_bits, n_scans);
}
void launch_prepare_small(const MapView& m, const BatchView& bv, float4* out, uint32_t n_scans, int key_bits, uint32_t max_kept, cudaStream_t st) {
    if (max_kept <= 2u * kSmallThreads) k_prepare_small<2><<<n_scans, kSmallThreads, 0, st>>>(m, bv, out, key_bits);
    else k_prepare_small<4><<<n_scans, kSmallThreads, 0, st>>>(m, bv, out, key_bits);
}
void launch_scan_gather(const float4* in, const uint32_t* vals, const uint64_t* keys, size_t first, const uint32_t* offset, size_t total, float4* out,
                        int cell_bits, bool key32, cudaStream_t st) {
    const uint32_t grid = uint32_t((total + kThreads - 1) / kThreads);
    if (key32) k_scan_gather<uint32_t><<<grid, kThreads, 0, st>>>(in, vals + first, reinterpret_cast<const uint32_t*>(keys) + first, offset, total, out, cell_bits);
    else k_scan_gather<uint64_t><<<grid, kThreads, 0, st>>>(in, vals + first, keys + first, offset, total, out, cell_bits);
}
// Correspondence stage of one ICP iteration = launch_match (search + fit of every scan point) + launch_first_eval (first
// evaluation of the new solve, the edge kernel when an edge cloud is present, and the optimiser's iteration zero).
// medge / eb / grid_e: edge branch (grid_e == 0: idle); k_lm_step sums the partials of both branches.
void launch_match(const MapView& m, const BatchView& bv, const CorrBuf& cb, const NnBuf& nb, uint32_t grid_x, uint32_t n_scans, cudaStream_t st, int part) {
    if (!grid_x) return;
#if SO_FUSE_KNN_FIT
    (void)part;
    k_knn_fit<<<dim3(grid_x, n_scans), kThreads, 0, st>>>(m, bv, cb, nb);
#else
    if (part != 2) {
        if (bv.coop_knn) k_knn_scan_coop<<<dim3(grid_x * (kThreads / kCoopWarps), n_scans), kThreads, 0, st>>>(m, bv, nb);
        else k_knn_scan<<<dim3(grid_x * (kThreads / kTileThreads), n_scans), kTileThreads, 0, st>>>(m, bv, nb);
    }
    const uint32_t gf = (grid_x * kThreads + kFitPts * kFitThreads - 1) / (kFitPts * kFitThreads);
    if (part != 1) k_fit<<<dim3(gf, n_scans), kFitThreads, 0, st>>>(m, bv, cb, nb);
#endif
}
void launch_inject(const MapView& m, const float4* by_id, uint32_t n_map, const BatchView& bv, const NnBuf& nb, const uint32_t* ids, int n_trace_iters,
                   uint32_t grid_x, uint32_t n_scans, cudaStream_t st) {
    if (grid_x) k_knn_inject<<<dim3(grid_x, n_scans), kThreads, 0, st>>>(m, by_id, n_map, bv, nb, ids, n_trace_iters);
}
void launch_first_eval(const BatchView& bv, const CorrBuf& cb, uint32_t grid_x, uint32_t n_scans, cudaStream_t st, const MapView* medge, const EdgeBuf* eb,
                       uint32_t grid_e) {
    const uint32_t gp = grid_x ? eval_grid(grid_x * kThreads) : 0;
    if (bv.counters && gp && !grid_e) { k_evaluate_lm<PH_CORR><<<dim3(gp, n_scans), kThreads, 0, st>>>(bv, cb, bv.counters); return; }
    if (gp) k_evaluate<PH_CORR><<<dim3(gp, n_scans), kThreads, 0, st>>>(bv, cb);
    if (grid_e) k_edge_fit<<<dim3(grid_e, n_scans), kThreads, 0, st>>>(*medge, bv, *eb, bv.edge_partial_offset);
    k_lm_step<PH_CORR><<<n_scans, 128, 0, st>>>(bv, gp, bv.edge_partial_offset);
}
void launch_correspond(const MapView& m, const BatchView& bv, const CorrBuf& cb, const NnBuf& nb, uint32_t grid_x, uint32_t n_scans, cudaStream_t st,
                       const MapView* medge, const EdgeBuf* eb, uint32_t grid_e) {
    launch_match(m, bv, cb, nb, grid_x, n_scans, st);
    launch_first_eval(bv, cb, grid_x, n_scans, st, medge, eb, grid_e);
}
void launch_evaluate(const BatchView& bv, const CorrBuf& cb, uint32_t grid_x, uint32_t n_scans, cudaStream_t st, const EdgeBuf* eb, uint32_t grid_e) {
    const uint32_t gx = grid_x ? eval_grid(grid_x * kThreads) : 0;
    if (bv.counters && gx && !grid_e) { k_evaluate_lm<PH_EVAL><<<dim3(gx, n_scans), kThreads, 0, st>>>(bv, cb, bv.counters); return; }
    if (gx) k_evaluate<PH_EVAL><<<dim3(gx, n_scans), kThreads, 0, st>>>(bv, cb);
    if (grid_e) k_edge_evaluate<<<dim3(grid_e, n_scans), kThreads, 0, st>>>(bv, *eb, bv.edge_partial_offset);
    k_lm_step<PH_EVAL><<<n_scans, 128, 0, st>>>(bv, gx, bv.edge_partial_offset);
}
void launch_loop_cond(const BatchView& bv, uint32_t n_scans, cudaGraphConditionalHandle handle, cudaStream_t st) {
    k_loop_cond<<<1, 32, 0, st>>>(bv.st, n_scans, handle);
}
void launch_pack_poses(const IcpState* st, uint32_t n_scans, double* rows, cudaStream_t stream) {
    k_pack_poses<<<(n_scans + 63) / 64, 64, 0, stream>>>(st, n_scans, rows);
}
void launch_query_keys(const MapView& m, const float4* q, size_t nq, uint32_t* keys, uint32_t* vals, cudaStream_t st) {
    k_query_keys<<<uint32_t((nq + kThreads - 1) / kThreads), kThreads, 0, st>>>(m, q, nq, keys, vals);
}
template <int K>
static void launch_knn_k(const MapView& m, const float4* q, const uint32_t* order, size_t nq, float max_d2, uint32_t* idx, float* d2, cudaStream_t st) {
    const uint32_t grid = uint32_t((nq + kTileThreads - 1) / kTileThreads);
    if (order) k_knn<K, true><<<grid, kTileThreads, 0, st>>>(m, q, order, nq, max_d2, idx, d2);
    else k_knn<K, false><<<grid, kTileThreads, 0, st>>>(m, q, order, nq, max_d2, idx, d2);
}
int launch_knn(const MapView& m, const float4* q, const uint32_t* order, size_t nq, int k, float max_d2, uint32_t* idx, float* d2, cudaStream_t st) {
    switch (k) {
        case 1: launch_knn_k<1>(m, q, order, nq, max_d2, idx, d2, st); break;
        case 2: launch_knn_k<2>(m, q, order, nq, max_d2, idx, d2, st); break;
        case 3: launch_knn_k<3>(m, q, order, nq, max_d2, idx, d2, st); break;
        case 4: launch_knn_k<4>(m, q, order, nq, max_d2, idx, d2, st); break;
        case 5: launch_knn_k<5>(m, q, order, nq, max_d2, idx, d2, st); break;
        case 6: launch_knn_k<6>(m, q, order, nq, max_d2, idx, d2, st); break;
        case 7: launch_knn_k<7>(m, q, order, nq, max_d2, idx, d2, st); break;
        case 8: launch_knn_k<8>(m, q, order, nq, max_d2, idx, d2, st); break;
        default: return -1;
    }
    return 0;
}

}  // namespace so
