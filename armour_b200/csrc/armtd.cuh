// ARMTD comparison planner (SURVEY.md 8f-3; reference directory kinova_planner_realtime_armtd_comparison = "KPA") on the
// kernels of the main path.  KPA differs from the main planner in two places only: the trajectory class
// (KPA/Trajectory.cu: constant-acceleration trajectories whose cos / sin reach sets come from an OFFLINE table handed in by the
// caller) and the NLP (KPA/NLPclass.cu: no torque rows, other joint-limit rows, other cost); its PZ arithmetic, forward
// kinematics, reduce_link_PZ and collision kernels are copies of the main planner's.  So the build is k_armtd_jrs (the offline
// table rotated by q0) followed by k_reachsets with the joint reachable set imported (Batch::jrs_ext, csrc/k1_reachsets.cuh:
// jrs_joint; forward kinematics only) and k_hyperplanes; an evaluation is k_constraints followed by k_armtd_assemble, which
// lays the collision rows out as KPA does and adds its joint-limit rows.  Every kernel here works on a batch of problems.
// KPA uses 100 time steps (KPA/Parameters.h:17); the constraint kernels work on chunks of 8 intervals, so the context runs 104
// with the last interval repeated and the padding rows are dropped here.
#pragma once
#include <cuda_runtime.h>

#include "device_constants.cuh"
#include "layout.h"
#include "bezier.cuh"

namespace armour {

constexpr int ARMTD_T = 100;       // NUM_TIME_STEPS of KPA
constexpr int ARMTD_T_PADDED = 104;

// rows of one problem in KPA's layout: collision rows (l * 100 + t) * O + o, then 4 * NF joint-limit rows
__host__ __device__ inline int armtd_m(int NJ, int O) { return NJ * ARMTD_T * O + 4 * NF; }

// ConstantAccelerationCurve::makePolyZono, KPA/Trajectory.cu:29-62: the cos / sin models of joint i over interval t, from the
// offline table jrs [nprob][6][NF][100] (c_cos, g_cos, r_cos, c_sin, g_sin, r_sin) into ext [nprob][104][NF][6]; the padding
// intervals 100..103 repeat interval 99.  cs [nprob][NF][2] = cos q0, sin q0 as the caller computed them (the host-pointer
// build: the host's libm, bit-identical to the reference's host code); nullptr: the device's sincos of q0.  The expression order
// is the reference's (the library is compiled with -fmad=false, so no product is contracted into a fused multiply-add).
__global__ void __launch_bounds__(256)
k_armtd_jrs(int nprob, const double* __restrict__ q0, const double* __restrict__ cs, const double* __restrict__ jrs,
            double* __restrict__ ext) {
    const int n = nprob * ARMTD_T_PADDED * NF;
    for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < n; x += gridDim.x * blockDim.x) {
        const int i = x % NF, t = (x / NF) % ARMTD_T_PADDED, p = x / (NF * ARMTD_T_PADDED);
        const int ts = t < ARMTD_T ? t : ARMTD_T - 1;
        double cos_q0, sin_q0;
        if (cs) {
            cos_q0 = cs[(size_t(p) * NF + i) * 2];
            sin_q0 = cs[(size_t(p) * NF + i) * 2 + 1];
        } else {
            sincos(q0[size_t(p) * NF + i], &sin_q0, &cos_q0);
        }
        const double* a = jrs + size_t(p) * 6 * NF * ARMTD_T + size_t(i) * ARMTD_T + ts;  // a[c * NF * 100]: array c
        const size_t A = size_t(NF) * ARMTD_T;
        double* o = ext + size_t(x) * 6;
        o[0] = cos_q0 * a[0 * A] - sin_q0 * a[3 * A];
        o[1] = cos_q0 * a[1 * A] - sin_q0 * a[4 * A];
        double e = fabs(cos_q0) * a[2 * A] + fabs(sin_q0) * a[5 * A];
        e *= 4.0;
        o[2] = e;
        o[3] = cos_q0 * a[3 * A] + sin_q0 * a[0 * A];
        o[4] = cos_q0 * a[4 * A] + sin_q0 * a[1 * A];
        e = fabs(cos_q0) * a[5 * A] + fabs(sin_q0) * a[2 * A];
        e *= 4.0;
        o[5] = e;
    }
}

// ConstantAccelerationCurve::returnJointStateExtremum and ...Gradient for one joint (KPA/Trajectory.cu:88-384):
// ext / grad = {q_min, q_max, qd_min, qd_max}; the gradients are with respect to k_range * k, as the reference writes them
__host__ __device__ inline void armtd_joint_extremum(double q0, double qd0, double k_actual, double* ext, double* grad) {
    const double t_move = 0.5, t_total = 1.0, t_to_stop = t_total - t_move;
    const double q_peak = q0 + qd0 * t_move + k_actual * t_move * t_move * 0.5;
    const double q_dot_peak = qd0 + k_actual * t_move;
    const double q_ddot_to_stop = -q_dot_peak / t_to_stop;
    const double q_stop = q_peak + q_dot_peak * t_to_stop + 0.5 * q_ddot_to_stop * t_to_stop * t_to_stop;
    const double t_mm = -qd0 / k_actual;  // interior extremum of the first phase; inf / nan at k = 0 fails both tests below
    double q_lo, q_hi, g_lo, g_hi;
    if (q_peak >= q0) {
        q_lo = q0; q_hi = q_peak; g_lo = 0; g_hi = 0.5 * t_move * t_move;
    } else {
        q_lo = q_peak; q_hi = q0; g_lo = 0.5 * t_move * t_move; g_hi = 0;
    }
    double q_min_p = q_lo, q_max_p = q_hi, gq_min_p = g_lo, gq_max_p = g_hi;
    if (t_mm > 0 && t_mm < t_move) {
        const double q_int = q0 + qd0 * t_mm + 0.5 * k_actual * t_mm * t_mm;
        const double g_int = (0.5 * qd0 * qd0) / (k_actual * k_actual);
        if (k_actual >= 0) {
            q_min_p = q_int; gq_min_p = g_int;
        } else {
            q_max_p = q_int; gq_max_p = g_int;
        }
    }
    double v_min_p, v_max_p, gv_min_p, gv_max_p;
    if (q_dot_peak >= qd0) {
        v_min_p = qd0; v_max_p = q_dot_peak; gv_min_p = 0; gv_max_p = t_move;
    } else {
        v_min_p = q_dot_peak; v_max_p = qd0; gv_min_p = t_move; gv_max_p = 0;
    }
    double q_min_s, q_max_s, gq_min_s, gq_max_s;
    if (q_stop >= q_peak) {
        q_min_s = q_peak; q_max_s = q_stop;
        gq_min_s = 0.5 * t_move * t_move; gq_max_s = 0.5 * t_move * t_move + 0.5 * t_move * t_to_stop;
    } else {
        q_min_s = q_stop; q_max_s = q_peak;
        gq_min_s = 0.5 * t_move * t_move + 0.5 * t_move * t_to_stop; gq_max_s = 0.5 * t_move * t_move;
    }
    double v_min_s, v_max_s, gv_min_s, gv_max_s;
    if (q_dot_peak >= 0) {
        v_min_s = 0; v_max_s = q_dot_peak; gv_min_s = 0; gv_max_s = t_move;
    } else {
        v_min_s = q_dot_peak; v_max_s = 0; gv_min_s = t_move; gv_max_s = 0;
    }
    const bool a = q_min_p <= q_min_s, b = q_max_p >= q_max_s, c = v_min_p <= v_min_s, d = v_max_p >= v_max_s;
    ext[0] = a ? q_min_p : q_min_s;
    ext[1] = b ? q_max_p : q_max_s;
    ext[2] = c ? v_min_p : v_min_s;
    ext[3] = d ? v_max_p : v_max_s;
    grad[0] = a ? gq_min_p : gq_min_s;
    grad[1] = b ? gq_max_p : gq_max_s;
    grad[2] = c ? gv_min_p : gv_min_s;
    grad[3] = d ? gv_max_p : gv_max_s;
}

// g_full / j_full: the main planner's layout with Tp = 104 intervals (torque rows, collision rows (l * Tp + t) * O + o, Bezier
// rows), B.m() rows per problem; g / jac: KPA's layout, armtd_m() rows per problem, collision rows (l * 100 + t) * O + o then
// 4 * NF joint-limit rows (KPA/NLPclass.cu:43-44, 248-336).  The joint-limit rows of the Jacobian are diagonal: the reference
// writes only the diagonal entries and clears 4*NF*NF BYTES of those rows (KPA/Trajectory.cu:262), i.e. it relies on a
// zero-filled buffer.  Problem plist[blockIdx.y] (B.plist, or blockIdx.y); q0 / qd0 from B, k_range [p][NF] (per world).
__global__ void __launch_bounds__(256)
k_armtd_assemble(Batch B, const double* __restrict__ k_range, const double* __restrict__ k, const double* __restrict__ g_full,
                 const double* __restrict__ j_full, double* __restrict__ g, double* __restrict__ jac) {
    const int p = B.plist ? B.plist[blockIdx.y] : int(blockIdx.y);
    const int NJ = B.NJ, O = B.O, Tp = B.T;
    const int rows = NJ * ARMTD_T * O;
    const size_t mf = size_t(B.m()), ma = size_t(armtd_m(NJ, O));
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += gridDim.x * blockDim.x) {
        const int o = r % O, lt = r / O, t = lt % ARMTD_T, l = lt / ARMTD_T;
        const size_t src = p * mf + size_t(NF) * Tp + (size_t(l) * Tp + t) * O + o;
        if (g) g[p * ma + r] = g_full[src];
        if (jac)
            for (int v = 0; v < NF; v++) jac[(p * ma + r) * NF + v] = j_full[src * NF + v];
    }
    if (blockIdx.x == 0 && threadIdx.x < NF) {
        const int i = threadIdx.x;
        double ext[4], grad[4];
        armtd_joint_extremum(B.q0[size_t(p) * NF + i], B.qd0[size_t(p) * NF + i], k_range[size_t(p) * NF + i] * k[size_t(p) * NF + i],
                             ext, grad);
        for (int q = 0; q < 4; q++) {
            const size_t row = p * ma + rows + q * NF + i;
            if (g) g[row] = ext[q];
            if (jac)
                for (int v = 0; v < NF; v++) jac[row * NF + v] = (v == i) ? grad[q] : 0.0;
        }
    }
}
inline cudaError_t launch_armtd_assemble(const Batch& B, const double* k_range, const double* d_k, const double* g_full,
                                         const double* j_full, double* g, double* jac, cudaStream_t st) {
    const int rows = B.NJ * ARMTD_T * B.O;
    k_armtd_assemble<<<dim3(rows > 0 ? (rows + 255) / 256 : 1, B.nprob), 256, 0, st>>>(B, k_range, d_k, g_full, j_full, g, jac);
    return cudaGetLastError();
}

// finalize_solution's predicate (KPA/NLPclass.cu:366-455) for each problem of KPA-layout g [nprob][armtd_m]: feasible[p], and
// first[p] = the first violated row in the reference's check order or -1.  The reference's collision loop runs over
// NUM_FACTORS - 1 links (KPA/NLPclass.cu:400), so the rows of links NF-1.. are not checked; the check order is ascending row
// index otherwise, so the first violation is the smallest violating index among the checked rows.  One CTA per problem.
__global__ void __launch_bounds__(256)
k_armtd_verdict(int NJ, int O, const double* __restrict__ g, int* __restrict__ feasible, int* __restrict__ first) {
    const int p = blockIdx.x;
    const int m = armtd_m(NJ, O), ncol = NJ * ARMTD_T * O, nchecked = (NF - 1) * ARMTD_T * O;
    const double* gp = g + size_t(p) * m;
    const RobotConstants& R = c_robot;
    int best = m;
    for (int r = threadIdx.x; r < m; r += blockDim.x) {
        const double v = gp[r];
        bool bad;
        if (r < ncol) {
            bad = r < nchecked && v > R.collision_violation_threshold;
        } else {
            const int q = r - ncol, j = q % NF;
            if (q < 2 * NF)
                bad = v < R.state_limits_lb[j] + R.qe || v > R.state_limits_ub[j] - R.qe;
            else
                bad = v < -R.speed_limits[j] + R.qde || v > R.speed_limits[j] - R.qde;
        }
        if (bad && r < best) best = r;
    }
    __shared__ int s_best;
    if (threadIdx.x == 0) s_best = m;
    __syncthreads();
    atomicMin(&s_best, best);
    __syncthreads();
    if (threadIdx.x == 0) {
        feasible[p] = (s_best == m) ? 1 : 0;
        first[p] = (s_best == m) ? -1 : s_best;
    }
}

// KPA's cost (KPA/NLPclass.cu:178-243): q(t_plan) = q0 + 0.5 qd0 + 0.125 k_range k; host arithmetic for armour_armtd_batch_cost
// and device arithmetic for the batched solver, the same expressions
__host__ __device__ inline double armtd_wrap(double a) {
    while (a < -M_PI) a += 2 * M_PI;
    while (a > M_PI) a -= 2 * M_PI;
    return a;
}
__host__ __device__ inline double armtd_cost(const double* q0, const double* qd0, const double* k_range, const double* q_des,
                                             const double* k, double cost_scale, double* grad) {
    double qp[NF];
    for (int i = 0; i < NF; i++) qp[i] = q0[i] + qd0[i] * 0.5 + k_range[i] * k[i] * 0.125;
    if (grad)
        for (int i = 0; i < NF; i++) {
            const double dk = k_range[i] * 0.125;
            grad[i] = (i % 2 == 0) ? (2 * armtd_wrap(qp[i] - q_des[i]) * dk) : (2 * (qp[i] - q_des[i]) * dk);
            grad[i] *= cost_scale;
        }
    const double v = pw2(armtd_wrap(q_des[0] - qp[0])) + pw2(armtd_wrap(q_des[2] - qp[2])) + pw2(armtd_wrap(q_des[4] - qp[4])) +
                     pw2(armtd_wrap(q_des[6] - qp[6])) + pw2(q_des[1] - qp[1]) + pw2(q_des[3] - qp[3]) + pw2(q_des[5] - qp[5]);
    return v * cost_scale;
}

// NLP policy of the batched solver (csrc/k4_solver.cuh) for KPA's armtd_NLP, as local_solve drives it in armtd_main
// (host/armtd_main.cpp, host/local_solver.cpp): collision rows one-sided with collision_tol, limit rows two-sided with
// tolerance 0 and the bounds of armour_armtd_get_bounds, KPA's cost.  The solver's violation measure counts the collision rows
// of ALL links, the last one included, while the final verdict (k_armtd_verdict) skips the last link as the reference's
// finalize_solution does.  The difference is deliberate: it is what the host solver over armtd_NLP does, so both give the same
// iterates; a plan is only ever more conservative than the verdict asks.
struct ArmtdNlp {
    const double* k_range;  // [p][NF]
    __device__ int m(const Batch& B) const { return armtd_m(B.NJ, B.O); }
    __device__ void row_bounds(const Batch& B, int, int i, double, double ctol, double* gl, double* gu, double* tol) const {
        const RobotConstants& R = c_robot;
        const int ncol = B.NJ * ARMTD_T * B.O;
        if (i < ncol) {
            *gl = -1e19;
            *gu = 0;
            *tol = ctol;
            return;
        }
        const int q = i - ncol, j = q % NF;
        if (q < 2 * NF) {
            *gl = R.state_limits_lb[j] + R.qe;
            *gu = R.state_limits_ub[j] - R.qe;
        } else {
            *gl = -R.speed_limits[j] + R.qde;
            *gu = R.speed_limits[j] - R.qde;
        }
        *tol = 0.0;
    }
    __device__ double cost(const Batch& B, int p, const double* q_des, const double* k, double* grad) const {
        return armtd_cost(B.q0 + size_t(p) * NF, B.qd0 + size_t(p) * NF, k_range + size_t(p) * NF, q_des, k, c_robot.cost_scale,
                          grad);
    }
};

}  // namespace armour
