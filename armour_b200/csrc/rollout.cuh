// Closed-loop replanning episodes on the device (armour_batch_rollout*, armour_armtd_batch_rollout*) and the exact clearance
// of arm configurations (armour_batch_clearance*).  The semantics are those of include/armour_b200.h and DESIGN.md section 3
// ("Closed-loop episodes"); the host loop that sequences these kernels around the device build and solve is rollout_run in
// armour_capi.cu, templated over the planner like the batched solver over its NLP.
//
// Per replan: k_rollout_plan (compaction list -> dense planning inputs, waypoint, log rows), the planner's build and solve on
// the running worlds, k_rollout_advance (verdict -> executed segment, next state, audit samples; its trajectory class is a
// template parameter), k_clearance over the audit samples, k_rollout_finish (stop tests, stable compaction of the running worlds
// in ascending world index).
#pragma once
#include <climits>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "../../include/armour_b200.h"
#include "armtd.cuh"
#include "bezier.cuh"
#include "device_constants.cuh"

namespace armour {

constexpr int ROLL_STATE = 3 * NF;  // q, qd, qdd
constexpr int ROLL_PLAN = 4 * NF;   // q0, qd0, qdd0 (real time), k (rad): the Bezier of an executed plan; ARMTD: q0, qd0, 0, k_a
constexpr int ROLL_THREADS = 128;
constexpr int CLEAR_THREADS = 128;
constexpr int FINISH_THREADS = 1024;

// Device view of one rollout: inputs, per-world state (indexed by world w) and the dense batch (indexed by batch position i).
struct RolloutDev {
    int n, R, nobs, S;
    double lookahead, goal_radius, collision_tol;
    const double* start;      // [n][NF]
    const double* goal;       // [n][NF]
    const double* obstacles;  // [n][nobs][12]
    double* state;            // [n][21] planning state of the next replan (the end of the last executed segment)
    double* plan;             // [n][28] current plan
    double* minc;             // [n]
    int* outcome;             // [n] -1 while running, then ARMOUR_ROLLOUT_*
    int* replans;             // [n]
    int* infeasible;          // [n]
    int* limit;               // [n] the audit of the last segment found a limit exceeded
    double *dq0, *dqd0, *dqdd0, *dq_des, *dk, *dobs;  // [i][NF] / [i][nobs][12]
    double* samp;             // [i][S][NF] configurations of the audit samples
    double* dclear;           // [i]
    int *dfeas, *dfirst, *diters;
    double* log_state;        // [R][n][21], any log pointer may be null
    double* log_q_des;        // [R][n][NF]
    double* log_k;            // [R][n][NF]
    int* log_int;             // [R][n][4]
    double* log_clearance;    // [R][n]
};

__device__ __forceinline__ bool roll_continuous(int j) { return (j % 2) == 0; }  // joints 0, 2, 4, 6

// MATLAB angdiff(a, b) = b - a wrapped to [-pi, pi), as numpy computes (d + pi) % (2 pi) - pi (fmod, then the sign fix)
__device__ __forceinline__ double roll_angdiff(double a, double b) {
    double m = fmod((b - a) + M_PI, 2 * M_PI);
    if (m != 0.0 && m < 0.0) m += 2 * M_PI;
    return m - M_PI;
}
__device__ __forceinline__ double roll_goal_diff(const double* q, const double* goal, int j) {
    return roll_continuous(j) ? roll_angdiff(q[j], goal[j]) : goal[j] - q[j];
}

// every world starts at rest at its start configuration, its current plan the rest plan there; log rows not planned stay
// NaN (doubles) / -1 (ints)
__global__ void k_rollout_init(RolloutDev D, int* list) {
    const size_t stride = size_t(gridDim.x) * blockDim.x;
    const size_t tid = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const size_t rn = size_t(D.R) * D.n;
    for (size_t e = tid; e < rn; e += stride) {
        if (D.log_state)
            for (int j = 0; j < ROLL_STATE; j++) D.log_state[e * ROLL_STATE + j] = nan;
        for (int j = 0; j < NF; j++) {
            if (D.log_q_des) D.log_q_des[e * NF + j] = nan;
            if (D.log_k) D.log_k[e * NF + j] = nan;
        }
        if (D.log_int)
            for (int j = 0; j < 4; j++) D.log_int[e * 4 + j] = -1;
        if (D.log_clearance) D.log_clearance[e] = nan;
    }
    for (size_t w = tid; w < size_t(D.n); w += stride) {
        for (int j = 0; j < NF; j++) {
            const double q = D.start[w * NF + j];
            D.state[w * ROLL_STATE + j] = q;
            D.state[w * ROLL_STATE + NF + j] = 0.0;
            D.state[w * ROLL_STATE + 2 * NF + j] = 0.0;
            D.plan[w * ROLL_PLAN + j] = q;
            D.plan[w * ROLL_PLAN + NF + j] = 0.0;
            D.plan[w * ROLL_PLAN + 2 * NF + j] = 0.0;
            D.plan[w * ROLL_PLAN + 3 * NF + j] = 0.0;
        }
        D.minc[w] = CUDART_INF;
        D.outcome[w] = -1;
        D.replans[w] = 0;
        D.infeasible[w] = 0;
        D.limit[w] = 0;
        list[w] = int(w);
    }
}

// batch position i <- world list[i]: planning state, straight-line waypoint, obstacles; the replan's log rows
__global__ void k_rollout_plan(RolloutDev D, int r, int nrun, const int* __restrict__ list) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrun) return;
    const int w = list[i];
    const double* st = D.state + size_t(w) * ROLL_STATE;
    const double* goal = D.goal + size_t(w) * NF;
    double d[NF], nrm2 = 0.0;
    for (int j = 0; j < NF; j++) {
        d[j] = roll_goal_diff(st, goal, j);
        nrm2 += d[j] * d[j];
    }
    const double nrm = sqrt(nrm2);
    const bool at_goal = nrm <= D.lookahead;  // the waypoint is the goal itself: an arriving arm is not pulled past it
    const size_t row = size_t(r) * D.n + w;
    for (int j = 0; j < NF; j++) {
        const double qd = at_goal ? st[j] + d[j] : st[j] + D.lookahead * d[j] / nrm;
        D.dq0[size_t(i) * NF + j] = st[j];
        D.dqd0[size_t(i) * NF + j] = st[NF + j];
        D.dqdd0[size_t(i) * NF + j] = st[2 * NF + j];
        D.dq_des[size_t(i) * NF + j] = qd;
        if (D.log_q_des) D.log_q_des[row * NF + j] = qd;
    }
    if (D.log_state)
        for (int j = 0; j < ROLL_STATE; j++) D.log_state[row * ROLL_STATE + j] = st[j];
    const size_t no = size_t(D.nobs) * 12;
    for (size_t e = 0; e < no; e++) D.dobs[size_t(i) * no + e] = D.obstacles[size_t(w) * no + e];
}

// q, qd, qdd (real time) of the plan P = (q0, qd0, qdd0, k) at normalised time s
__device__ __forceinline__ void roll_eval_plan(const double* P, double s, double* q, double* qd, double* qdd) {
    const double Dur = c_robot.duration;
    for (int j = 0; j < NF; j++) {
        const double q0 = P[j], a = P[NF + j] * Dur, b = P[2 * NF + j] * Dur * Dur, k = P[3 * NF + j];
        if (q) q[j] = bez_q(q0, a, b, k, s);
        if (qd) qd[j] = bez_qd(q0, a, b, k, s) / Dur;
        if (qdd) qdd[j] = bez_qdd(q0, a, b, k, s) / (Dur * Dur);
    }
}

// Trajectory classes of k_rollout_advance: the scale of a solved k into the plan's last slot for batch position i and joint j,
// the normalised time t_move of the segment split, and (q, qd, qdd) of a stored plan at normalised time s.
// The main planner's: the Bezier of roll_eval_plan, k scaled by the robot model's k_range.
struct RollBezier {
    __device__ __forceinline__ double k_scale(int, int j) const { return c_robot.k_range[j]; }
    __device__ __forceinline__ double s_move() const { return c_robot.t_plan / c_robot.duration; }
    __device__ __forceinline__ void eval(const double* P, double s, double* q, double* qd, double* qdd) const {
        roll_eval_plan(P, s, q, qd, qdd);
    }
};
// The ARMTD comparison planner's: the constant-acceleration curve of armtd_curve over t in [0, 1] (t_move 0.5), k scaled by the
// k_range of the replan ([i][NF], dense), the plan stored as (q0, qd0, 0, k_a).  The planner has no acceleration input: qdd is 0.
struct RollConstAcc {
    const double* k_range;
    __device__ __forceinline__ double k_scale(int i, int j) const { return k_range[size_t(i) * NF + j]; }
    __device__ __forceinline__ double s_move() const { return 0.5; }
    __device__ __forceinline__ void eval(const double* P, double s, double* q, double* qd, double* qdd) const {
        for (int j = 0; j < NF; j++) {
            double a, b;
            armtd_curve(P[j], P[NF + j], P[3 * NF + j], s, &a, &b);
            if (q) q[j] = a;
            if (qd) qd[j] = b;
            if (qdd) qdd[j] = 0.0;
        }
    }
};

// the solve's verdict -> executed segment (the new plan over [0, t_move] or the current plan's braking half [t_move, 1]),
// next state, current plan, counters, audit samples and the joint-limit audit
template <class Traj>
__global__ void k_rollout_advance(RolloutDev D, int r, int nrun, const int* __restrict__ list, const int* __restrict__ build_status,
                                  int epoch, Traj traj) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrun) return;
    const RobotConstants& R = c_robot;
    const int w = list[i];
    const bool ok = D.dfeas[i] != 0;
    const int bs = (build_status[i] >> 3) == epoch && (build_status[i] & 7) != 0 ? ARMOUR_ERR_CAPACITY : ARMOUR_OK;
    const size_t row = size_t(r) * D.n + w;
    if (D.log_k)
        for (int j = 0; j < NF; j++) D.log_k[row * NF + j] = D.dk[size_t(i) * NF + j];
    if (D.log_int) {
        D.log_int[row * 4 + 0] = ok ? 1 : 0;
        D.log_int[row * 4 + 1] = D.dfirst[i];
        D.log_int[row * 4 + 2] = D.diters[i];
        D.log_int[row * 4 + 3] = bs;
    }
    double* P = D.plan + size_t(w) * ROLL_PLAN;
    double* st = D.state + size_t(w) * ROLL_STATE;
    const double s_move = traj.s_move();
    if (ok) {  // the new plan becomes the current plan
        for (int j = 0; j < NF; j++) {
            P[j] = st[j];
            P[NF + j] = st[NF + j];
            P[2 * NF + j] = st[2 * NF + j];
            P[3 * NF + j] = traj.k_scale(i, j) * D.dk[size_t(i) * NF + j];
        }
    }
    const double s0 = ok ? 0.0 : s_move, s1 = ok ? s_move : 1.0;
    // audit samples (both ends included) and the raw joint limits
    int lim = 0;
    for (int m = 0; m < D.S; m++) {
        const double s = s0 + (s1 - s0) * double(m) / double(D.S - 1);
        double q[NF], qd[NF];
        traj.eval(P, s, q, qd, nullptr);
        for (int j = 0; j < NF; j++) {
            D.samp[(size_t(i) * D.S + m) * NF + j] = q[j];
            if (!roll_continuous(j) && (q[j] < R.state_limits_lb[j] || q[j] > R.state_limits_ub[j])) lim = 1;
            if (fabs(qd[j]) > R.speed_limits[j]) lim = 1;
        }
    }
    D.limit[w] = lim;
    if (ok) {
        double q[NF], qd[NF], qdd[NF];
        traj.eval(P, s_move, q, qd, qdd);
        for (int j = 0; j < NF; j++) {
            st[j] = q[j];
            st[NF + j] = qd[j];
            st[2 * NF + j] = qdd[j];
        }
    } else {  // braked to rest at s = 1: the current plan becomes the rest plan there (constant in both trajectory classes)
        double q[NF];
        traj.eval(P, 1.0, q, nullptr, nullptr);
        for (int j = 0; j < NF; j++) {
            st[j] = q[j];
            st[NF + j] = 0.0;
            st[2 * NF + j] = 0.0;
            P[j] = q[j];
            P[NF + j] = 0.0;
            P[2 * NF + j] = 0.0;
            P[3 * NF + j] = 0.0;
        }
        D.infeasible[w]++;
    }
    D.replans[w] = r + 1;
}

// Signed clearance of two parallelepipeds (centre + 3 generator columns) by the separating-axis test: 3 + 3 face normals
// and 9 edge x edge cross products, axes of norm below 1e-12 skipped; the largest gap over the axes.  > 0: separated (a
// lower bound on the distance), <= 0: intersecting (-penetration along the best axis).
__device__ __forceinline__ double sat_axis(const double* n, const double* d, const double (*A)[3], const double (*B)[3], double best) {
    const double nn = sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    if (nn < 1e-12) return best;
    double ra = 0.0, rb = 0.0;
    for (int e = 0; e < 3; e++) {
        ra += fabs(A[e][0] * n[0] + A[e][1] * n[1] + A[e][2] * n[2]);
        rb += fabs(B[e][0] * n[0] + B[e][1] * n[1] + B[e][2] * n[2]);
    }
    const double gap = (fabs(d[0] * n[0] + d[1] * n[1] + d[2] * n[2]) - ra - rb) / nn;
    return gap > best ? gap : best;
}
__device__ __forceinline__ void sat_cross(const double* a, const double* b, double* n) {
    n[0] = a[1] * b[2] - a[2] * b[1];
    n[1] = a[2] * b[0] - a[0] * b[2];
    n[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ inline double sat_clearance(const double* ca, const double (*A)[3], const double* cb, const double (*B)[3]) {
    const double d[3] = {cb[0] - ca[0], cb[1] - ca[1], cb[2] - ca[2]};
    double best = -CUDART_INF, n[3];
    const int pa[3] = {0, 1, 0}, pb[3] = {1, 2, 2};
    for (int f = 0; f < 3; f++) {
        sat_cross(A[pa[f]], A[pb[f]], n);
        best = sat_axis(n, d, A, B, best);
    }
    for (int f = 0; f < 3; f++) {
        sat_cross(B[pa[f]], B[pb[f]], n);
        best = sat_axis(n, d, A, B, best);
    }
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 3; b++) {
            sat_cross(A[a], B[b], n);
            best = sat_axis(n, d, A, B, best);
        }
    return best;
}

// Link box l of configuration q by the scalar chain of k_reachsets' kinematics: FK_T += FK_R trans_i,
// FK_R = FK_R rrpy_i Rz(q_i) (fixed joints beyond NF: rrpy_i only); centre FK_T + FK_R c_l, generators FK_R diag(g_l).
__device__ inline void fk_link_box(const double* q, int l, double* c, double (*G)[3]) {
    const RobotConstants& R = c_robot;
    double Rm[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, T[3] = {0, 0, 0};  // column-major
    for (int i = 0; i <= l; i++) {
        const double* tr = &R.trans[3 * i];
        for (int e = 0; e < 3; e++) T[e] += Rm[e] * tr[0] + Rm[3 + e] * tr[1] + Rm[6 + e] * tr[2];
        double J[9];
        const double* Rr = &R.rrpy[i * 9];
        if (i < NF) {
            double sn, cs;
            sincos(q[i], &sn, &cs);
            const double Z[9] = {cs, sn, 0, -sn, cs, 0, 0, 0, 1};
            for (int a = 0; a < 3; a++)
                for (int b = 0; b < 3; b++) J[a + 3 * b] = Rr[a] * Z[3 * b] + Rr[3 + a] * Z[3 * b + 1] + Rr[6 + a] * Z[3 * b + 2];
        } else {
            for (int e = 0; e < 9; e++) J[e] = Rr[e];
        }
        double N[9];
        for (int a = 0; a < 3; a++)
            for (int b = 0; b < 3; b++) N[a + 3 * b] = Rm[a] * J[3 * b] + Rm[3 + a] * J[3 * b + 1] + Rm[6 + a] * J[3 * b + 2];
        for (int e = 0; e < 9; e++) Rm[e] = N[e];
    }
    const double* lc = &R.link_zonotope_center[3 * l];
    const double* lg = &R.link_zonotope_generators[3 * l];
    for (int e = 0; e < 3; e++) {
        c[e] = T[e] + Rm[e] * lc[0] + Rm[3 + e] * lc[1] + Rm[6 + e] * lc[2];
        for (int g = 0; g < 3; g++) G[g][e] = Rm[3 * g + e] * lg[g];
    }
}

// One block per group of ns configurations q[b][ns][NF] against obstacle set world[b] (null: set 0); one thread per
// (configuration, link, obstacle).  out[b] = the smallest clearance, which[b] = l * nobs + o of the pair that attains it
// (ties: the first configuration, then the lowest l * nobs + o); +inf and -1 without obstacles.  The block reduction is
// in a fixed order, so the result does not depend on the schedule.
__global__ void __launch_bounds__(CLEAR_THREADS) k_clearance(const double* __restrict__ q, int ns, const int* __restrict__ world,
                                                             const double* __restrict__ obstacles, int nobs, double* __restrict__ out,
                                                             int* __restrict__ which) {
    __shared__ double s_v[CLEAR_THREADS];
    __shared__ long long s_k[CLEAR_THREADS];
    const int b = blockIdx.x;
    const int NJ = c_robot.num_joints;
    const long long per = (long long)NJ * nobs, items = per * ns;
    const double* obs = obstacles + (world ? size_t(world[b]) : 0) * size_t(nobs) * 12;
    double best = CUDART_INF;
    long long bk = LLONG_MAX;
    for (long long it = threadIdx.x; it < items; it += CLEAR_THREADS) {
        const int m = int(it / per), lo = int(it % per), l = lo / nobs, o = lo % nobs;
        double c[3], G[3][3], cb[3], Gb[3][3];
        fk_link_box(q + (size_t(b) * ns + m) * NF, l, c, G);
        const double* z = obs + size_t(o) * 12;
        for (int e = 0; e < 3; e++) {
            cb[e] = z[e];
            for (int g = 0; g < 3; g++) Gb[g][e] = z[3 + 3 * g + e];
        }
        const double v = sat_clearance(c, G, cb, Gb);
        if (v < best || (v == best && it < bk)) {  // items ascend per thread: the first of equal values is kept
            best = v;
            bk = it;
        }
    }
    s_v[threadIdx.x] = best;
    s_k[threadIdx.x] = bk;
    __syncthreads();
    for (int h = CLEAR_THREADS / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h) {
            const double v = s_v[threadIdx.x + h];
            const long long k = s_k[threadIdx.x + h];
            if (v < s_v[threadIdx.x] || (v == s_v[threadIdx.x] && k < s_k[threadIdx.x])) {
                s_v[threadIdx.x] = v;
                s_k[threadIdx.x] = k;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[b] = s_v[0];
        if (which) which[b] = s_k[0] == LLONG_MAX ? -1 : int(s_k[0] % per);
    }
}

// One block: the stop tests of the running worlds (clearance below -collision_tol: collision; a joint limit exceeded:
// limit; the segment's end within goal_radius of the goal: arrived; max_replans used: budget, in this order), then the
// worlds still running in ascending world index into next[] (a stable compaction of list[]) and their number into *count.
__global__ void __launch_bounds__(FINISH_THREADS) k_rollout_finish(RolloutDev D, int r, int nrun, const int* __restrict__ list,
                                                                   int* __restrict__ next, int* __restrict__ count) {
    __shared__ int s_warp[FINISH_THREADS / 32];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int base = 0; base < nrun; base += FINISH_THREADS) {
        const int i = base + threadIdx.x;
        int w = -1;
        bool keep = false;
        if (i < nrun) {
            w = list[i];
            const double cl = D.dclear[i];
            if (D.log_clearance) D.log_clearance[size_t(r) * D.n + w] = cl;
            if (cl < D.minc[w]) D.minc[w] = cl;
            const double* st = D.state + size_t(w) * ROLL_STATE;
            const double* goal = D.goal + size_t(w) * NF;
            double e2 = 0.0;
            for (int j = 0; j < NF; j++) {
                const double d = roll_goal_diff(st, goal, j);
                e2 += d * d;
            }
            int oc = -1;
            if (cl < -D.collision_tol) oc = ARMOUR_ROLLOUT_COLLISION;
            else if (D.limit[w]) oc = ARMOUR_ROLLOUT_LIMIT;
            else if (sqrt(e2) <= D.goal_radius) oc = ARMOUR_ROLLOUT_ARRIVED;
            else if (r + 1 >= D.R) oc = ARMOUR_ROLLOUT_BUDGET;
            D.outcome[w] = oc;
            keep = oc < 0;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        if (threadIdx.x == 0) {  // exclusive scan of the warp counts
            int acc = 0;
            for (int k = 0; k < FINISH_THREADS / 32; k++) {
                const int c = s_warp[k];
                s_warp[k] = acc;
                acc += c;
            }
        }
        __syncthreads();
        if (keep) next[s_base + s_warp[warp] + __popc(bal & ((1u << lane) - 1u))] = w;
        __syncthreads();
        if (threadIdx.x == FINISH_THREADS - 1) s_base += s_warp[warp] + __popc(bal);
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = s_base;
}

}  // namespace armour
