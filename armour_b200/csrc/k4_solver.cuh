// K4: batched trust-region SQP on the device — the caller of the hot path (SURVEY.md 8f-1).
//
// The reference hands ONE armtd_NLP to Ipopt (KPR/armour_main.cu:237-278); every iteration crosses PCIe twice
// (eval_g, eval_jac_g) and Ipopt is serial.  With the constraint kernel at ~0.65 us per evaluation the solver loop
// is what bounds "planning iterations per second", so the loop itself runs on the device for a whole batch: one
// CTA per planning problem, thousands in step, only k_opt and the verdict leave the GPU.
//
// The algorithm is the one of armour_b200/host/local_solver.cpp (the stand-in for Ipopt of the C++ host side),
// statement for statement, so that both give the same iterates: the planner's cost is an exactly spherical
// quadratic in k (KPR/NLPclass.cu:207-268), each iteration solves
//     min 1/2 h |d|^2 + grad_f . d   s.t.  g_l <= g + J d <= g_u,  -1 <= x + d <= 1,  |d|_inf <= Delta
// exactly, by the dual active-set method of host/active_set_qp.h over the rows that can become active inside the trust
// region (the CTA searches the most violated row, one thread does the 7 x 7 algebra of taking it in), then accepts /
// rejects on (violation, cost).  Per iteration: k_constraints (g, J at x),
// k_solver_step, k_constraints (g at the trial point), k_solver_accept.
//
// The kernels are templates over an NLP policy: m(B) rows per problem, row_bounds(B, p, i, ...) = bounds and acceptance
// tolerance of row i, cost(B, p, q_des, k, grad) = cost and its gradient.  ArmourNlp below is the main planner's armtd_NLP;
// ArmtdNlp (csrc/armtd.cuh) is the one of the ARMTD comparison planner, whose evaluation step assembles KPA's row layout
// behind k_constraints.
#pragma once
#include <cuda_runtime.h>

#include "../host/active_set_qp.h"
#include "bezier.cuh"
#include "device_constants.cuh"
#include "layout.h"

namespace armour {

#ifndef ARMOUR_SOLVER_THREADS
#define ARMOUR_SOLVER_THREADS 256
#endif
constexpr int SOLVER_THREADS = ARMOUR_SOLVER_THREADS;
constexpr int SOLVER_WARPS = SOLVER_THREADS / 32;
// steps of 32 rows per warp so that SOLVER_WARPS segments cover m rows; dynamic shared memory of k_solver_step
__host__ __device__ inline int solver_steps(int m) { return ((m + SOLVER_WARPS - 1) / SOLVER_WARPS + 31) / 32; }
__host__ __device__ inline size_t solver_step_smem(int m) { return size_t(SOLVER_WARPS) * solver_steps(m) * 2 * sizeof(unsigned); }
constexpr int SOLVER_ROWCAP = 2048;   // linearised rows kept per problem; more -> status ROW_OVERFLOW
constexpr int SOLVER_ROWW = 9;        // doubles per row: a[7], b, 1 / |a|
enum { SOLVER_RUNNING = 0, SOLVER_SUCCESS = 1, SOLVER_MAXITER = 2, SOLVER_TINY_STEP = 3, SOLVER_INFEASIBLE = 4,
       SOLVER_ROW_OVERFLOW = 5 };

struct SolverState {   // structure of arrays, [nprob] or [nprob][NF]
    double* x;         // current iterate
    double* xt;        // trial point
    double* best;      // best accepted feasible point
    double* f;         // cost at x
    double* viol;      // violation at x (<= 0: finalize_solution would accept)
    double* fbest;
    double* delta;     // trust-region radius
    int* have_best;
    int* status;       // SOLVER_*
    int* iters;
    int* evals;
    int* dbg;          // [nprob][3]: rows, active-set iterations, dropped rows of the last step (diagnostics)
    double* rows;      // [nprob][SOLVER_ROWW][SOLVER_ROWCAP]: component-major, the scan of a QP round reads it lane-contiguously
    const double* q_des;  // [nprob][NF]
    double tol, torque_tol, collision_tol;
    int max_iter;
    int qp_sweeps;
    int qp_update_budget;
};

// cost and gradient of one problem (KPR/NLPclass.cu:207-268; same expressions as armour_cost in armour_capi.cu)
__device__ __forceinline__ double solver_wrap(double a) {
    while (a < -M_PI) a += 2 * M_PI;
    while (a > M_PI) a -= 2 * M_PI;
    return a;
}
__device__ inline double solver_cost(const Batch& B, int p, const double* q_des, const double* k, double* grad) {
    const RobotConstants& R = c_robot;
    const double tp = R.t_plan, D = R.duration;
    double qp[NF];
    for (int i = 0; i < NF; i++)
        qp[i] = bez_q(B.q0[size_t(p) * NF + i], B.qd0[size_t(p) * NF + i] * D, B.qdd0[size_t(p) * NF + i] * D * D,
                      R.k_range[i] * k[i], tp);
    const double v = pw2(solver_wrap(q_des[0] - qp[0])) + pw2(solver_wrap(q_des[2] - qp[2])) + pw2(solver_wrap(q_des[4] - qp[4])) +
                     pw2(solver_wrap(q_des[6] - qp[6])) + pw2(q_des[1] - qp[1]) + pw2(q_des[3] - qp[3]) + pw2(q_des[5] - qp[5]);
    if (grad) {
        for (int i = 0; i < NF; i++) {
            const double dk = pw3(tp) * (6 * pw2(tp) - 15 * tp + 10) * R.k_range[i];
            grad[i] = (i % 2 == 0) ? (2 * solver_wrap(qp[i] - q_des[i]) * dk) : (2 * (qp[i] - q_des[i]) * dk);
            grad[i] *= R.cost_scale;
        }
    }
    return v * R.cost_scale;
}

// bounds of row i (armour_batch_get_bounds / KPR/NLPclass.cu:116-165) and the acceptance tolerance of its class
__device__ __forceinline__ void solver_row_bounds(const Batch& B, int p, int i, double ttol, double ctol, double* gl,
                                                  double* gu, double* tol) {
    const RobotConstants& R = c_robot;
    const int T = B.T, NJ = B.NJ, O = B.O;
    if (i < NF * T) {
        const int t = i / NF, j = i % NF;
        const double tr = B.torque_radius[size_t(p) * NF * T + size_t(j) * T + t];
        *gl = -R.torque_limits[j] + tr;
        *gu = R.torque_limits[j] - tr;
        *tol = ttol;
    } else if (i < NF * T + NJ * T * O) {
        *gl = -1e19;
        *gu = 0;
        *tol = ctol;
    } else {
        const int q = i - (NF * T + NJ * T * O), j = q % NF;
        if (q < 2 * NF) {
            *gl = R.state_limits_lb[j] + R.qe;
            *gu = R.state_limits_ub[j] - R.qe;
        } else {
            *gl = -R.speed_limits[j] + R.qde;
            *gu = R.speed_limits[j] - R.qde;
        }
        *tol = 0.0;
    }
}

// the main planner's NLP (KPR/NLPclass.cu)
struct ArmourNlp {
    __device__ int m(const Batch& B) const { return B.m(); }
    __device__ void row_bounds(const Batch& B, int p, int i, double ttol, double ctol, double* gl, double* gu, double* tol) const {
        solver_row_bounds(B, p, i, ttol, ctol, gl, gu, tol);
    }
    __device__ double cost(const Batch& B, int p, const double* q_des, const double* k, double* grad) const {
        return solver_cost(B, p, q_des, k, grad);
    }
};

// block-wide maximum (all threads get it)
__device__ inline double solver_block_max(double v, double* s_red) {
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = s_red[0];
    for (int w = 1; w < SOLVER_THREADS / 32; w++) r = fmax(r, s_red[w]);
    return r;
}
// violation with the verdict's tolerances folded in: <= 0 means "finalize_solution would accept"
template <class Nlp>
__device__ inline double solver_violation(const Batch& B, const Nlp& nlp, int p, const double* g, double ttol, double ctol,
                                          double* s_red) {
    const int m = nlp.m(B);
    double v = -1e300;
    for (int i = threadIdx.x; i < m; i += SOLVER_THREADS) {
        double gl, gu, tol;
        nlp.row_bounds(B, p, i, ttol, ctol, &gl, &gu, &tol);
        v = fmax(v, g[i] - gu - tol);
        if (gl > -1e18) v = fmax(v, gl - g[i] - tol);
    }
    return solver_block_max(v, s_red);
}

// start: x = 0 (armtd_NLP::get_starting_point), cost and violation there from g(0)
template <class Nlp>
__global__ void __launch_bounds__(SOLVER_THREADS) k_solver_start(Batch B, Nlp nlp, SolverState S, const double* __restrict__ g) {
    const int p = blockIdx.x;
    __shared__ double s_red[SOLVER_THREADS / 32];
    const double viol = solver_violation(B, nlp, p, g + size_t(p) * nlp.m(B), S.torque_tol, S.collision_tol, s_red);
    if (threadIdx.x == 0) {
        double x[NF];
        for (int j = 0; j < NF; j++) x[j] = S.x[size_t(p) * NF + j];
        const double f = nlp.cost(B, p, S.q_des + size_t(p) * NF, x, nullptr);
        S.f[p] = f;
        S.viol[p] = viol;
        S.have_best[p] = viol <= 0;
        S.fbest[p] = f;
        if (viol <= 0)
            for (int j = 0; j < NF; j++) S.best[size_t(p) * NF + j] = x[j];
        S.delta[p] = 0.5;
        S.status[p] = SOLVER_RUNNING;
        S.iters[p] = 0;
        S.evals[p] = 1;
    }
}

// row `at` of the component-major row buffer of one problem
__device__ __forceinline__ void solver_store_row(double* rows, int at, const double* a, double sign, double b) {
    double r[NF];
    for (int j = 0; j < NF; j++) {
        r[j] = sign * a[j];
        rows[size_t(j) * SOLVER_ROWCAP + at] = r[j];
    }
    rows[size_t(7) * SOLVER_ROWCAP + at] = b;
    rows[size_t(8) * SOLVER_ROWCAP + at] = asqp::row_scale(r, NF);
}
__device__ __forceinline__ void solver_load_row(const double* rows, int i, double* a, double* b, double* scale) {
    for (int j = 0; j < NF; j++) a[j] = rows[size_t(j) * SOLVER_ROWCAP + i];
    *b = rows[size_t(7) * SOLVER_ROWCAP + i];
    *scale = rows[size_t(8) * SOLVER_ROWCAP + i];
}

// one SQP step from (g, J) at x: writes the trial point xt, or ends the problem (step below tolerance)
template <class Nlp>
__global__ void __launch_bounds__(SOLVER_THREADS)
k_solver_step(Batch B, Nlp nlp, SolverState S, const double* __restrict__ g_all, const double* __restrict__ jac_all, int it) {
    const int p = B.plist ? B.plist[blockIdx.x] : int(blockIdx.x), tid = threadIdx.x;
    if (S.status[p] != SOLVER_RUNNING) return;  // uniform per CTA
#ifdef SOLVER_PROFILE
    const long long pc0 = clock64();
#endif
    const int m = nlp.m(B);
    const double* g = g_all + size_t(p) * m;
    const double* J = jac_all + size_t(p) * m * NF;
    __shared__ double s_x[NF], s_gf[NF], s_h, s_delta;
    __shared__ int s_cnt[SOLVER_THREADS], s_total;
    if (tid == 0) {
        double x[NF], gf[NF], xt[NF];
        for (int j = 0; j < NF; j++) x[j] = S.x[size_t(p) * NF + j];
        const double* qd = S.q_des + size_t(p) * NF;
        nlp.cost(B, p, qd, x, gf);
        // curvature of the cost along the gradient from one extra evaluation (exact for the planner's quadratic cost)
        double h = 1.0, gn2 = 0;
        for (int j = 0; j < NF; j++) gn2 += gf[j] * gf[j];
        if (gn2 > 0) {
            const double eps = 1e-3 / sqrt(gn2);
            for (int j = 0; j < NF; j++) xt[j] = x[j] - eps * gf[j];
            const double f2 = nlp.cost(B, p, qd, xt, nullptr);
            const double curv = 2.0 * (f2 - S.f[p] + eps * gn2) / (eps * eps * gn2);
            if (curv > 1e-8) h = curv;
        }
        for (int j = 0; j < NF; j++) {
            s_x[j] = x[j];
            s_gf[j] = gf[j];
        }
        s_h = h;
        s_delta = S.delta[p];
        S.iters[p] = it + 1;
    }
    __syncthreads();
    const double h = s_h, delta = s_delta;
    // rows that can be reached inside the trust region, linearised, in row order (upper side, then lower side).
    // Warp w owns the contiguous segment [w * seg, (w + 1) * seg) of the m rows, its lanes take consecutive rows (coalesced
    // reads of g and J, four steps of 32 rows in flight).  Pass 0 only decides: the ballots of "upper side kept" / "lower
    // side kept" go to shared memory; the warp totals give every warp its base; pass 1 revisits the steps that keep
    // anything (a few per cent of them) and writes the rows at base + (kept entries before it), which is row order.
    extern __shared__ unsigned s_keep[];  // [SOLVER_WARPS][steps][2]
    const int warp = tid >> 5, lane = tid & 31;
    const int steps = solver_steps(m), seg = steps * 32;
    const int w0 = warp * seg;
    unsigned* keep = s_keep + size_t(warp) * steps * 2;
    double* rows = S.rows + size_t(p) * SOLVER_ROWCAP * SOLVER_ROWW;
    int wcount = 0;
    for (int st0 = 0; st0 < steps; st0 += 4) {
        bool pu[4], pl[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int i = w0 + (st0 + q) * 32 + lane;
            pu[q] = pl[q] = false;
            if (st0 + q < steps && i < m) {
                double gl, gu, tol;
                nlp.row_bounds(B, p, i, S.torque_tol, S.collision_tol, &gl, &gu, &tol);
                tol *= 0.5;  // aim inside the acceptance band
                double l1 = 0;
                for (int j = 0; j < NF; j++) l1 += fabs(J[size_t(i) * NF + j]);
                const double gi = g[i];
                const double bu = gu + tol - gi;
                const double bl = gi - (gl - tol);
                pu[q] = !(bu > l1 * delta);
                pl[q] = gl > -1e18 && !(bl > l1 * delta);
            }
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const unsigned mu = __ballot_sync(0xffffffffu, pu[q]), ml = __ballot_sync(0xffffffffu, pl[q]);
            if (st0 + q < steps && lane == 0) {
                keep[(st0 + q) * 2] = mu;
                keep[(st0 + q) * 2 + 1] = ml;
            }
            wcount += __popc(mu) + __popc(ml);
        }
    }
    s_cnt[tid] = wcount;  // (the same number in every lane of a warp)
    __syncthreads();
    int base = 0;
    for (int w = 0; w < warp; w++) base += s_cnt[w * 32];
    if (tid == 0) {
        int tot = 0;
        for (int w = 0; w < SOLVER_WARPS; w++) tot += s_cnt[w * 32];
        s_total = tot;
    }
    for (int st = 0; st < steps; st++) {
        const unsigned mu = keep[st * 2], ml = keep[st * 2 + 1];
        if ((mu | ml) == 0) continue;
        const unsigned below = (1u << lane) - 1u;
        const int at = base + __popc(mu & below) + __popc(ml & below);
        const bool ku = (mu >> lane) & 1u, kl = (ml >> lane) & 1u;
        if (ku || kl) {
            const int i = w0 + st * 32 + lane;
            double gl, gu, tol;
            nlp.row_bounds(B, p, i, S.torque_tol, S.collision_tol, &gl, &gu, &tol);
            tol *= 0.5;
            double a[NF];
            for (int j = 0; j < NF; j++) a[j] = J[size_t(i) * NF + j];
            if (ku && at < SOLVER_ROWCAP) solver_store_row(rows, at, a, 1.0, gu + tol - g[i]);
            if (kl && at + (ku ? 1 : 0) < SOLVER_ROWCAP) solver_store_row(rows, at + (ku ? 1 : 0), a, -1.0, g[i] - (gl - tol));
        }
        base += __popc(mu) + __popc(ml);
    }
    __syncthreads();
    __shared__ int s_nrows;
    if (tid == 0) {
        int nrows = s_total;
        if (nrows + 2 * NF > SOLVER_ROWCAP) {
            S.status[p] = SOLVER_ROW_OVERFLOW;
            nrows = -1;
        } else {
            // variable bounds and trust region: e_j . d <= min(delta, xu - x), -e_j . d <= min(delta, x - xl)
            for (int j = 0; j < NF; j++) {
                for (int sgn = 0; sgn < 2; sgn++) {
                    const double b = sgn == 0 ? fmin(delta, 1.0 - s_x[j]) : fmin(delta, s_x[j] - (-1.0));
                    if (b > 1.0 * delta) continue;  // push(): l1 = 1, the row is kept unless b > delta
                    double e[NF];
                    for (int q = 0; q < NF; q++) e[q] = 0.0;
                    e[j] = 1.0;
                    solver_store_row(rows, nrows, e, sgn == 0 ? 1.0 : -1.0, b);
                    nrows++;
                }
            }
        }
        s_nrows = nrows;
    }
    __syncthreads();
    const int nrows = s_nrows;
    if (nrows < 0) return;
#ifdef SOLVER_PROFILE
    const long long pc1 = clock64();
#endif
    // exact QP (host/active_set_qp.h; same statements as solve_qp() of the host solver): every round the CTA finds the
    // most violated row at the current d (scaled by 1 / |a|; ties: lowest index — what the host's ascending scan with a
    // strict comparison picks), thread 0 takes it into the active set
    __shared__ asqp::State<NF> s_qp;
    __shared__ double s_bv[SOLVER_THREADS / 32];
    __shared__ int s_bi[SOLVER_THREADS / 32], s_stop;
    if (tid == 0) {
        asqp::init(s_qp, NF, h, s_gf);
        s_stop = 0;
    }
    __syncthreads();
    int qp_it = 0;
    for (; qp_it < S.qp_sweeps; qp_it++) {
        double d[NF];
        for (int j = 0; j < NF; j++) d[j] = s_qp.d[j];
        double bv = asqp::VIOLATION_TOL;
        int bi = -1;
        for (int i = tid; i < nrows; i += SOLVER_THREADS) {
            double a[NF], b, sc;
            solver_load_row(rows, i, a, &b, &sc);
            const double v = asqp::row_violation(a, b, sc, d, NF);
            if (v > bv && !asqp::is_excluded(s_qp, i)) {
                bv = v;
                bi = i;
            }
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) {
                bv = ov;
                bi = oi;
            }
        }
        if ((tid & 31) == 0) {
            s_bv[tid >> 5] = bv;
            s_bi[tid >> 5] = bi;
        }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < SOLVER_THREADS / 32; w++) {
                const double ov = s_bv[w];
                const int oi = s_bi[w];
                if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) {
                    bv = ov;
                    bi = oi;
                }
            }
            if (bi < 0) {
                s_stop = 1;
            } else {
                double a[NF], b, sc;
                solver_load_row(rows, bi, a, &b, &sc);
                if (asqp::add_row(s_qp, bi, a, b) == 2) s_stop = 2;
            }
        }
        __syncthreads();
        if (s_stop) break;
    }
    if (tid != 0) return;
    double d[NF];
    for (int j = 0; j < NF; j++) d[j] = s_qp.d[j];
    const int n_sweeps = qp_it, n_moves = s_qp.drops;
    {
        S.dbg[p * 3 + 0] = nrows;
        S.dbg[p * 3 + 1] = n_sweeps;
        S.dbg[p * 3 + 2] = n_moves;
#ifdef SOLVER_PROFILE
        S.dbg[p * 3 + 0] = int((pc1 - pc0) >> 4);        // row building, cycles / 16
        S.dbg[p * 3 + 2] = int((clock64() - pc1) >> 4);  // QP, cycles / 16
#endif
        double dn = 0;
        for (int j = 0; j < NF; j++) {
            d[j] = fmax(-delta, fmin(delta, d[j]));
            const double xt = fmax(-1.0, fmin(1.0, s_x[j] + d[j]));
            S.xt[size_t(p) * NF + j] = xt;
            dn = fmax(dn, fabs(xt - s_x[j]));
        }
        if (dn < S.tol) {
            S.status[p] = (S.viol[p] <= 0) ? SOLVER_SUCCESS : SOLVER_INFEASIBLE;
            for (int j = 0; j < NF; j++) S.xt[size_t(p) * NF + j] = s_x[j];
        }
    }
}

// acceptance test of the trial point from g(xt): filter-style — feasible points must lower the cost, infeasible ones
// must lower the violation
template <class Nlp>
__global__ void __launch_bounds__(SOLVER_THREADS) k_solver_accept(Batch B, Nlp nlp, SolverState S, const double* __restrict__ gt_all,
                                                                  int last) {
    const int p = B.plist ? B.plist[blockIdx.x] : int(blockIdx.x);
    if (S.status[p] != SOLVER_RUNNING) return;
    __shared__ double s_red[SOLVER_THREADS / 32];
    const double vt = solver_violation(B, nlp, p, gt_all + size_t(p) * nlp.m(B), S.torque_tol, S.collision_tol, s_red);
    if (threadIdx.x == 0) {
        double xt[NF];
        for (int j = 0; j < NF; j++) xt[j] = S.xt[size_t(p) * NF + j];
        const double ft = nlp.cost(B, p, S.q_des + size_t(p) * NF, xt, nullptr);
        S.evals[p] += 1;
        const double f = S.f[p], viol = S.viol[p];
        const bool accept = (vt <= 0 && (viol > 0 || ft < f - 1e-12)) || (vt > 0 && viol > 0 && vt < viol - 1e-12);
        if (accept) {
            for (int j = 0; j < NF; j++) S.x[size_t(p) * NF + j] = xt[j];
            S.f[p] = ft;
            S.viol[p] = vt;
            S.delta[p] = fmin(1.0, S.delta[p] * 1.5);
            if (vt <= 0 && (!S.have_best[p] || ft < S.fbest[p])) {
                S.have_best[p] = 1;
                S.fbest[p] = ft;
                for (int j = 0; j < NF; j++) S.best[size_t(p) * NF + j] = xt[j];
            }
        } else {
            const double nd = S.delta[p] * 0.4;
            S.delta[p] = nd;
            if (nd < S.tol) S.status[p] = (viol <= 0) ? SOLVER_TINY_STEP : SOLVER_INFEASIBLE;
        }
        if (last && S.status[p] == SOLVER_RUNNING) S.status[p] = SOLVER_MAXITER;
    }
}

// the point handed to finalize_solution: the best accepted feasible point if there is one, else the last iterate
__global__ void k_solver_final(SolverState S, int nprob, double* __restrict__ k_opt, int* __restrict__ running) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nprob) return;
    const bool hb = S.have_best[p] != 0;
    for (int j = 0; j < NF; j++) k_opt[size_t(p) * NF + j] = hb ? S.best[size_t(p) * NF + j] : S.x[size_t(p) * NF + j];
    if (running && S.status[p] == SOLVER_RUNNING) atomicAdd(running, 1);
}
// the problems still running, as a list for the next launches (any order: the problems are independent)
__global__ void k_solver_compact(SolverState S, int nprob, int* __restrict__ running, int* __restrict__ list) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < nprob && S.status[p] == SOLVER_RUNNING) list[atomicAdd(running, 1)] = p;
}

}  // namespace armour
