// Constraint-side kernels of the hot path (sm_100a, FP64 SIMT, HBM-streaming):
//
//   k_hyperplanes  — K3a: buffered obstacle zonotope -> the half-spaces that can attain the maximum of a
//                    (link, interval, obstacle) row for some k in the box.  Replaces bufferObstaclesKernel +
//                    polytope_PH (reference KPR/CollisionChecking.cu:136-228, 14 launches).
//   k_constraints  — K3: slice every link / torque reach set at k (value and d/dk), evaluate the
//                    collision rows and their gradients, append the Bezier joint-limit rows; writes the
//                    whole g(k) and dense Jacobian.  Replaces PZsparse::slice (KPR/PZsparse.cu:404-555),
//                    checkCollisionKernel (KPR/CollisionChecking.cu:230-299) and the row assembly of
//                    armtd_NLP::eval_g / eval_jac_g (KPR/NLPclass.cu:272-396): 1 launch instead of
//                    7 launches + 8-9 blocking PCIe copies per call.
//   k_constraints_slow — the few collision rows without a stored candidate list, or all of them when k lies outside
//                    the box the lists were built for: full 72-plane scan from the generators.  Its own launch, so that
//                    k_constraints carries no stack frame for it.
//   k_verdict      — feasibility predicate of armtd_NLP::finalize_solution (KPR/NLPclass.cu:449-537).
//
// One CTA handles TB = 8 consecutive intervals of one problem, so that each output run per link is
// TB*O contiguous doubles (g) or TB*O*7 (Jacobian) and the hyper-plane chunk it streams is contiguous.
// Included by kernels.cu (one translation unit, so all kernels share the __constant__ block).
// Compiled with -fmad=false: coefficient arithmetic is plain round-to-nearest like the host reference.
#pragma once
#include <cuda_runtime.h>

#include "bezier.cuh"
#include "device_constants.cuh"
#include "layout.h"

namespace armour {

// tuning knobs of k_constraints (see the sweep quoted at the kernel)
#ifndef K3_CH
#define K3_CH 2   // monomials of a table fetched together by a slicing thread
#endif
#ifndef K3_CQ
#define K3_CQ 2   // candidate records in flight per collision row (2.05 stored per row on average)
#endif
#ifndef K3_MINB
#define K3_MINB 4 // resident CTAs per SM the register budget is sized for (48 registers per thread)
#endif

// ---------------------------------------------------------------------------------------------------
// Collision half-spaces of one (link, interval, obstacle) row.
//
// The buffered obstacle zonotope has 9 generators: 3 of the obstacle, the <= 3 pure link-generator
// columns and diag(radius) of the link reach set (KPR/CollisionChecking.cu:136-167).  Each of the
// C(9,2) = 36 generator pairs gives a unit normal C = g_a x g_b / |g_a x g_b| (zero if degenerate),
// an offset d = C . c_obs and a half-width delta = sum_j |C . g_j| (polytope_PH, :169-228); the
// constraint of the row is h(k) = -max_i max(C_i.p(k) - (d_i + delta_i), -C_i.p(k) - (-d_i + delta_i))
// with strict '>' in the scan order pos_0, neg_0, pos_1, ... (checkCollisionKernel, :230-299).
// for_each_plane() enumerates the pairs in the reference order (0,1),(0,2)...(7,8) with every index a
// compile-time constant, so the 27 generator components stay in registers.
template <class F>
__device__ __forceinline__ void for_each_plane(const double (&G)[9][3], const double (&oc)[3], F f) {
    int i = 0;
#pragma unroll
    for (int a = 0; a < 8; a++) {
#pragma unroll
        for (int b = a + 1; b < 9; b++) {
            const double cx = G[a][1] * G[b][2] - G[a][2] * G[b][1];
            const double cy = G[a][2] * G[b][0] - G[a][0] * G[b][2];
            const double cz = G[a][0] * G[b][1] - G[a][1] * G[b][0];
            const double nrm = sqrt(cx * cx + cy * cy + cz * cz);
            double C0 = 0, C1 = 0, C2 = 0;
            if (nrm > 0) {
                C0 = cx / nrm;
                C1 = cy / nrm;
                C2 = cz / nrm;
            }
            const double d = C0 * oc[0] + C1 * oc[1] + C2 * oc[2];
            double delta = 0.0;
#pragma unroll
            for (int gI = 0; gI < 9; gI++) delta += fabs(C0 * G[gI][0] + C1 * G[gI][1] + C2 * G[gI][2]);
            const bool nz = sqrt(C0 * C0 + C1 * C1 + C2 * C2) > 0;  // the test of checkCollisionKernel (:259)
            f(i, C0, C1, C2, d, delta, nz);
            i++;
        }
    }
}

__device__ __forceinline__ void load_row_generators(const double* __restrict__ ob, const double* __restrict__ LG,
                                                    double (&G)[9][3], double (&oc)[3]) {
#pragma unroll
    for (int e = 0; e < 3; e++) {
        oc[e] = ob[e];
#pragma unroll
        for (int gI = 0; gI < 3; gI++) G[gI][e] = ob[(gI + 1) * 3 + e];
#pragma unroll
        for (int gI = 0; gI < 6; gI++) G[gI + 3][e] = LG[e + gI * 3];
    }
}

// ---------------------------------------------------------------------------------------------------
// K3a: half-space candidate lists.  Replaces bufferObstaclesKernel + polytope_PH (14 launches in the
// reference).  The reference stores all 72 half-spaces of every row (12.9 MB per problem at 10
// obstacles) and scans them at every constraint evaluation.  Here the scan is bounded at build time:
// the link centre p(k) is a polynomial in k with known coefficients, so each half-space value
//     v_i(k) = s_i C_i . p(k) - b_i     lies in   [vc_i - rho_i, vc_i + rho_i]   for all |k_j| <= K_DOMAIN,
// rho_i = sum_m |C_i . g_m|.  A half-space whose upper bound is below the best lower bound can never
// be the maximum; neither can one that repeats the normal of an earlier candidate with a larger
// offset.  Only the survivors are stored, in scan order, as 32-byte records (s_i C_i, b_i), so that the
// evaluation kernel returns bit-identical values and gradients while reading ~100 B per row instead
// of 1440 B.  Rows with more than HP_CAP survivors are flagged and evaluated from the generators.
// One thread per (row, generator pair): HP_ROWS rows per CTA.  Step 1 computes the pair's two half-spaces and
// their value bounds, step 2 the row's best guaranteed lower bound, step 3 decides per candidate (bound
// filter + "an earlier candidate with the same normal and a smaller offset dominates"; dominance is
// transitive, so testing against all earlier candidates that pass the filter equals the sequential rule),
// step 4 writes the survivors at their scan-order positions.  Bit-identical lists to a sequential scan.
constexpr int HP_ROWS = 8;
constexpr int HP_STAGE = 24;  // link monomials staged in shared memory per row (longer tables are read from global)
constexpr int HP_THREADS = HP_ROWS * NCOMB;  // 288
// Two optional extras of the latency path (one planning problem, device pointers):
//   * unit_flag: the kernel was launched as a programmatic dependent of k_reachsets and may start before that grid has
//     finished; a CTA then waits until the intervals of ITS rows are flagged complete (acquire) — the half-space stage of
//     the early intervals runs under the tail of the reach-set kernel;
//   * stage: B.q0 / qd0 / qdd0 / obstacles point at the CALLER's buffers during the build; the first CTA of each problem
//     copies them into the context's own buffers (for the evaluations that follow), which saves four copies in front of
//     the build.
struct HpStage {
    double* q0;
    double* qd0;
    double* qdd0;
    double* obstacles;
};
__global__ void __launch_bounds__(HP_THREADS) k_hyperplanes(Batch B, const int* __restrict__ unit_flag, HpStage stage) {
    const int p = blockIdx.y;
    if (stage.q0 && blockIdx.x == 0) {
        for (int i = threadIdx.x; i < NF; i += HP_THREADS) {
            stage.q0[size_t(p) * NF + i] = B.q0[size_t(p) * NF + i];
            stage.qd0[size_t(p) * NF + i] = B.qd0[size_t(p) * NF + i];
            stage.qdd0[size_t(p) * NF + i] = B.qdd0[size_t(p) * NF + i];
        }
        for (int i = threadIdx.x; i < B.O * 12; i += HP_THREADS)
            stage.obstacles[size_t(p) * B.O * 12 + i] = B.obstacles[size_t(p) * B.O * 12 + i];
    }
    if (unit_flag) {
        if (threadIdx.x == 0) {
            const int per = B.NJ * TB * B.O, total = per * (B.T / TB);
            int r0 = blockIdx.x * HP_ROWS, r1 = r0 + HP_ROWS - 1;
            if (r1 >= total) r1 = total - 1;
            // rows are chunk-major, x = (l*TB + tt)*O + o inside a chunk
            int t_seen = -1;
            for (int r = r0; r <= r1; r++) {
                const int t = (r / per) * TB + ((r % per) / B.O) % TB;
                if (t == t_seen) continue;
                t_seen = t;
                const int* f = unit_flag + size_t(p) * B.T + t;
                int v;
                for (;;) {
                    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
                    if (v == B.epoch) break;
                    __nanosleep(200);
                }
            }
        }
        __syncthreads();
    }
    const int NJ = B.NJ, O = B.O, T = B.T;
    const int per_pair = NJ * TB * O;          // rows of one (problem, TB intervals) chunk
    const int rows_total = per_pair * (T / TB);
    const int lr = threadIdx.x / NCOMB, pi = threadIdx.x % NCOMB;  // local row, pair index
    const int r = blockIdx.x * HP_ROWS + lr;   // row of the problem, chunk-major
    __shared__ double s_G[HP_ROWS][9][3], s_oc[HP_ROWS][3], s_c[HP_ROWS][3];
    __shared__ double s_A[HP_ROWS][NCOMB][3], s_b[HP_ROWS][2 * NCOMB], s_up[HP_ROWS][2 * NCOMB], s_lo[HP_ROWS][NCOMB];
    __shared__ double s_lomax[HP_ROWS];
    __shared__ double s_vc[HP_ROWS][2 * NCOMB];           // value of each signed half-space at the centre of the k box
    __shared__ double s_gm[HP_ROWS][HP_STAGE][3];        // monomial coefficients of the row's link reach set
    __shared__ int s_best[HP_ROWS];                        // signed half-space with the best guaranteed lower bound
    __shared__ unsigned char s_flag[HP_ROWS][2 * NCOMB], s_list[HP_ROWS][2 * NCOMB];
    __shared__ int s_nlist[HP_ROWS];
    const bool live = r < rows_total;
    int tb = 0, x = 0;
    size_t idx = 0;
    if (live) {
        tb = r / per_pair;
        x = r - tb * per_pair;
        const int o = x % O, ltt = x / O, tt = ltt % TB, l = ltt / TB;
        idx = (size_t(p) * T + size_t(tb) * TB + tt) * NJ + l;
        if (pi < 27) {  // 9 generators x 3 components: 3 of the obstacle, then the 3x6 link matrix (column-major)
            const int gI = pi / 3, e = pi % 3;
            s_G[lr][gI][e] = (gI < 3) ? B.obstacles[(size_t(p) * O + o) * 12 + (gI + 1) * 3 + e] : B.link_gens[idx * 18 + e + (gI - 3) * 3];
        } else if (pi < 30) {
            s_oc[lr][pi - 27] = B.obstacles[(size_t(p) * O + o) * 12 + (pi - 27)];
        } else if (pi < 33) {
            s_c[lr][pi - 30] = B.link_c[idx * 3 + (pi - 30)];
        } else if (pi == 33) {
            s_nlist[lr] = 0;
        }
        const int n = B.link_n[idx];
        const int ns = n < HP_STAGE ? n : HP_STAGE;
        for (int q = pi; q < ns * 3; q += NCOMB) s_gm[lr][q / 3][q % 3] = B.link_g[idx * B.capL * 3 + q];
    }
    __syncthreads();
    bool nz = false;
    if (live) {  // step 1: same expressions as for_each_plane / the bounds of the sequential version
        const int a = c_combA[pi], b = c_combB[pi];
        const double(*G)[3] = s_G[lr];
        const double cx = G[a][1] * G[b][2] - G[a][2] * G[b][1];
        const double cy = G[a][2] * G[b][0] - G[a][0] * G[b][2];
        const double cz = G[a][0] * G[b][1] - G[a][1] * G[b][0];
        const double nrm = sqrt(cx * cx + cy * cy + cz * cz);
        double C0 = 0, C1 = 0, C2 = 0;
        if (nrm > 0) {
            C0 = cx / nrm;
            C1 = cy / nrm;
            C2 = cz / nrm;
        }
        const double d = C0 * s_oc[lr][0] + C1 * s_oc[lr][1] + C2 * s_oc[lr][2];
        double delta = 0.0;
#pragma unroll 1
        for (int gI = 0; gI < 9; gI++) delta += fabs(C0 * G[gI][0] + C1 * G[gI][1] + C2 * G[gI][2]);
        nz = sqrt(C0 * C0 + C1 * C1 + C2 * C2) > 0;  // the test of checkCollisionKernel (:259)
        const double dot = C0 * s_c[lr][0] + C1 * s_c[lr][1] + C2 * s_c[lr][2];
        const double vpos = dot - (d + delta);
        const double vneg = -dot - (-d + delta);
        const int n = B.link_n[idx];
        const int ns = n < HP_STAGE ? n : HP_STAGE;
        const double* __restrict__ lg = B.link_g + idx * B.capL * 3;
        double rr = 0.0;
#pragma unroll 1
        for (int mI = 0; mI < ns; mI++) rr += fabs(C0 * s_gm[lr][mI][0] + C1 * s_gm[lr][mI][1] + C2 * s_gm[lr][mI][2]);
#pragma unroll 1
        for (int mI = ns; mI < n; mI++) rr += fabs(C0 * lg[mI * 3 + 0] + C1 * lg[mI * 3 + 1] + C2 * lg[mI * 3 + 2]);
        // |k_j| <= K_DOMAIN, total degree <= 21; plus evaluation round-off (values are O(1))
        const double rho = rr * HP_RHO_SCALE + (1e-10 + 1e-12 * (fabs(dot) + fabs(d) + delta));
        s_A[lr][pi][0] = C0;
        s_A[lr][pi][1] = C1;
        s_A[lr][pi][2] = C2;
        s_b[lr][2 * pi] = d + delta;
        s_b[lr][2 * pi + 1] = -d + delta;
        s_up[lr][2 * pi] = nz ? vpos + rho : -1e300;
        s_up[lr][2 * pi + 1] = nz ? vneg + rho : -1e300;
        s_lo[lr][pi] = nz ? fmax(vpos, vneg) - rho : -1e300;
        s_vc[lr][2 * pi] = vpos;
        s_vc[lr][2 * pi + 1] = vneg;
    }
    __syncthreads();
    if (live && pi == 0) {  // step 2: the best guaranteed lower bound of the row, and who holds it
        double lo_max = -100000000;
        int best = -1;
#pragma unroll 1
        for (int i = 0; i < NCOMB; i++) {
            if (s_lo[lr][i] > lo_max) {
                lo_max = s_lo[lr][i];
                best = 2 * i + (s_vc[lr][2 * i + 1] > s_vc[lr][2 * i] ? 1 : 0);
            }
        }
        s_lomax[lr] = lo_max;
        s_best[lr] = best;
    }
    __syncthreads();
    // step 2b: pairwise test against that half-space j.  v_j(k) - v_i(k) = (vc_j - vc_i) + (A_j - A_i) . sum_m g_m mono_m(k)
    // >= (vc_j - vc_i) - sum_m |(A_j - A_i) . g_m| for every k of the box: the variation the two half-spaces share
    // cancels, so this removes the half-spaces that are nearly parallel to j but further out, which the separate
    // bounds of step 1 cannot.  i is dropped only when the difference is positive by a margin (never on a tie), so
    // the maximum over the survivors and its first attaining index are those of the full scan.
    bool drop[2] = {false, false};
    if (live && nz && s_best[lr] >= 0) {
        const int jb = s_best[lr];
        const double sj = (jb & 1) ? -1.0 : 1.0;
        const double J0 = sj * s_A[lr][jb >> 1][0], J1 = sj * s_A[lr][jb >> 1][1], J2 = sj * s_A[lr][jb >> 1][2];
        const double vj = s_vc[lr][jb];
        const int n = B.link_n[idx];
        const int ns = n < HP_STAGE ? n : HP_STAGE;
        const double* __restrict__ lg = B.link_g + idx * B.capL * 3;
#pragma unroll 1
        for (int sgn = 0; sgn < 2; sgn++) {
            const int sI = 2 * pi + sgn;
            if (sI == jb || !(s_up[lr][sI] >= s_lomax[lr])) continue;
            const double sg = sgn ? -1.0 : 1.0;
            const double D0 = J0 - sg * s_A[lr][pi][0], D1 = J1 - sg * s_A[lr][pi][1], D2 = J2 - sg * s_A[lr][pi][2];
            double rd = 0.0;
#pragma unroll 1
            for (int mI = 0; mI < ns; mI++) rd += fabs(D0 * s_gm[lr][mI][0] + D1 * s_gm[lr][mI][1] + D2 * s_gm[lr][mI][2]);
#pragma unroll 1
            for (int mI = ns; mI < n; mI++) rd += fabs(D0 * lg[mI * 3 + 0] + D1 * lg[mI * 3 + 1] + D2 * lg[mI * 3 + 2]);
            const double vi = s_vc[lr][sI];
            const double margin = rd * HP_RHO_SCALE + (1e-10 + 1e-12 * (fabs(vi) + fabs(vj) + fabs(s_b[lr][sI]) + fabs(s_b[lr][jb])));
            drop[sgn] = (vj - vi) > margin;
        }
    }
    __syncthreads();
    if (live) {
        if (drop[0]) s_up[lr][2 * pi] = -1e300;
        if (drop[1]) s_up[lr][2 * pi + 1] = -1e300;
    }
    __syncthreads();
    // step 3: the candidates that pass the filters enter a short list per row (a handful of the 72; arrival order,
    // the tests below do not depend on it)
    if (live) {
        const double lo_max = s_lomax[lr];
#pragma unroll 1
        for (int sgn = 0; sgn < 2; sgn++) {
            const int sI = 2 * pi + sgn;  // position in the scan order pos_0, neg_0, pos_1, ...
            if (nz && s_up[lr][sI] >= lo_max) s_list[lr][atomicAdd(&s_nlist[lr], 1)] = (unsigned char)sI;
        }
    }
    __syncthreads();
    // step 3b: a listed candidate is dropped when a listed candidate EARLIER in the scan order has the same normal and
    // a smaller or equal offset (it can never win the strict '>' scan).  Dominance is transitive, so testing against
    // all earlier listed candidates equals the sequential rule.
    bool keep[2] = {false, false};
    if (live) {
        const double lo_max = s_lomax[lr];
        const int nl = s_nlist[lr];
#pragma unroll 1
        for (int sgn = 0; sgn < 2; sgn++) {
            const int sI = 2 * pi + sgn;
            bool k = nz && s_up[lr][sI] >= lo_max;
            if (k) {
                const double sg = sgn ? -1.0 : 1.0;
                const double A0 = sg * s_A[lr][pi][0], A1 = sg * s_A[lr][pi][1], A2 = sg * s_A[lr][pi][2], bb = s_b[lr][sI];
#pragma unroll 1
                for (int c = 0; c < nl && k; c++) {
                    const int q = s_list[lr][c];
                    if (q >= sI) continue;
                    const double sq = (q & 1) ? -1.0 : 1.0;
                    const int qi = q >> 1;
                    if (sq * s_A[lr][qi][0] == A0 && sq * s_A[lr][qi][1] == A1 && sq * s_A[lr][qi][2] == A2 && s_b[lr][q] <= bb)
                        k = false;
                }
            }
            keep[sgn] = k;
            s_flag[lr][sI] = k ? 1 : 0;
        }
    }
    __syncthreads();
    if (live) {  // step 4: survivors to their scan-order positions (counted over the short list)
        const size_t chunk = size_t(p) * (T / TB) + tb;
        // the row's fixed run of HP_CAP records in the chunk's evaluation image; k_pack_image compacts the runs
        double* row = reinterpret_cast<double*>(B.img + chunk * B.img_chunk() + B.img_hdr()) + size_t(x) * HP_CAP * 4;
        const size_t cstride = 4;
        const int nl = s_nlist[lr];
        if (keep[0] || keep[1] || pi == 0) {
            int count = 0, before[2] = {0, 0};
#pragma unroll 1
            for (int c = 0; c < nl; c++) {
                const int q = s_list[lr][c];
                if (s_flag[lr][q]) {
                    count++;
                    before[0] += (q < 2 * pi);
                    before[1] += (q < 2 * pi + 1);
                }
            }
            if (count <= HP_CAP) {
#pragma unroll 1
                for (int sgn = 0; sgn < 2; sgn++) {
                    if (keep[sgn]) {
                        const double sg = sgn ? -1.0 : 1.0;
                        double* e = row + size_t(before[sgn]) * cstride;
                        e[0] = sg * s_A[lr][pi][0];
                        e[1] = sg * s_A[lr][pi][1];
                        e[2] = sg * s_A[lr][pi][2];
                        e[3] = s_b[lr][2 * pi + sgn];
                    }
                }
            }
            if (pi == 0) B.hp_cnt[chunk * per_pair + x] = (count > HP_CAP) ? (unsigned char)HP_OVERFLOW : (unsigned char)count;
            if (pi == 0 && count > HP_CAP) atomicAdd(&B.hp_slow[p], 1);  // k_constraints_slow evaluates the row
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Pack the evaluation image of one chunk (layout: Batch::img) at the end of a build.  One CTA per (chunk, problem):
//   1. the rows are taken in tiles of PK_TILE: exclusive prefix of the tile's stored candidate counts (HP_OVERFLOW rows store
//      none) in shared memory, continued from the previous tiles;
//   2. the tile's records move from the rows' fixed runs of HP_CAP (k_hyperplanes) to their CSR positions, in place: the
//      record with CSR index c comes from run position x * HP_CAP + q >= c, so passes over increasing CSR indices
//      [c0, c0 + PK_THREADS) that read all their records before they write any never overwrite a record a later pass (of
//      this tile or a later one) still has to read;
//   3. header, then the link and torque tables at their exact lengths behind the records.
// Problems whose build failed are skipped: k_constraints writes their fail-safe rows without reading the image.
constexpr int PK_THREADS = 256;
constexpr int PK_TILE = 1024;  // rows per tile (a multiple of 32: the row-group bases are written tile by tile)
constexpr int PK_ROWS_PER_THREAD = PK_TILE / PK_THREADS;
__global__ void __launch_bounds__(PK_THREADS) k_pack_image(Batch B) {
    const int tb = blockIdx.x, p = blockIdx.y, tid = threadIdx.x;
    if (B.failed(p) != 0) return;
    const int NJ = B.NJ, T = B.T, rows = B.img_rows();
    const size_t chunk = size_t(p) * (T / TB) + tb;
    unsigned char* img = B.img + chunk * B.img_chunk();
    double* imgd = reinterpret_cast<double*>(img);
    const unsigned char* cnt = B.hp_cnt + chunk * rows;
    __shared__ unsigned s_off[PK_TILE + 1];  // first CSR record of each row of the tile, then the tile's end
    __shared__ unsigned s_part[PK_THREADS];
    __shared__ unsigned s_carry;             // records of the rows before the tile
    __shared__ int s_loff[TB * MAXJ + 1], s_uoff[TB * NF + 1];
    if (tid == 0) {
        s_carry = 0;
        // table offsets (counts clamped to the capacities: a valid build never exceeds them)
        int a = 0;
        for (int i = 0; i < TB * NJ; i++) {
            s_loff[i] = a;
            a += min(B.link_n[(size_t(p) * T + tb * TB) * NJ + i], B.capL);
        }
        s_loff[TB * NJ] = a;
        a = 0;
        for (int i = 0; i < TB * NF; i++) {
            s_uoff[i] = a;
            a += min(B.u_n[(size_t(p) * T + tb * TB) * NF + i], B.capU);
        }
        s_uoff[TB * NF] = a;
    }
    double4* rec = reinterpret_cast<double4*>(img + B.img_hdr());
    unsigned* grp = reinterpret_cast<unsigned*>(img + B.img_grp());
    for (int t0 = 0; t0 < rows; t0 += PK_TILE) {
        const int n = min(PK_TILE, rows - t0);
        // 1. prefix of the tile's counts: each thread PK_ROWS_PER_THREAD consecutive rows, then the thread sums
        const int r0 = min(tid * PK_ROWS_PER_THREAD, n), r1 = min(r0 + PK_ROWS_PER_THREAD, n);
        unsigned sum = 0;
        for (int x = r0; x < r1; x++) sum += cnt[t0 + x] == HP_OVERFLOW ? 0u : cnt[t0 + x];
        s_part[tid] = sum;
        __syncthreads();  // (also publishes s_carry and the table offsets, or the previous tile's carry)
        if (tid == 0) {
            unsigned run = s_carry;
            for (int i = 0; i < PK_THREADS; i++) {
                const unsigned v = s_part[i];
                s_part[i] = run;
                run += v;
            }
            s_off[n] = run;
        }
        __syncthreads();
        sum = s_part[tid];
        for (int x = r0; x < r1; x++) {
            s_off[x] = sum;
            if (((t0 + x) & 31) == 0) grp[(t0 + x) >> 5] = sum;
            sum += cnt[t0 + x] == HP_OVERFLOW ? 0u : cnt[t0 + x];
        }
        __syncthreads();
        // 2. the tile's records to their CSR positions
        const unsigned first = s_off[0], end = s_off[n];
        for (unsigned c0 = first; c0 < end; c0 += PK_THREADS) {
            const unsigned c = c0 + tid;
            double4 v;
            if (c < end) {
                int lo = 0, hi = n - 1;  // last row of the tile whose first record is <= c (the row that holds c)
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (s_off[mid] <= c) lo = mid; else hi = mid - 1;
                }
                v = rec[size_t(t0 + lo) * HP_CAP + (c - s_off[lo])];
            }
            __syncthreads();
            if (c < end) rec[c] = v;
            __syncthreads();
        }
        if (tid == 0) s_carry = end;  // read by thread 0 only, after the next tile's first barrier
        __syncthreads();
    }
    __syncthreads();
    const unsigned total = s_carry;
    // 3. header and tables
    const int nlink = s_loff[TB * NJ], ntorque = s_uoff[TB * NF];
    const size_t l0 = B.img_hdr() / 8 + size_t(total) * 4;  // first double of the link records
    const size_t u0 = l0 + size_t(nlink) * 4;                // first torque coefficient
    const size_t k0 = (u0 + ntorque) * 4;                    // first torque key (uint16 units)
    const size_t lidx = (size_t(p) * T + tb * TB) * NJ, uidx = (size_t(p) * T + tb * TB) * NF;
    for (int i = tid; i < TB * NJ; i += PK_THREADS)
        reinterpret_cast<int2*>(img)[i] = make_int2(int(l0) + 4 * s_loff[i], s_loff[i + 1] - s_loff[i]);
    for (int i = tid; i < TB * NF; i += PK_THREADS)
        reinterpret_cast<int4*>(img + B.img_ut())[i] = make_int4(int(u0) + s_uoff[i], int(k0) + s_uoff[i], s_uoff[i + 1] - s_uoff[i], 0);
    for (int i = tid; i < TB * NJ * 3; i += PK_THREADS) {
        reinterpret_cast<double*>(img + B.img_lc())[i] = B.link_c[lidx * 3 + i];
        reinterpret_cast<double*>(img + B.img_lr())[i] = B.link_r[lidx * 3 + i];
    }
    for (int i = tid; i < TB * NF; i += PK_THREADS) {
        reinterpret_cast<double*>(img + B.img_uc())[i] = B.u_c[uidx + i];
        reinterpret_cast<double*>(img + B.img_ur())[i] = B.u_r[uidx + i];
    }
    for (int x = tid; x < rows; x += PK_THREADS) img[B.img_cnt() + x] = cnt[x];
    for (int q = tid; q < TB * NJ * B.capL; q += PK_THREADS) {
        const int i = q / B.capL, mI = q - i * B.capL;
        if (mI >= s_loff[i + 1] - s_loff[i]) continue;
        const size_t src = (lidx + i) * B.capL + mI;
        double* dst = imgd + l0 + size_t(s_loff[i] + mI) * 4;
        dst[0] = B.link_g[src * 3 + 0];
        dst[1] = B.link_g[src * 3 + 1];
        dst[2] = B.link_g[src * 3 + 2];
        dst[3] = __longlong_as_double((long long)B.link_key[src]);  // key in the low half-word (little-endian)
    }
    for (int q = tid; q < TB * NF * B.capU; q += PK_THREADS) {
        const int i = q / B.capU, mI = q - i * B.capU;
        if (mI >= s_uoff[i + 1] - s_uoff[i]) continue;
        const size_t src = (uidx + i) * B.capU + mI;
        imgd[u0 + s_uoff[i] + mI] = B.u_g[src];
        reinterpret_cast<uint16_t*>(img)[k0 + s_uoff[i] + mI] = B.u_key[src];
    }
}
cudaError_t launch_pack_image(const Batch& B, cudaStream_t st) {
    if (B.nprob == 0) return cudaSuccess;
    k_pack_image<<<dim3(B.T / TB, B.nprob), PK_THREADS, 0, st>>>(B);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// K3
// Slow path of one collision row: scan all 72 half-spaces computed from the generators
// (checkCollisionKernel, KPR/CollisionChecking.cu:230-299).  Only k_constraints_slow calls it.
__device__ __noinline__ void row_from_generators(const double* __restrict__ ob, const double* __restrict__ LG,
                                                 double c0, double c1, double c2, double* max_out, double* A0o,
                                                 double* A1o, double* A2o) {
    double G[9][3], oc[3];
    load_row_generators(ob, LG, G, oc);
    double max_elt = -100000000, A0 = 0, A1 = 0, A2 = 0;
    for_each_plane(G, oc, [&](int, double a0, double a1, double a2, double d, double dl, bool nz) {
        if (!nz) return;
        const double dot = a0 * c0 + a1 * c1 + a2 * c2;
        const double pos = dot - (d + dl);
        const double neg = -dot - (-d + dl);
        if (pos > max_elt) {
            max_elt = pos;
            A0 = -a0; A1 = -a1; A2 = -a2;
        }
        if (neg > max_elt) {
            max_elt = neg;
            A0 = a0; A1 = a1; A2 = a2;
        }
    });
    *max_out = max_elt;
    *A0o = A0;
    *A1o = A1;
    *A2o = A2;
}

// One component of one reach set sliced at k: value and all seven d/dk in a single pass over the
// monomials.  Per monomial the factors k_j^{d_j} are applied in ascending j exactly like
// PZsparse::slice (KPR/PZsparse.cu:404-435) and its gradient overloads (:477-555); a factor with
// d_j = 0 is 1.0 and is skipped (exact).  D[v] carries coef * prod_{j<v} f_j * f'_v * prod_{v<j} f_j.
__device__ __forceinline__ void slice_component(const uint16_t* __restrict__ keys, const double* __restrict__ coef,
                                                int n, int kstride, int cstride, const double2 (*kpd)[4], double& value,
                                                double (&grad)[NF]) {
    constexpr int CH = K3_CH;  // monomials fetched together: the loads of a chunk are independent and overlap
    for (int m0 = 0; m0 < n; m0 += CH) {
        unsigned kk[CH];
        double cc[CH];
#pragma unroll
        for (int i = 0; i < CH; i++) {
            const bool on = m0 + i < n;
            kk[i] = on ? keys[(m0 + i) * kstride] : 0u;
            cc[i] = on ? coef[(m0 + i) * cstride] : 0.0;
        }
#pragma unroll 1
        for (int i = 0; i < CH; i++) {
            if (m0 + i >= n) break;
            // (dynamic index into kk / cc would spill: rotate instead)
            const unsigned key = kk[0];
            double val = cc[0];
#pragma unroll
            for (int q = 0; q + 1 < CH; q++) {
                kk[q] = kk[q + 1];
                cc[q] = cc[q + 1];
            }
            // No branch on the degree: kpd[j][0] = {1, 0}, and x * 1.0 is exact, val * 0.0 adds a zero to the
            // gradient: the same values as skipping the factor, without seven divergent branches per monomial.
            double D[NF];
#pragma unroll
            for (int j = 0; j < NF; j++) {
                const double2 fd = kpd[j][(key >> (2 * j)) & 3];
                D[j] = val * fd.y;
#pragma unroll
                for (int v = 0; v < j; v++) D[v] *= fd.x;
                val *= fd.x;
            }
            value += val;
#pragma unroll
            for (int v = 0; v < NF; v++) grad[v] += D[v];
        }
    }
}

// Warp roles: warps [0, 6) slice the link reach sets (one thread per (interval, link, component)), warps
// [6, 10) slice the torque reach sets, two lanes per (interval, joint) table (the torque tables are ~3x longer).
// The link warps meet on named barrier 1 and go straight to the collision rows; the torque warps write their
// rows, then join through barrier 2 (on which the link warps only arrive), so nobody waits for the slowest
// slice.  Collision rows are handed out in chunks of 32 from a shared counter.
#ifndef K3_DIRECT_J
#define K3_DIRECT_J 1      // 1: a lane stores the 7 Jacobian entries of its row itself (56 contiguous bytes); 0: transposition
#endif
#ifndef K3_SKIP_ZERO_DK
#define K3_SKIP_ZERO_DK 0   // 1: no look-ups / products for d/dk_v with v above the link index (exactly zero); measured: no gain
#endif
#ifndef K3_STREAM_STORES
#define K3_STREAM_STORES 0  // 1: Jacobian rows with st.global.cs (evict-first)
#endif
#if K3_STREAM_STORES
#define K3_ST2(p, a, b) __stcs(reinterpret_cast<double2*>(p), make_double2(a, b))
#define K3_ST1(p, a) __stcs(p, a)
#else
#define K3_ST2(p, a, b) (*reinterpret_cast<double2*>(p) = make_double2(a, b))
#define K3_ST1(p, a) (*(p) = (a))
#endif
#ifndef K3_LD_NOALLOC
#define K3_LD_NOALLOC 0     // 1: candidate records with ld.global.nc.L1::no_allocate
#endif
#ifndef K3_LD256
#define K3_LD256 1
#endif
#ifndef K3_POWER_TABLES
#define K3_POWER_TABLES 1  // 1: slices against two power-product tables built per CTA (2 products + 8 fused multiply-adds + 5
                           // look-ups per monomial); 0: factor by factor like the reference (35 + 7 look-ups)
#endif
// Power-product tables of one k (built per CTA, one entry per thread, before the slices).  A k-only monomial key holds seven
// 2-bit degrees (SURVEY A.1): the key is split into its low 6 bits (k_0..k_2, 64 entries {M, dM/dk_0..2}) and its high 8 bits
// (k_3..k_6, 256 entries {M, dM/dk_3..6}).  A factor of degree 0 is the exact 1.0 and its derivative the exact 0.0, as in
// PZsparse::slice (KPR/PZsparse.cu:404-555); the association differs from the reference's coef * f_0 * f_1 * ... by a few ulp
// of each term (bar: 1e-9).
constexpr int PT_LO = 64, PT_LO_STRIDE = 4;    // doubles per entry: 32 B, two 16-byte loads
constexpr int PT_HI = 256, PT_HI_STRIDE = 6;   // 5 used + 1 pad: 48 B, three 16-byte loads
__device__ __forceinline__ void power_and_slope(double k, int d, double& f, double& fp) {
    f = d == 0 ? 1.0 : d == 1 ? k : d == 2 ? k * k : k * k * k;
    fp = d == 0 ? 0.0 : d == 1 ? 1.0 : d == 2 ? 2.0 * k : 3.0 * (k * k);
}
// entry `e` of the table over the NV variables v0 .. v0+NV-1: out[0] = prod f_v, out[1+i] = f'_{v0+i} prod_{u != i} f_u
template <int NV>
__device__ __forceinline__ void power_table_entry(const double* __restrict__ k, int v0, int e, double* out) {
    double f[NV], fp[NV];
#pragma unroll
    for (int i = 0; i < NV; i++) power_and_slope(k[v0 + i], (e >> (2 * i)) & 3, f[i], fp[i]);
    double M = f[0];
#pragma unroll
    for (int i = 1; i < NV; i++) M *= f[i];
    out[0] = M;
#pragma unroll
    for (int i = 0; i < NV; i++) {
        double G = fp[i];
#pragma unroll
        for (int u = 0; u < NV; u++)
            if (u != i) G *= f[u];
        out[1 + i] = G;
    }
}
__device__ __forceinline__ void slice_component_pt(const uint16_t* __restrict__ keys, const double* __restrict__ coef, int n,
                                                   int kstride, int cstride, const double* __restrict__ pt_lo,
                                                   const double* __restrict__ pt_hi, double& value, double (&grad)[NF]) {
    constexpr int CH = K3_CH;
    for (int m0 = 0; m0 < n; m0 += CH) {
        unsigned kk[CH];
        double cc[CH];
#pragma unroll
        for (int i = 0; i < CH; i++) {
            const bool on = m0 + i < n;
            kk[i] = on ? keys[(m0 + i) * kstride] : 0u;
            cc[i] = on ? coef[(m0 + i) * cstride] : 0.0;
        }
        // a monomial past the end has coefficient 0 and key 0: it adds exact zeros, so the chunk needs no tail test
#pragma unroll
        for (int i = 0; i < CH; i++) {
            const double2* L = reinterpret_cast<const double2*>(pt_lo + (kk[i] & (PT_LO - 1)) * PT_LO_STRIDE);
            const double2* H = reinterpret_cast<const double2*>(pt_hi + ((kk[i] >> 6) & (PT_HI - 1)) * PT_HI_STRIDE);
            const double2 l0 = L[0], l1 = L[1], h0 = H[0], h1 = H[1], h2 = H[2];
            const double cl = cc[i] * l0.x, ch = cc[i] * h0.x;
            value = fma(cl, h0.x, value);
            grad[0] = fma(ch, l0.y, grad[0]);
            grad[1] = fma(ch, l1.x, grad[1]);
            grad[2] = fma(ch, l1.y, grad[2]);
            grad[3] = fma(cl, h0.y, grad[3]);
            grad[4] = fma(cl, h1.x, grad[4]);
            grad[5] = fma(cl, h1.y, grad[5]);
            grad[6] = fma(cl, h2.x, grad[6]);
        }
    }
}
constexpr int K3_LINK_THREADS = ((TB * 3 * MAXJ + 31) / 32) * 32;  // 192 for TB = 8
#ifndef K3_TORQUE_LANES_N
#define K3_TORQUE_LANES_N 2
#endif
constexpr int K3_TORQUE_LANES = K3_TORQUE_LANES_N;  // lanes per torque table in the slice phase (a power of two)
constexpr int K3_THREADS = K3_LINK_THREADS + ((TB * NF * K3_TORQUE_LANES + 31) / 32) * 32;
constexpr int K3_CNT_SMEM = 2048;  // rows per CTA whose candidate counts are staged in shared memory
constexpr int K3_WARPS = K3_THREADS / 32;
constexpr int K3_TORQUE_T0 = K3_LINK_THREADS;
static_assert(TB * 3 * MAXJ <= K3_LINK_THREADS && K3_TORQUE_T0 + TB * NF * K3_TORQUE_LANES <= K3_THREADS,
              "thread map of the slice phase");

// Register budget (round-1 sweep on B200, 1 024 worlds, ms per launch): 64 registers / 3 CTAs per SM with 8 monomials and
// 4 candidate records in flight per thread 0.81; the same at 96 registers / 2 CTAs 0.98, at 48 / 4 CTAs 1.68 (spills);
// 2 monomials + 2 records in flight at 64 / 3 CTAs 0.73, at 48 / 4 CTAs 0.66, at 40 / 5 CTAs 0.81.  The kernel lives
// on resident warps, not on loads in flight per warp: anything that spills or costs a CTA per SM loses.
#if K3_POWER_TABLES
#define K3_SLICE slice_component_pt
#define K3_SLICE_TABLES pt_lo, pt_hi
#else
#define K3_SLICE slice_component
#define K3_SLICE_TABLES kpd
#endif
__global__ void __launch_bounds__(K3_THREADS, K3_MINB)
k_constraints(Batch B, const double* __restrict__ kin, double* __restrict__ g, double* __restrict__ jac) {
    const int tb = blockIdx.x, p = B.plist ? B.plist[blockIdx.y] : int(blockIdx.y);
    const int NJ = B.NJ, O = B.O, T = B.T;
    const int m = B.m();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#if K3_POWER_TABLES
    __shared__ __align__(16) double pt_lo[PT_LO * PT_LO_STRIDE];  // power products of k_0..k_2 and their slopes
    __shared__ __align__(16) double pt_hi[PT_HI * PT_HI_STRIDE];  // the same for k_3..k_6
#else
    __shared__ double2 kpd[NF][4];  // {k_j^d, d/dk_j k_j^d} for d = 0..3
#endif
    __shared__ __align__(4) unsigned char s_cnt[K3_CNT_SMEM];  // candidate counts of this CTA's rows
    __shared__ double s_lc[TB][MAXJ][3];
    __shared__ double s_dlc[TB][MAXJ][NF][3];
#if !K3_DIRECT_J
    __shared__ double s_stage[K3_WARPS][32 * NF];  // per-warp transpose buffer: Jacobian rows leave coalesced
#endif
    __shared__ double s_tj[TB * NF * NF];          // torque rows of the Jacobian: leave as one contiguous run
    __shared__ int s_in_domain;
    __shared__ int s_next;  // next chunk of 32 collision rows

    if (B.failed(p) != 0) {
        // the build of this problem overflowed a table (ARMOUR_ERR_CAPACITY): its reach sets are not valid.  Fail-safe rows:
        // every torque and collision row violated, zero Jacobian -> no caller can take the problem for feasible.
        double* gp0 = g ? g + size_t(p) * m : nullptr;
        double* jp0 = jac ? jac + size_t(p) * m * NF : nullptr;
        for (int i = tid; i < TB * NF; i += K3_THREADS) {
            if (gp0) gp0[size_t(tb) * TB * NF + i] = 1e300;
            if (jp0)
                for (int v = 0; v < NF; v++) jp0[(size_t(tb) * TB * NF + i) * NF + v] = 0.0;
        }
        for (int x = tid; x < NJ * TB * O; x += K3_THREADS) {
            const int o = x % O, ltt = x / O, tt = ltt % TB, l = ltt / TB;
            const size_t r = size_t(NF) * T + (size_t(l) * T + tb * TB + tt) * O + o;
            if (gp0) gp0[r] = 1e300;
            if (jp0)
                for (int v = 0; v < NF; v++) jp0[r * NF + v] = 0.0;
        }
        if (tb == 0 && tid < 4 * NF) {
            const size_t r = size_t(NF) * T + size_t(NJ) * T * O + tid;
            if (gp0) gp0[r] = 0.0;
            if (jp0)
                for (int v = 0; v < NF; v++) jp0[r * NF + v] = 0.0;
        }
        return;
    }
    if (tid == 32) {
        bool in = true;
        for (int j = 0; j < NF; j++) in = in && (fabs(kin[size_t(p) * NF + j]) <= K_DOMAIN);
        s_in_domain = in ? 1 : 0;
        s_next = 0;
    }
#if K3_POWER_TABLES
    for (int q = tid; q < PT_HI + PT_LO; q += K3_THREADS) {  // one table entry per thread (320 entries)
        if (q < PT_HI) {
            power_table_entry<4>(kin + size_t(p) * NF, 3, q, pt_hi + q * PT_HI_STRIDE);
            pt_hi[q * PT_HI_STRIDE + 5] = 0.0;
        } else {
            power_table_entry<3>(kin + size_t(p) * NF, 0, q - PT_HI, pt_lo + (q - PT_HI) * PT_LO_STRIDE);
        }
    }
#else
    if (tid < NF) {
        const double k = kin[size_t(p) * NF + tid];
        kpd[tid][0] = make_double2(1.0, 0.0);
        kpd[tid][1] = make_double2(k, 1.0);
        kpd[tid][2] = make_double2(k * k, 2.0 * k);
        kpd[tid][3] = make_double2(k * k * k, 3.0 * (k * k));
    }
#endif
    const int per_pair = NJ * TB * O;
    const size_t chunk = size_t(p) * (T / TB) + tb;
    const unsigned char* __restrict__ img = B.img + chunk * B.img_chunk();  // everything this CTA reads of the build
    const double* __restrict__ imgd = reinterpret_cast<const double*>(img);
    const bool cnt_in_smem = per_pair <= K3_CNT_SMEM;
    __syncthreads();

    double* gp = g ? g + size_t(p) * m : nullptr;
    double* jp = jac ? jac + size_t(p) * m * NF : nullptr;

    // ---- phase 1: slices
    if (tid < K3_LINK_THREADS) {
        // candidate counts of the CTA's rows: fetched now, parked in shared memory after the slice (the loads are in
        // flight meanwhile), visible to everybody through barriers 1 and 2.  per_pair is a multiple of 8: whole words
        constexpr int CW = (K3_CNT_SMEM / 4 + K3_LINK_THREADS - 1) / K3_LINK_THREADS;
        unsigned cw[CW];
        if (cnt_in_smem) {
            const unsigned* src = reinterpret_cast<const unsigned*>(img + B.img_cnt());
#pragma unroll
            for (int q = 0; q < CW; q++) cw[q] = (tid + q * K3_LINK_THREADS < per_pair / 4) ? __ldg(src + tid + q * K3_LINK_THREADS) : 0u;
        }
        const bool slicer = tid < TB * NJ * 3;
        const int e = tid % 3;
        const int l = (tid / 3) % NJ;
        const int tt = slicer ? tid / (3 * NJ) : 0;
        const int li = tt * NJ + l;  // table of the chunk
        const int2 lt = slicer ? reinterpret_cast<const int2*>(img)[li] : make_int2(0, 0);
        if (slicer) {
            double value = reinterpret_cast<const double*>(img + B.img_lc())[li * 3 + e];
            double grad[NF] = {0, 0, 0, 0, 0, 0, 0};
            // 32-byte records: coefficient e at double e, the key in the low half-word of double 3 (half-word 12)
            K3_SLICE(reinterpret_cast<const uint16_t*>(imgd + lt.x) + 12, imgd + lt.x + e, lt.y, 16, 4, K3_SLICE_TABLES, value, grad);
            // centre of Interval(c - r, c + r), as getCenter(slice()) does (KPR/NLPclass.cu:313)
            const double r = reinterpret_cast<const double*>(img + B.img_lr())[li * 3 + e];
            const double c = ((value - r) + (value + r)) * 0.5;
            s_lc[tt][l][e] = c;
            if (p == 0) B.link_sliced[((size_t(tb) * TB + tt) * NJ + l) * 3 + e] = c;  // armtd_NLP::link_sliced_center
#pragma unroll
            for (int v = 0; v < NF; v++) s_dlc[tt][l][v][e] = grad[v];
        }
        if (cnt_in_smem) {
#pragma unroll
            for (int q = 0; q < CW; q++)
                if (tid + q * K3_LINK_THREADS < per_pair / 4) reinterpret_cast<unsigned*>(s_cnt)[tid + q * K3_LINK_THREADS] = cw[q];
        }
        asm volatile("bar.sync 1, %0;" ::"n"(K3_LINK_THREADS) : "memory");    // link slices complete
        asm volatile("bar.arrive 2, %0;" ::"n"(K3_THREADS) : "memory");       // tell the torque warps, do not wait
    } else {
        const int tq = tid - K3_TORQUE_T0;
        const int i = tq / K3_TORQUE_LANES, part = tq % K3_TORQUE_LANES;  // table tt*NF + j, lane of the table
        double value = 0.0;
        double grad[NF] = {0, 0, 0, 0, 0, 0, 0};
        const bool on = i < TB * NF;
        const int4 ut = on ? reinterpret_cast<const int4*>(img + B.img_ut())[i] : make_int4(0, 0, 0, 0);
        if (on) {
            // lane `part` takes the monomials part, part + 2, ...; the two partial sums are added below
            // (the oracle adds the monomials one after the other: a difference of a few ulp)
            const int n = ut.z;
            const int mine = (n - part + K3_TORQUE_LANES - 1) / K3_TORQUE_LANES;
            K3_SLICE(reinterpret_cast<const uint16_t*>(img) + ut.y + part, imgd + ut.x + part, mine > 0 ? mine : 0,
                            K3_TORQUE_LANES, K3_TORQUE_LANES, K3_SLICE_TABLES, value, grad);
        }
#pragma unroll
        for (int d = 1; d < K3_TORQUE_LANES; d <<= 1) {
            value += __shfl_xor_sync(0xffffffffu, value, d);
#pragma unroll
            for (int v = 0; v < NF; v++) grad[v] += __shfl_xor_sync(0xffffffffu, grad[v], d);
        }
        double* st = s_tj;
        if (on && part == 0) {
            value = reinterpret_cast<const double*>(img + B.img_uc())[i] + value;
            const double r = reinterpret_cast<const double*>(img + B.img_ur())[i];
            if (gp) gp[tb * TB * NF + i] = ((value - r) + (value + r)) * 0.5;
#pragma unroll
            for (int v = 0; v < NF; v++) st[i * NF + v] = grad[v];
        }
        asm volatile("bar.sync 3, %0;" ::"n"(K3_THREADS - K3_LINK_THREADS) : "memory");
        if (jp) {  // rows tb*TB*NF + i, i < 56: 392 contiguous doubles
            double* dst = jp + size_t(tb) * TB * NF * NF;
            for (int q = tq; q < TB * NF * NF; q += K3_THREADS - K3_TORQUE_T0) dst[q] = st[q];
        }
        asm volatile("bar.sync 3, %0;" ::"n"(K3_THREADS - K3_LINK_THREADS) : "memory");  // stage free again
        asm volatile("bar.sync 2, %0;" ::"n"(K3_THREADS) : "memory");                      // link slices are complete
    }

    // ---- phase 2: collision rows.  x = (l*TB + tt)*O + o; 32 consecutive rows per warp pass
    // the stored records of the chunk, row after row; grp[g] = records of the rows before row 32 g
    const double2* __restrict__ cand = reinterpret_cast<const double2*>(img + B.img_hdr());
    const unsigned* __restrict__ grp = reinterpret_cast<const unsigned*>(img + B.img_grp());
    const unsigned char* cnt = img + B.img_cnt();
    const bool in_domain = s_in_domain != 0;
    const float inv_O = O > 0 ? 1.0f / float(O) : 0.0f;
#if !K3_DIRECT_J
    double* stage = &s_stage[warp][0];
#endif
    for (;;) {
        int x0 = 0;
        if (lane == 0) x0 = atomicAdd(&s_next, 1) * 32;
        x0 = __shfl_sync(0xffffffffu, x0, 0);
        if (x0 >= per_pair) break;
        const int x = x0 + lane;
        bool active = x < per_pair;
        const unsigned base = grp[x0 >> 5];
        double max_elt = -100000000;
        double A0 = 0, A1 = 0, A2 = 0;  // minus the winning signed normal
        int l = 0, tt = 0, o = 0;
        const int n = active ? (cnt_in_smem ? s_cnt[x] : cnt[x]) : 0;
        // first record of the row: base + the records of the warp's earlier rows (inclusive scan over the lanes)
        const int stored = n == HP_OVERFLOW ? 0 : n;
        int before = stored;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, before, d);
            if (lane >= d) before += t;
        }
        before -= stored;
        if (active) {
            const int ltt = __float2int_rz((float(x) + 0.5f) * inv_O);  // x / O, exact for x < 2^22
            o = x - ltt * O;
            tt = ltt % TB;
            l = ltt / TB;
            const double c0 = s_lc[tt][l][0], c1 = s_lc[tt][l][1], c2 = s_lc[tt][l][2];
            if (n != HP_OVERFLOW && in_domain) {
                const double2* row = cand + size_t(base + unsigned(before)) * 2;
                // K3_CQ candidate records in flight per thread (the scan itself stays in order)
                for (int q0 = 0; q0 < n; q0 += K3_CQ) {
                    double2 u[K3_CQ], w[K3_CQ];
#pragma unroll
                    for (int i = 0; i < K3_CQ; i++) {
                        if (q0 + i < n) {
#if K3_LD256
                            // one 32-byte record = one 256-bit load (sm_100: ld.global.v4.f64)
#if K3_LD_NOALLOC
                            asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0, %1, %2, %3}, [%4];"
#else
                            asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];"
#endif
                                         : "=d"(u[i].x), "=d"(u[i].y), "=d"(w[i].x), "=d"(w[i].y)
                                         : "l"(row + (q0 + i) * 2));
#else
                            u[i] = __ldg(row + (q0 + i) * 2);
                            w[i] = __ldg(row + (q0 + i) * 2 + 1);
#endif
                        }
                    }
#pragma unroll
                    for (int i = 0; i < K3_CQ; i++) {
                        if (q0 + i < n) {
                            const double v = (u[i].x * c0 + u[i].y * c1 + w[i].x * c2) - w[i].y;
                            if (v > max_elt) {  // strict '>' in scan order: KPR/CollisionChecking.cu:264-276
                                max_elt = v;
                                A0 = -u[i].x; A1 = -u[i].y; A2 = -w[i].x;
                            }
                        }
                    }
                }
            } else {
                active = false;  // no stored list, or k outside the box the lists were built for: k_constraints_slow
            }
        }
        const long long row_i = active ? (long long)(size_t(NF) * T + (size_t(l) * T + tb * TB + tt) * O + o) : -1;
        if (gp && active) gp[row_i] = -max_elt;
#if K3_DIRECT_J
#if K3_SKIP_ZERO_DK
        // the centre of link l depends on k_0 .. k_l only: d/dk_v is exactly zero for v > l, those products are not made
        // (the rows of a warp pass belong to at most two consecutive links: the bound is the larger one)
        const int lmax = __reduce_max_sync(0xffffffffu, active ? l : 0);
#endif
        if (jp && active) {
            double* out = jp + row_i * NF;
            double jv[NF];
#pragma unroll
            for (int v = 0; v < NF; v++) {
#if K3_SKIP_ZERO_DK
                if (v > lmax) {
                    jv[v] = 0.0;
                    continue;
                }
#endif
                const double* dk = s_dlc[tt][l][v];
                // -(C.dk) for a 'pos' winner, +(C.dk) for 'neg' (:286-295); the sign is folded into A
                jv[v] = A0 * dk[0] + A1 * dk[1] + A2 * dk[2];
            }
            // 56 contiguous bytes per row, 16-byte aligned for even rows (the Jacobian of a problem starts 16-byte aligned and
            // m is even): three 16-byte stores and one 8-byte store instead of seven 8-byte stores
            if ((row_i & 1) == 0) {
                K3_ST2(out, jv[0], jv[1]);
                K3_ST2(out + 2, jv[2], jv[3]);
                K3_ST2(out + 4, jv[4], jv[5]);
                K3_ST1(out + 6, jv[6]);
            } else {
                K3_ST1(out, jv[0]);
                K3_ST2(out + 1, jv[1], jv[2]);
                K3_ST2(out + 3, jv[3], jv[4]);
                K3_ST2(out + 5, jv[5], jv[6]);
            }
        }
#else
        if (jp) {
            if (active) {
#pragma unroll
                for (int v = 0; v < NF; v++) {
                    const double* dk = s_dlc[tt][l][v];
                    // -(C.dk) for a 'pos' winner, +(C.dk) for 'neg' (:286-295); the sign is folded into A
                    stage[lane * NF + v] = A0 * dk[0] + A1 * dk[1] + A2 * dk[2];
                }
            }
            __syncwarp();
#pragma unroll
            for (int q = 0; q < NF; q++) {
                const int e = q * 32 + lane;
                const int r = e / NF;
                const long long rr = __shfl_sync(0xffffffffu, row_i, r);
                if (rr >= 0) jp[rr * NF + (e - r * NF)] = stage[e];
            }
            __syncwarp();
        }
#endif
    }

    // Bezier joint-limit rows (KPR/Trajectory.cu:256-540), once per problem
    if (tb == 0 && tid < NF) {
        const int i = tid;
        const double D = c_robot.duration;
        const double q0 = B.q0[size_t(p) * NF + i];
        const double a = B.qd0[size_t(p) * NF + i] * D;
        const double b = B.qdd0[size_t(p) * NF + i] * D * D;
        const double kn = kin[size_t(p) * NF + i];
        const int off = NF * T + NJ * T * O;
        for (int vel = 0; vel < 2; vel++) {
            double mn, mx, dmn, dmx;
            bez_extrema(vel == 1, q0, a, b, c_robot.k_range[i], D, kn, &mn, &mx, &dmn, &dmx);
            const int r0 = off + vel * 2 * NF + i;
            if (gp) {
                gp[r0] = mn;
                gp[r0 + NF] = mx;
            }
            if (jp) {
                for (int j = 0; j < NF; j++) {
                    jp[size_t(r0) * NF + j] = (j == i) ? dmn : 0.0;
                    jp[size_t(r0 + NF) * NF + j] = (j == i) ? dmx : 0.0;
                }
            }
        }
    }
}

#undef K3_SLICE
#undef K3_SLICE_TABLES
// k_constraints_slow: the collision rows k_constraints leaves out — rows without a stored candidate list (more than HP_CAP
// survivors, or no room left in the chunk) and every row of a problem whose k lies outside the box the lists were built
// for.  One CTA per problem, which returns at once in the usual case (no such row); otherwise one thread per row slices
// the link reach set in the reference's factor order (KPR/PZsparse.cu:404-555) and scans all 72 half-spaces computed from
// the generators (KPR/CollisionChecking.cu:169-299).
constexpr int K3S_PROBLEMS = 16;  // problems per CTA of k_constraints_slow
__global__ void __launch_bounds__(128)
k_constraints_slow(Batch B, const double* __restrict__ kin, double* __restrict__ g, double* __restrict__ jac) {
    // k_constraints is launched right behind this kernel as a programmatic dependent and runs BESIDE it: the two share no
    // data (this kernel writes only the rows that one leaves out), so whatever this kernel has to do — usually nothing, a few
    // dozen rows for some batches — is hidden under the 0.6 ms of the main kernel instead of being added to it
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int NJ = B.NJ, O = B.O, T = B.T;
    __shared__ int s_list[K3S_PROBLEMS], s_n;
    __shared__ double2 kpd[NF][4];  // {k_j^d, d/dk_j k_j^d} for d = 0..3
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    if (threadIdx.x < K3S_PROBLEMS) {  // one thread per problem: does it have anything for this kernel?  (usually not)
        const int i = blockIdx.x * K3S_PROBLEMS + threadIdx.x;
        if (i < B.nprob && O > 0) {
            const int p = B.plist ? B.plist[i] : i;
            if (B.failed(p) == 0) {
                bool in = true;
                for (int j = 0; j < NF; j++) in = in && (fabs(kin[size_t(p) * NF + j]) <= K_DOMAIN);
                if (!in || B.hp_slow[p] != 0) s_list[atomicAdd(&s_n, 1)] = p;
            }
        }
    }
    __syncthreads();
    const int nlist = s_n;
    for (int li = 0; li < nlist; li++) {
    const int p = s_list[li];
    bool in = true;
    for (int j = 0; j < NF; j++) in = in && (fabs(kin[size_t(p) * NF + j]) <= K_DOMAIN);
    __syncthreads();
    if (threadIdx.x < NF) {
        const double k = kin[size_t(p) * NF + threadIdx.x];
        kpd[threadIdx.x][0] = make_double2(1.0, 0.0);
        kpd[threadIdx.x][1] = make_double2(k, 1.0);
        kpd[threadIdx.x][2] = make_double2(k * k, 2.0 * k);
        kpd[threadIdx.x][3] = make_double2(k * k * k, 3.0 * (k * k));
    }
    __syncthreads();
    const int m = B.m();
    const int per_chunk = NJ * TB * O;
    double* gp = g ? g + size_t(p) * m : nullptr;
    double* jp = jac ? jac + size_t(p) * m * NF : nullptr;
    for (int r = threadIdx.x; r < per_chunk * (T / TB); r += blockDim.x) {
        const int tb = r / per_chunk, x = r - tb * per_chunk;
        const size_t chunk = size_t(p) * (T / TB) + tb;
        if (in && B.hp_cnt[chunk * per_chunk + x] != HP_OVERFLOW) continue;
        const int o = x % O, ltt = x / O, tt = ltt % TB, l = ltt / TB;
        const size_t idx = (size_t(p) * T + tb * TB + tt) * NJ + l;
        double c[3], dk[NF][3];
        const int n = B.link_n[idx];
        for (int e = 0; e < 3; e++) {
            double value = B.link_c[idx * 3 + e];
            double grad[NF] = {0, 0, 0, 0, 0, 0, 0};
            for (int mI = 0; mI < n; mI++) {
                const unsigned key = B.link_key[idx * B.capL + mI];
                double val = B.link_g[(idx * B.capL + mI) * 3 + e];
                double D[NF];
#pragma unroll
                for (int j = 0; j < NF; j++) {
                    const double2 fd = kpd[j][(key >> (2 * j)) & 3];
                    D[j] = val * fd.y;
#pragma unroll
                    for (int v = 0; v < j; v++) D[v] *= fd.x;
                    val *= fd.x;
                }
                value += val;
#pragma unroll
                for (int v = 0; v < NF; v++) grad[v] += D[v];
            }
            const double rr = B.link_r[idx * 3 + e];
            c[e] = ((value - rr) + (value + rr)) * 0.5;
#pragma unroll
            for (int v = 0; v < NF; v++) dk[v][e] = grad[v];
        }
        double r_max, A0, A1, A2;
        row_from_generators(B.obstacles + (size_t(p) * O + o) * 12, B.link_gens + idx * 18, c[0], c[1], c[2], &r_max, &A0, &A1, &A2);
        const size_t row = size_t(NF) * T + (size_t(l) * T + tb * TB + tt) * O + o;
        if (gp) gp[row] = -r_max;
        if (jp)
            for (int v = 0; v < NF; v++) jp[row * NF + v] = A0 * dk[v][0] + A1 * dk[v][1] + A2 * dk[v][2];
    }
    }
}

// ---------------------------------------------------------------------------------------------------
// Structured Jacobian.  The reference declares the Jacobian dense (KPR/NLPclass.cu:348-357), but its pattern is fixed by the
// kinematics: a collision row of link l depends on k_0..k_l only (the link's reach set has no monomial in a later joint's
// parameter: those entries are exact zeros), a Bezier row on its own joint only; torque rows are full.  jac_row_width() is
// that pattern; k_pack_jacobian gathers the non-zeros of the dense rows (row-major, columns ascending) so that a caller
// which gives Ipopt the sparse structure moves 39 % fewer Jacobian bytes over PCIe (10 obstacles: 42 140 of 69 188 values).
__host__ __device__ inline int jac_link_width(int l) { return l + 1 < NF ? l + 1 : NF; }
__host__ __device__ inline long long jac_nnz(int T, int NJ, int O) {
    long long w = 0;
    for (int l = 0; l < NJ; l++) w += jac_link_width(l);
    return (long long)NF * NF * T + (long long)T * O * w + 4 * NF;
}
__global__ void __launch_bounds__(256)
k_pack_jacobian(Batch B, const double* __restrict__ jac, double* __restrict__ out, long long nnz) {
    const int p = blockIdx.y;
    const int T = B.T, NJ = B.NJ, O = B.O;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nnz) return;
    const double* jp = jac + size_t(p) * B.m() * NF;
    long long row, col;
    const long long n_t = (long long)NF * NF * T;
    if (idx < n_t) {
        row = idx / NF;
        col = idx % NF;
    } else {
        long long r = idx - n_t;
        int l = 0;
        for (; l < NJ; l++) {
            const long long blk = (long long)T * O * jac_link_width(l);
            if (r < blk) break;
            r -= blk;
        }
        if (l < NJ) {
            const int w = jac_link_width(l);
            row = (long long)NF * T + (long long)l * T * O + r / w;
            col = r % w;
        } else {  // Bezier rows: min / max position, min / max velocity of joint i -> column i
            row = (long long)NF * T + (long long)NJ * T * O + r;
            col = r % NF;
        }
    }
    out[size_t(p) * nnz + idx] = jp[row * NF + col];
}
cudaError_t launch_pack_jacobian(const Batch& B, const double* d_jac, double* d_out, cudaStream_t st) {
    if (B.nprob == 0) return cudaSuccess;
    const long long nnz = jac_nnz(B.T, B.NJ, B.O);
    dim3 grid((unsigned)((nnz + 255) / 256), B.nprob);
    k_pack_jacobian<<<grid, 256, 0, st>>>(B, d_jac, d_out, nnz);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// verdict: first violated row in the reference's check order (= ascending row index), one CTA per problem
__global__ void __launch_bounds__(256)
k_verdict(Batch B, const double* __restrict__ g, int* __restrict__ feasible, int* __restrict__ first) {
    const int p = blockIdx.x;
    const int T = B.T, NJ = B.NJ, O = B.O, m = B.m();
    const double* gp = g + size_t(p) * m;
    const double* tr = B.torque_radius + size_t(p) * NF * T;
    int best = m;
    for (int r = threadIdx.x; r < m; r += blockDim.x) {
        const double v = gp[r];
        bool bad;
        if (r < NF * T) {
            const int t = r / NF, j = r % NF;
            const double rad = tr[j * T + t];
            bad = v < -c_robot.torque_limits[j] + rad - c_robot.torque_violation_threshold ||
                  v > c_robot.torque_limits[j] - rad + c_robot.torque_violation_threshold;
        } else if (r < NF * T + NJ * T * O) {
            bad = v > c_robot.collision_violation_threshold;
        } else {
            const int q = r - (NF * T + NJ * T * O);
            const int j = q % NF;
            if (q < 2 * NF)
                bad = v < c_robot.state_limits_lb[j] + c_robot.qe || v > c_robot.state_limits_ub[j] - c_robot.qe;
            else
                bad = v < -c_robot.speed_limits[j] + c_robot.qde || v > c_robot.speed_limits[j] - c_robot.qde;
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

// ---------------------------------------------------------------------------------------------------
// host launchers (called from capi.cu)
cudaError_t launch_hyperplanes(const Batch& B, cudaStream_t st, const int* unit_flag = nullptr, HpStage stage = HpStage{nullptr, nullptr, nullptr, nullptr}) {
    if (B.O == 0 || B.nprob == 0) return cudaSuccess;
    // (B.hp_slow was zeroed by k_reachsets, or by the caller when the tables were imported)
    const int rows = B.NJ * B.T * B.O;
    dim3 grid((rows + HP_ROWS - 1) / HP_ROWS, B.nprob);
    if (unit_flag) {  // programmatic dependent of the reach-set kernel launched just before on this stream
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid;
        cfg.blockDim = dim3(HP_THREADS);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, k_hyperplanes, B, unit_flag, stage);
    }
    k_hyperplanes<<<grid, HP_THREADS, 0, st>>>(B, unit_flag, stage);
    return cudaGetLastError();
}
cudaError_t launch_constraints(const Batch& B, const double* d_k, double* d_g, double* d_jac, cudaStream_t st) {
    if (B.nprob == 0) return cudaSuccess;
#ifdef K3_CARVEOUT_KNOB
    {  // experiment: shared-memory carve-out of the main kernel in per cent of the maximum (ARMOUR_K3_CARVEOUT)
        static int done = 0;
        if (!done) {
            done = 1;
            const char* v = std::getenv("ARMOUR_K3_CARVEOUT");
            if (v) {
                cudaError_t ec = cudaFuncSetAttribute(k_constraints, cudaFuncAttributePreferredSharedMemoryCarveout, std::atoi(v));
                std::printf("k_constraints carve-out %s %%: %s\n", v, cudaGetErrorString(ec));
            }
        }
    }
#endif
    dim3 grid(B.T / TB, B.nprob);
    if (B.O == 0) {
        k_constraints<<<grid, K3_THREADS, 0, st>>>(B, d_k, d_g, d_jac);
        return cudaGetLastError();
    }
    // slow path first (a normal launch: it waits for whatever precedes it on the stream), the main kernel behind it as a
    // programmatic dependent: it starts as soon as the slow kernel's few CTAs are resident and runs beside them
    k_constraints_slow<<<(B.nprob + K3S_PROBLEMS - 1) / K3S_PROBLEMS, 128, 0, st>>>(B, d_k, d_g, d_jac);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(K3_THREADS);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, k_constraints, B, d_k, d_g, d_jac);
}
cudaError_t launch_verdict(const Batch& B, const double* d_g, int* d_feasible, int* d_first, cudaStream_t st) {
    if (B.nprob == 0) return cudaSuccess;
    k_verdict<<<B.nprob, 256, 0, st>>>(B, d_g, d_feasible, d_first);
    return cudaGetLastError();
}

}  // namespace armour
