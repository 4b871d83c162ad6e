// K1/K2: reach-set construction on the device.  One CTA builds ALL reach sets of one
// (planning problem, time interval): the joint reachable set of the Bezier trajectory (K2, prologue),
// the PZ forward kinematics of the link volumes, one pass of PZ recursive Newton-Euler carrying the
// nominal and the interval-parameter radius lanes, and the robust-input radius (epilogue).
//
// Replaces, per time interval, BezierCurve::makePolyZono (KPR/Trajectory.cu:63-254),
// KinematicsDynamics::fk / rnea_nominal / rnea_interval (KPR/Dynamics.cu:69-181), reduce_link_PZ / reduce
// (KPR/PZsparse.cu:352-402) and sections II.B-II.C of main() (KPR/armour_main.cu:96-210), which the
// reference runs on the host under OpenMP.  Operation order and every simplify() point follow the
// reference (see k1_pz.cuh for how a simplify() is carried out here).
//
// CTAs are persistent: each takes (problem, interval) units from a global counter, so a batch of
// worlds x replans fills the 148 SMs without any cross-CTA communication.
#ifndef ARMOUR_EMU
#include "../../include/armour_b200.h"
#endif
#include "bezier.cuh"
#include "device_constants.cuh"
#include "k1_pz.cuh"
#undef set_fail
#define set_fail(code) set_fail_at(code, 10000 + __LINE__)
#include "k1_interval.cuh"
#include "layout.h"

namespace armour {
namespace K1_NS {

// fixed shared-memory region for the joint reachable set of the current interval
constexpr int ROT_WORDS = 27 + 3 + 27;  // 3x3 PZ with at most 3 monomials
constexpr int SCL_WORDS = 3 + 2 + 2;    // scalar PZ with at most 2 monomials
constexpr int JRS_WORDS = (MAXJ + 1) * ROT_WORDS + 3 * NF * SCL_WORDS;
constexpr double RADIUS_SLACK = 1.0 + 0x1p-40;  // outward slack on exported radii (see DESIGN.md "soundness")

struct K1Params {
    Batch B;
    int* work;          // [2]: global unit counter and count of finished CTAs; the last CTA to finish resets both, so
                        // a launch needs no memset in front of it
    int* unit_flag;     // optional [p*T + t]: set to B.epoch when the unit is complete (release); lets the half-space
                        // kernel, launched as a programmatic dependent, start on finished intervals.  nullptr: unused
    double* gscr;       // [grid][gscr_words]: per CTA [arena spill space | F / N blocks of one unit]
    int gscr_words;
    int fn_words;       // words of the F / N part (the last fn_words of a CTA's scratch)
    char* gtab;         // [grid][gtab_bytes], all zero between launches
    int gtab_bytes;
    int arena_words;    // shared-memory working arena per CTA (behind the fixed JRS region)
    int tab_s_bytes;    // shared-memory table pool per group
    int group_bytes;    // shared memory per group (control block + JRS region + arena + table pool)
    const int* units;   // optional explicit unit list (p*T + t); nullptr = all units of the batch
    int nunits;
    int* stats;         // [4]: max arena words used, tables placed in global memory, failed units, units done
    double* mbox;       // MG mode: [grid][mbox_words] mailboxes
    int mbox_words;
};

// handles of the joint reachable set blocks (fixed places at the bottom of the virtual arena)
K1_DI PZ8 jrs_R(int i) {
    PZ8 h;
    h.off = i * ROT_WORDS;
    h.n = k1s().jrs_n[i];
    return h;
}
K1_DI PZ8 jrs_scalar(int g, int i) {  // g = 0: qd_des, 1: qda_des, 2: qdda_des
    PZ8 h;
    h.off = (MAXJ + 1) * ROT_WORDS + (g * NF + i) * SCL_WORDS;
    h.n = k1s().jrs_n[16 + 8 * g + i];
    return h;
}

K1_DI void indep_range(double v_lb, double v_ub, double s_lb, double s_ub, double e1s, double e1v, double e2s,
                       double e2v, double* radius, double* center) {  // KPR/Trajectory.cu:80-94
    double lb = v_lb, ub = v_ub;
    if (lb > ub) {
        const double x = lb;
        lb = ub;
        ub = x;
    }
    if (s_lb < e1s && e1s < s_ub) {
        lb = fmin(lb, e1v);
        ub = fmax(ub, e1v);
    }
    if (s_lb < e2s && e2s < s_ub) {
        lb = fmin(lb, e2v);
        ub = fmax(ub, e2v);
    }
    *radius = (ub - lb) * 0.5;
    *center = (lb + ub) * 0.5;
}

// scalar PZ  c + coef0 * x_{key0} + coef1 * x_{key1}, simplified (KPR/PZsparse.cu:120-136)
K1_DI void write_scalar_pz(double* p, int* n_out, double thr, double center, double c0, u64 k0, double c1, u64 k1_) {
    double rad = 0.0;
    int n = 0;
    u64 keys[2];
    double cf[2];
    const double cc[2] = {c0, c1};
    const u64 kk[2] = {k0, k1_};
    for (int i = 0; i < 2; i++) {
        if (sqrt(cc[i] * cc[i]) <= thr) {
            rad = __dadd_ru(rad, fabs(cc[i]));
        } else {
            keys[n] = kk[i];
            cf[n] = cc[i];
            n++;
        }
    }
    p[0] = center;
    p[1] = rad;
    p[2] = rad;
    u64* pk = reinterpret_cast<u64*>(p + 3);
    for (int i = 0; i < n; i++) pk[i] = keys[i];
    for (int i = 0; i < n; i++) p[3 + n + i] = cf[i];
    *n_out = n;
}

// Joint reachable set of joint i over interval t (KPR/Trajectory.cu:15-61 for the extrema of the
// k-independent parts, :63-254 for the interval itself).  Executed by one thread per joint.
K1_OP void jrs_joint(int i, int t, int T, double q0, double qd0, double qdd0, double thr, double* rot_blk, int* rot_n,
                     double* qd_blk, int* qd_n, double* qda_blk, int* qda_n, double* qdda_blk, int* qdda_n, const double* ext) {
    const RobotConstants& rc = c_robot;
    const double D = rc.duration;
    const double a = qd0 * D, b = qdd0 * D * D;
    const double kr = rc.k_range[i];
    const double ds = 1.0 / T;
    const double s_lb = t * ds, s_ub = (t + 1) * ds;
    // interior extrema of the k-independent parts (BezierCurve ctor)
    double es[3][2], ev[3][2];
    {
        const double sq = sqrt(64 * pw2(a) + 14 * a * b + pw2(b));
        es[0][0] = (2 * a + b + sq) / (5 * (6 * a + b));
        es[0][1] = (2 * a + b - sq) / (5 * (6 * a + b));
        ev[0][0] = bez_q_indep(q0, a, b, es[0][0]);
        ev[0][1] = bez_q_indep(q0, a, b, es[0][1]);
    }
    {
        const double sq = sqrt(6 * (54 * pw2(a) + 14 * a * b + pw2(b)));
        es[1][0] = (18 * a + 4 * b + sq) / (10 * (6 * a + b));
        es[1][1] = (18 * a + 4 * b - sq) / (10 * (6 * a + b));
        ev[1][0] = bez_qd_indep(a, b, es[1][0], D);
        ev[1][1] = bez_qd_indep(a, b, es[1][1], D);
    }
    {
        const double sq = sqrt(2 * (152 * pw2(a) + 42 * a * b + 3 * pw2(b)));
        es[2][0] = (32 * a + 6 * b + sq) / (10 * (6 * a + b));
        es[2][1] = (32 * a + 6 * b - sq) / (10 * (6 * a + b));
        ev[2][0] = bez_qdd_indep(a, b, es[2][0], D);
        ev[2][1] = bez_qdd_indep(a, b, es[2][1], D);
    }

    // Part 1: position -> cos / sin Taylor models (:75-134) — or, for the ARMTD comparison planner, the six numbers the caller
    // derived from its offline joint reachable set (KPA/Trajectory.cu:34-62): same form  c + k-coefficient * k_i + e * cosqe_i
    double cos_c, cos_k, cos_e, sin_c, sin_k, sin_e;
    double kd_lb, kd_ub, kd_center, kd_radius, ki_radius;
    if (ext) {
        cos_c = ext[0];
        cos_k = ext[1];
        cos_e = ext[2];
        sin_c = ext[3];
        sin_k = ext[4];
        sin_e = ext[5];
    } else {
        kd_lb = pw3(s_lb) * (6 * pw2(s_lb) - 15 * s_lb + 10);
        kd_ub = pw3(s_ub) * (6 * pw2(s_ub) - 15 * s_ub + 10);
        kd_center = (kd_ub + kd_lb) * 0.5;
        kd_radius = (kd_ub - kd_lb) * 0.5 * kr;
        double q_c;
        indep_range(bez_q_indep(q0, a, b, s_lb), bez_q_indep(q0, a, b, s_ub), s_lb, s_ub, es[0][0], ev[0][0], es[0][1],
                    ev[0][1], &ki_radius, &q_c);
        const Itv qr = iv(-kd_radius - ki_radius - rc.qe, kd_radius + ki_radius + rc.qe);
        const Itv kint = iv(-kr, kr);
        const double sq_c = sin(q_c), cq_c = cos(q_c);
        const Itv arg = iv_add(iv_addd(q_c, iv_muld(kd_center, kint)), qr);
        const Itv e2 = iv_pow2(iv_add(qr, iv_muld(kd_center, kint)));
        Itv cos_r = iv_sub(iv_muld(sq_c, iv_neg(qr)), iv_mul(iv_muld(0.5, iv_cos(arg)), e2));
        cos_c = cq_c + iv_mid(cos_r);
        cos_r = iv_subd(cos_r, iv_mid(cos_r));
        cos_k = -kd_center * kr * sq_c;
        cos_e = iv_rad(cos_r);
        Itv sin_r = iv_sub(iv_muld(cq_c, qr), iv_mul(iv_muld(0.5, iv_sin(arg)), e2));
        sin_c = sq_c + iv_mid(sin_r);
        sin_r = iv_subd(sin_r, iv_mid(sin_r));
        sin_k = kd_center * kr * cq_c;
        sin_e = iv_rad(sin_r);
    }

    // 3x3 rotation about z from the cos / sin models (KPR/PZsparse.cu:179-250), simplified, then
    // R = Rrpy * Rz (KPR/Trajectory.cu:136-144): a product with a constant left operand.
    {
        double rotc[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        rotc[0] = cos_c;
        rotc[3] = -1.0 * sin_c;
        rotc[1] = sin_c;
        rotc[4] = cos_c;
        double rot_rad[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        double M[3][9];
        u64 mk[3];
        int nm = 0;
        for (int which = 0; which < 3; which++) {
            double m[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
            if (which == 0) {  // the two k_i monomials merged
                m[0] = cos_k;
                m[1] = sin_k;
                m[3] = -0.0 + (-1.0 * sin_k);
                m[4] = cos_k;
            } else if (which == 1) {
                m[0] = cos_e;
                m[3] = -0.0;
                m[4] = cos_e;
            } else {
                m[1] = sin_e;
                m[3] = -1.0 * sin_e;
            }
            if (frobN<9>(m) <= thr) {
                for (int e = 0; e < 9; e++) rot_rad[e] = __dadd_ru(rot_rad[e], fabs(m[e]));
            } else {
                for (int e = 0; e < 9; e++) M[nm][e] = m[e];
                mk[nm] = which == 0 ? key_k(i) : (which == 1 ? key_cosqe(i) : key_sinqe(i));
                nm++;
            }
        }
        const double* Rr = &rc.rrpy[i * 9];
        double cen[9], absR[9], rad[9];
        matmul3<3, false>(Rr, rotc, cen);
        for (int e = 0; e < 9; e++) absR[e] = fabs(Rr[e]);
        matmul3_up<3, false>(absR, rot_rad, rad);
        double outM[3][9];
        u64 outk[3];
        int no = 0;
        for (int j = 0; j < nm; j++) {
            double v[9];
            matmul3<3, false>(Rr, M[j], v);
            if (frobN<9>(v) <= thr) {
                for (int e = 0; e < 9; e++) rad[e] = __dadd_ru(rad[e], fabs(v[e]));
            } else {
                for (int e = 0; e < 9; e++) outM[no][e] = v[e];
                outk[no] = mk[j];
                no++;
            }
        }
        for (int e = 0; e < 9; e++) {
            rot_blk[e] = cen[e];
            rot_blk[9 + e] = rad[e];
            rot_blk[18 + e] = rad[e];
        }
        u64* pk = reinterpret_cast<u64*>(rot_blk + 27);
        for (int j = 0; j < no; j++) pk[j] = outk[j];
        for (int j = 0; j < no; j++)
            for (int e = 0; e < 9; e++) rot_blk[27 + no + j * 9 + e] = outM[j][e];
        *rot_n = no;
    }

    if (ext) {  // forward kinematics only: the velocity / acceleration sets stay empty (zero scalars)
        write_scalar_pz(qd_blk, qd_n, thr, 0.0, 0.0, key_k(i), 0.0, key_qde(i));
        write_scalar_pz(qda_blk, qda_n, thr, 0.0, 0.0, key_k(i), 0.0, key_qdae(i));
        write_scalar_pz(qdda_blk, qdda_n, thr, 0.0, 0.0, key_k(i), 0.0, key_qddae(i));
        return;
    }
    // Part 2: velocity (:151-192)
    kd_lb = (30 * pw2(s_lb) * pw2(s_lb - 1)) / D;
    kd_ub = (30 * pw2(s_ub) * pw2(s_ub - 1)) / D;
    if (kd_ub < kd_lb) {
        const double x = kd_lb;
        kd_lb = kd_ub;
        kd_ub = x;
    }
    kd_center = (kd_ub + kd_lb) * 0.5 * kr;
    kd_radius = (kd_ub - kd_lb) * 0.5 * kr;
    double qd_c;
    indep_range(bez_qd_indep(a, b, s_lb, D), bez_qd_indep(a, b, s_ub, D), s_lb, s_ub, es[1][0], ev[1][0], es[1][1],
                ev[1][1], &ki_radius, &qd_c);
    write_scalar_pz(qd_blk, qd_n, thr, qd_c, kd_center, key_k(i), kd_radius + ki_radius + rc.qde, key_qde(i));
    write_scalar_pz(qda_blk, qda_n, thr, qd_c, kd_center, key_k(i), kd_radius + ki_radius + rc.qdae, key_qdae(i));

    // Part 3: acceleration (:195-244)
    const double kQddMax = 0.5 - sqrt(3.0) / 6, kQddMin = 0.5 + sqrt(3.0) / 6;  // KPR/Trajectory.h:7-8
    const double temp_lb = (60 * s_lb * (2 * pw2(s_lb) - 3 * s_lb + 1)) / D / D;
    const double temp_ub = (60 * s_ub * (2 * pw2(s_ub) - 3 * s_ub + 1)) / D / D;
    if (s_ub <= kQddMax) {
        kd_lb = temp_lb;
        kd_ub = temp_ub;
    } else if (s_lb <= kQddMax) {
        kd_lb = fmin(temp_lb, temp_ub);
        kd_ub = (60 * kQddMax * (2 * pw2(kQddMax) - 3 * kQddMax + 1)) / D / D;
    } else if (s_ub <= kQddMin) {
        kd_lb = temp_ub;
        kd_ub = temp_lb;
    } else if (s_lb <= kQddMin) {
        kd_lb = (60 * kQddMin * (2 * pw2(kQddMin) - 3 * kQddMin + 1)) / D / D;
        kd_ub = fmax(temp_lb, temp_ub);
    } else {
        kd_lb = temp_lb;
        kd_ub = temp_ub;
    }
    kd_center = (kd_ub + kd_lb) * 0.5 * kr;
    kd_radius = (kd_ub - kd_lb) * 0.5 * kr;
    double qdd_c;
    indep_range(bez_qdd_indep(a, b, s_lb, D), bez_qdd_indep(a, b, s_ub, D), s_lb, s_ub, es[2][0], ev[2][0], es[2][1],
                ev[2][1], &ki_radius, &qdd_c);
    write_scalar_pz(qdda_blk, qdda_n, thr, qdd_c, kd_center, key_k(i), kd_radius + ki_radius + rc.qddae, key_qddae(i));
}

// ---- exports --------------------------------------------------------------------------------------
// reduce_link_PZ (KPR/PZsparse.cu:370-402) + the k-only table of one link reach set, sorted by key.
K1_OP void export_link(PZ8 L8, const Batch& B, int p, int t, int l) {
    K1S& S = k1s();
    if (S.fail) return;
    const int tid = k1_tid(), lane = tid & 31, warp = tid >> 5;
    const PZH L = view<3>(L8);
    const u64* keys = pz_keys(L);
    const double* cf = pz_coef(L);
    const size_t idx = (size_t(p) * B.T + t) * B.NJ + l;
    double rad[3] = {0, 0, 0};
    int nk = 0;
    for (int m = 0; m < L.n; m++) nk += (keys[m] < KEY_K_ONLY);  // uniform (broadcast reads)
    if (nk > B.capL) {
        set_fail(FAIL_LINK_CAP);
        return;
    }
    double* gens = B.link_gens + idx * 18;
    if (tid < 18) gens[tid] = 0.0;
    k1_sync();
    for (int m = tid; m < L.n; m += NT) {
        const u64 key = keys[m];
        const bool konly = key < KEY_K_ONLY;
        const bool gen = !konly && key < KEY_K_LINKS && (key & KEY_K_MASK) == 0;
        if (konly || gen) {
            int rank = 0;
            for (int q = 0; q < L.n; q++) {
                const u64 kq = keys[q];
                const bool same = konly ? (kq < KEY_K_ONLY) : (kq >= KEY_K_ONLY && kq < KEY_K_LINKS && (kq & KEY_K_MASK) == 0);
                rank += (same && kq < key);
            }
            if (konly) {
                B.link_key[idx * B.capL + rank] = uint16_t(key);
                for (int e = 0; e < 3; e++) B.link_g[(idx * B.capL + rank) * 3 + e] = cf[size_t(m) * 3 + e];
            } else if (rank < 3) {
                for (int e = 0; e < 3; e++) gens[e + rank * 3] = cf[size_t(m) * 3 + e];
            } else {
                for (int e = 0; e < 3; e++) rad[e] = __dadd_ru(rad[e], fabs(cf[size_t(m) * 3 + e]));
            }
        } else {
            for (int e = 0; e < 3; e++) rad[e] = __dadd_ru(rad[e], fabs(cf[size_t(m) * 3 + e]));
        }
    }
    for (int e = 0; e < 3; e++) rad[e] = warp_sum_up(rad[e]);
    if (lane == 0)
        for (int e = 0; e < 3; e++) S.red[warp * RED_STRIDE + e] = rad[e];
    k1_sync();
    if (tid < 3) {
        const int e = tid;
        double v = pz_r(L, 0)[e];
        for (int w = 0; w < NW; w++) v = __dadd_ru(v, S.red[w * RED_STRIDE + e]);
        gens[e + (3 + e) * 3] = __dmul_ru(v, RADIUS_SLACK);
        B.link_r[idx * 3 + e] = gens[e + (3 + e) * 3];  // the diagonal alone, contiguous: what k_constraints streams
        B.link_c[idx * 3 + e] = pz_c(L)[e];
    }
    if (tid == 0) B.link_n[idx] = nk;
    k1_sync();
}

// u_nom.reduce() (KPR/PZsparse.cu:352-368) + the k-only table of one torque reach set; leaves in S.misc the
// radius of the reduced nominal PZ ([j]) and the disturbance radius toInterval(u_nom_int - u_nom) =
// r_int + r_nom before the reduce ([8 + j]) (KPR/armour_main.cu:134-141).
K1_OP void export_torque(PZ8 U8, const Batch& B, int p, int t, int j) {
    K1S& S = k1s();
    if (S.fail) return;
    const int tid = k1_tid(), lane = tid & 31, warp = tid >> 5;
    const PZH U = view<1>(U8);
    const u64* keys = pz_keys(U);
    const double* cf = pz_coef(U);
    const size_t idx = (size_t(p) * B.T + t) * NF + j;
    int nk = 0;
    for (int m = 0; m < U.n; m++) nk += (keys[m] < KEY_K_ONLY);
    if (nk > B.capU) {
        set_fail(FAIL_TORQUE_CAP);
        return;
    }
    double rad = 0.0;
    for (int m = tid; m < U.n; m += NT) {
        const u64 key = keys[m];
        if (key < KEY_K_ONLY) {
            int rank = 0;
            for (int q = 0; q < U.n; q++) rank += (keys[q] < key);  // every smaller key is k-only too
            B.u_key[idx * B.capU + rank] = uint16_t(key);
            B.u_g[idx * B.capU + rank] = cf[m];
        } else {
            rad = __dadd_ru(rad, fabs(cf[m]));
        }
    }
    rad = warp_sum_up(rad);
    if (lane == 0) S.red[warp * RED_STRIDE] = rad;
    k1_sync();
    if (tid == 0) {
        double v = 0.0;
        for (int w = 0; w < NW; w++) v = __dadd_ru(v, S.red[w * RED_STRIDE]);
        const double r_nom = pz_r(U, 0)[0], r_int = pz_r(U, 1)[0];
        const double reduced = __dadd_ru(r_nom, v);
        double* misc = MG ? k1x().misc : S.misc;  // MG: the torque tasks of a unit run on different groups
        misc[j] = reduced;
        misc[8 + j] = __dadd_ru(r_int, r_nom);
        B.u_n[idx] = nk;
        B.u_c[idx] = pz_c(U)[0];
        B.u_r[idx] = __dmul_ru(reduced, RADIUS_SLACK);
    }
    k1_sync();
}

// ---- K2: joint reachable set of interval t into the fixed region at the bottom of the arena ----
K1_DI void build_jrs(const Batch& B, int p, int t) {
    const RobotConstants& rc = c_robot;
    K1S& S = k1s();
    const int tid = k1_tid();
    const int NJ = B.NJ, T = B.T;
    const double thr = S.thr;
    double* rot_mem = arena0();
    double* scl_mem = arena0() + (MAXJ + 1) * ROT_WORDS;
    if (tid < NF) {
        const int i = tid;
        jrs_joint(i, t, T, B.q0[size_t(p) * NF + i], B.qd0[size_t(p) * NF + i], B.qdd0[size_t(p) * NF + i], thr,
                  rot_mem + i * ROT_WORDS, &S.jrs_n[i], scl_mem + (0 * NF + i) * SCL_WORDS, &S.jrs_n[16 + i],
                  scl_mem + (1 * NF + i) * SCL_WORDS, &S.jrs_n[24 + i], scl_mem + (2 * NF + i) * SCL_WORDS,
                  &S.jrs_n[32 + i], B.jrs_ext ? B.jrs_ext + ((size_t(p) * T + t) * NF + i) * 6 : nullptr);
    } else if (tid >= 32 && tid < 32 + (NJ + 1 - NF)) {  // fixed joints and the identity after the last one
        const int i = NF + (tid - 32);
        double* blk = rot_mem + i * ROT_WORDS;
        for (int e = 0; e < 9; e++) {
            blk[e] = (i < NJ) ? rc.rrpy[i * 9 + e] : ((e % 4 == 0) ? 1.0 : 0.0);
            blk[9 + e] = 0.0;
            blk[18 + e] = 0.0;
        }
        S.jrs_n[i] = 0;
    }
    k1_sync();

}

// link box zonotope of joint i as a 3x1 PZ at `top`: centre + diag(generators) on the x / y / z generator
// variables, which reuse the hash slots of qde_0 / qdae_0 / qddae_0 (KPR/Dynamics.cu:51-66)
K1_DI PZ8 make_link_box(int top, int i) {
    const RobotConstants& rc = c_robot;
    K1S& S = k1s();
    const int tid = k1_tid();
    const double thr = S.thr;
    bool ok;
    PZ8 box = pz_alloc<3>(top, 3, &ok);
    if (ok && tid == 0) {
        double* bp = vptr(box.off);
        double rad[3] = {0, 0, 0};
        int n = 0;
        u64 kk[3];
        double gg[3][3];
        for (int jx = 0; jx < 3; jx++) {
            const double g = rc.link_zonotope_generators[i * 3 + jx];
            if (sqrt(g * g) <= thr) {
                rad[jx] = fabs(g);
            } else {
                kk[n] = 1ull << (14 + 7 * jx);
                for (int e = 0; e < 3; e++) gg[n][e] = (e == jx) ? g : 0.0;
                n++;
            }
        }
        for (int e = 0; e < 3; e++) {
            bp[e] = rc.link_zonotope_center[i * 3 + e];
            bp[3 + e] = rad[e];
            bp[6 + e] = rad[e];
        }
        u64* pk = reinterpret_cast<u64*>(bp + 9);
        for (int q = 0; q < n; q++) pk[q] = kk[q];
        for (int q = 0; q < n; q++)
            for (int e = 0; e < 3; e++) bp[9 + n + q * 3 + e] = gg[q][e];
        S.cnt[0] = n;
    }
    k1_sync();
    box.n = ok ? S.cnt[0] : 0;
    k1_sync();
    return box;
}

// ---- one (problem, interval) unit -----------------------------------------------------------------
// `top` (the arena top, a CTA-uniform register) is threaded through the operations: every operation
// allocates exactly one block at `top` and the new top is the end of the block it returns.
// K1_PROFILE (developer builds only, tools/k1_profile.py): thread 0 of a unit accumulates the cycles of every
// operation site into g_k1prof[interval][site] = {cycles, source line}
#ifdef K1_PROFILE
#define K1_PROF_T0 const long long _pt0 = clock64()
#define K1_PROF_T1(_h)                                                           \
    if (k1_tid() == 0) {                                                         \
        long long* _pp = g_k1prof + (size_t(t) * K1_PROF_SITES + (__COUNTER__ % K1_PROF_SITES)) * 2; \
        _pp[0] += clock64() - _pt0;                                              \
        const long long _n = (_pp[1] >> 32) > _h.n ? (_pp[1] >> 32) : _h.n;      \
        _pp[1] = __LINE__ | (_n << 32);                                          \
    }
#else
#define K1_PROF_T0
#define K1_PROF_T1(_h)
#endif
#define K1_OP_DO(h, SZ, ...)      \
    PZ8 h;                        \
    {                             \
        K1_PROF_T0;               \
        h = (__VA_ARGS__);        \
        K1_PROF_T1(h)             \
    }                             \
    k1_sync_cta();                \
    top = end_of<SZ>(h);          \
    top_max = top > top_max ? top : top_max
#define K1_OP_VAR(h, SZ, ...) \
    {                         \
        K1_PROF_T0;           \
        h = (__VA_ARGS__);    \
        K1_PROF_T1(h)         \
    }                         \
    k1_sync_cta();            \
    top = end_of<SZ>(h);      \
    top_max = top > top_max ? top : top_max

// FK_ONLY: the ARMTD comparison planner (B.jrs_ext set): forward kinematics only, as mg_task_list_fk in the latency
// configuration; with an imported joint reachable set the Newton-Euler pass would run on meaningless Bezier models.  A template
// parameter rather than a test of B.jrs_ext, so that the main planner's kernel is the same code as without the ARMTD path.
template <bool FK_ONLY>
K1_DI int build_unit(const Batch& B, int p, int t) {
    const RobotConstants& rc = c_robot;
    K1S& S = k1s();
    const int tid = k1_tid();
    const int NJ = B.NJ, T = B.T;
    constexpr int B0 = JRS_WORDS;  // bottom of the working arena
    int top = B0, top_max = B0, gtop = 0;

    build_jrs(B, p, t);

    // ---- forward kinematics of the link volumes (KPR/Dynamics.cu:69-81) ----
    {
        bool ok;
        PZ8 FK_R = pz_alloc<9>(top, 0, &ok);
        top = end_of<9>(FK_R);
        PZ8 FK_T = pz_alloc<3>(top, 0, &ok);
        top = end_of<3>(FK_T);
        if (ok) {
            if (tid < 27) vptr(FK_R.off)[tid] = (tid < 9 && tid % 4 == 0) ? 1.0 : 0.0;
            if (tid >= 32 && tid < 41) vptr(FK_T.off)[tid - 32] = 0.0;
        }
        k1_sync();
        for (int i = 0; i < NJ; i++) {
            K1_OP_DO(t1, 3, op_const_mul<2>(top, &rc.trans[3 * i], 0.0, FK_R));
            PZ8 FK_T2, FK_R2;
            K1_OP_VAR(FK_T2, 3, op_add<3>(top, FK_T, t1));
            K1_OP_VAR(FK_R2, 9, op_mul33<3, false>(top, FK_R, jrs_R(i)));
            const PZ8 box = make_link_box(top, i);
            top = box.off + pz_words(3, 3);  // the block was sized for three generators
            K1_OP_DO(l1, 3, op_mul33<1, false>(top, FK_R2, box));
            K1_OP_DO(link, 3, op_add<3>(top, l1, FK_T2));
            export_link(link, B, p, t, i);
            int cur = B0;  // slide over the old FK_R / FK_T
            keep<3>(cur, FK_T2);
            keep<9>(cur, FK_R2);
            top = cur;
            FK_T = FK_T2;
            FK_R = FK_R2;
        }
    }
    if (FK_ONLY) return top_max;

    // ---- recursive Newton-Euler, forward pass (KPR/Dynamics.cu:83-155) ----
    top = B0;
    PZ8 la, w, wa, wd;
    K1_OP_VAR(la, 3, pz_zero<3>(top));
    K1_OP_VAR(w, 3, pz_zero<3>(top));
    K1_OP_VAR(wa, 3, pz_zero<3>(top));
    K1_OP_VAR(wd, 3, pz_zero<3>(top));
    if (!S.fail && tid == 0) vptr(la.off)[2] = rc.gravity;
    k1_sync();
    for (int i = 0; i < NJ; i++) {
        const double* pI = &rc.trans[3 * i];
        const double* cI = &rc.com[3 * i];
        const PZ8 Rt = jrs_R(i);  // used transposed
        // state blocks sit at the bottom of the arena in the order of the keep lists below; each step
        // drops what has just died so the live set stays small
        const int mark = top;
        PZ8 la2;
        {
            K1_OP_DO(t1, 3, op_cross_const(top, wd, pI, false));
            PZ8 t2;
            K1_OP_VAR(t2, 3, op_add<3>(top, la, t1));
            int cur = mark;
            keep<3>(cur, t2);
            top = cur;
            K1_OP_DO(t3, 3, op_cross_const(top, wa, pI, false));
            K1_OP_DO(t4, 3, op_cross(top, w, t3));
            PZ8 t5;
            K1_OP_VAR(t5, 3, op_add<3>(top, t2, t4));
            cur = mark;
            keep<3>(cur, t5);
            top = cur;
            K1_OP_VAR(la2, 3, op_mul33<1, true>(top, Rt, t5));
        }
        PZ8 w2, wa2, wd3;
        if (rc.axes[i] != 0) {
            const int ax = abs(rc.axes[i]) - 1;
            int cur = B0;  // la is dead
            keep<3>(cur, w);
            keep<3>(cur, wa);
            keep<3>(cur, wd);
            keep<3>(cur, la2);
            top = cur;
            K1_OP_DO(w1, 3, op_mul33<1, true>(top, Rt, w));
            K1_OP_VAR(w2, 3, op_add_one_dim(top, w1, jrs_scalar(0, i), ax));
            cur = B0;  // w, w1 are dead
            keep<3>(cur, wa);
            keep<3>(cur, wd);
            keep<3>(cur, la2);
            keep<3>(cur, w2);
            top = cur;
            PZ8 wa1, wd1;
            K1_OP_VAR(wa1, 3, op_mul33<1, true>(top, Rt, wa));
            K1_OP_VAR(wd1, 3, op_mul33<1, true>(top, Rt, wd));
            cur = B0;  // wa, wd are dead
            keep<3>(cur, la2);
            keep<3>(cur, w2);
            keep<3>(cur, wa1);
            keep<3>(cur, wd1);
            top = cur;
            const int m2 = top;
            K1_OP_DO(zero3, 3, pz_zero<3>(top));
            K1_OP_DO(tmp, 3, op_add_one_dim(top, zero3, jrs_scalar(0, i), ax));
            K1_OP_DO(t6, 3, op_cross(top, wa1, tmp));
            PZ8 wd2;
            K1_OP_VAR(wd2, 3, op_add<3>(top, wd1, t6));
            cur = m2;
            keep<3>(cur, wd2);
            top = cur;
            K1_OP_VAR(wa2, 3, op_add_one_dim(top, wa1, jrs_scalar(1, i), ax));
            K1_OP_VAR(wd3, 3, op_add_one_dim(top, wd2, jrs_scalar(2, i), ax));
            cur = B0;  // wa1, wd1, wd2 are dead
            keep<3>(cur, la2);
            keep<3>(cur, w2);
            keep<3>(cur, wa2);
            keep<3>(cur, wd3);
            top = cur;
        } else {
            K1_OP_VAR(w2, 3, op_mul33<1, true>(top, Rt, w));
            K1_OP_VAR(wa2, 3, op_mul33<1, true>(top, Rt, wa));
            K1_OP_VAR(wd3, 3, op_mul33<1, true>(top, Rt, wd));
            int cur = B0;
            keep<3>(cur, la2);
            keep<3>(cur, w2);
            keep<3>(cur, wa2);
            keep<3>(cur, wd3);
            top = cur;
        }
        {
            const int m3 = top;
            K1_OP_DO(t7, 3, op_cross_const(top, wd3, cI, false));
            PZ8 t8;
            K1_OP_VAR(t8, 3, op_add<3>(top, la2, t7));
            int cur = m3;
            keep<3>(cur, t8);
            top = cur;
            K1_OP_DO(t9, 3, op_cross_const(top, wa2, cI, false));
            K1_OP_DO(t10, 3, op_cross(top, w2, t9));
            PZ8 t11;
            K1_OP_VAR(t11, 3, op_add<3>(top, t8, t10));
            cur = m3;
            keep<3>(cur, t11);
            top = cur;
            K1_OP_DO(F, 3, op_const_mul<0>(top, &rc.mass[i], rc.mass_uncertainty, t11));
            const PZ8 Fs = spill_global<3>(gtop, F);
            top = m3;
            K1_OP_DO(t12, 3, op_const_mul<1>(top, &rc.inertia[i * 9], rc.inertia_uncertainty, wd3));
            K1_OP_DO(t13, 3, op_const_mul<1>(top, &rc.inertia[i * 9], rc.inertia_uncertainty, w2));
            K1_OP_DO(t14, 3, op_cross(top, wa2, t13));
            K1_OP_DO(N, 3, op_add<3>(top, t12, t14));
            const PZ8 Ns = spill_global<3>(gtop, N);
            if (tid == 0) {
                S.Fg[i] = Fs;
                S.Ng[i] = Ns;
            }
            top = m3;
        }
        la = la2;
        w = w2;
        wd = wd3;
        wa = wa2;
    }

    // ---- backward pass (KPR/Dynamics.cu:157-180) ----
    top = B0;
    PZ8 f, n;
    K1_OP_VAR(f, 3, pz_zero<3>(top));  // the barrier inside also publishes S.Fg / S.Ng
    K1_OP_VAR(n, 3, pz_zero<3>(top));
    for (int i = NJ - 1; i >= 0; i--) {
        const PZ8 Rn = jrs_R(i + 1);
        const PZ8 Fi = S.Fg[i], Ni = S.Ng[i];
        const int mark = top;
        K1_OP_DO(a1, 3, op_mul33<1, false>(top, Rn, n));
        PZ8 a2;
        K1_OP_VAR(a2, 3, op_add<3>(top, Ni, a1));
        int cur = mark;
        keep<3>(cur, a2);
        top = cur;
        K1_OP_DO(a3, 3, op_cross_const(top, Fi, &rc.com[3 * i], true));
        PZ8 a4;
        K1_OP_VAR(a4, 3, op_add<3>(top, a2, a3));
        cur = mark;
        keep<3>(cur, a4);
        top = cur;
        K1_OP_DO(a5, 3, op_mul33<1, false>(top, Rn, f));
        K1_OP_DO(a6, 3, op_cross_const(top, a5, &rc.trans[3 * (i + 1)], true));
        PZ8 n2, f2;
        K1_OP_VAR(n2, 3, op_add<3>(top, a4, a6));
        K1_OP_VAR(f2, 3, op_add<3>(top, a5, Fi));
        cur = B0;
        keep<3>(cur, n2);
        keep<3>(cur, f2);
        top = cur;
        n = n2;
        f = f2;
        if (rc.axes[i] != 0) {
            const int ax = abs(rc.axes[i]) - 1;
            const int m2 = top;
            K1_OP_DO(u1, 1, op_lin2<1>(top, n, 3, ax, 0, 1.0, jrs_scalar(2, i), 1, 0, 0, rc.armature[i]));
            K1_OP_DO(u2, 1, op_lin2<1>(top, u1, 1, 0, 0, 1.0, jrs_scalar(0, i), 1, 0, 0, rc.damping[i]));
            export_torque(u2, B, p, t, i);
            top = m2;
        }
    }

    // ---- robust-input radius (KPR/armour_main.cu:172-201) ----
    if (!S.fail && tid == 0) {
        const double* s_unom_r = S.misc;
        const double* s_dist = S.misc + 8;
        double rho = 0.0;
        for (int j = 0; j < NF; j++) rho = __dadd_ru(rho, __dmul_ru(s_dist[j], s_dist[j]));
        const double nrm = __dsqrt_ru(rho);
        for (int j = 0; j < NF; j++) {
            double v = __dadd_ru(__dmul_ru(__dmul_ru(rc.alpha, rc.M_max - rc.M_min), rc.eps), 0.5 * s_dist[j]);
            v = __dadd_ru(v, 0.5 * nrm);
            v = __dadd_ru(v, s_unom_r[j]);
            v = __dadd_ru(v, rc.friction[j]);
            B.torque_radius[size_t(p) * NF * T + size_t(j) * T + t] = __dmul_ru(v, RADIUS_SLACK);
        }
    }
    k1_sync();
    return top_max;
}
#undef K1_OP_DO
#undef K1_OP_VAR


// ---- MG mode, host-checkable part: mailbox slots, task kinds and the claim order (pure integer code; the CPU
// suite checks through tests/emu that the order is topological for the dependencies of run_task) ----
enum {
    MB_W, MB_WA1, MB_WA2, MB_WD, MB_T4, MB_LA, MB_T10, MB_F, MB_A3, MB_N, MB_FKR, MB_FKT, MB_A6, MB_F2, MB_N2,
    EV_FKL, EV_U, MB_KINDS
};
static_assert(MB_KINDS * (MAXJ + 1) <= MB_SLOTS, "mailbox slots");
enum { TK_W, TK_WA, TK_WD, TK_T4, TK_LA, TK_T10, TK_TF, TK_TN, TK_FKC, TK_FKL, TK_FB, TK_NB, TK_U, TK_EPI };
// Claim order of the tasks of one unit (a topological order).  The forward Newton-Euler pass keeps the three groups
// busy on its own; the backward pass is a chain (FB, one group) with a follower (NB, U), so the kinematics tasks -
// which nothing inside the kernel consumes - are dealt out there: round r of the backward pass offers FB(NJ-1-r),
// FKC(r), FKL(r-1), NB(NJ-r), U(NJ+1-r), all of which depend only on results of round r-1.
#ifndef K1_FK_EARLY
#define K1_FK_EARLY 3
#endif
K1_DI int mg_task_list(unsigned short* tasks, int NJ) {
    int n = 0;
    const int fwd[8] = {TK_W, TK_WA, TK_T4, TK_WD, TK_LA, TK_T10, TK_TN, TK_TF};
    // the forward pass ends in a chain (T10 -> TF of the last joint, the biggest cross product of the unit) on which
    // two groups would wait: the kinematics of the first K1_FK_EARLY joints is offered there
    const int early = K1_FK_EARLY < NJ ? K1_FK_EARLY : NJ;
    for (int i = 0; i < NJ; i++)
        for (int q = 0; q < 8; q++) {
            if (i == NJ - 1 && fwd[q] == TK_TF)
                for (int r = 0; r < early; r++) {
                    tasks[n++] = (unsigned short)((TK_FKC << 8) | r);
                    tasks[n++] = (unsigned short)((TK_FKL << 8) | r);
                }
            tasks[n++] = (unsigned short)((fwd[q] << 8) | i);
        }
    // backward rounds; the remaining kinematics joints are spread over them
    for (int r = 0; r <= NJ + 1; r++) {
        const int fk = early + r;  // FKC(fk) and FKL(fk - 1) in round r
        if (NJ - 1 - r >= 0) tasks[n++] = (unsigned short)((TK_FB << 8) | (NJ - 1 - r));
        if (fk < NJ) tasks[n++] = (unsigned short)((TK_FKC << 8) | fk);
        if (fk - 1 >= early && fk - 1 < NJ) tasks[n++] = (unsigned short)((TK_FKL << 8) | (fk - 1));
        if (NJ - r >= 0 && NJ - r < NJ) tasks[n++] = (unsigned short)((TK_NB << 8) | (NJ - r));
        if (NJ + 1 - r >= 0 && NJ + 1 - r < NJ) tasks[n++] = (unsigned short)((TK_U << 8) | (NJ + 1 - r));
    }
    tasks[n++] = (unsigned short)(TK_EPI << 8);
    return n;
}

// forward kinematics only (ARMTD comparison planner: no Newton-Euler pass, KPA/Dynamics.cu): the chain FKC(0..NJ-1) with the
// link volume FKL(i) offered right behind FKC(i); every task depends on tasks before it in the list only
K1_DI int mg_task_list_fk(unsigned short* tasks, int NJ) {
    int n = 0;
    for (int i = 0; i < NJ; i++) {
        tasks[n++] = (unsigned short)((TK_FKC << 8) | i);
        tasks[n++] = (unsigned short)((TK_FKL << 8) | i);
    }
    return n;
}

#if K1_MG
// ---- MG mode: one unit built by all groups of the CTA ------------------------------------------------
// The unit is a list of tasks; operands and results travel through the CTA's mailbox (global memory, written
// once per unit, L2-resident), so a task is a pure function mailbox -> mailbox and any group can run it.
// Operation order inside every chain of the recursion and every simplify() point are those of build_unit().
K1_DI int mb_slot(int kind, int i) { return kind * (MAXJ + 1) + i; }

K1_DI void ev_signal(int slot) {  // called by all threads of the group after a barrier that follows the writes
    if (k1_tid() == 0) {
        K1X& X = k1x();
        __threadfence_block();
        reinterpret_cast<volatile int*>(X.ev)[slot] = X.seq;
    }
}
K1_DI void ev_wait(int slot) {
    if (k1_tid() == 0) {
        K1X& X = k1x();
        const int seq = X.seq;
#ifdef K1_PROFILE
        const long long _w0 = clock64();
#endif
        while (reinterpret_cast<volatile int*>(X.ev)[slot] != seq) __nanosleep(40);
        __threadfence_block();
#ifdef K1_PROFILE
        k1s().red2[NW * RED_STRIDE - 1] += double(clock64() - _w0);  // (thread 0 only; last word is otherwise unused)
#endif
    }
    k1_sync();
}
// copy block h into the mailbox and announce it under `slot`
template <int SZ>
K1_DI void mb_publish(int slot, PZ8 h) {
    K1S& S = k1s();
    K1X& X = k1x();
    const int tid = k1_tid();
    const int w = pz_words(h.n, SZ);
    const bool ok = !S.fail && w <= X.mbox_words;  // mbox_words: words of ONE slot
    if (ok) {
        const double* src = vptr(h.off);
        double* dst = X.mbox + size_t(slot) * X.mbox_words;
        for (int i = tid; i < w; i += NT) dst[i] = src[i];
    } else {
        set_fail(FAIL_SCRATCH);
    }
    if (tid == 0) {
        PZ8 m;
        m.off = ok ? 0 : -1;
        m.n = ok ? h.n : 0;
        X.mb[slot] = m;
    }
    k1_sync();
    ev_signal(slot);
}
// wait for block `slot` and copy it into the arena at `top`
template <int SZ>
K1_DI PZ8 mb_import(int slot, int top) {
    K1X& X = k1x();
    const int tid = k1_tid();
    ev_wait(slot);
    const PZ8 m = X.mb[slot];
    if (m.off < 0) set_fail(FAIL_SCRATCH);  // the producer failed
    bool ok;
    const PZ8 h = pz_alloc<SZ>(top, m.off < 0 ? 0 : m.n, &ok);
    if (ok) {
        const int w = pz_words(h.n, SZ);
        const double* src = X.mbox + size_t(slot) * X.mbox_words;
        double* dst = vptr(h.off);
        for (int i = tid; i < w; i += NT) dst[i] = src[i];
    }
    k1_sync();
    return h;
}
// the block of joint i - 1, or the recursion's zero start value for the first joint
template <int SZ>
K1_DI PZ8 mb_prev(int kind, int i, int top) {
    if (i == 0) return pz_zero<SZ>(top);
    return mb_import<SZ>(mb_slot(kind, i - 1), top);
}

#define MG_DO(h, SZ, ...)        \
    const PZ8 h = (__VA_ARGS__); \
    top = end_of<SZ>(h);         \
    top_max = top > top_max ? top : top_max

K1_DI int run_task(const Batch& B, int p, int t, int kind, int i) {
    const RobotConstants& rc = c_robot;
    K1S& S = k1s();
    const int tid = k1_tid();
    const int NJ = B.NJ;
    constexpr int B0 = JRS_WORDS;
    int top = B0, top_max = B0;
    const int ax = (kind != TK_EPI && rc.axes[i] != 0) ? abs(rc.axes[i]) - 1 : -1;  // -1: fixed joint
    switch (kind) {
    case TK_W: {  // w_i = R_i^T w_{i-1} + qd_i e_axis   (KPR/Dynamics.cu:95-103)
        MG_DO(w, 3, mb_prev<3>(MB_W, i, top));
        MG_DO(w1, 3, op_mul33<1, true>(top, jrs_R(i), w));
        if (ax >= 0) {
            MG_DO(w2, 3, op_add_one_dim(top, w1, jrs_scalar(0, i), ax));
            mb_publish<3>(mb_slot(MB_W, i), w2);
        } else {
            mb_publish<3>(mb_slot(MB_W, i), w1);
        }
    } break;
    case TK_WA: {  // auxiliary angular velocity
        MG_DO(wa, 3, mb_prev<3>(MB_WA2, i, top));
        MG_DO(wa1, 3, op_mul33<1, true>(top, jrs_R(i), wa));
        if (ax >= 0) {
            mb_publish<3>(mb_slot(MB_WA1, i), wa1);
            MG_DO(wa2, 3, op_add_one_dim(top, wa1, jrs_scalar(1, i), ax));
            mb_publish<3>(mb_slot(MB_WA2, i), wa2);
        } else {
            mb_publish<3>(mb_slot(MB_WA2, i), wa1);
        }
    } break;
    case TK_WD: {  // angular acceleration
        MG_DO(wd, 3, mb_prev<3>(MB_WD, i, top));
        MG_DO(wd1, 3, op_mul33<1, true>(top, jrs_R(i), wd));
        if (ax >= 0) {
            MG_DO(wa1, 3, mb_import<3>(mb_slot(MB_WA1, i), top));
            MG_DO(zero3, 3, pz_zero<3>(top));
            MG_DO(tmp, 3, op_add_one_dim(top, zero3, jrs_scalar(0, i), ax));
            MG_DO(t6, 3, op_cross(top, wa1, tmp));
            MG_DO(wd2, 3, op_add<3>(top, wd1, t6));
            MG_DO(wd3, 3, op_add_one_dim(top, wd2, jrs_scalar(2, i), ax));
            mb_publish<3>(mb_slot(MB_WD, i), wd3);
        } else {
            mb_publish<3>(mb_slot(MB_WD, i), wd1);
        }
    } break;
    case TK_T4: {  // w_{i-1} x (wa_{i-1} x p_i)
        MG_DO(wa, 3, mb_prev<3>(MB_WA2, i, top));
        MG_DO(t3, 3, op_cross_const(top, wa, &rc.trans[3 * i], false));
        MG_DO(w, 3, mb_prev<3>(MB_W, i, top));
        MG_DO(t4, 3, op_cross(top, w, t3));
        mb_publish<3>(mb_slot(MB_T4, i), t4);
    } break;
    case TK_LA: {  // linear acceleration of the joint frame
        PZ8 la;
        if (i == 0) {
            la = pz_zero<3>(top);
            if (!S.fail && tid == 0) vptr(la.off)[2] = rc.gravity;
            k1_sync();
        } else {
            la = mb_import<3>(mb_slot(MB_LA, i - 1), top);
        }
        top = end_of<3>(la);
        MG_DO(wd, 3, mb_prev<3>(MB_WD, i, top));
        MG_DO(t1, 3, op_cross_const(top, wd, &rc.trans[3 * i], false));
        MG_DO(t2, 3, op_add<3>(top, la, t1));
        MG_DO(t4, 3, mb_import<3>(mb_slot(MB_T4, i), top));
        MG_DO(t5, 3, op_add<3>(top, t2, t4));
        MG_DO(la2, 3, op_mul33<1, true>(top, jrs_R(i), t5));
        mb_publish<3>(mb_slot(MB_LA, i), la2);
    } break;
    case TK_T10: {  // w_i x (wa_i x c_i)
        MG_DO(wa2, 3, mb_import<3>(mb_slot(MB_WA2, i), top));
        MG_DO(t9, 3, op_cross_const(top, wa2, &rc.com[3 * i], false));
        MG_DO(w2, 3, mb_import<3>(mb_slot(MB_W, i), top));
        MG_DO(t10, 3, op_cross(top, w2, t9));
        mb_publish<3>(mb_slot(MB_T10, i), t10);
    } break;
    case TK_TF: {  // F_i = m_i (la_i + wd_i x c_i + w_i x (wa_i x c_i)), and c_i x F_i for the backward pass
        MG_DO(wd3, 3, mb_import<3>(mb_slot(MB_WD, i), top));
        MG_DO(t7, 3, op_cross_const(top, wd3, &rc.com[3 * i], false));
        MG_DO(la2, 3, mb_import<3>(mb_slot(MB_LA, i), top));
        MG_DO(t8, 3, op_add<3>(top, la2, t7));
        MG_DO(t10, 3, mb_import<3>(mb_slot(MB_T10, i), top));
        MG_DO(t11, 3, op_add<3>(top, t8, t10));
        MG_DO(F, 3, op_const_mul<0>(top, &rc.mass[i], rc.mass_uncertainty, t11));
        mb_publish<3>(mb_slot(MB_F, i), F);
        MG_DO(a3, 3, op_cross_const(top, F, &rc.com[3 * i], true));
        mb_publish<3>(mb_slot(MB_A3, i), a3);
    } break;
    case TK_TN: {  // N_i = I_i wd_i + wa_i x (I_i w_i)
        MG_DO(wd3, 3, mb_import<3>(mb_slot(MB_WD, i), top));
        MG_DO(t12, 3, op_const_mul<1>(top, &rc.inertia[i * 9], rc.inertia_uncertainty, wd3));
        MG_DO(w2, 3, mb_import<3>(mb_slot(MB_W, i), top));
        MG_DO(t13, 3, op_const_mul<1>(top, &rc.inertia[i * 9], rc.inertia_uncertainty, w2));
        MG_DO(wa2, 3, mb_import<3>(mb_slot(MB_WA2, i), top));
        MG_DO(t14, 3, op_cross(top, wa2, t13));
        MG_DO(N, 3, op_add<3>(top, t12, t14));
        mb_publish<3>(mb_slot(MB_N, i), N);
    } break;
    case TK_FKC: {  // forward-kinematics chain (KPR/Dynamics.cu:69-81)
        bool ok;
        PZ8 FK_R, FK_T;
        if (i == 0) {
            FK_R = pz_alloc<9>(top, 0, &ok);
            top = end_of<9>(FK_R);
            FK_T = pz_alloc<3>(top, 0, &ok);
            top = end_of<3>(FK_T);
            if (ok) {
                if (tid < 27) vptr(FK_R.off)[tid] = (tid < 9 && tid % 4 == 0) ? 1.0 : 0.0;
                if (tid >= 32 && tid < 41) vptr(FK_T.off)[tid - 32] = 0.0;
            }
            k1_sync();
        } else {
            FK_R = mb_import<9>(mb_slot(MB_FKR, i - 1), top);
            top = end_of<9>(FK_R);
            FK_T = mb_import<3>(mb_slot(MB_FKT, i - 1), top);
            top = end_of<3>(FK_T);
        }
        top_max = top > top_max ? top : top_max;
        MG_DO(t1, 3, op_const_mul<2>(top, &rc.trans[3 * i], 0.0, FK_R));
        MG_DO(FK_T2, 3, op_add<3>(top, FK_T, t1));
        mb_publish<3>(mb_slot(MB_FKT, i), FK_T2);
        MG_DO(FK_R2, 9, op_mul33<3, false>(top, FK_R, jrs_R(i)));
        mb_publish<9>(mb_slot(MB_FKR, i), FK_R2);
    } break;
    case TK_FKL: {  // link volume i: FK_R box + FK_T, reduce_link_PZ
        MG_DO(FK_R2, 9, mb_import<9>(mb_slot(MB_FKR, i), top));
        MG_DO(FK_T2, 3, mb_import<3>(mb_slot(MB_FKT, i), top));
        MG_DO(box, 3, make_link_box(top, i));
        MG_DO(l1, 3, op_mul33<1, false>(top, FK_R2, box));
        MG_DO(link, 3, op_add<3>(top, l1, FK_T2));
        export_link(link, B, p, t, i);
    } break;
    case TK_FB: {  // backward pass, force chain: f_i = R_{i+1} f_{i+1} + F_i; also p_{i+1} x (R_{i+1} f_{i+1})
        MG_DO(Fi, 3, mb_import<3>(mb_slot(MB_F, i), top));  // published long ago: fetched while the chain value is awaited
        PZ8 f;
        if (i == NJ - 1) f = pz_zero<3>(top); else f = mb_import<3>(mb_slot(MB_F2, i + 1), top);
        top = end_of<3>(f);
        MG_DO(a5, 3, op_mul33<1, false>(top, jrs_R(i + 1), f));
        MG_DO(f2, 3, op_add<3>(top, a5, Fi));
        mb_publish<3>(mb_slot(MB_F2, i), f2);  // the chain moves on before the side product is made
        MG_DO(a6, 3, op_cross_const(top, a5, &rc.trans[3 * (i + 1)], true));
        mb_publish<3>(mb_slot(MB_A6, i), a6);
    } break;
    case TK_NB: {  // backward pass, moment chain: n_i = ((N_i + R_{i+1} n_{i+1}) + c_i x F_i) + p_{i+1} x (R f)
        MG_DO(Ni, 3, mb_import<3>(mb_slot(MB_N, i), top));
        MG_DO(a3, 3, mb_import<3>(mb_slot(MB_A3, i), top));
        PZ8 n;
        if (i == NJ - 1) n = pz_zero<3>(top); else n = mb_import<3>(mb_slot(MB_N2, i + 1), top);
        top = end_of<3>(n);
        MG_DO(a1, 3, op_mul33<1, false>(top, jrs_R(i + 1), n));
        MG_DO(a2, 3, op_add<3>(top, Ni, a1));
        MG_DO(a4, 3, op_add<3>(top, a2, a3));
        MG_DO(a6, 3, mb_import<3>(mb_slot(MB_A6, i), top));
        MG_DO(n2, 3, op_add<3>(top, a4, a6));
        mb_publish<3>(mb_slot(MB_N2, i), n2);
    } break;
    case TK_U: {  // joint torque u_i = n_i[axis] + armature qdda + damping qd, its k-only table
        if (ax >= 0) {
            MG_DO(n, 3, mb_import<3>(mb_slot(MB_N2, i), top));
            MG_DO(u1, 1, op_lin2<1>(top, n, 3, ax, 0, 1.0, jrs_scalar(2, i), 1, 0, 0, rc.armature[i]));
            MG_DO(u2, 1, op_lin2<1>(top, u1, 1, 0, 0, 1.0, jrs_scalar(0, i), 1, 0, 0, rc.damping[i]));
            export_torque(u2, B, p, t, i);
        }
        k1_sync();
        ev_signal(mb_slot(EV_U, i));
    } break;
    case TK_EPI: {  // robust-input radius (KPR/armour_main.cu:172-201), after every torque task
        for (int j = 0; j < NJ; j++) ev_wait(mb_slot(EV_U, j));
        bool any_fail = S.fail != 0;
        if (tid == 0) {
            const K1X& X = k1x();
            const double* s_unom_r = X.misc;
            const double* s_dist = X.misc + 8;
            double rho = 0.0;
            for (int j = 0; j < NF; j++) rho = __dadd_ru(rho, __dmul_ru(s_dist[j], s_dist[j]));
            const double nrm = __dsqrt_ru(rho);
            for (int j = 0; j < NF && !any_fail; j++) {
                double v = __dadd_ru(__dmul_ru(__dmul_ru(rc.alpha, rc.M_max - rc.M_min), rc.eps), 0.5 * s_dist[j]);
                v = __dadd_ru(v, 0.5 * nrm);
                v = __dadd_ru(v, s_unom_r[j]);
                v = __dadd_ru(v, rc.friction[j]);
                B.torque_radius[size_t(p) * NF * B.T + size_t(j) * B.T + t] = __dmul_ru(v, RADIUS_SLACK);
            }
        }
        k1_sync();
    } break;
    }
    return top_max;
}
#undef MG_DO

#endif  // K1_MG

// ---- kernel ---------------------------------------------------------------------------------------
#if K1_JRS_GLOBAL
constexpr int K1_FIXED_BYTES = K1S_BYTES;  // per group: the control block only (the JRS region is in the global scratch)
static_assert(!MG, "K1_JRS_GLOBAL is a knob of the throughput configuration");
#else
constexpr int K1_FIXED_BYTES = K1S_BYTES + JRS_WORDS * 8;  // per group: control block + joint reachable set region
#endif

// FK_ONLY (throughput configuration only): see build_unit; the latency configuration reads B.jrs_ext for its task list
template <bool FK_ONLY>
K1_DI void reachsets_body(const K1Params& P) {
#ifndef ARMOUR_EMU
    // a kernel launched behind this one with programmatic stream serialisation (k_hyperplanes in the latency path) may
    // start as soon as every CTA of this grid is resident; it synchronises on P.unit_flag, not on this grid's end
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
#if K1_MG
    if (threadIdx.x == 0) {
        K1X& X0 = k1x();
        X0.group_bytes = P.group_bytes;
        X0.seq = 0;
        X0.mbox = P.mbox + size_t(blockIdx.x) * MB_SLOTS * P.mbox_words;
        X0.mbox_words = P.mbox_words;
        X0.ntasks = P.B.jrs_ext ? mg_task_list_fk(X0.tasks, P.B.NJ) : mg_task_list(X0.tasks, P.B.NJ);
    }
    for (int i = threadIdx.x; i < MB_SLOTS; i += NT * GROUPS) k1x().ev[i] = 0;
#else
    if (threadIdx.x == 0) *reinterpret_cast<int*>(smem_cta()) = P.group_bytes;
#endif
    __syncthreads();
    K1S& S = k1s();
    const int tid = k1_tid();
    const int slot = blockIdx.x * GROUPS + k1_group();  // scratch slot of this group
    if (tid == 0) {
#if K1_JRS_GLOBAL
        S.gbase = P.gscr + size_t(slot) * P.gscr_words + JRS_WORDS;  // [JRS region | spill space | F/N scratch]
        S.AW = JRS_WORDS;
        S.GW = P.gscr_words - P.fn_words - JRS_WORDS;
#else
        S.gbase = P.gscr + size_t(slot) * P.gscr_words;
        S.AW = JRS_WORDS + P.arena_words;
        S.GW = P.gscr_words - P.fn_words;
#endif
        S.tab_g = P.gtab + size_t(slot) * P.gtab_bytes;
        S.thr = c_robot.simplify_threshold;
        S.thr2 = threshold_sq(S.thr);
        S.FW = P.fn_words;
        S.tab_s_bytes = P.tab_s_bytes;
        S.tab_g_bytes = P.gtab_bytes;
        S.fail = 0;
        S.n_tab_global = 0;
        S.flip = 0;
    }
    for (int i = tid; i < 2 * MASK_WORDS; i += NT) (&S.mask[0][0])[i] = 0u;
    k1_sync();
    u64* s_tab = reinterpret_cast<u64*>(tab_s0());
    for (int i = tid; i < P.tab_s_bytes / 8; i += NT) s_tab[i] = 0;
    k1_sync();

    const int nunits = P.units ? P.nunits : P.B.nprob * P.B.T;
    int nfail = 0, ndone = 0, top_max = 0;
    int* cta_unit = reinterpret_cast<int*>(smem_cta()) + 1;
    for (;;) {
#if K1_MG
        // one unit per CTA, built by all groups: claim it, reset the mailbox and the task cursor
        if (threadIdx.x == 0) {
            K1X& X0 = k1x();
            *cta_unit = atomicAdd(P.work, 1);
            X0.seq++;
            X0.next = 0;
            X0.bump = 0;
        }
        if (tid == 0) S.fail = 0;
        __syncthreads();
        int unit = *cta_unit;
        if (unit >= nunits) break;
        const bool extra = false;
        int p, t;
        if (P.units) {
            unit = P.units[unit];
            p = unit / P.B.T;
            t = unit % P.B.T;
        } else {
            t = P.B.T - 1 - (unit / P.B.nprob);  // long intervals first
            p = unit % P.B.nprob;
        }
#ifdef K1_PROFILE
        const long long _u0 = clock64();
#endif
        // joint reachable set: group 0 computes, the others copy its fixed region
        if (k1_group() == 0) build_jrs(P.B, p, t);
        __syncthreads();
        if (k1_group() != 0) {
            const unsigned char* g0 = smem_cta() + K1_HDR_BYTES;
            const K1S* S0 = reinterpret_cast<const K1S*>(g0);
            const double* a0 = reinterpret_cast<const double*>(g0 + K1S_BYTES);
            for (int i = tid; i < JRS_WORDS; i += NT) arena0()[i] = a0[i];
            for (int i = tid; i < 40; i += NT) S.jrs_n[i] = S0->jrs_n[i];
        }
        k1_sync();
        int tm = 0;
        for (;;) {
            if (tid == 0) S.cnt[0] = atomicAdd(&k1x().next, 1);
            k1_sync();
            const int k = S.cnt[0];
            k1_sync();
            if (k >= k1x().ntasks) break;
            const int code = k1x().tasks[k];
#ifdef K1_PROFILE
            const long long _c0 = clock64();
            if (tid == 0) S.red2[NW * RED_STRIDE - 1] = 0.0;
#endif
            const int tk = run_task(P.B, p, t, code >> 8, code & 255);
#ifdef K1_PROFILE
            if (tid == 0 && k < 255) {
                long long* pp = g_k1prof + (size_t(t) * K1_PROF_SITES * 2) + size_t(k) * 4;
                pp[0] = _c0 - _u0;
                pp[1] = clock64() - _u0;
                pp[2] = (long long)S.red2[NW * RED_STRIDE - 1];
                pp[3] = code | (k1_group() << 16);
            }
#endif
            tm = tk > tm ? tk : tm;
        }
        top_max = tm > top_max ? tm : top_max;
        if (k1_group() == 0) ndone++;
#else
        // one tile of GROUPS consecutive units per CTA; consecutive units are the SAME interval of consecutive
        // problems, i.e. equally long, so the groups stay in step
        if (threadIdx.x == 0) *cta_unit = atomicAdd(P.work, GROUPS);
        if (tid == 0) S.fail = 0;
        __syncthreads();
        const int unit0 = *cta_unit;
        __syncthreads();
        if (unit0 >= nunits) break;
        int unit = unit0 + k1_group();
        const bool extra = unit >= nunits;  // a partial last tile: the spare groups redo its last unit (same results)
        if (extra) unit = nunits - 1;
        int p, t;
        if (P.units) {
            unit = P.units[unit];
            p = unit / P.B.T;
            t = unit % P.B.T;
        } else {
            t = P.B.T - 1 - (unit / P.B.nprob);  // long intervals first
            p = unit % P.B.nprob;
        }
#ifdef K1_PROFILE
        const long long _u0 = clock64();
#endif
        const int tm = build_unit<FK_ONLY>(P.B, p, t);
#ifdef K1_PROFILE
        if (tid == 0) {
            g_k1prof[(size_t(t) * K1_PROF_SITES + K1_PROF_SITES - 1) * 2] += clock64() - _u0;
            g_k1prof[(size_t(t) * K1_PROF_SITES + K1_PROF_SITES - 1) * 2 + 1] = 0;
        }
#endif
        top_max = tm > top_max ? tm : top_max;
        if (!extra) ndone++;
#endif
        const int failed = S.fail;
        if (failed) {
            if (!extra && (!MG || k1_group() == 0)) nfail++;
            if (tid == 0) {
                atomicMax(&P.B.status[p], P.B.epoch * 8 + failed);  // (epochs grow: no reset between builds)
                if (P.stats && atomicMax(&P.stats[6], P.B.epoch) < P.B.epoch) {  // first failing unit of this build
                    P.stats[4] = S.fail_line * 8 + failed;
                    P.stats[5] = p * P.B.T + t;
                }
            }
            // a failed operation may leave a table half-built: restore the all-zero invariant
            for (int i = tid; i < P.tab_s_bytes / 8; i += NT) s_tab[i] = 0;
            for (int i = tid; i < P.gtab_bytes / 8; i += NT) reinterpret_cast<u64*>(S.tab_g)[i] = 0;
            for (int i = tid; i < 2 * MASK_WORDS; i += NT) (&S.mask[0][0])[i] = 0u;
        }
        k1_sync();
        if (MG) __syncthreads();  // the unit is complete in every group before the mailbox is reused
#ifndef ARMOUR_EMU
        if (MG ? threadIdx.x == 0 : (tid == 0 && !extra)) {
            if (t == 0 && P.B.hp_slow) P.B.hp_slow[p] = 0;  // rows without a candidate list are counted by k_hyperplanes
            if (P.unit_flag) {
                __threadfence();
                atomicExch(&P.unit_flag[size_t(p) * P.B.T + t], P.B.epoch);
            }
        }
#endif
#if defined(K1_PROFILE) && K1_MG
        if (threadIdx.x == 0) g_k1prof[(size_t(t) * 256 + 255) * 4] = clock64() - _u0;
#endif
    }
#ifndef ARMOUR_EMU
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(P.work + 1, 1) == int(gridDim.x) - 1) {  // every other CTA is past its last fetch
        P.work[0] = 0;
        P.work[1] = 0;
    }
#endif
    if (tid == 0 && P.stats) {
        atomicMax(&P.stats[0], top_max - JRS_WORDS);
        atomicAdd(&P.stats[1], S.n_tab_global);
        atomicAdd(&P.stats[2], nfail);
        atomicAdd(&P.stats[3], ndone);
    }
}

__global__ void __launch_bounds__(NT * GROUPS, CTAS_PER_SM) k_reachsets(K1Params P) { reachsets_body<false>(P); }
#if !K1_MG
// the ARMTD comparison planner's build (B.jrs_ext set) in the throughput configuration: forward kinematics only
__global__ void __launch_bounds__(NT * GROUPS, CTAS_PER_SM) k_reachsets_fk(K1Params P) { reachsets_body<true>(P); }
#endif

#ifndef ARMOUR_EMU
// ---- host side: scratch buffers and launch ----------------------------------------------------------
#ifndef K1_DYN_CAP
#define K1_DYN_CAP -1
#endif
#ifndef K1_TAB_EIGHTHS
#define K1_TAB_EIGHTHS 5
#endif
#ifndef K1_TAB_16THS
#define K1_TAB_16THS (2 * K1_TAB_EIGHTHS)
#endif
struct K1Scratch {
    int* work = nullptr;
    int* stats = nullptr;
    double* gscr = nullptr;
    char* gtab = nullptr;
    int grid = 0;
    int gscr_words = 0, fn_words = 0, gtab_bytes = 0;
    int arena_words = 0, tab_s_bytes = 0, group_bytes = 0;
    size_t smem_bytes = 0;
    double* mbox = nullptr;
    int mbox_words = 0;
    int h_stats[4] = {0, 0, 0, 0};
};

inline void k1_scratch_destroy(K1Scratch* s) {
    if (s->work) cudaFree(s->work);
    if (s->stats) cudaFree(s->stats);
    if (s->gscr) cudaFree(s->gscr);
    if (s->gtab) cudaFree(s->gtab);
    if (s->mbox) cudaFree(s->mbox);
    *s = K1Scratch();
}

inline cudaError_t k1_scratch_create(K1Scratch* s, const armour_config& cfg, const RobotConstants&, cudaStream_t st) {
    cudaError_t e;
    int dev = 0, sms = 0, smem_optin = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
    // CTAS_PER_SM CTAs per SM: an equal share of the SM's shared memory each (1 KB per CTA is reserved by the system)
    int per_cta = (smem_optin + 1024) / CTAS_PER_SM - 1024;
    per_cta &= ~1023;
    const int per_group = ((per_cta - K1_HDR_BYTES) / GROUPS) & ~15;
    int dyn = per_group - K1_FIXED_BYTES;
    // K1_DYN_CAP: at most this much shared memory per group beyond the fixed region.  What the arena and the scratch do
    // not hold in shared memory lives in the group's global scratch, i.e. in the L1 cache, which gets the shared memory
    // the CTAs do not claim (the spill slots of the kernel go through the same cache): see DESIGN.md section 6.
    if (K1_DYN_CAP >= 0 && dyn > K1_DYN_CAP) dyn = K1_DYN_CAP;
#if K1_JRS_GLOBAL
    if (dyn > 0) dyn = 0;  // the arena must start right behind the JRS region, in the global scratch
#endif
    if (dyn < 0) return cudaErrorInvalidConfiguration;  // the fixed region of GROUPS groups does not fit
    s->tab_s_bytes = (dyn * K1_TAB_16THS / 16) & ~1023;  // scratch of the merge / hash passes; the rest is the PZ arena
    s->arena_words = (dyn - s->tab_s_bytes) / 8;
    s->group_bytes = K1_FIXED_BYTES + s->arena_words * 8 + s->tab_s_bytes;
    s->smem_bytes = K1_HDR_BYTES + size_t(GROUPS) * s->group_bytes;
    s->grid = CTAS_PER_SM * sms;  // CTAs; each holds GROUPS scratch slots
    // per-CTA global scratch: arena spill space, then F_i / N_i of one unit; and the overflow hash-table pool
    const int capw = cfg.cap_work_monomials;
    s->fn_words = 2 * MAXJ * (9 + capw * 2);
    s->gscr_words = s->fn_words + 24 * capw + (K1_JRS_GLOBAL ? ((JRS_WORDS + 15) & ~15) : 0);
    s->gtab_bytes = 16 * capw * 8 * 7;  // a cross product table for up to ~10 * capw candidate keys
    if ((e = cudaMalloc(&s->work, 2 * sizeof(int))) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(s->work, 0, 2 * sizeof(int), st)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&s->stats, 8 * sizeof(int))) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(s->stats, 0, 8 * sizeof(int), st)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&s->gscr, size_t(s->grid) * GROUPS * s->gscr_words * 8)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&s->gtab, size_t(s->grid) * GROUPS * s->gtab_bytes)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(s->gtab, 0, size_t(s->grid) * GROUPS * s->gtab_bytes, st)) != cudaSuccess) return e;
    if (MG) {  // mailbox of a CTA: one fixed slot per published block
        s->mbox_words = 27 + 4 * capw;
        if ((e = cudaMalloc(&s->mbox, size_t(s->grid) * MB_SLOTS * s->mbox_words * 8)) != cudaSuccess) return e;
    }
    if ((e = cudaMemsetAsync(s->stats, 0, 4 * sizeof(int), st)) != cudaSuccess) return e;
#if !K1_MG
    if ((e = cudaFuncSetAttribute(k_reachsets_fk, cudaFuncAttributeMaxDynamicSharedMemorySize, int(s->smem_bytes))) != cudaSuccess)
        return e;
#endif
    return cudaFuncSetAttribute(k_reachsets, cudaFuncAttributeMaxDynamicSharedMemorySize, int(s->smem_bytes));
}

inline cudaError_t launch_reachsets(const Batch& B, K1Scratch& s, cudaStream_t st, int* nlaunch, int* unit_flag = nullptr) {
    *nlaunch = 0;
    if (B.nprob == 0) return cudaSuccess;
    // nothing in front of the kernel: the unit counter is reset by the previous launch's last CTA, the build status and the
    // unit flags carry the build epoch
    K1Params P;
    P.B = B;
    P.work = s.work;
    P.unit_flag = unit_flag;
    P.gscr = s.gscr;
    P.gscr_words = s.gscr_words;
    P.fn_words = s.fn_words;
    P.gtab = s.gtab;
    P.gtab_bytes = s.gtab_bytes;
    P.arena_words = s.arena_words;
    P.tab_s_bytes = s.tab_s_bytes;
    P.group_bytes = s.group_bytes;
    P.stats = s.stats;
    P.mbox = s.mbox;
    P.mbox_words = s.mbox_words;
    P.units = nullptr;
    P.nunits = 0;
    const int ntiles = MG ? B.nprob * B.T : (B.nprob * B.T + GROUPS - 1) / GROUPS;
    const int grid = ntiles < s.grid ? ntiles : s.grid;
#if !K1_MG
    if (B.jrs_ext) {
        k_reachsets_fk<<<grid, NT * GROUPS, s.smem_bytes, st>>>(P);
        *nlaunch = 1;
        return cudaGetLastError();
    }
#endif
    k_reachsets<<<grid, NT * GROUPS, s.smem_bytes, st>>>(P);
    *nlaunch = 1;
    return cudaGetLastError();
}
#endif  // ARMOUR_EMU

}  // namespace K1_NS

}  // namespace armour
