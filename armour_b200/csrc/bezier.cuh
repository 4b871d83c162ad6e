// Degree-5 Bezier desired trajectory helpers (device + host).
//
// q(s; k) = B(s) k + q_indep(s), s in [0,1], with q(0)=q0, q'(0)=qd0 T, q''(0)=qdd0 T^2 and
// q(1)=q0+k, q'(1)=q''(1)=0 — the parameterisation of the reference planner
// (KPR/Trajectory.h:10-31, KPR/Trajectory.cu:542-572, 812-822).
#pragma once
#include <cmath>

#ifndef __CUDACC__
#define ARMOUR_HD
#else
#define ARMOUR_HD __host__ __device__ __forceinline__
#endif

namespace armour {

ARMOUR_HD double pw2(double x) { return x * x; }
ARMOUR_HD double pw3(double x) { return x * x * x; }
ARMOUR_HD double pw4(double x) { const double y = x * x; return y * y; }
ARMOUR_HD double pw5(double x) { const double y = x * x; return y * y * x; }

// Bernstein form, KPR/Trajectory.cu:542-556
ARMOUR_HD double bez_q(double q0, double Tqd0, double TTqdd0, double k, double t) {
    const double B0 = -pw5(t - 1);
    const double B1 = 5 * t * pw4(t - 1);
    const double B2 = -10 * pw2(t) * pw3(t - 1);
    const double B3 = 10 * pw3(t) * pw2(t - 1);
    const double B4 = -5 * pw4(t) * (t - 1);
    const double B5 = pw5(t);
    const double beta1 = q0 + Tqd0 / 5;
    const double beta2 = q0 + (2 * Tqd0) / 5 + TTqdd0 / 20;
    const double beta3 = q0 + k;
    return B0 * q0 + B1 * beta1 + B2 * beta2 + B3 * beta3 + B4 * beta3 + B5 * beta3;
}
// derivative w.r.t. normalised time, KPR/Trajectory.cu:558-572
ARMOUR_HD double bez_qd(double q0, double Tqd0, double TTqdd0, double k, double t) {
    const double dB0 = pw4(t - 1.0) * -5.0;
    const double dB1 = t * pw3(t - 1.0) * 2.0E+1 + pw4(t - 1.0) * 5.0;
    const double dB2 = t * pw3(t - 1.0) * -2.0E+1 - (t * t) * pw2(t - 1.0) * 3.0E+1;
    const double dB3 = pw3(t) * (t * 2.0 - 2.0) * 1.0E+1 + (t * t) * pw2(t - 1.0) * 3.0E+1;
    const double dB4 = pw3(t) * (t - 1.0) * -2.0E+1 - pw4(t) * 5.0;
    const double dB5 = pw4(t) * 5.0;
    const double beta1 = q0 + Tqd0 / 5;
    const double beta2 = q0 + (2 * Tqd0) / 5 + TTqdd0 / 20;
    const double beta3 = q0 + k;
    return dB0 * q0 + dB1 * beta1 + dB2 * beta2 + dB3 * beta3 + dB4 * beta3 + dB5 * beta3;
}
// second derivative w.r.t. normalised time (the reference has none: the closed-loop rollout needs qdd at the end of the
// executed segment); q''(0) = TTqdd0, q''(1) = 0
ARMOUR_HD double bez_qdd(double q0, double Tqd0, double TTqdd0, double k, double t) {
    const double u = 1.0 - t;
    const double ddB0 = 20.0 * pw3(u);
    const double ddB1 = -40.0 * pw3(u) + 60.0 * t * pw2(u);
    const double ddB2 = 20.0 * pw3(u) - 120.0 * t * pw2(u) + 60.0 * pw2(t) * u;
    const double ddB3 = 60.0 * t * pw2(u) - 120.0 * pw2(t) * u + 20.0 * pw3(t);
    const double ddB4 = 60.0 * pw2(t) * u - 40.0 * pw3(t);
    const double ddB5 = 20.0 * pw3(t);
    const double beta1 = q0 + Tqd0 / 5;
    const double beta2 = q0 + (2 * Tqd0) / 5 + TTqdd0 / 20;
    const double beta3 = q0 + k;
    return ddB0 * q0 + ddB1 * beta1 + ddB2 * beta2 + ddB3 * beta3 + ddB4 * beta3 + ddB5 * beta3;
}
// k-independent parts, KPR/Trajectory.cu:812-822
ARMOUR_HD double bez_q_indep(double q0, double a, double b, double s) {
    return q0 + a * s - 6 * a * pw3(s) + 8 * a * pw4(s) - 3 * a * pw5(s) + (b * pw2(s)) * 0.5 - (3 * b * pw3(s)) * 0.5 +
           (3 * b * pw4(s)) * 0.5 - (b * pw5(s)) * 0.5;
}
ARMOUR_HD double bez_qd_indep(double a, double b, double s, double D) {
    return (pw2(s - 1) * (2 * a + 4 * a * s + 2 * b * s - 30 * a * pw2(s) - 5 * b * pw2(s))) * 0.5 / D;
}
ARMOUR_HD double bez_qdd_indep(double a, double b, double s, double D) {
    return -(s - 1.0) * (b - (36 * a + 8 * b) * s + (60 * a + 10 * b) * pw2(s)) / (D * D);
}

// Horizon extrema of joint position (vel == false) or velocity (vel == true) for one joint, and the
// derivative of each extremum w.r.t. the normalised parameter k_i in [-1, 1].
// Restates BezierCurve::returnJointPositionExtremum[Gradient] / returnJointVelocityExtremum[Gradient]
// (KPR/Trajectory.cu:256-540).  At an interior stationary point the derivative is dq/dk = B(s*)
// (position) or B'(s*) (velocity) — the envelope-theorem value of the reference's generated total
// derivative (:601-810).  The reference's `1.0` for the s = 1 velocity candidate is kept as is.
ARMOUR_HD void bez_extrema(bool vel, double q0, double a, double b, double k_range, double D, double kn, double* mn,
                           double* mx, double* dmn, double* dmx) {
    const double k = k_range * kn;
    double s[4], v[4];
    s[0] = 0;
    s[3] = 1;
    if (!vel) {
        const double sq = sqrt(64 * pw2(a) + 14 * a * b - 120 * k * a + pw2(b));
        s[1] = (2 * a + b + sq) / (5 * (6 * a - 12 * k + b));
        s[2] = (2 * a + b - sq) / (5 * (6 * a - 12 * k + b));
        for (int i = 0; i < 4; i++) v[i] = bez_q(q0, a, b, k, s[i]);
    } else {
        const double sq = sqrt(6 * (150 * pw2(k) - 180 * k * a - 20 * k * b + 54 * pw2(a) + 14 * a * b + pw2(b)));
        s[1] = (18 * a - 30 * k + 4 * b + sq) / (10 * (6 * a - 12 * k + b));
        s[2] = (18 * a - 30 * k + 4 * b - sq) / (10 * (6 * a - 12 * k + b));
        for (int i = 0; i < 4; i++) v[i] = bez_qd(q0, a, b, k, s[i]);
    }
    double vmin, vmax;
    int imin, imax;
    if (v[0] < v[3]) {
        vmin = v[0]; imin = 0; vmax = v[3]; imax = 3;
    } else {
        vmin = v[3]; imin = 3; vmax = v[0]; imax = 0;
    }
    for (int c = 1; c <= 2; c++) {
        if (0 <= s[c] && s[c] <= 1) {
            if (v[c] < vmin) { vmin = v[c]; imin = c; }
            if (vmax < v[c]) { vmax = v[c]; imax = c; }
        }
    }
    double gr[4];
    gr[0] = 0.0;
    gr[3] = 1.0;
    for (int c = 1; c <= 2; c++) {
        const double x = s[c];
        gr[c] = !vel ? (10 * pw3(x) * pw2(x - 1) - 5 * pw4(x) * (x - 1) + pw5(x))
                     : ((pw3(x) * (x * 2.0 - 2.0) * 1.0E+1 + (x * x) * pw2(x - 1.0) * 3.0E+1) +
                        (pw3(x) * (x - 1.0) * -2.0E+1 - pw4(x) * 5.0) + pw4(x) * 5.0);
    }
    const double scale = vel ? 1.0 / D : 1.0;
    *mn = vel ? vmin / D : vmin;
    *mx = vel ? vmax / D : vmax;
    *dmn = vel ? gr[imin] * k_range / D : gr[imin] * k_range;
    *dmx = vel ? gr[imax] * k_range / D : gr[imax] * k_range;
    (void)scale;
}

}  // namespace armour
