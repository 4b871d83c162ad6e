// C ABI of the robust-controller path (include/armour_b200.h, "robust controller" section): the batched twin of the
// reference's MEX entry kinova_controller(Kr, alpha, V_max, r_norm_threshold, q, qd, q_des, qd_des, qdd_des)
// (MEX/kinova_controller.cpp) and of the two Newton-Euler passes under it (MEX/rnea.cpp).  The model file is the
// reference's own text format (MEX/kinova_without_gripper.txt, written by its URDF exporter); reading it and the
// conversion to Featherstone's CoM-to-CoM form (MEX/robot_models.cpp:20-156) is load-time host work in doubles, the
// interval model (:175-237) is made from it, everything per state runs in csrc/controller.cuh on the device.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include "../../include/armour_b200.h"
#include "controller.cuh"
#include "device_buffer.h"

using armour::DeviceBuffer;
using namespace armour::ctl;

struct armour_controller {
    int device = 0;
    Model host;                 // the model as uploaded (derived blocks filled on the device)
    DeviceBuffer<Model> d_model;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    DeviceBuffer<double> d_buf;  // staging of the host-pointer entry points
    std::vector<double> h_trig;
    std::string last_error;
    long long launches = 0;
};

namespace {

thread_local std::string g_create_error;

int cfail(armour_controller* c, int code, const std::string& msg) {
    if (c) c->last_error = msg; else g_create_error = msg;
    return code;
}
#define CCU(expr)                                                                                         \
    do {                                                                                                  \
        cudaError_t e__ = (expr);                                                                         \
        if (e__ != cudaSuccess)                                                                           \
            return cfail(ctl, ARMOUR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));     \
    } while (0)

// ---- host doubles: 3x3 algebra of the model conversion (products coefficient by coefficient, p0 + (p1 + p2)) ----
struct HM {
    double a[9];
};
struct HV {
    double x[3];
};
struct HX {
    HM R;
    HV p;
};
double s3(double p0, double p1, double p2) { return p0 + (p1 + p2); }
HM hmm(const HM& A, const HM& B) {
    HM r;
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) r.a[3 * i + j] = s3(A.a[3 * i] * B.a[j], A.a[3 * i + 1] * B.a[3 + j], A.a[3 * i + 2] * B.a[6 + j]);
    return r;
}
HM htr(const HM& A) {
    HM r;
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) r.a[3 * i + j] = A.a[3 * j + i];
    return r;
}
HV hmv(const HM& A, const HV& b) {
    HV r;
    for (int i = 0; i < 3; i++) r.x[i] = s3(A.a[3 * i] * b.x[0], A.a[3 * i + 1] * b.x[1], A.a[3 * i + 2] * b.x[2]);
    return r;
}
HM hscale(double s, const HM& A) {
    HM r;
    for (int i = 0; i < 9; i++) r.a[i] = s * A.a[i];
    return r;
}
HM hadd(const HM& A, const HM& B) {
    HM r;
    for (int i = 0; i < 9; i++) r.a[i] = A.a[i] + B.a[i];
    return r;
}
HM hsub(const HM& A, const HM& B) {
    HM r;
    for (int i = 0; i < 9; i++) r.a[i] = A.a[i] - B.a[i];
    return r;
}
HM hneg(const HM& A) { return hscale(-1.0, A); }
HM hhat(const HV& p) {
    HM r = {{0, -p.x[2], p.x[1], p.x[2], 0, -p.x[0], -p.x[1], p.x[0], 0}};
    return r;
}
HV hcross(const HV& a, const HV& b) {
    HV r = {{a.x[1] * b.x[2] - a.x[2] * b.x[1], a.x[2] * b.x[0] - a.x[0] * b.x[2], a.x[0] * b.x[1] - a.x[1] * b.x[0]}};
    return r;
}
HX hidentity() {
    HX X;
    std::memset(&X, 0, sizeof(X));
    X.R.a[0] = X.R.a[4] = X.R.a[8] = 1.0;
    return X;
}
HX hx_apply(const HX& X, const HX& x2) {  // Transform::apply(Transform), MEX/spatial.cpp:239-246
    HX r;
    r.R = hmm(X.R, x2.R);
    const HV t = hmv(htr(x2.R), X.p);
    for (int k = 0; k < 3; k++) r.p.x[k] = x2.p.x[k] + t.x[k];
    return r;
}
HX hx_inverse(const HX& X) {  // :248-253
    HX r;
    r.R = htr(X.R);
    r.p = hmv(hneg(X.R), X.p);
    return r;
}

struct FileModel {
    int nj = 0;
    std::vector<HV> Sw, Sv, com;
    std::vector<HX> X;
    std::vector<double> m, transI, friction, damping;
    std::vector<HM> Ibar, mch;
    std::vector<int> parent;
    double gravity[3] = {0, 0, 0};
};

// "<field> [index] <v0 v1 ...>" per line (MEX/robot_models.cpp:28-124)
bool parse_model(const std::string& path, FileModel& F, std::string& err) {
    std::ifstream in(path);
    if (!in.is_open()) {
        err = "cannot open robot model file " + path;
        return false;
    }
    std::string line;
    auto need = [&](size_t have, size_t want, const std::string& field) {
        if (have < want) {
            err = "robot model file: field '" + field + "' has " + std::to_string(have) + " values, needs " + std::to_string(want);
            return false;
        }
        return true;
    };
    while (std::getline(in, line)) {
        const size_t lt = line.find('<'), gt = line.find('>');
        if (lt == std::string::npos || gt == std::string::npos || gt < lt) continue;
        std::istringstream head(line.substr(0, lt));
        std::string field;
        int ind = -1;
        head >> field;
        head >> ind;
        std::istringstream body(line.substr(lt + 1, gt - lt - 1));
        std::vector<double> v;
        double x;
        while (body >> x) v.push_back(x);
        if (field == "numJoints") {
            if (!need(v.size(), 1, field)) return false;
            F.nj = int(v[0]);
            if (F.nj < 1 || F.nj > MAXJ) {
                err = "robot model file: numJoints must be 1.." + std::to_string(MAXJ);
                return false;
            }
            const size_t n = size_t(F.nj);
            F.Sw.assign(n, HV{{0, 0, 0}});
            F.Sv.assign(n, HV{{0, 0, 0}});
            F.com.assign(n, HV{{0, 0, 0}});
            F.X.assign(n, hidentity());
            F.m.assign(n, 0.0);
            F.transI.assign(n, 0.0);
            F.friction.assign(n, 0.0);
            F.damping.assign(n, 0.0);
            HM z;
            std::memset(&z, 0, sizeof(z));
            F.Ibar.assign(n, z);
            F.mch.assign(n, z);
            F.parent.assign(n, -1);
            continue;
        }
        if (F.nj == 0) {
            err = "robot model file: numJoints must come first";
            return false;
        }
        const bool indexed = field == "twist" || field == "inertia" || field == "Xtree" || field == "CoM";
        if (indexed && (ind < 0 || ind >= F.nj)) {
            err = "robot model file: index of '" + field + "' out of range";
            return false;
        }
        if (field == "twist") {
            if (!need(v.size(), 6, field)) return false;
            for (int k = 0; k < 3; k++) {
                F.Sw[ind].x[k] = v[k];
                F.Sv[ind].x[k] = v[3 + k];
            }
        } else if (field == "gravity") {
            if (!need(v.size(), 3, field)) return false;
            for (int k = 0; k < 3; k++) F.gravity[k] = v[k];
        } else if (field == "inertia") {
            if (!need(v.size(), 19, field)) return false;
            F.m[ind] = v[0];
            for (int k = 0; k < 9; k++) {
                F.Ibar[ind].a[k] = v[1 + k];
                F.mch[ind].a[k] = v[10 + k];
            }
        } else if (field == "Xtree") {
            if (!need(v.size(), 12, field)) return false;
            for (int k = 0; k < 9; k++) F.X[ind].R.a[k] = v[k];
            for (int k = 0; k < 3; k++) F.X[ind].p.x[k] = v[9 + k];
        } else if (field == "parent") {
            if (!need(v.size(), size_t(F.nj), field)) return false;
            for (int j = 0; j < F.nj; j++) F.parent[j] = int(v[j]);
        } else if (field == "CoM") {
            if (!need(v.size(), 3, field)) return false;
            for (int k = 0; k < 3; k++) F.com[ind].x[k] = v[k];
        } else if (field == "transI" || field == "friction" || field == "damping") {
            if (!need(v.size(), size_t(F.nj), field)) return false;
            std::vector<double>& dst = field == "transI" ? F.transI : (field == "friction" ? F.friction : F.damping);
            for (int j = 0; j < F.nj; j++) dst[j] = v[j];
        }  // torque_limits, joint_limits, gear_ratios: read by the reference, not used by it either
    }
    if (F.nj == 0) {
        err = "robot model file: no numJoints line";
        return false;
    }
    for (int j = 0; j < F.nj; j++)
        if (F.parent[j] < -1 || F.parent[j] >= j) {
            err = "robot model file: parent[j] must be -1 or a joint before j";
            return false;
        }
    return true;
}

// MEX/robot_models.cpp:126-156: joint frame -> Featherstone's CoM-to-CoM form; then the interval model with +-eps on the
// mass and on every entry of the inertia (:213-232)
void convert_model(const FileModel& F, double eps, Model& M) {
    std::memset(&M, 0, sizeof(M));
    M.nj = F.nj;
    M.chain = 1;
    for (int i = 0; i < F.nj; i++)
        if (F.parent[i] != i - 1) M.chain = 0;
    for (int k = 0; k < 3; k++) M.gravity[k] = F.gravity[k];
    const double lowP = 1 - eps, highP = 1 + eps;
    for (int i = 0; i < F.nj; i++) {
        M.parent[i] = F.parent[i];
        M.friction[i] = F.friction[i];
        M.damping[i] = F.damping[i];
        // twist from the joint frame to the world frame
        HX Xwj = F.X[i];
        for (int pind = F.parent[i]; pind > -1; pind = F.parent[pind]) Xwj = hx_apply(Xwj, F.X[pind]);
        const HV newW = hmv(htr(Xwj.R), F.Sw[i]);  // Transform::invapply(Twist), spatial.cpp:205-209
        const HV c = hcross(Xwj.p, newW);
        const HV rv = hmv(htr(Xwj.R), F.Sv[i]);
        HV newV;
        for (int k = 0; k < 3; k++) newV.x[k] = rv.x[k] + c.x[k];
        // inertia from the joint frame to the body CoM frame: CoM[i].apply(I[i]) with R = identity (spatial.cpp:221-237)
        HX C = hidentity();
        C.p = F.com[i];
        const HM p_hat = hhat(C.p);
        const HM mRp_hat = hmm(hscale(F.m[i], C.R), p_hat);
        const HM Rt = htr(C.R);
        const HM new_mch = hsub(hmm(hmm(C.R, F.mch[i]), Rt), hmm(hmm(hscale(F.m[i], C.R), p_hat), Rt));
        const HM new_Ibar = hmm(hsub(hmm(C.R, hadd(F.Ibar[i], hmm(hscale(2.0, F.mch[i]), p_hat))), hmm(mRp_hat, p_hat)), Rt);
        // Xtree from joint-to-joint to CoM-to-CoM
        HX prevCoM = hidentity();
        if (F.parent[i] != -1) prevCoM.p = F.com[F.parent[i]];
        HX nextCoM = hidentity();
        nextCoM.p = F.com[i];
        const HX newX = hx_apply(prevCoM, hx_apply(hx_inverse(F.X[i]), hx_inverse(nextCoM)));

        JointModel<double>& N = M.nom[i];
        JointModel<Itv>& I = M.iv[i];
        for (int k = 0; k < 3; k++) {
            N.S.w.x[k] = newW.x[k];
            N.S.v.x[k] = newV.x[k];
            N.X.p.x[k] = newX.p.x[k];
            I.S.w.x[k] = Itv{newW.x[k], newW.x[k]};
            I.S.v.x[k] = Itv{newV.x[k], newV.x[k]};
            I.X.p.x[k] = Itv{newX.p.x[k], newX.p.x[k]};
        }
        N.m = F.m[i];
        I.m = Itv{F.m[i] * lowP, F.m[i] * highP};
        N.transI = F.transI[i];
        I.transI = Itv{F.transI[i], F.transI[i]};
        for (int k = 0; k < 9; k++) {
            N.X.R.a[k] = newX.R.a[k];
            I.X.R.a[k] = Itv{newX.R.a[k], newX.R.a[k]};
            N.Ibar.a[k] = new_Ibar.a[k];
            N.mch.a[k] = new_mch.a[k];
            I.mch.a[k] = Itv{new_mch.a[k], new_mch.a[k]};
            const double val = new_Ibar.a[k];
            I.Ibar.a[k] = val >= 0 ? Itv{val * lowP, val * highP} : Itv{val * highP, val * lowP};
        }
    }
}

// sin(-q), cos(-q) with the host's libm, as the reference computes them (spatial_interval.cpp:150-151 with theta = -q);
// large batches are split over the host's threads (each value depends on its own angle only)
void host_trig(const double* q, size_t count, std::vector<double>& out) {
    out.resize(count * 2);
    double* o = out.data();
    auto run = [q, o](size_t i0, size_t i1) {
        for (size_t i = i0; i < i1; i++) {
            const double theta = -q[i];
            o[2 * i] = std::sin(theta);
            o[2 * i + 1] = std::cos(theta);
        }
    };
    const size_t min_chunk = 1 << 14;
    unsigned nt = std::thread::hardware_concurrency();
    if (nt > 16) nt = 16;
    if (nt < 2 || count < 2 * min_chunk) {
        run(0, count);
        return;
    }
    if (count / min_chunk < nt) nt = unsigned(count / min_chunk);
    std::vector<std::thread> pool;
    const size_t per = (count + nt - 1) / nt;
    for (unsigned t = 1; t < nt; t++) pool.emplace_back(run, std::min(count, t * per), std::min(count, (t + 1) * per));
    run(0, std::min(count, per));
    for (auto& th : pool) th.join();
}
int grid(int n) { return (n + CTL_THREADS - 1) / CTL_THREADS; }

}  // namespace

extern "C" {

const char* armour_controller_create_error(void) { return g_create_error.c_str(); }

int armour_controller_create(const char* model_file, double model_uncertainty, int device, armour_controller** out) {
    armour_controller* ctl = nullptr;
    if (!model_file || !out) return cfail(nullptr, ARMOUR_ERR_ARG, "null argument");
    if (!(model_uncertainty >= 0) || !(model_uncertainty < 1)) return cfail(nullptr, ARMOUR_ERR_ARG, "model_uncertainty must be in [0, 1)");
    FileModel F;
    std::string err;
    if (!parse_model(model_file, F, err)) return cfail(nullptr, ARMOUR_ERR_ARG, err);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1 || device < 0 || device >= ndev)
        return cfail(nullptr, ARMOUR_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    armour_controller* c = new armour_controller;
    c->device = device;
    convert_model(F, model_uncertainty, c->host);
    auto bail = [&](cudaError_t e, const char* what) {
        const std::string msg = std::string(what) + ": " + cudaGetErrorString(e);
        if (c->stream) cudaStreamDestroy(c->stream);
        delete c;
        return cfail(nullptr, ARMOUR_ERR_CUDA, msg);
    };
    cudaError_t e;
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(e, "cudaSetDevice");
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    if ((e = c->d_model.reserve(1)) != cudaSuccess) return bail(e, "cudaMalloc(model)");
    if ((e = cudaMemcpyAsync(c->d_model.get(), &c->host, sizeof(Model), cudaMemcpyHostToDevice, c->stream)) != cudaSuccess) return bail(e, "upload");
    k_model_setup<<<1, 32, 0, c->stream>>>(c->d_model.get());
    if ((e = cudaGetLastError()) != cudaSuccess) return bail(e, "k_model_setup");
    if ((e = cudaMemcpyAsync(&c->host, c->d_model.get(), sizeof(Model), cudaMemcpyDeviceToHost, c->stream)) != cudaSuccess) return bail(e, "download");
    if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return bail(e, "k_model_setup");
    c->launches = 1;
    (void)ctl;
    *out = c;
    return ARMOUR_OK;
}

void armour_controller_destroy(armour_controller* ctl) {
    if (!ctl) return;
    cudaSetDevice(ctl->device);
    if (ctl->stream && ctl->own_stream) cudaStreamDestroy(ctl->stream);
    delete ctl;  // frees the buffers
}

int armour_controller_num_joints(const armour_controller* ctl) { return ctl ? ctl->host.nj : ARMOUR_ERR_ARG; }
const char* armour_controller_last_error(const armour_controller* ctl) { return ctl ? ctl->last_error.c_str() : g_create_error.c_str(); }
long long armour_controller_kernel_launches(const armour_controller* ctl) { return ctl ? ctl->launches : 0; }
int armour_controller_set_stream(armour_controller* ctl, void* cuda_stream) {
    if (!ctl || !cuda_stream) return ARMOUR_ERR_ARG;
    cudaSetDevice(ctl->device);
    if (ctl->stream && ctl->own_stream) cudaStreamDestroy(ctl->stream);
    ctl->stream = static_cast<cudaStream_t>(cuda_stream);
    ctl->own_stream = false;
    return ARMOUR_OK;
}
int armour_controller_synchronize(armour_controller* ctl) {
    if (!ctl) return ARMOUR_ERR_ARG;
    CCU(cudaSetDevice(ctl->device));
    CCU(cudaStreamSynchronize(ctl->stream));
    return ARMOUR_OK;
}

// the interval model after conversion, in the layout of oracle's refctl_int_model (tests): per joint S.w[3] S.v[3] | X.R[9]
// X.p[3] | m | I_bar[9] | m_c_hat[9], each (lower, upper): 2 * 37 doubles per joint
int armour_controller_get_interval_model(const armour_controller* ctl, double* out) {
    if (!ctl || !out) return ARMOUR_ERR_ARG;
    int k = 0;
    auto put = [&](const Itv& x) {
        out[k++] = x.lo;
        out[k++] = x.hi;
    };
    for (int i = 0; i < ctl->host.nj; i++) {
        const JointModel<Itv>& J = ctl->host.iv[i];
        for (int a = 0; a < 3; a++) put(J.S.w.x[a]);
        for (int a = 0; a < 3; a++) put(J.S.v.x[a]);
        for (int a = 0; a < 9; a++) put(J.X.R.a[a]);
        for (int a = 0; a < 3; a++) put(J.X.p.x[a]);
        put(J.m);
        for (int a = 0; a < 9; a++) put(J.Ibar.a[a]);
        for (int a = 0; a < 9; a++) put(J.mch.a[a]);
    }
    return ARMOUR_OK;
}

int armour_controller_rnea_device(armour_controller* ctl, int n, const double* d_q, const double* d_qd, const double* d_qda,
                                  const double* d_qdd, const double* d_sincos, int apply_friction, int apply_gravity,
                                  double* d_tau, double* d_tau_lo, double* d_tau_hi) {
    if (!ctl || !d_q || !d_qd || !d_qda || !d_qdd) return ARMOUR_ERR_ARG;
    if (n < 1) return cfail(ctl, ARMOUR_ERR_ARG, "n must be positive");
    if (!d_tau && !(d_tau_lo && d_tau_hi)) return cfail(ctl, ARMOUR_ERR_ARG, "no output requested");
    if ((d_tau_lo == nullptr) != (d_tau_hi == nullptr)) return cfail(ctl, ARMOUR_ERR_ARG, "tau_lo and tau_hi go together");
    CCU(cudaSetDevice(ctl->device));
    TrigSrc trig{d_sincos};
    k_rnea<<<grid(n), CTL_THREADS, 0, ctl->stream>>>(ctl->d_model.get(), n, d_q, d_qd, d_qda, d_qdd, trig, apply_friction, apply_gravity,
                                                      d_tau, d_tau_lo, d_tau_hi);
    CCU(cudaGetLastError());
    ctl->launches++;
    return ARMOUR_OK;
}

int armour_controller_rnea(armour_controller* ctl, int n, const double* q, const double* qd, const double* qda, const double* qdd,
                           int apply_friction, int apply_gravity, double* tau, double* tau_lo, double* tau_hi) {
    if (!ctl || !q || !qd || !qda || !qdd) return ARMOUR_ERR_ARG;
    if (n < 1) return cfail(ctl, ARMOUR_ERR_ARG, "n must be positive");
    CCU(cudaSetDevice(ctl->device));
    const size_t N = size_t(n) * ctl->host.nj;
    CCU(ctl->d_buf.reserve(N * 9));
    double* d = ctl->d_buf.get();  // q qd qda qdd | sincos (2N) | tau lo hi
    host_trig(q, N, ctl->h_trig);
    cudaStream_t st = ctl->stream;
    CCU(cudaMemcpyAsync(d, q, N * sizeof(double), cudaMemcpyHostToDevice, st));
    CCU(cudaMemcpyAsync(d + N, qd, N * sizeof(double), cudaMemcpyHostToDevice, st));
    CCU(cudaMemcpyAsync(d + 2 * N, qda, N * sizeof(double), cudaMemcpyHostToDevice, st));
    CCU(cudaMemcpyAsync(d + 3 * N, qdd, N * sizeof(double), cudaMemcpyHostToDevice, st));
    CCU(cudaMemcpyAsync(d + 4 * N, ctl->h_trig.data(), 2 * N * sizeof(double), cudaMemcpyHostToDevice, st));
    const bool want_iv = tau_lo && tau_hi;
    int rc = armour_controller_rnea_device(ctl, n, d, d + N, d + 2 * N, d + 3 * N, d + 4 * N, apply_friction, apply_gravity,
                                           tau ? d + 6 * N : nullptr, want_iv ? d + 7 * N : nullptr, want_iv ? d + 8 * N : nullptr);
    if (rc) return rc;
    if (tau) CCU(cudaMemcpyAsync(tau, d + 6 * N, N * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (want_iv) {
        CCU(cudaMemcpyAsync(tau_lo, d + 7 * N, N * sizeof(double), cudaMemcpyDeviceToHost, st));
        CCU(cudaMemcpyAsync(tau_hi, d + 8 * N, N * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CCU(cudaStreamSynchronize(st));
    return ARMOUR_OK;
}

static int fill_gains(armour_controller* ctl, const armour_controller_gains* g, ControllerGains& G) {
    if (!g || !g->Kr) return cfail(ctl, ARMOUR_ERR_ARG, "gains");
    for (int i = 0; i < ctl->host.nj; i++) G.Kr[i] = g->Kr[i];
    G.alpha = g->alpha;
    G.V_max = g->V_max;
    G.r_norm_threshold = g->r_norm_threshold;
    G.friction = g->apply_friction;
    return ARMOUR_OK;
}

int armour_controller_update_device(armour_controller* ctl, int n, const armour_controller_gains* gains, const double* d_q,
                                    const double* d_qd, const double* d_q_des, const double* d_qd_des, const double* d_qdd_des,
                                    const double* d_sincos, double* d_u, double* d_u_nominal, double* d_v, int* d_status) {
    if (!ctl || !d_q || !d_qd || !d_q_des || !d_qd_des || !d_qdd_des || !d_u) return ARMOUR_ERR_ARG;
    if (n < 1) return cfail(ctl, ARMOUR_ERR_ARG, "n must be positive");
    ControllerGains G;
    int rc = fill_gains(ctl, gains, G);
    if (rc) return rc;
    CCU(cudaSetDevice(ctl->device));
    TrigSrc trig{d_sincos};
    k_controller_update<<<grid(n), CTL_THREADS, 0, ctl->stream>>>(ctl->d_model.get(), n, G, d_q, d_qd, d_q_des, d_qd_des, d_qdd_des, trig, d_u,
                                                                   d_u_nominal, d_v, d_status);
    CCU(cudaGetLastError());
    ctl->launches++;
    return ARMOUR_OK;
}

int armour_controller_update(armour_controller* ctl, int n, const armour_controller_gains* gains, const double* q, const double* qd,
                             const double* q_des, const double* qd_des, const double* qdd_des, double* u, double* u_nominal, double* v,
                             int* status) {
    if (!ctl || !q || !qd || !q_des || !qd_des || !qdd_des || !u) return ARMOUR_ERR_ARG;
    if (n < 1) return cfail(ctl, ARMOUR_ERR_ARG, "n must be positive");
    CCU(cudaSetDevice(ctl->device));
    const size_t N = size_t(n) * ctl->host.nj;
    CCU(ctl->d_buf.reserve(N * 10 + size_t(n)));
    double* d = ctl->d_buf.get();  // q qd q_des qd_des qdd_des | sincos (2N) | u u_nominal v | status (ints in n doubles)
    host_trig(q, N, ctl->h_trig);
    cudaStream_t st = ctl->stream;
    const double* src[5] = {q, qd, q_des, qd_des, qdd_des};
    for (int k = 0; k < 5; k++) CCU(cudaMemcpyAsync(d + k * N, src[k], N * sizeof(double), cudaMemcpyHostToDevice, st));
    CCU(cudaMemcpyAsync(d + 5 * N, ctl->h_trig.data(), 2 * N * sizeof(double), cudaMemcpyHostToDevice, st));
    int* d_status = reinterpret_cast<int*>(d + 10 * N);
    int rc = armour_controller_update_device(ctl, n, gains, d, d + N, d + 2 * N, d + 3 * N, d + 4 * N, d + 5 * N, d + 7 * N,
                                             d + 8 * N, d + 9 * N, d_status);
    if (rc) return rc;
    CCU(cudaMemcpyAsync(u, d + 7 * N, N * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (u_nominal) CCU(cudaMemcpyAsync(u_nominal, d + 8 * N, N * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (v) CCU(cudaMemcpyAsync(v, d + 9 * N, N * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (status) CCU(cudaMemcpyAsync(status, d_status, size_t(n) * sizeof(int), cudaMemcpyDeviceToHost, st));
    CCU(cudaStreamSynchronize(st));
    return ARMOUR_OK;
}

}  // extern "C"
