"""Host-side mirror of the reference's ARMTD comparison planner (kinova_planner_realtime_armtd_comparison: armtd_main.cu +
armtd_NLP) over the `armour_armtd_*` section of the C ABI: ArmtdPlanner has the same method names as the TNLP members the
reference's Ipopt run calls (one problem); ArmtdBatch runs many worlds in one context.  All compute is in libarmour_b200.so;
there is no CPU fallback."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import NF, ArmourError, Config, dp, ip

T = 100  # KPA/Parameters.h:17


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _dp(a):
    return a.ctypes.data_as(dp)


class ArmtdPlanner:
    def __init__(self, max_obstacles=40, simplify_threshold=5e-4, device=0):
        self.lib = _lib.load()
        cfg = Config()
        self.lib.armour_config_default(C.byref(cfg))
        cfg.max_obstacles = int(max_obstacles)
        cfg.simplify_threshold = float(simplify_threshold)
        cfg.device = int(device)
        h = C.c_void_p()
        rc = self.lib.armour_armtd_ctx_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise ArmourError(rc, self.lib.armour_status_string(rc).decode())
        self._h = h
        self.NJ = self.lib.armour_num_joints(h)
        self.m = 0

    def close(self):
        if getattr(self, "_h", None):
            self.lib.armour_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise ArmourError(rc, self.lib.armour_status_string(rc).decode() + ": " + self.lib.armour_last_error(self._h).decode())

    @property
    def kernel_launches(self):
        return int(self.lib.armour_kernel_launches(self._h))

    def build(self, q0, qd0, jrs, k_range, obstacles):
        """jrs: [6, 7, 100] = c_cos, g_cos, r_cos, c_sin, g_sin, r_sin (the arrays of KPA's input file)"""
        q0, qd0, jrs, k_range = _f64(q0), _f64(qd0), _f64(jrs), _f64(k_range)
        if jrs.shape != (6, NF, T):
            raise ValueError("jrs must be [6, 7, 100]")
        obs = _f64(obstacles).reshape(-1, 12)
        self._check(self.lib.armour_armtd_build(self._h, _dp(q0), _dp(qd0), _dp(jrs), _dp(k_range), _dp(obs), obs.shape[0]))
        self.m = self.lib.armour_armtd_num_constraints(self._h)
        return self

    def eval_g(self, k):
        k, g = _f64(k), np.empty(self.m)
        self._check(self.lib.armour_armtd_eval(self._h, _dp(k), _dp(g), None))
        return g

    def eval_jac_g(self, k):
        k, v = _f64(k), np.empty((self.m, NF))
        self._check(self.lib.armour_armtd_eval(self._h, _dp(k), None, _dp(v)))
        return v

    def eval(self, k):
        k, g, v = _f64(k), np.empty(self.m), np.empty((self.m, NF))
        self._check(self.lib.armour_armtd_eval(self._h, _dp(k), _dp(g), _dp(v)))
        return g, v

    def get_bounds_info(self):
        gl, gu = np.empty(self.m), np.empty(self.m)
        self._check(self.lib.armour_armtd_get_bounds(self._h, _dp(gl), _dp(gu)))
        return gl, gu

    def finalize_solution(self, g):
        g = _f64(g)
        ok, first = C.c_int(0), C.c_int(-1)
        self._check(self.lib.armour_armtd_verdict(self._h, _dp(g), C.byref(ok), C.byref(first)))
        return bool(ok.value), first.value

    def eval_f(self, q_des, k):
        q_des, k = _f64(q_des), _f64(k)
        f = C.c_double(0)
        self._check(self.lib.armour_armtd_cost(self._h, _dp(q_des), _dp(k), C.cast(C.byref(f), dp), None))
        return f.value

    def eval_grad_f(self, q_des, k):
        q_des, k, grad = _f64(q_des), _f64(k), np.empty(NF)
        self._check(self.lib.armour_armtd_cost(self._h, _dp(q_des), _dp(k), None, _dp(grad)))
        return grad

    def link_sliced_center(self):
        out = np.empty((T, self.NJ, 3))
        self._check(self.lib.armour_armtd_get_link_sliced_center(self._h, _dp(out)))
        return out

    def link_independent_generators(self):
        out = np.empty((T, self.NJ, 18))
        self._check(self.lib.armour_armtd_get_link_independent_generators(self._h, _dp(out)))
        return out


def _ip(a):
    return a.ctypes.data_as(ip)


class ArmtdBatch:
    """A batch of ARMTD comparison-planner problems (worlds) in one context, over the `armour_armtd_batch_*` calls: build,
    evaluation, verdict, cost and the batched device solver for every problem at once.  Arrays are problem-major: q0, qd0,
    k_range, k, q_des [n, 7]; jrs [n, 6, 7, 100]; obstacles [n, O, 12]; g [n, m]; J [n, m, 7]."""

    def __init__(self, max_problems, max_obstacles=40, simplify_threshold=5e-4, device=0, cap_link_monomials=None):
        self.lib = _lib.load()
        cfg = Config()
        self.lib.armour_config_default(C.byref(cfg))
        cfg.max_problems = int(max_problems)
        cfg.max_obstacles = int(max_obstacles)
        cfg.simplify_threshold = float(simplify_threshold)
        cfg.device = int(device)
        if cap_link_monomials is not None:
            cfg.cap_link_monomials = int(cap_link_monomials)
        h = C.c_void_p()
        rc = self.lib.armour_armtd_batch_ctx_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise ArmourError(rc, self.lib.armour_status_string(rc).decode())
        self._h = h
        self.device = int(device)
        self.NJ = self.lib.armour_num_joints(h)
        self.nprob, self.nobs, self.m = 0, 0, 0

    def close(self):
        if getattr(self, "_h", None):
            self.lib.armour_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise ArmourError(rc, self.lib.armour_status_string(rc).decode() + ": " + self.lib.armour_last_error(self._h).decode())

    @property
    def kernel_launches(self):
        return int(self.lib.armour_kernel_launches(self._h))

    def _built(self, nprob, nobs):
        self.nprob, self.nobs = int(nprob), int(nobs)
        self.m = self.NJ * T * self.nobs + 4 * NF

    def build(self, q0, qd0, jrs, k_range, obstacles):
        """Host-pointer build of n problems.  A capacity failure of some problems raises ArmourError (ARMOUR_ERR_CAPACITY)
        after the build: build_status() names them and their rows are fail-safe."""
        q0, qd0, k_range = (_f64(a).reshape(-1, NF) for a in (q0, qd0, k_range))
        n = q0.shape[0]
        jrs = _f64(jrs)
        if jrs.shape != (n, 6, NF, T):
            raise ValueError(f"jrs must be [{n}, 6, 7, 100], got {list(jrs.shape)}")
        if qd0.shape[0] != n or k_range.shape[0] != n:
            raise ValueError("q0, qd0 and k_range must have one row per problem")
        obs = _f64(obstacles)
        obs = obs.reshape(n, -1, 12) if obs.size else np.zeros((n, 0, 12))
        rc = self.lib.armour_armtd_batch_build(self._h, n, _dp(q0), _dp(qd0), _dp(jrs), _dp(k_range), _dp(obs), obs.shape[1])
        if rc in (0, _lib.ERR_CAPACITY):
            self._built(n, obs.shape[1])
        self._check(rc)
        return self

    def offline_jrs(self, qd0, k_range):
        """The offline table the episodes build from (armour_armtd_offline_jrs): this repository's synthetic stand-in for the
        reference's CORA tables, computed on the device; worlds.armtd_offline_jrs_batch restated to a few ulp.  qd0, k_range
        [n, 7] -> [n, 6, 7, 100]."""
        qd0, k_range = _f64(qd0).reshape(-1, NF), _f64(k_range).reshape(-1, NF)
        if qd0.shape != k_range.shape:
            raise ValueError("qd0 and k_range must have one row per problem")
        out = np.empty((qd0.shape[0], 6, NF, T))
        self._check(self.lib.armour_armtd_offline_jrs(self._h, qd0.shape[0], _dp(qd0), _dp(k_range), _dp(out)))
        return out

    def offline_jrs_device(self, n, d_qd0, d_k_range, d_jrs):
        """Asynchronous armour_armtd_offline_jrs_device on device pointers (ints)."""
        self._check(self.lib.armour_armtd_offline_jrs_device(self._h, n, d_qd0, d_k_range, d_jrs))

    def build_device(self, nprob, nobs, d_q0, d_qd0, d_jrs, d_k_range, d_obstacles, d_sincos=None):
        """Asynchronous build from device pointers (ints, e.g. torch.Tensor.data_ptr()); d_sincos [n, 7, 2] = cos q0, sin q0,
        or None for the device's sincos."""
        self._check(self.lib.armour_armtd_batch_build_device(self._h, nprob, d_q0, d_qd0, d_jrs, d_k_range, d_obstacles or None,
                                                             nobs, d_sincos or None))
        self._built(nprob, nobs)

    def synchronize(self):
        self._check(self.lib.armour_ctx_synchronize(self._h))

    def build_status(self):
        out = np.zeros(self.nprob, np.int32)
        self._check(self.lib.armour_batch_get_build_status(self._h, self.nprob, _ip(out)))
        return out

    def monomial_counts(self):
        """link_n [n, 104, NJ]: stored k-only monomials of every link reach set (the context's 104 intervals)."""
        ln = np.zeros((self.nprob, self.lib.armour_num_time_steps(self._h), self.NJ), np.int32)
        self._check(self.lib.armour_batch_get_monomial_counts(self._h, self.nprob, _ip(ln), None))
        return ln

    def eval(self, k, want_g=True, want_jac=True):
        k = _f64(k).reshape(-1, NF)
        n = k.shape[0]
        g = np.empty((n, self.m)) if want_g else None
        jac = np.empty((n, self.m, NF)) if want_jac else None
        self._check(self.lib.armour_armtd_batch_eval(self._h, n, _dp(k), _dp(g) if want_g else None,
                                                     _dp(jac) if want_jac else None))
        return g, jac

    def eval_device(self, nprob, d_k, d_g, d_jac):
        """Asynchronous evaluation on device pointers (ints; 0/None to skip an output)."""
        self._check(self.lib.armour_armtd_batch_eval_device(self._h, nprob, d_k, d_g or None, d_jac or None))

    def verdict_device(self, nprob, d_g, d_feasible, d_first):
        self._check(self.lib.armour_armtd_batch_verdict_device(self._h, nprob, d_g, d_feasible, d_first))

    def finalize_solution(self, g):
        """KPA's finalize_solution predicate for every row of g [n, m], on the device: (feasible [n] bool, first [n])."""
        import torch

        dev = torch.device("cuda", self.device)
        dg = torch.as_tensor(_f64(g).reshape(-1, self.m), device=dev)
        n = dg.shape[0]
        out = torch.empty((2, n), dtype=torch.int32, device=dev)
        torch.cuda.synchronize(dev)
        self.verdict_device(n, dg.data_ptr(), out[0].data_ptr(), out[1].data_ptr())
        self.synchronize()
        out = out.cpu().numpy()
        return out[0].astype(bool), out[1]

    def cost(self, q_des, k):
        """eval_f / eval_grad_f of every problem: (obj [n], grad [n, 7])."""
        q_des, k = _f64(q_des).reshape(-1, NF), _f64(k).reshape(-1, NF)
        n = k.shape[0]
        obj, grad = np.empty(n), np.empty((n, NF))
        self._check(self.lib.armour_armtd_batch_cost(self._h, n, _dp(q_des), _dp(k), _dp(obj), _dp(grad)))
        return obj, grad

    def link_independent_generators(self):
        """[n, 100, NJ, 18], column-major 3x6 per link and interval"""
        out = np.empty((self.nprob, T, self.NJ, 18))
        self._check(self.lib.armour_armtd_batch_get_link_independent_generators(self._h, self.nprob, _dp(out)))
        return out

    def solve(self, q_des, max_iter=None, tol=1e-7, qp_sweeps=None, collision_tol=None):
        """Batched planning on the device (armour_armtd_batch_solve) from k = 0 for every built problem: KPA's NLP, KPA's
        tolerance.  Returns (k_opt [n, 7], feasible [n] bool, first violated row [n], iterations [n])."""
        q_des = _f64(q_des).reshape(self.nprob, NF)
        opt = _lib.SolverOptions()
        self.lib.armour_solver_options_default(C.byref(opt))
        opt.tol = float(tol)
        if max_iter is not None:
            opt.max_iter = int(max_iter)
        if qp_sweeps is not None:
            opt.qp_sweeps = int(qp_sweeps)
        if collision_tol is not None:
            opt.collision_tol = float(collision_tol)
        k = np.empty((self.nprob, NF))
        ok, first, iters = (np.zeros(self.nprob, np.int32) for _ in range(3))
        self._check(self.lib.armour_armtd_batch_solve(self._h, self.nprob, _dp(q_des), C.byref(opt), _dp(k), _ip(ok), _ip(first),
                                                      _ip(iters)))
        return k, ok.astype(bool), first, iters

    def rollout(self, start, goal, obstacles, max_replans=100, goal_radius=0.05, lookahead=0.1, audit_samples=16, max_iter=None,
                tol=1e-7, collision_tol=None, qp_sweeps=None):
        """Closed-loop episodes of this planner for a batch of worlds on the device (armour_armtd_batch_rollout; semantics in
        include/armour_b200.h): the same worlds, options, audit and returned dict as ReachSetEngine.rollout, KPA's tolerance by
        default.  The context's reach sets afterwards are those of the last replan's sub-batch: build again before evaluating."""
        from .planner import run_rollout
        res = run_rollout(self, self.lib.armour_armtd_batch_rollout, start, goal, obstacles, max_replans, goal_radius, lookahead,
                          audit_samples, dict(max_iter=max_iter, tol=tol, collision_tol=collision_tol, qp_sweeps=qp_sweeps))
        self.nprob, self.nobs, self.m = 0, 0, 0
        return res
