"""Host-side Python mirror of the reference planner's interface for the hot path.

`ReachSetEngine` wraps one C-ABI context (one CUDA device, one stream).  Its methods carry the names
of the reference calls they stand in for (reference KPR/armour_main.cu and KPR/NLPclass.{h,cu}):
build -> sections II.A-II.D of main(); eval_g / eval_jac_g / get_bounds_info / finalize_solution ->
the armtd_NLP members.  All arithmetic happens in the CUDA library; numpy / torch only carry buffers.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import NF, ArmourError


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _dp(a):
    return a.ctypes.data_as(_lib.dp)


def run_rollout(owner, fn, start, goal, obstacles, max_replans, goal_radius, lookahead, audit_samples, solver):
    """One call of an episode entry point with host pointers (armour_batch_rollout or armour_armtd_batch_rollout: the same
    arguments) for owner's context; solver: solver option name -> value, None keeps the default.  Returns the dict of
    ReachSetEngine.rollout."""
    start, goal = _f64(start).reshape(-1, NF), _f64(goal).reshape(-1, NF)
    n = start.shape[0]
    obs = _f64(obstacles)
    obs = obs.reshape(n, -1, 12) if obs.size else np.zeros((n, 0, 12))
    opt = _lib.RolloutOptions()
    owner.lib.armour_rollout_options_default(C.byref(opt))
    opt.max_replans, opt.goal_radius, opt.lookahead = int(max_replans), float(goal_radius), float(lookahead)
    opt.audit_samples = int(audit_samples)
    for name, v in solver.items():
        if v is not None:
            setattr(opt.solver, name, type(getattr(opt.solver, name))(v))
    R = opt.max_replans
    res = dict(outcome=np.zeros(n, np.int32), replans=np.zeros(n, np.int32), infeasible=np.zeros(n, np.int32),
               final_state=np.zeros((n, 3 * NF)), min_clearance=np.zeros(n), log_state=np.zeros((max(R, 0), n, 3 * NF)),
               log_q_des=np.zeros((max(R, 0), n, NF)), log_k=np.zeros((max(R, 0), n, NF)),
               log_int=np.zeros((max(R, 0), n, 4), np.int32), log_clearance=np.zeros((max(R, 0), n)))
    out = _lib.RolloutOut()
    for name, a in res.items():
        setattr(out, name, a.ctypes.data_as(_lib.ip if a.dtype == np.int32 else _lib.dp))
    owner._check(fn(owner._h, n, _dp(start), _dp(goal), _dp(obs), obs.shape[1], C.byref(opt), C.byref(out)))
    return res


class ReachSetEngine:
    def __init__(self, max_problems=1, max_obstacles=40, device=0, robot_model=0, num_time_steps=128,
                 simplify_threshold=5e-4, k_range=None, cap_link=32, cap_torque=64, cap_work=768,
                 mass_uncertainty=-1.0, inertia_uncertainty=-1.0):
        self.lib = _lib.load()
        cfg = _lib.Config()
        self.lib.armour_config_default(C.byref(cfg))
        cfg.device = device
        cfg.robot_model = robot_model
        cfg.num_time_steps = num_time_steps
        cfg.max_obstacles = max_obstacles
        cfg.max_problems = max_problems
        cfg.cap_link_monomials = cap_link
        cfg.cap_torque_monomials = cap_torque
        cfg.cap_work_monomials = cap_work
        cfg.simplify_threshold = simplify_threshold
        if k_range is not None:
            for i in range(NF):
                cfg.k_range[i] = float(k_range[i])
        cfg.mass_uncertainty = mass_uncertainty
        cfg.inertia_uncertainty = inertia_uncertainty
        self.cfg = cfg
        self._h = C.c_void_p()
        rc = self.lib.armour_ctx_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            self._h = None
            raise ArmourError(rc, "armour_ctx_create failed (" + self.lib.armour_status_string(rc).decode() +
                              "); a CUDA device is required, there is no CPU fallback")
        self.T = self.lib.armour_num_time_steps(self._h)
        self.NJ = self.lib.armour_num_joints(self._h)
        self.nobs = 0
        self.nprob = 0

    # -- plumbing ------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.armour_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise ArmourError(rc, self.lib.armour_status_string(rc).decode() + ": " +
                              self.lib.armour_last_error(self._h).decode())

    def set_stream(self, cuda_stream_handle):
        self._check(self.lib.armour_ctx_set_stream(self._h, C.c_void_p(cuda_stream_handle)))

    def synchronize(self):
        self._check(self.lib.armour_ctx_synchronize(self._h))

    @property
    def kernel_launches(self):
        return int(self.lib.armour_kernel_launches(self._h))

    @property
    def m(self):
        return self.lib.armour_num_constraints(self._h, self.nobs)

    # -- reach sets (armour_main.cu:86-216) ----------------------------------------------------------
    def build(self, q0, qd0, qdd0, obstacles):
        """Batched build.  q0/qd0/qdd0: [nprob, 7] (or [7]); obstacles: [nprob, nobs, 12] (or [nobs, 12])."""
        q0, qd0, qdd0 = _f64(q0).reshape(-1, NF), _f64(qd0).reshape(-1, NF), _f64(qdd0).reshape(-1, NF)
        nprob = q0.shape[0]
        obs = _f64(obstacles)
        obs = obs.reshape(nprob, -1, 12) if obs.size else np.zeros((nprob, 0, 12))
        nobs = obs.shape[1]
        self._check(self.lib.armour_batch_reachsets_build(self._h, nprob, _dp(q0), _dp(qd0), _dp(qdd0), _dp(obs), nobs))
        self.nprob, self.nobs = nprob, nobs
        return self

    def build_device(self, nprob, nobs, d_q0, d_qd0, d_qdd0, d_obstacles):
        """Asynchronous build from device pointers (ints, e.g. torch.Tensor.data_ptr())."""
        self._check(self.lib.armour_batch_reachsets_build_device(self._h, nprob, d_q0, d_qd0, d_qdd0, d_obstacles, nobs))
        self.nprob, self.nobs = nprob, nobs

    def build_status(self):
        out = np.zeros(self.nprob, np.int32)
        self._check(self.lib.armour_batch_get_build_status(self._h, self.nprob, out.ctypes.data_as(_lib.ip)))
        return out

    def monomial_counts(self):
        """(link_n [nprob, T, NJ], u_n [nprob, T, 7]) stored k-only monomial counts of the built reach sets."""
        ln = np.zeros((self.nprob, self.T, self.NJ), np.int32)
        un = np.zeros((self.nprob, self.T, NF), np.int32)
        self._check(self.lib.armour_batch_get_monomial_counts(self._h, self.nprob, ln.ctypes.data_as(_lib.ip),
                                                              un.ctypes.data_as(_lib.ip)))
        return ln, un

    def candidate_counts(self):
        """Stored collision half-space candidates per row, uint8 [nprob, T/C, NJ, C, O] with C intervals per kernel
        chunk (255: evaluated from the generators)."""
        C_ = self.lib.armour_chunk_intervals()
        out = np.zeros((self.nprob, self.T // C_, self.NJ, C_, max(self.nobs, 0)), np.uint8)
        if out.size:
            self._check(self.lib.armour_batch_get_candidate_counts(self._h, self.nprob, out.ctypes.data_as(C.c_void_p)))
        return out

    def eval_image_layout(self):
        """Byte offsets inside one chunk's evaluation image at the current obstacle count, and its size ("chunk").
        Layout in DESIGN.md."""
        lay = (C.c_longlong * 10)()
        self._check(self.lib.armour_eval_image_layout(self._h, lay))
        names = ("chunk", "link_tables", "torque_tables", "link_c", "link_r", "u_c", "u_r", "groups", "counts", "records")
        return dict(zip(names, (int(v) for v in lay)))

    def eval_images(self):
        """Evaluation images of the built problems: (uint8 [nprob, T/C, bytes per chunk], eval_image_layout()).  An
        inspection aid for tests and tools."""
        layout = self.eval_image_layout()
        C_ = self.lib.armour_chunk_intervals()
        out = np.zeros((self.nprob, self.T // C_, layout["chunk"]), np.uint8)
        self._check(self.lib.armour_batch_get_eval_images(self._h, self.nprob, out.ctypes.data_as(C.c_void_p)))
        return out, layout

    def solve(self, q_des, max_iter=None, tol=None, qp_sweeps=None, qp_update_budget=None):
        """Batched planning on the device (armour_batch_solve): the trust-region SQP of the C++ host solver run on the
        GPU for every built problem, from k = 0.  Returns (k_opt [nprob, 7], feasible [nprob] bool, first violated row
        [nprob], iterations [nprob])."""
        q_des = np.ascontiguousarray(np.asarray(q_des, dtype=np.float64).reshape(self.nprob, NF))
        opt = _lib.SolverOptions()
        self.lib.armour_solver_options_default(C.byref(opt))
        if max_iter is not None:
            opt.max_iter = int(max_iter)
        if tol is not None:
            opt.tol = float(tol)
        if qp_sweeps is not None:
            opt.qp_sweeps = int(qp_sweeps)
        if qp_update_budget is not None:
            opt.qp_update_budget = int(qp_update_budget)
        k = np.empty((self.nprob, NF))
        ok = np.zeros(self.nprob, np.int32)
        first = np.zeros(self.nprob, np.int32)
        iters = np.zeros(self.nprob, np.int32)
        self._check(self.lib.armour_batch_solve(self._h, self.nprob, _dp(q_des), C.byref(opt), _dp(k),
                                                ok.ctypes.data_as(_lib.ip), first.ctypes.data_as(_lib.ip),
                                                iters.ctypes.data_as(_lib.ip)))
        return k, ok.astype(bool), first, iters

    # -- closed-loop episodes (kinova_run_100_worlds.m -> simulator_armtd.run) ------------------------------------------
    def rollout(self, start, goal, obstacles, max_replans=100, goal_radius=0.05, lookahead=0.1, audit_samples=16,
                max_iter=None, tol=None, torque_tol=None, collision_tol=None, qp_sweeps=None):
        """Closed-loop replanning episodes of a batch of worlds on the device (armour_batch_rollout; semantics in
        include/armour_b200.h).  start, goal: [n, 7]; obstacles: [n, nobs, 12].  Returns a dict of numpy arrays: outcome,
        replans, infeasible [n], final_state [n, 21], min_clearance [n], log_state [R, n, 21], log_q_des, log_k [R, n, 7],
        log_int [R, n, 4] (feasible, first violated row, iterations, build status), log_clearance [R, n].  The context's
        reach sets afterwards are those of the last replan's sub-batch: build again before evaluating."""
        res = run_rollout(self, self.lib.armour_batch_rollout, start, goal, obstacles, max_replans, goal_radius, lookahead,
                          audit_samples, dict(max_iter=max_iter, tol=tol, torque_tol=torque_tol, collision_tol=collision_tol,
                                              qp_sweeps=qp_sweeps))
        self.nprob = 0
        return res

    def clearance(self, q, obstacles, world=None):
        """Exact signed clearance of arm configurations q [n, 7] (armour_batch_clearance): link boxes of this context's
        robot model against obstacle set world[i] of obstacles [nsets, nobs, 12] (or [nobs, 12]; world None: set 0) by the
        separating-axis test.  Returns (clearance [n], which [n] = l * nobs + o of the closest pair)."""
        q = _f64(q).reshape(-1, NF)
        n = q.shape[0]
        obs = _f64(obstacles)
        nobs = obs.shape[-2] if obs.size else 0
        obs = obs.reshape(-1, nobs, 12) if obs.size else np.zeros((1, 0, 12))
        w = None if world is None else np.ascontiguousarray(np.asarray(world, dtype=np.int32).reshape(n))
        if w is not None and (w.min() < 0 or w.max() >= obs.shape[0]):
            raise ValueError("world index outside the obstacle sets")
        clr = np.empty(n)
        which = np.empty(n, np.int32)
        self._check(self.lib.armour_batch_clearance(self._h, n, _dp(q), w.ctypes.data_as(_lib.ip) if w is not None else None,
                                                    _dp(obs), nobs, _dp(clr), which.ctypes.data_as(_lib.ip)))
        return clr, which

    def measure_fp64_peak(self):
        """Sustained non-tensor FP64 rate of the device in TFLOP/s (FMA probe kernel in the library)."""
        v = C.c_double(0)
        self._check(self.lib.armour_measure_fp64_peak(self._h, C.byref(v)))
        return v.value

    def torque_radius(self):
        out = np.empty((self.nprob, NF, self.T))
        self._check(self.lib.armour_batch_get_torque_radius(self._h, self.nprob, _dp(out)))
        return out

    def link_independent_generators(self):
        """[nprob, T, NJ, 3, 6]"""
        out = np.empty((self.nprob, self.T, self.NJ, 6, 3))
        self._check(self.lib.armour_batch_get_link_independent_generators(self._h, self.nprob, _dp(out)))
        return out.transpose(0, 1, 2, 4, 3)

    # -- NLP callbacks (NLPclass.cu) -----------------------------------------------------------------
    def get_bounds_info(self):
        gl, gu = np.empty((self.nprob, self.m)), np.empty((self.nprob, self.m))
        self._check(self.lib.armour_batch_get_bounds(self._h, self.nprob, _dp(gl), _dp(gu)))
        return gl, gu

    def eval(self, k, want_g=True, want_jac=True):
        """One eval_g + eval_jac_g per problem with host buffers.  k: [nprob, 7]."""
        k = _f64(k).reshape(-1, NF)
        n = k.shape[0]
        g = np.empty((n, self.m)) if want_g else None
        jac = np.empty((n, self.m, NF)) if want_jac else None
        self._check(self.lib.armour_batch_eval(self._h, n, _dp(k), _dp(g) if want_g else None,
                                               _dp(jac) if want_jac else None))
        return g, jac

    def eval_g(self, k):
        return self.eval(k, True, False)[0]

    def eval_jac_g(self, k):
        return self.eval(k, False, True)[1]

    def eval_into(self, k, g, jac):
        """Host-buffer evaluation into caller-owned (ideally pinned) numpy arrays."""
        n = k.shape[0]
        self._check(self.lib.armour_batch_eval(self._h, n, _dp(k), _dp(g) if g is not None else None,
                                               _dp(jac) if jac is not None else None))

    # -- structured Jacobian (offered beside the dense one) --------------------------------------------
    @property
    def jacobian_nnz(self):
        return int(self.lib.armour_jacobian_nnz(self._h, self.nobs))

    def jacobian_structure(self):
        """(iRow, jCol) of the non-zeros, C-style indices, in the order eval_structured returns the values."""
        n = self.jacobian_nnz
        ir, jc = np.zeros(n, np.int32), np.zeros(n, np.int32)
        self._check(self.lib.armour_jacobian_structure(self._h, self.nobs, ir.ctypes.data_as(_lib.ip), jc.ctypes.data_as(_lib.ip)))
        return ir, jc

    def eval_structured(self, k, want_g=True):
        """eval_g + the non-zeros of the Jacobian per problem with host buffers: (g [n, m] or None, values [n, nnz])."""
        k = _f64(k).reshape(-1, NF)
        n = k.shape[0]
        g = np.empty((n, self.m)) if want_g else None
        vals = np.empty((n, self.jacobian_nnz))
        self._check(self.lib.armour_batch_eval_structured(self._h, n, _dp(k), _dp(g) if want_g else None, _dp(vals)))
        return g, vals

    def eval_structured_into(self, k, g, vals):
        self._check(self.lib.armour_batch_eval_structured(self._h, k.shape[0], _dp(k), _dp(g) if g is not None else None, _dp(vals)))

    def eval_device(self, nprob, d_k, d_g, d_jac):
        """Asynchronous evaluation on device pointers (ints; 0/None to skip an output)."""
        self._check(self.lib.armour_batch_eval_device(self._h, nprob, d_k, d_g or None, d_jac or None))

    def verdict_device(self, nprob, d_g, d_feasible, d_first):
        self._check(self.lib.armour_batch_verdict_device(self._h, nprob, d_g, d_feasible, d_first))

    def finalize_solution(self, g):
        """Feasibility verdict of problem 0 for a host g (NLPclass.cu:449-537): (feasible, first_violated_row)."""
        g = _f64(g)
        ok, first = C.c_int(0), C.c_int(-1)
        self._check(self.lib.armour_verdict(self._h, _dp(g), C.byref(ok), C.byref(first)))
        return bool(ok.value), first.value

    def cost(self, q_des, k):
        q_des, k = _f64(q_des), _f64(k)
        obj, grad = C.c_double(0), np.empty(NF)
        self._check(self.lib.armour_cost(self._h, _dp(q_des), _dp(k), C.byref(obj), _dp(grad)))
        return obj.value, grad

    def link_sliced_center(self):
        out = np.empty((self.T, self.NJ, 3))
        self._check(self.lib.armour_get_link_sliced_center(self._h, _dp(out)))
        return out

    # -- reach-set tables ----------------------------------------------------------------------------
    def _tables(self, r):
        t = _lib.ReachsetTables()
        t.cap_link, t.cap_u = r["hl"].shape[1], r["hu"].shape[1]
        t.link_n = r["nl"].ctypes.data_as(_lib.ip)
        t.link_center = _dp(r["cl"])
        t.link_key = r["hl"].ctypes.data_as(_lib.up)
        t.link_coeff = _dp(r["gl"])
        t.u_n = r["nu"].ctypes.data_as(_lib.ip)
        t.u_center = _dp(r["cu"])
        t.u_key = r["hu"].ctypes.data_as(_lib.up)
        t.u_coeff = _dp(r["gu"])
        t.u_radius = _dp(r["ru"])
        t.torque_radius = _dp(r["torque_radius"])
        t.link_gens = _dp(r["link_gens"])
        return t

    def import_reachsets(self, prob, nprob_total, tables, q0, qd0, qdd0, obstacles):
        """Upload externally built k-only tables (dict in the neutral layout of the C ABI)."""
        obs = _f64(obstacles).reshape(-1, 12)
        q0, qd0, qdd0 = _f64(q0), _f64(qd0), _f64(qdd0)
        t = self._tables(tables)
        self._check(self.lib.armour_import_reachsets(self._h, prob, nprob_total, C.byref(t), _dp(q0), _dp(qd0),
                                                     _dp(qdd0), _dp(obs), obs.shape[0]))
        self.nobs = obs.shape[0]
        if prob == nprob_total - 1:
            self.nprob = nprob_total

    def export_reachsets(self, prob=0):
        T, NJ = self.T, self.NJ
        cl, cu = self.cfg.cap_link_monomials, self.cfg.cap_torque_monomials
        r = dict(nl=np.zeros(T * NJ, np.int32), cl=np.zeros((T * NJ, 3)), hl=np.zeros((T * NJ, cl), np.uint64),
                 gl=np.zeros((T * NJ, cl, 3)), nu=np.zeros(T * NF, np.int32), cu=np.zeros(T * NF),
                 hu=np.zeros((T * NF, cu), np.uint64), gu=np.zeros((T * NF, cu)), ru=np.zeros(T * NF),
                 torque_radius=np.zeros((NF, T)), link_gens=np.zeros((T, NJ, 18)))
        t = self._tables(r)
        self._check(self.lib.armour_export_reachsets(self._h, prob, C.byref(t)))
        return r
