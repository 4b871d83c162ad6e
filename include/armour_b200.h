/* armour_b200.h — C ABI of the B200-native ARMOUR reach-set / constraint-evaluation hot path.
 *
 * The reference planner (roahmlab/armour, kinova_planner_realtime = "KPR/") has no library ABI: its
 * boundaries are the Ipopt TNLP virtual interface implemented by armtd_NLP (KPR/NLPclass.h:11-184)
 * and the armour.in / armour*.out text files (KPR/armour_main.cu:36-78,312-372).  This header is the
 * thin C layer a maintainer binds instead of the bodies of those functions; every entry point names
 * the reference code it replaces.  Conventions:
 *   - plain pointers and sizes only; every function returns ARMOUR_OK (0) or a negative error code and
 *     never throws across the ABI (the reference throws int / aborts: KPR/CollisionChecking.cu:10-13);
 *   - the caller owns all host buffers; the context owns all device memory;
 *   - one context = one CUDA device + one stream; thread-compatible, not thread-safe (Ipopt calls
 *     eval_g / eval_jac_g serially from one thread);
 *   - there is NO CPU fallback: without a CUDA device armour_ctx_create fails with ARMOUR_ERR_CUDA;
 *   - several contexts may live on one device.  Contexts of identical configuration run side by side; switching
 *     between contexts whose configuration differs drains the device first (their constants share one block);
 *   - a problem whose build returned / recorded ARMOUR_ERR_CAPACITY has no valid reach sets: every evaluation of it
 *     returns fail-safe rows (torque and collision rows 1e300, zero Jacobian), so its verdict is always infeasible.
 *
 * Index conventions (T = num_time_steps = 128, NJ = links, NF = 7, O = obstacles of the problem):
 *   constraint rows m = NF*T + NJ*T*O + 4*NF            (KPR/NLPclass.cu:45-57)
 *     [0, NF*T)                     torque centre, row t*NF + j
 *     [NF*T, NF*T + NJ*T*O)         collision value, row NF*T + (l*T + t)*O + o   (link-major)
 *     next NF / NF                  min / max joint position over the horizon
 *     next NF / NF                  min / max joint velocity
 *   Jacobian: dense, values[row*NF + col]                (KPR/NLPclass.cu:348-357)
 *   obstacles: O x 12 doubles, zonotope centre then 3 generators (KPR/armour_main.cu:71-75)
 */
#ifndef ARMOUR_B200_H
#define ARMOUR_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define ARMOUR_NF 7
#define ARMOUR_ABI_VERSION 1

enum {
    ARMOUR_OK = 0,
    ARMOUR_ERR_ARG = -1,        /* null pointer / out-of-range argument */
    ARMOUR_ERR_CUDA = -2,       /* CUDA runtime error or no device (see armour_last_error) */
    ARMOUR_ERR_OBSTACLES = -3,  /* more obstacles than max_obstacles (reference: throw, CollisionChecking.cu:10-13) */
    ARMOUR_ERR_CAPACITY = -4,   /* a monomial table overflowed its configured capacity (never truncated silently) */
    ARMOUR_ERR_STATE = -5,      /* call order: eval before build, batch larger than max_problems, ... */
    ARMOUR_ERR_NOMEM = -6
};

typedef struct armour_ctx armour_ctx;

/* Run-time form of the reference's compile-time configuration (KPR/Parameters.h:10-58,
 * KPR/KinovaWithoutGripperInfo.h:41-61).  Fill with armour_config_default() first. */
typedef struct armour_config {
    int struct_size;            /* sizeof(armour_config), ABI check */
    int device;                 /* CUDA device ordinal */
    int robot_model;            /* 0: Kinova Gen3 without gripper (NUM_JOINTS 7); 1: with fixed gripper link (8) */
    int num_time_steps;         /* NUM_TIME_STEPS, even, <= 128 */
    int max_obstacles;          /* per problem (reference MAX_OBSTACLE_NUM = 40) */
    int max_problems;           /* batch capacity of this context (<= 65535) */
    int cap_link_monomials;     /* capacity of the stored k-only table of one link reach set (multiple of 8) */
    int cap_torque_monomials;   /* capacity of the stored k-only table of one torque reach set (multiple of 8) */
    int cap_work_monomials;     /* capacity of one intermediate PZ during reach-set construction */
    double simplify_threshold;  /* SIMPLIFY_THRESHOLD */
    double k_range[ARMOUR_NF];  /* k_range */
    double mass_uncertainty;    /* < 0: model default (0.03) */
    double inertia_uncertainty; /* < 0: model default (0.03) */
} armour_config;

int armour_config_default(armour_config* cfg);
int armour_ctx_create(const armour_config* cfg, armour_ctx** out);
int armour_ctx_destroy(armour_ctx* ctx);
/* Allocate now everything a batch of nprob problems with nobs obstacles will need (obstacle / half-space /
 * staging buffers), so that the first build is not charged for cudaMalloc.  If the reservation has to grow the
 * half-space buffers the current batch is dropped (build again before evaluating).  The reference allocates in the
 * Obstacles constructor, before its reach-set timer starts (KPR/armour_main.cu:86-88, CollisionChecking.cu:6-55). */
int armour_ctx_reserve(armour_ctx* ctx, int nprob, int nobs);
/* Launch everything on this cudaStream_t (default: a stream owned by the context). */
int armour_ctx_set_stream(armour_ctx* ctx, void* cuda_stream);
int armour_ctx_synchronize(armour_ctx* ctx);
const char* armour_status_string(int status);
const char* armour_last_error(const armour_ctx* ctx);
int armour_abi_version(void);
/* Number of kernels this library has launched on the context since creation (bench.py gpu_launches). */
long long armour_kernel_launches(const armour_ctx* ctx);

/* Problem dimensions: replaces armtd_NLP::get_nlp_info (KPR/NLPclass.cu:62-84). */
int armour_num_joints(const armour_ctx* ctx);
int armour_num_time_steps(const armour_ctx* ctx);
int armour_num_constraints(const armour_ctx* ctx, int nobs);

/* ---- single planning problem (a batch of one) --------------------------------------------------- */

/* Replaces sections II.A-II.D of main(): BezierCurve::makePolyZono, KinematicsDynamics::fk /
 * rnea_nominal / rnea_interval, the robust-input radius and Obstacles::initializeHyperPlane
 * (KPR/armour_main.cu:86-216).  Inputs as parsed from armour.in. */
int armour_reachsets_build(armour_ctx* ctx, const double q0[ARMOUR_NF], const double qd0[ARMOUR_NF],
                           const double qdd0[ARMOUR_NF], const double* obstacles, int nobs);
/* torque_radius(j, t) at out[j*T + t] (Eigen column = time; KPR/armour_main.cu:168-201). */
int armour_get_torque_radius(armour_ctx* ctx, double* out);
/* 3x6 column-major generator matrix of link l, interval t at out[(t*NJ + l)*18]
 * (link_independent_generators, KPR/armour_main.cu:113,126; written to armour_joint_position_radius.out). */
int armour_get_link_independent_generators(armour_ctx* ctx, double* out);
/* Replaces armtd_NLP::get_bounds_info rows g_l / g_u (KPR/NLPclass.cu:116-165). */
int armour_get_bounds(armour_ctx* ctx, double* g_l, double* g_u);
/* Replaces the body of armtd_NLP::eval_g (KPR/NLPclass.cu:272-324): g has m entries. */
int armour_eval_g(armour_ctx* ctx, const double k[ARMOUR_NF], double* g);
/* Replaces the body of armtd_NLP::eval_jac_g with values != NULL (KPR/NLPclass.cu:330-396): m*NF entries. */
int armour_eval_jac_g(armour_ctx* ctx, const double k[ARMOUR_NF], double* values);
/* Both at once (one launch); either output may be NULL. */
int armour_eval_g_jac(armour_ctx* ctx, const double k[ARMOUR_NF], double* g, double* values);
/* Structured Jacobian, offered BESIDE the dense one (the reference declares its Jacobian dense, KPR/NLPclass.cu:348-357, and
 * the calls above keep that contract).  The pattern is fixed by the kinematics: a collision row of link l depends on k_0..k_l
 * only, a Bezier row on its own joint, torque rows are full; every other entry of the dense Jacobian is an exact zero.  A
 * caller that hands Ipopt this structure (get_nlp_info: nnz_jac_g = armour_jacobian_nnz; eval_jac_g with values == NULL:
 * armour_jacobian_structure, C-style indices, row-major, columns ascending) receives the non-zeros alone: 42 140 instead of
 * 69 188 values per problem at 10 obstacles, 39 % fewer bytes over PCIe. */
long long armour_jacobian_nnz(const armour_ctx* ctx, int nobs);
int armour_jacobian_structure(const armour_ctx* ctx, int nobs, int* iRow, int* jCol);
int armour_eval_jac_g_structured(armour_ctx* ctx, const double k[ARMOUR_NF], double* values_nnz);
/* armtd_NLP::link_sliced_center of the last evaluation, out[(t*NJ + l)*3] (KPR/NLPclass.h:150). */
int armour_get_link_sliced_center(armour_ctx* ctx, double* out);
/* Feasibility predicate of armtd_NLP::finalize_solution (KPR/NLPclass.cu:449-537) applied to g:
 * *feasible = 1/0, *first_violation = first violated row in the reference's check order, or -1. */
int armour_verdict(armour_ctx* ctx, const double* g, int* feasible, int* first_violation);
/* Cost and its gradient: armtd_NLP::eval_f / eval_grad_f (KPR/NLPclass.cu:207-268); host arithmetic. */
int armour_cost(armour_ctx* ctx, const double q_des[ARMOUR_NF], const double k[ARMOUR_NF], double* obj,
                double grad[ARMOUR_NF]);

/* ---- batched planning problems (worlds x replans), problem-major arrays ------------------------- */

/* nprob independent problems with the same obstacle count: q0/qd0/qdd0 [nprob*NF],
 * obstacles [nprob*nobs*12].  Host pointers; the H2D copy is part of the call. */
int armour_batch_reachsets_build(armour_ctx* ctx, int nprob, const double* q0, const double* qd0, const double* qdd0,
                                 const double* obstacles, int nobs);
/* One eval_g + eval_jac_g per problem: k [nprob*NF] -> g [nprob*m], values [nprob*m*NF] (either may be
 * NULL).  Host pointers; H2D of k and D2H of the results are part of the call. */
int armour_batch_eval(armour_ctx* ctx, int nprob, const double* k, double* g, double* values);
/* Structured variants: values_nnz [nprob * armour_jacobian_nnz] instead of the dense values (g may be NULL). */
int armour_batch_eval_structured(armour_ctx* ctx, int nprob, const double* k, double* g, double* values_nnz);
int armour_batch_eval_structured_device(armour_ctx* ctx, int nprob, const double* d_k, double* d_g, double* d_values_nnz);
/* Same with DEVICE pointers; asynchronous on the context's stream, no copies. */
int armour_batch_eval_device(armour_ctx* ctx, int nprob, const double* d_k, double* d_g, double* d_values);
/* Inputs already on the device (same layout as the host variant); asynchronous. */
int armour_batch_reachsets_build_device(armour_ctx* ctx, int nprob, const double* d_q0, const double* d_qd0,
                                        const double* d_qdd0, const double* d_obstacles, int nobs);
/* Per-problem verdict on the device from device g: feasible[nprob], first_violation[nprob] (int32). */
int armour_batch_verdict_device(armour_ctx* ctx, int nprob, const double* d_g, int* d_feasible, int* d_first);
int armour_batch_get_torque_radius(armour_ctx* ctx, int nprob, double* out /* [nprob][NF*T] */);
int armour_batch_get_link_independent_generators(armour_ctx* ctx, int nprob, double* out /* [nprob][T*NJ*18] */);
int armour_batch_get_bounds(armour_ctx* ctx, int nprob, double* g_l, double* g_u);
/* Batched planning on the device (SURVEY.md 8f-1; replaces, for a batch, the IpoptApplication::OptimizeTNLP call of
 * KPR/armour_main.cu:237-278 and the PCIe round trips of its eval_g / eval_jac_g callbacks): every problem of the
 * batch runs the trust-region SQP of armour_b200/host/local_solver.cpp on the GPU, in step, from k = 0.  Outputs (device
 * pointers in the _device variant): k_opt[nprob*7] = the point finalize_solution would receive, feasible[nprob] and
 * first_violation[nprob] = its verdict (KPR/NLPclass.cu:449-537), iterations[nprob] (may be NULL).  q_des[nprob*7].
 * No wall-clock limit (the reference's max_wall_time makes results machine dependent); max_iter bounds the work. */
typedef struct armour_solver_options {
    int max_iter;          /* 60, as the host solver */
    double tol;            /* 1e-4 = IPOPT_OPTIMIZATION_TOLERANCE (KPR/Parameters.h:51): step-size stopping test */
    double torque_tol;     /* 1e-2 N m, the verdict's tolerances (KPR/Parameters.h:40-43) */
    double collision_tol;  /* 1e-4 m */
    int qp_sweeps;         /* 200: cap on the active-set iterations of one QP (a guard: the QP of a step is solved exactly
                              by a dual active-set method, which is finite; typical QPs take 2-15 iterations) */
    int qp_update_budget;  /* ignored since round 2 (was the update budget of the Hildreth iteration); kept for the layout */
} armour_solver_options;
void armour_solver_options_default(armour_solver_options* opt);
int armour_batch_solve_device(armour_ctx* ctx, int nprob, const double* d_q_des, const armour_solver_options* opt,
                              double* d_k_opt, int* d_feasible, int* d_first_violation, int* d_iterations);
int armour_batch_solve(armour_ctx* ctx, int nprob, const double* q_des, const armour_solver_options* opt, double* k_opt,
                       int* feasible, int* first_violation, int* iterations);
/* Status of the last build per problem (ARMOUR_OK or ARMOUR_ERR_CAPACITY), out[nprob]. */
int armour_batch_get_build_status(armour_ctx* ctx, int nprob, int* out);
/* Stored k-only monomial counts of the built reach sets: link_n[nprob*T*NJ], u_n[nprob*T*NF] (either may
 * be NULL).  bench.py derives the algorithmic bytes of one evaluation from them (SURVEY.md 8d B_eval). */
int armour_batch_get_monomial_counts(armour_ctx* ctx, int nprob, int* link_n, int* u_n);
/* Stored collision half-space candidates per (link, interval, obstacle) row, out[nprob][T/C][NJ][C][O] bytes in
 * the kernel's chunk order, C = armour_chunk_intervals() (255 = row evaluated from the generators).  bench.py reports
 * the candidate bytes one evaluation streams; there is no counterpart in the reference, which stores all 72
 * half-spaces per row (KPR/CollisionChecking.cu:169-228). */
int armour_batch_get_candidate_counts(armour_ctx* ctx, int nprob, unsigned char* out);
int armour_chunk_intervals(void);
/* Evaluation images (inspection aid): at the end of every build the reach-set tables and candidate lists of each chunk of
 * C intervals are packed into one contiguous image, which is all the evaluation kernel reads.  layout receives 10 byte
 * counts: image bytes per chunk, then the offsets of the link-table entries, torque-table entries, link centres, link
 * radii, torque centres, torque radii, row-group bases, candidate counts and candidate records (see DESIGN.md).
 * armour_batch_get_eval_images copies the images of problems 0..nprob-1 ([p][T/C] chunks of that size) into out.
 * Images of problems whose build failed are not written. */
int armour_eval_image_layout(armour_ctx* ctx, long long* layout);
int armour_batch_get_eval_images(armour_ctx* ctx, int nprob, void* out);
/* Measurement aid: runs a dependent-chain-free FP64 FMA kernel on the context's device and returns the
 * sustained non-tensor FP64 rate in TFLOP/s (the FP64 roofline denominator; BASELINE.md section 2). */
int armour_measure_fp64_peak(armour_ctx* ctx, double* tflops);

/* ---- closed-loop replanning episodes (worlds replanned in sequence) --------------------------------------------------------
 *
 * The loop of the reference's system test (kinova_run_100_worlds.m -> simulator_armtd.run): waypoint, plan, execute the plan up
 * to t_move, replan from where the executed motion ends; run for a batch of worlds on the device, with an exact collision and
 * joint-limit audit of every executed segment.  A world has a start and a goal configuration and nobs obstacles ([nobs][12]
 * zonotopes as everywhere else); the arm starts at rest; nworlds <= max_problems.  Replan r of world w:
 *   1. planning state (q0, qd0, qdd0): (start, 0, 0) at r = 0, afterwards the state step 5 of replan r - 1 produced;
 *   2. q_des: the straight-line waypoint of armour_b200.worlds.straight_line_waypoint (angdiff on the continuous joints 0, 2,
 *      4, 6; lookahead rad along d = goal - q), except that when |d| <= lookahead the waypoint is the goal itself (q + d), so
 *      that an arriving arm is not pulled past it.  The clamp is this library's choice (the reference's high-level planner,
 *      robot_arm_straight_line_HLP.m, is not part of the reference tree this library restates);
 *   3. plan: armour_batch_reachsets_build_device + armour_batch_solve_device on the running worlds, from k = 0, with
 *      opt->solver as given.  A build that overflowed a table evaluates fail-safe: an infeasible replan, logged separately;
 *   4. executed segment: after a feasible plan the new plan over s in [0, t_move], and it becomes the world's current plan;
 *      otherwise the current plan's braking half s in [t_move, 1], after which the current plan is the rest plan at its end
 *      (q = q(1), qd = qdd = 0, k = 0; its Bezier is constant, so repeated failures keep the arm still).  The initial current
 *      plan is the rest plan at the start.  t_move = t_plan = 0.5 s of the robot model (duration 1 s);
 *   5. next state: (q, qd, qdd) of the executed plan at the segment's end, time derivatives in real time;
 *   6. audit: audit_samples evenly spaced samples of the executed segment, both ends included.  At each sample the exact link
 *      boxes (forward kinematics of all num_joints links) against every obstacle: the signed clearance of two parallelepipeds
 *      by the separating-axis test (15 axes; > 0 separated, a lower bound on the distance; <= 0 intersecting, -penetration);
 *      the non-continuous joints against the raw position limits and |qd| against the raw speed limits (without the margins of
 *      the verdict);
 *   7. stop: clearance below -opt->solver.collision_tol -> ARMOUR_ROLLOUT_COLLISION, else a limit exceeded -> _LIMIT, else the
 *      segment's end within goal_radius of the goal (2-norm of the difference, angdiff on the continuous joints) -> _ARRIVED,
 *      else max_replans used -> _BUDGET.  The loop ends when no world is running.
 * Stopped worlds leave the later builds and solves: the running worlds are gathered in ascending world index into the dense
 * batch (the sub-batch of replan r is the worlds with replans > r, in order).  Continuous joints are not wrapped; there is no
 * %.10f quantisation inside the loop.  Log rows are indexed by world; world w planned at replan r exactly when r < replans[w];
 * the rows of replans it did not plan are NaN (doubles) and -1 (ints).  The context's reach sets after the call are those of
 * the last replan's sub-batch.  Not modelled: tracking error and the low-level controller, torque audits, warm starts.
 * Errors: ARMOUR_ERR_STATE for nworlds > max_problems and for a context of the ARMTD comparison planner, ARMOUR_ERR_OBSTACLES for
 * nobs > max_obstacles, ARMOUR_ERR_ARG for bad options and null inputs. */
enum { ARMOUR_ROLLOUT_BUDGET = 0, ARMOUR_ROLLOUT_ARRIVED = 1, ARMOUR_ROLLOUT_COLLISION = 2, ARMOUR_ROLLOUT_LIMIT = 3 };
typedef struct armour_rollout_options {
    int struct_size;               /* sizeof(armour_rollout_options) */
    int max_replans;               /* >= 1, default 100 */
    double lookahead;              /* > 0, default 0.1 rad (the reference's straight-line waypoint) */
    double goal_radius;            /* >= 0, default 0.05 rad: this library's choice, the reference's goal test is not in its tree */
    int audit_samples;             /* >= 2, default 16 */
    armour_solver_options solver;  /* the solve of every replan; collision_tol is also the audit's tolerance */
} armour_rollout_options;
void armour_rollout_options_default(armour_rollout_options* opt);
/* Outputs; any pointer may be NULL.  [n] = nworlds, [R] = max_replans. */
typedef struct armour_rollout_out {
    int* outcome;            /* [n] ARMOUR_ROLLOUT_* */
    int* replans;            /* [n] replans planned */
    int* infeasible;         /* [n] replans that executed the braking half */
    double* final_state;     /* [n][21] q, qd, qdd at the end of the last executed segment */
    double* min_clearance;   /* [n] smallest audited clearance over the episode, m (+inf without obstacles) */
    double* log_state;       /* [R][n][21] planning state q0, qd0, qdd0 of replan r */
    double* log_q_des;       /* [R][n][7] */
    double* log_k;           /* [R][n][7] k_opt */
    int* log_int;            /* [R][n][4] feasible, first violated row, solver iterations, build status (0 / ARMOUR_ERR_CAPACITY) */
    double* log_clearance;   /* [R][n] smallest audited clearance of the segment executed after replan r */
} armour_rollout_out;
/* start, goal [nworlds][7], obstacles [nworlds][nobs][12]; DEVICE pointers, in *out too.  One device-to-host copy of the
 * running count and one synchronisation per replan. */
int armour_batch_rollout_device(armour_ctx* ctx, int nworlds, const double* d_start, const double* d_goal, const double* d_obstacles,
                                int nobs, const armour_rollout_options* opt, const armour_rollout_out* d_out);
/* The same with host pointers (the copies are part of the call). */
int armour_batch_rollout(armour_ctx* ctx, int nworlds, const double* start, const double* goal, const double* obstacles, int nobs,
                         const armour_rollout_options* opt, const armour_rollout_out* out);
/* Episodes of the ARMTD comparison planner (section "ARMTD comparison planner" below), on the same worlds, options, outputs and
 * audit as the episodes above, on a context of armour_armtd_batch_ctx_create.  Replan r of world w, step by step:
 *   1. planning state (q0, qd0): (start, 0) at r = 0, afterwards the end of the last executed segment.  The planner has no
 *      acceleration input: the qdd slots of log_state and final_state are 0 (the 21-wide layout is kept so that
 *      armour_rollout_out is shared);
 *   2. q_des: as step 2 above (the same straight-line waypoint and the same clamp at the goal);
 *   3. plan: k_range = max(pi / 24, |qd0| / 3) per joint (armour_b200.worlds.armtd_k_range) and the offline table of
 *      armour_armtd_offline_jrs (this library's synthetic stand-in, not the reference's CORA table) for every running world,
 *      armour_armtd_batch_build_device with the device's sincos (d_sincos NULL) + armour_armtd_batch_solve_device, from k = 0
 *      with opt->solver as given (armour_rollout_options_default leaves its tol at the main planner's default; KPA's is 1e-7).
 *      The verdict is KPA's finalize_solution (armour_armtd_batch_verdict_device), so the collision rows of the last link are not
 *      checked, as in the reference.  A build that overflowed a table is an infeasible replan, logged with its build status;
 *   4. executed segment: after a feasible plan the new plan over t in [0, 0.5], and it becomes the world's current plan;
 *      otherwise the current plan's braking half t in [0.5, 1], after which the current plan is the rest plan at q_stop
 *      (qd0 = 0, k_a = 0).  The trajectory is the constant-acceleration curve of KPA (the one armour_armtd_eval's joint-limit
 *      rows bound): q0 + qd0 t + k_a t^2 / 2 for t <= 0.5, then q_peak + qd_peak tau - qd_peak tau^2 with tau = t - 0.5, braking
 *      to rest at t = 1; k_a = k_range * k_opt.  The end points at t = 0.5 and t = 1 are computed by the expressions of those
 *      rows (q_peak, q_dot_peak, q_stop).  A plan is stored as (q0, qd0, 0, k_a); the initial current plan is the rest plan at
 *      the start;
 *   5. next state: (q, qd, 0) at the segment's end;
 *   6. audit and stop: steps 6 and 7 above unchanged (all num_joints links by the separating-axis test, the raw position and
 *      speed limits; collision, limit, arrived, budget in this order).
 * Compaction, log rows and the context's reach sets afterwards: as above.  Rollout scratch grows by 4 207 doubles per world
 * (the table and k_range of the dense batch).  Errors: ARMOUR_ERR_STATE on a context of the main planner and for
 * nworlds > max_problems, ARMOUR_ERR_OBSTACLES for nobs > max_obstacles, ARMOUR_ERR_ARG for bad options and null inputs. */
int armour_armtd_batch_rollout_device(armour_ctx* ctx, int nworlds, const double* d_start, const double* d_goal,
                                      const double* d_obstacles, int nobs, const armour_rollout_options* opt,
                                      const armour_rollout_out* d_out);
int armour_armtd_batch_rollout(armour_ctx* ctx, int nworlds, const double* start, const double* goal, const double* obstacles,
                               int nobs, const armour_rollout_options* opt, const armour_rollout_out* out);
/* Exact clearance of nconf arm configurations q [nconf][7]: the link boxes of the context's robot model against obstacle set
 * world[i] of obstacles [nsets][nobs][12] (world NULL: set 0 for all) by the audit's separating-axis test.  clearance[nconf]
 * = the smallest over links and obstacles, which[nconf] (may be NULL) = l * nobs + o of the pair attaining it (ties: the lowest),
 * +inf and -1 without obstacles.  The _device call does not check world[] against the number of sets. */
int armour_batch_clearance_device(armour_ctx* ctx, int nconf, const double* d_q, const int* d_world, const double* d_obstacles,
                                  int nobs, double* d_clearance, int* d_which);
int armour_batch_clearance(armour_ctx* ctx, int nconf, const double* q, const int* world, const double* obstacles, int nobs,
                           double* clearance, int* which);

/* ---- reach-set tables (k-only monomials after reduce / reduce_link_PZ) -------------------------- */

/* Padded neutral layout shared with the test oracle:
 *   links : n[t*NJ+l], center[(t*NJ+l)*3+e], key[(t*NJ+l)*cap_link+m], coeff[((t*NJ+l)*cap_link+m)*3+e]
 *   torque: n[t*NF+j], center[t*NF+j],       key[(t*NF+j)*cap_u+m],    coeff[(t*NF+j)*cap_u+m]
 * key = the reference's degree hash (KPR/PZsparse.h:23-40), < 2^14 for k-only monomials. */
typedef struct armour_reachset_tables {
    int cap_link, cap_u;
    int* link_n;
    double* link_center;
    unsigned long long* link_key;
    double* link_coeff;
    int* u_n;
    double* u_center;
    unsigned long long* u_key;
    double* u_coeff;
    double* u_radius;        /* [t*NF + j] radius of the reduced nominal torque PZ (u_nom.independent) */
    double* torque_radius;   /* [j*T + t] */
    double* link_gens;       /* [(t*NJ + l)*18] */
} armour_reachset_tables;

/* Download the tables of problem `prob` (debugging / parity tests / *_joint_position_*.out files). */
int armour_export_reachsets(armour_ctx* ctx, int prob, armour_reachset_tables* out);
/* Upload externally built tables for problem `prob` together with the inputs the Bezier rows need, then
 * build its collision hyper-planes.  Lets the constraint kernels be exercised in isolation. */
int armour_import_reachsets(armour_ctx* ctx, int prob, int nprob_total, const armour_reachset_tables* in,
                            const double q0[ARMOUR_NF], const double qd0[ARMOUR_NF], const double qdd0[ARMOUR_NF],
                            const double* obstacles, int nobs);

/* ---- robust controller: interval Newton-Euler pass and robust input, batched over states (SURVEY.md 8f-4) -------------
 *
 * Replaces, for a batch of n sampled states, what the reference's MEX entry computes for ONE state per call:
 *   [u, tau, v] = kinova_controller(Kr, alpha, V_max, r_norm_threshold, q, qd, q_des, qd_des, qdd_des [, eps])
 * (MEX/kinova_controller.cpp:19-99): Robot(RobotFilePath, eps) -> armour_controller_create, RobustController::update
 * (MEX/robust_controller.cpp:67-181, ARMOUR method) -> armour_controller_update, and the two passes under it, passRNEA /
 * passRNEA_Int (MEX/rnea.cpp:6-94 / 96-187) -> armour_controller_rnea.  All state arrays are [n][numJoints] row-major.
 * Interval end points are outward rounded at every operation exactly as Boost.Interval does in the reference.
 * The host-pointer calls compute sin / cos of the joint angles with the host's libm like the reference and are bit-exact
 * against it for the interval outputs; the *_device calls take device pointers and, when d_sincos is NULL, use the device's
 * sincos (end points within a few ulp).  d_sincos: [n][numJoints][2] = sin(-q), cos(-q).
 * A controller object is thread-compatible, not thread-safe; it owns one stream (armour_controller_set_stream adopts the
 * caller's).  There is no CPU fallback. */
typedef struct armour_controller armour_controller;
typedef struct armour_controller_gains {
    const double* Kr;          /* [numJoints] diagonal of Kr (kinova_controller.cpp:36-40) */
    double alpha;              /* ARMOUR robust input: lambda = max(0, -alpha (V_max - sup V) / |r| + |bound|) */
    double V_max;
    double r_norm_threshold;   /* v = 0 below this |r| */
    int apply_friction;        /* RobustController::applyFriction; the MEX entry sets 0 */
} armour_controller_gains;
/* model_file: the reference's robot text format (MEX/kinova_without_gripper.txt); model_uncertainty: eps of the interval
 * model (0.03 in the MEX entry).  On failure *out is untouched and armour_controller_create_error() tells why. */
int armour_controller_create(const char* model_file, double model_uncertainty, int device, armour_controller** out);
const char* armour_controller_create_error(void);
void armour_controller_destroy(armour_controller* ctl);
int armour_controller_num_joints(const armour_controller* ctl);
const char* armour_controller_last_error(const armour_controller* ctl);
long long armour_controller_kernel_launches(const armour_controller* ctl);
int armour_controller_set_stream(armour_controller* ctl, void* cuda_stream);
int armour_controller_synchronize(armour_controller* ctl);
/* The interval model after the conversion of IntModel::IntModel (MEX/robot_models.cpp:175-237), per joint
 * S.w[3] S.v[3] XTree.R[9] XTree.p[3] m I_bar[9] m_c_hat[9], each as (lower, upper): out[numJoints * 74]. */
int armour_controller_get_interval_model(const armour_controller* ctl, double* out);
/* passRNEA (tau, may be NULL) and / or passRNEA_Int (tau_lo, tau_hi, may both be NULL) of n states. */
int armour_controller_rnea(armour_controller* ctl, int n, const double* q, const double* qd, const double* qda,
                           const double* qdd, int apply_friction, int apply_gravity, double* tau, double* tau_lo,
                           double* tau_hi);
int armour_controller_rnea_device(armour_controller* ctl, int n, const double* d_q, const double* d_qd,
                                  const double* d_qda, const double* d_qdd, const double* d_sincos, int apply_friction,
                                  int apply_gravity, double* d_tau, double* d_tau_lo, double* d_tau_hi);
/* RobustController::update for n states: u = u_nominal - v; u_nominal, v, status may be NULL.  status[i] = 1 where the
 * nominal torque is outside the interval torque (the reference throws there), else 0. */
int armour_controller_update(armour_controller* ctl, int n, const armour_controller_gains* gains, const double* q,
                             const double* qd, const double* q_des, const double* qd_des, const double* qdd_des, double* u,
                             double* u_nominal, double* v, int* status);
int armour_controller_update_device(armour_controller* ctl, int n, const armour_controller_gains* gains, const double* d_q,
                                    const double* d_qd, const double* d_q_des, const double* d_qd_des,
                                    const double* d_qdd_des, const double* d_sincos, double* d_u, double* d_u_nominal,
                                    double* d_v, int* d_status);

/* ---- ARMTD comparison planner (SURVEY.md 8f-3) ---------------------------------------------------------------------------
 *
 * The reference's second planner (kinova_planner_realtime_armtd_comparison/, "KPA": armtd_main.cu, Trajectory.cu, NLPclass.cu):
 * constant-acceleration trajectories whose cos / sin joint reachable sets come from an OFFLINE table the caller slices and hands
 * in (the six arrays of KPA's input file, armtd_main.cu:70-88), forward kinematics only, 100 time steps, no torque rows.  It runs
 * on the kernels of the main path: the build is k_armtd_jrs (the table rotated by q0) + k_reachsets with the joint reachable set
 * imported + k_hyperplanes, an evaluation is k_constraints + a kernel that lays the rows out as KPA's armtd_NLP does.  A context
 * holds a batch of problems (worlds), problem-major arrays as in the armour_batch_* family; the single-problem calls below act
 * on problem 0 and are batches of one.
 *   rows of g: collision (l * 100 + t) * nobs + o  (l < num_joints, t < 100), then 7 minimum joint positions, 7 maximum joint
 *   positions, 7 minimum joint velocities, 7 maximum joint velocities (KPA/NLPclass.cu:43-44, 248-283);
 *   values: dense m x 7 row-major like the main planner's; the joint-limit rows are diagonal and, as in the reference, hold the
 *   derivative with respect to k_range * k (KPA/Trajectory.cu:262-384 writes no k_range factor).
 * armour_armtd_ctx_create: cfg may be NULL (defaults); num_time_steps, max_problems (1) and robot_model are set by the call.
 * jrs: [6][7][100] = c_cos, g_cos, r_cos, c_sin, g_sin, r_sin, each joint-major over the 100 intervals. */
int armour_armtd_ctx_create(const armour_config* cfg, armour_ctx** out);
int armour_armtd_build(armour_ctx* ctx, const double q0[ARMOUR_NF], const double qd0[ARMOUR_NF], const double* jrs,
                       const double k_range[ARMOUR_NF], const double* obstacles, int nobs);   /* armtd_main.cu:107-160 */
int armour_armtd_num_constraints(const armour_ctx* ctx);                                      /* NLPclass.cu:43-44 */
int armour_armtd_eval(armour_ctx* ctx, const double k[ARMOUR_NF], double* g, double* values); /* eval_g / eval_jac_g; either NULL */
int armour_armtd_get_bounds(armour_ctx* ctx, double* g_l, double* g_u);                       /* NLPclass.cu:75-142; any problem */
int armour_armtd_verdict(armour_ctx* ctx, const double* g, int* feasible, int* first_violation);  /* :366-455 */
int armour_armtd_cost(armour_ctx* ctx, const double q_des[ARMOUR_NF], const double k[ARMOUR_NF], double* obj, double* grad);
/* [100][num_joints][3] of the last evaluation, of problem 0 only (in a batch too, like armour_get_link_sliced_center) */
int armour_armtd_get_link_sliced_center(armour_ctx* ctx, double* out);
int armour_armtd_get_link_independent_generators(armour_ctx* ctx, double* out);  /* [100][num_joints][18], column-major 3x6 */

/* Batches of ARMTD problems (worlds x replans), the counterpart of the armour_batch_* family: nprob independent problems with the
 * same obstacle count, each with its own q0 / qd0 / offline table / k_range (KPA's k_range depends on the world).  Shapes:
 * q0, qd0, k_range, q_des, k, k_opt [nprob][7]; jrs [nprob][6][7][100]; obstacles [nprob][nobs][12]; g [nprob][m];
 * values [nprob][m][7]; m = armour_armtd_num_constraints.  The *_device calls take device pointers and are asynchronous on the
 * context's stream.  Errors as in the armour_batch_* family: ARMOUR_ERR_STATE for a batch larger than max_problems and for an
 * evaluation / verdict / solve before a build; ARMOUR_ERR_OBSTACLES above max_obstacles; on a context of the main planner
 * ARMOUR_ERR_STATE from the build, eval, verdict and solve calls and ARMOUR_ERR_ARG from armour_armtd_batch_cost and
 * armour_armtd_batch_get_link_independent_generators (as from their single-problem counterparts).  A problem whose build
 * overflowed a table (ARMOUR_ERR_CAPACITY; armour_batch_get_build_status names it) evaluates to collision rows 1e300 with a
 * zero Jacobian and is never feasible; the other problems of the batch are unaffected.
 * armour_armtd_batch_ctx_create: as armour_armtd_ctx_create but honours cfg->max_problems. */
int armour_armtd_batch_ctx_create(const armour_config* cfg, armour_ctx** out);
/* ConstantAccelerationCurve (KPA/Trajectory.cu:29-62) + forward kinematics + hyper-planes for the batch.  The host-pointer call
 * computes cos q0 / sin q0 with the host's libm like the reference; the device call takes them from d_sincos [nprob][7][2] =
 * (cos q0, sin q0), or, when d_sincos is NULL, uses the device's sincos (a few ulp from the host's). */
int armour_armtd_batch_build(armour_ctx* ctx, int nprob, const double* q0, const double* qd0, const double* jrs,
                             const double* k_range, const double* obstacles, int nobs);
int armour_armtd_batch_build_device(armour_ctx* ctx, int nprob, const double* d_q0, const double* d_qd0, const double* d_jrs,
                                    const double* d_k_range, const double* d_obstacles, int nobs, const double* d_sincos);
/* The offline table as this library generates it: a SYNTHETIC STAND-IN for the reference's offline tables (MATLAB / CORA output
 * that is not in the reference tree), NOT the reference's CORA table.  qd0, k_range [n][7] -> jrs [n][6][7][100] in the layout the
 * builds take: per joint and interval the centre and slope of cos / sin of q(t) - q0 = qd0 t + k_range k t^2 / 2 (braking to rest
 * after t = 0.5, the curve of armour_armtd_batch_rollout) at the interval's mid-time, and the radius 1.1 * the largest residual
 * over 9 x 33 samples of (t, k) + 1e-6.  It restates armour_b200.worlds.armtd_offline_jrs_batch operation for operation; the
 * device's sincos stands in for numpy's cos / sin, so entries differ from numpy's by a few ulp.  The episodes build from this
 * table at every replan; these calls let a logged replan be rebuilt from exactly that table.  ARMTD contexts only
 * (ARMOUR_ERR_STATE otherwise), n >= 1, no limit from max_problems. */
int armour_armtd_offline_jrs(armour_ctx* ctx, int n, const double* qd0, const double* k_range, double* jrs);
int armour_armtd_offline_jrs_device(armour_ctx* ctx, int n, const double* d_qd0, const double* d_k_range, double* d_jrs);
/* eval_g / eval_jac_g of every problem at k (either output may be NULL) */
int armour_armtd_batch_eval(armour_ctx* ctx, int nprob, const double* k, double* g, double* values);
int armour_armtd_batch_eval_device(armour_ctx* ctx, int nprob, const double* d_k, double* d_g, double* d_values);
/* finalize_solution's predicate (KPA/NLPclass.cu:366-455) per problem: d_feasible[nprob], d_first[nprob] (int32).  As in the
 * reference the collision rows of the last link are not checked (its loop runs over NUM_FACTORS - 1 links). */
int armour_armtd_batch_verdict_device(armour_ctx* ctx, int nprob, const double* d_g, int* d_feasible, int* d_first);
/* eval_f / eval_grad_f (KPA/NLPclass.cu:178-243) per problem: obj[nprob], grad[nprob][7] (either may be NULL); host arithmetic */
int armour_armtd_batch_cost(armour_ctx* ctx, int nprob, const double* q_des, const double* k, double* obj, double* grad);
/* out [nprob][100][num_joints][18] (the padding intervals of the context are left out) */
int armour_armtd_batch_get_link_independent_generators(armour_ctx* ctx, int nprob, double* out);
/* Batched planning on the device: replaces, for a batch, the Ipopt run of KPA/armtd_main.cu:162-207 (armtd_main's local
 * solver with its PCIe round trips per callback).  The trust-region SQP of armour_batch_solve over KPA's NLP: collision rows
 * one-sided with collision_tol (all links), joint-limit rows two-sided with tolerance 0, KPA's cost; the verdict is
 * armour_armtd_batch_verdict_device's.  opt == NULL: armour_solver_options_default with tol = 1e-7 (IPOPT_OPTIMIZATION_TOLERANCE,
 * KPA/Parameters.h:43).  No wall-clock limit.  Outputs as armour_batch_solve. */
int armour_armtd_batch_solve(armour_ctx* ctx, int nprob, const double* q_des, const armour_solver_options* opt, double* k_opt,
                             int* feasible, int* first_violation, int* iterations);
int armour_armtd_batch_solve_device(armour_ctx* ctx, int nprob, const double* d_q_des, const armour_solver_options* opt,
                                    double* d_k_opt, int* d_feasible, int* d_first_violation, int* d_iterations);

#ifdef __cplusplus
}
#endif
#endif /* ARMOUR_B200_H */
