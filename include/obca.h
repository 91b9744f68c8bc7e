/*
 * obca.h -- C ABI of the B200-native batched OBCA solver (libobca_b200.so).
 *
 * The reference (XuShenLZ/conflict_rez) has no FFI: its boundary is the CasADi ``Opti`` protocol used
 * inside the planner classes.  Each entry point below names the reference call it replaces:
 *
 *   obca_create / obca_set_static   <- building the Opti graph: Vehicle.setup_single_final_problem
 *                                      (confrez/control/vehicle.py:360-640) and the joint assembly in
 *                                      MultiVehiclePlanner.solve_final_problem_obca
 *                                      (confrez/control/multi_vehicle_planner.py:365-451)
 *   obca_set_init_pose              <- the initial-state equalities (vehicle.py:424-434) per instance
 *   obca_set_initial                <- opti.set_initial(...) (vehicle.py:482-485,629-636;
 *                                      multi_vehicle_planner.py:367,426-428)
 *   obca_solve                      <- opti.solver("ipopt", ...); opti.solve()
 *                                      (vehicle.py:657-658; multi_vehicle_planner.py:464-465)
 *   obca_get_solution               <- sol.value(...) (vehicle.py:668-716)
 *   obca_get_stats                  <- sol.stats()["return_status"] (vehicle.py:659)
 *
 * Conventions: every array is FP64, C-contiguous; "dev" pointers are device pointers owned by the
 * caller (torch tensors in the Python host layer), "host" pointers are plain host memory.  All calls
 * return 0 on success and a negative code on error (obca_last_error() gives the text).  No exception
 * crosses the ABI, there is no CPU fallback: obca_create fails when no CUDA device is usable.
 * A handle is not thread-safe; different handles may be used concurrently.
 */
#ifndef OBCA_H_
#define OBCA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OBCA_MAX_V 8      /* vehicles per instance */
#define OBCA_MAX_O 32     /* obstacles (4 half-planes each) */
#define OBCA_MAX_SETS 64  /* strategy sets per vehicle */
#define OBCA_MODE_COLLOCATION 0
#define OBCA_MODE_MPC 1   /* VehicleFollower.setup_controller NLP (confrez/control/vehicle_follower.py:146-368) */
#define OBCA_MODE_STATE_WS 2 /* Vehicle.state_ws: Euler-discretised tube-following NLP (confrez/control/vehicle.py:99-231); one vehicle,
                                n_sets[0] strategy sets, n_per_set = Euler steps per move (the reference's N), nodes 0 .. N (S - 1);
                                the sample time is ObcaStatic.mpc_dt, the initial state goes in through obca_set_mpc_params (cur) */

/* per-instance return status, mirroring IPOPT's ApplicationReturnStatus strings */
#define OBCA_SOLVE_SUCCEEDED 0
#define OBCA_SOLVED_TO_ACCEPTABLE_LEVEL 1   /* search direction below machine precision at the smallest mu */
#define OBCA_MAXITER_EXCEEDED (-1)
#define OBCA_RESTORATION_FAILED (-2)
#define OBCA_ERROR_IN_STEP_COMPUTATION (-3)
#define OBCA_INVALID_NUMBER_DETECTED (-4)
#define OBCA_SEARCH_DIRECTION_TOO_SMALL (-5)   /* two consecutive tiny steps at the smallest mu without an acceptable point */
#define OBCA_INFEASIBLE_PROBLEM_DETECTED (-6) /* converged with an active elastic variable: the reference problem (hard distance rows) is infeasible */
#define OBCA_NOT_SOLVED (-100)

typedef struct ObcaDims {
  int32_t batch;                 /* B: independent instances */
  int32_t V;                     /* vehicles per instance */
  int32_t O;                     /* obstacles */
  int32_t K;                     /* collocation degree (must be 5) */
  int32_t n_per_set;             /* collocation intervals per strategy move (must be >= 1) */
  int32_t n_sets[OBCA_MAX_V];    /* S_a: strategy sets of vehicle a; N_a = n_per_set * (S_a - 1) */
  int32_t mode;                  /* OBCA_MODE_COLLOCATION (default 0) or OBCA_MODE_MPC */
  int32_t horizon;               /* MPC: nodes N (vehicle_follower.py:146, N = 30) */
  int32_t n_others;              /* MPC: other vehicles whose predictions are parameters */
  int32_t bounded_input;         /* STATE_WS: a / w limits enforced (state_ws(bounded_input=True), vehicle.py:155-167) */
} ObcaDims;

typedef struct ObcaOptions {
  double tol, constr_viol_tol, dual_inf_tol, compl_inf_tol;
  double mu_init;
  double dmin, shrink_tube;
  double elastic_weight;         /* rho of the exact l1 penalty on the elastic variables of the distance rows */
  int32_t max_iter;
  int32_t refine_steps;          /* iterative-refinement solves per Newton system (IPOPT: max_refinement_steps); -1 = automatic:
                                    0 when tol > 1e-5 (the reference's 1e-2), 2 at tight tolerances */
} ObcaOptions;

typedef struct ObcaStatic {       /* host pointers; copied by obca_set_static */
  const double* obs_A;           /* (O,4,2) */
  const double* obs_b;           /* (O,4) */
  const double* tube_A;          /* (V,Smax,2[back,front],4,2), Smax = max n_sets */
  const double* tube_b;          /* (V,Smax,2,4) raw b (shrink_tube is subtracted inside) */
  const double* body_G;          /* (4,2) */
  const double* body_g;          /* (4) */
  const double* region;          /* xmin,xmax,ymin,ymax */
  const double* limits;          /* v,delta,a,w (min,max) */
  const double* final_heading;   /* (V) NaN = unconstrained */
  double wb;
  double mpc_dt;                 /* MPC sample time (vehicle_follower.py:146, dt = 0.1); unused in collocation mode */
  const double* colloc_A;        /* (K+1,K+1) A[j][k] = L_j'(tau_k) as Vehicle.collocation_coefficients computes it (vehicle.py:54-97), */
  const double* colloc_B;        /* (K+1) quadrature weights; NULL = computed inside from the Radau points (same values to ~1e-14) */
} ObcaStatic;

typedef struct ObcaHandle ObcaHandle;

const char* obca_version(void);
const char* obca_last_error(void);
void obca_default_options(ObcaOptions* opts);

int obca_create(const ObcaDims* dims, const ObcaOptions* opts, int device, ObcaHandle** out);
int obca_destroy(ObcaHandle* h);
int obca_set_static(ObcaHandle* h, const ObcaStatic* st);
int obca_set_options(ObcaHandle* h, const ObcaOptions* opts);

/* dev: (B,V,3) x,y,psi including the initial offsets */
int obca_set_init_pose(ObcaHandle* h, const double* init_pose_dev, void* stream);

/* dev, node-major like CollocationGuess: z (B,V,Mmax,7); lam, mu (B,V,Mmax,O,4); dt (B);
 * pair_lam, pair_mu (B,P,Mmax,4); pair_s (B,P,Mmax,2) -- pair pointers may be NULL when V == 1. */
int obca_set_initial(ObcaHandle* h, const double* z, const double* lam, const double* mu, const double* dt,
                     const double* pair_lam, const double* pair_mu, const double* pair_s, void* stream);

/* MPC mode, replaces opti.set_value(...) of VehicleFollower.step (vehicle_follower.py:432-456): dev pointers
 * cur (B,5) current state, ref (B,N,3) reference x,y,psi, others (B,n_others,N,3) neighbours' shifted predictions.
 * obca_set_initial takes z (B,1,N,7), lam/mu (B,1,N,O,4), dt (B, ignored), pair_* (B,n_others,N,.) in this mode. */
int obca_set_mpc_params(ObcaHandle* h, const double* cur, const double* ref, const double* others, void* stream);

/* Dual warm starts in closed form for 4-face polytopes, on the device (all pointers dev, node-major like obca_set_initial):
 * obca_dual_ws replaces Vehicle.dual_ws (confrez/control/vehicle.py:233-296): poses z (B,V,Mmax,7) -> lam, mu (B,V,Mmax,O,4);
 * obca_joint_dual_ws replaces MultiVehiclePlanner.joint_dual_ws (confrez/control/multi_vehicle_planner.py:208-341):
 * z -> pair_lam, pair_mu (B,P,Mmax,4), pair_s (B,P,Mmax,2).  Entries of padding nodes are set to zero. */
int obca_dual_ws(ObcaHandle* h, const double* z, double* lam, double* mu, void* stream);
int obca_joint_dual_ws(ObcaHandle* h, const double* z, double* pair_lam, double* pair_mu, double* pair_s, void* stream);

/* ---- trajectory-side kernels (csrc/obca_traj.h); no handle needed, all pointers dev unless noted ------------------------ */
/* replaces Vehicle.get_interpolator / interpolate_states (confrez/control/vehicle.py:722-829), one thread per sample:
 * z (B,V,Mmax,7) collocation solution, dt (B) -- or (B,V) when dt_per_vehicle != 0 (separately planned vehicles) --,
 * n_intervals (V, HOST), tau (K+1 = 6, HOST) collocation nodes on [0,1];
 * times (T) shared by all vehicles, or (B,V,T) when per_vehicle_times != 0; out (B,V,T,7) = x y psi v delta a w.
 * States: degree-K Lagrange polynomial of the interval that contains t, final state held beyond the horizon;
 * inputs: piecewise constant between the collocation nodes (ca.pw_const semantics). */
int obca_interpolate(int device, const double* z, const double* dt, const int32_t* n_intervals, const double* tau, int B, int V, int Mmax,
                     const double* times, int T, int per_vehicle_times, int dt_per_vehicle, double* out, void* stream);
/* replaces Vehicle.interp_ws_for_collocation (confrez/control/vehicle.py:298-358): C warm-start signals sampled on the time grid
 * t (T, dev) are interpolated linearly (scipy interp1d) onto the collocation times (i + tau_k) / N * t[T-1], i < N, k <= K:
 * in (B,T,C) -> out (B,N*(K+1),C); tau (K+1 = 6, HOST). */
int obca_interp_ws(int device, const double* in, const double* t, const double* tau, int B, int T, int C, int N, double* out, void* stream);
/* replaces the time lookup of VehicleFollower.get_current_ref (confrez/control/vehicle_follower.py:370-404): for every vehicle
 * (B,V) the N sample times  t_ref[argmin |t_ref - clock|] + k * dt_mpc  of the dense reference grid linspace(t_first, t_last, n_ref);
 * grid (B,V,3) = t_first, t_last, n_ref (as double), clock (B,V) -> times (B,V,N) (feed to obca_interpolate, per_vehicle_times = 1) */
int obca_mpc_ref_times(int device, const double* grid, const double* clock, int B, int V, int N, double dt_mpc, double* times, void* stream);
/* replaces simulator (confrez/control/dynamic_model.py:61-93): state (B,5), input (B,2) -> next (B,5) after dt under constant input
 * (fixed-step RK4, `substeps` sub-steps; the reference integrates the same ODE with IDAS) */
int obca_plant_step(int device, const double* state, const double* input, int B, double dt, double wb, int substeps, double* next, void* stream);
/* replaces VehicleFollower._adv_onestep (vehicle_follower.py:413-426) for a (B,N,W) array: out[b][n] = in[b][min(n+1, N-1)] */
int obca_shift_horizon(int device, const double* in, int B, int N, int W, double* out, void* stream);

/* DFMA micro-benchmark: sustained FP64 FMA throughput of `device` in TFLOP/s (the FP64 roofline denominator of bench.py;
 * SURVEY.md 8d asks for a measured figure next to the data-sheet 37 TFLOP/s) */
int obca_measure_dfma_peak(int device, double* tflops);

/* Processing order of the batch: order_dev (B int32, a permutation, dev pointer, copied) tells which instance the k-th free
 * CTA picks up.  Instances are independent, so results do not depend on it; putting the instances that are expected to need
 * the most iterations first shortens the tail of the persistent-CTA queue (longest-processing-time-first).  NULL = 0..B-1. */
int obca_set_order(ObcaHandle* h, const int32_t* order_dev, void* stream);

/* run the batched interior-point solve, asynchronously on `stream`; no host sync inside */
int obca_solve(ObcaHandle* h, void* stream);

/* same shapes as obca_set_initial, dev pointers, any may be NULL */
int obca_get_solution(ObcaHandle* h, double* z, double* lam, double* mu, double* dt, double* pair_lam,
                      double* pair_mu, double* pair_s, void* stream);

/* dev pointers (B): any may be NULL.  cviol is the violation of the REFERENCE problem: max(|c|, largest elastic variable);
 * elastic is the largest elastic variable alone (0 at a solution of the reference problem). */
int obca_get_stats(ObcaHandle* h, int32_t* status, int32_t* iters, double* obj, double* cviol, double* dual_inf,
                   double* compl_inf, double* elastic, void* stream);

/* ---- iteration record ---------------------------------------------------------------------------------------------------
 * With recording on, obca_solve writes one row of OBCA_HIST_FIELDS doubles per head of the interior-point loop of every
 * instance, i.e. per evaluation of the error measures and the convergence test -- IPOPT's iteration table.  Row r describes
 * iterate r and the step taken from it (the convention of IPOPT's own table shifts the step columns down by one row; see
 * solver.format_history).  Rows are stored instance-major (B, capacity, OBCA_HIST_FIELDS), independent of obca_set_order.
 *
 *   #  field      value
 *   0  ITER       iteration counter at the head (it accumulates over the attempts of an instance)
 *   1  ATTEMPT    0 for the first interior-point run of the instance, +1 per restart (dual restoration or raise of rho)
 *   2  OBJ        objective f
 *   3  INF_PR     max |c|
 *   4  THETA      sum |c| (the filter's constraint-violation measure)
 *   5  INF_DU     max |grad f + J'y - zL + zU|
 *   6  COMPL      max complementarity gap * multiplier (at mu = 0)
 *   7  MU         barrier parameter at the head, before this iteration's update
 *   8  ERR        scaled overall error E_0 of the convergence test
 *   9  REG        delta_w of the inertia correction used for the step (0: none)
 *  10  D_NORM     max |dx|
 *  11  ALPHA_PR   accepted primal step (0 when the line search failed)
 *  12  ALPHA_DU   step of the bound multipliers (0 when the line search failed)
 *  13  LS_TRIALS  trial points evaluated by the filter line search (0 for a tiny step)
 *  14  FLAGS      OBCA_HIST_F_* bits
 *  15  RHO        elastic penalty weight in force
 *
 * A row without a step (the last head of a solve, a failed step computation) has NaN in fields 9..13.  Rows past the capacity are
 * not written but are counted; unwritten rows read back as NaN. */
#define OBCA_HIST_FIELDS 16
#define OBCA_HIST_ITER 0
#define OBCA_HIST_ATTEMPT 1
#define OBCA_HIST_OBJ 2
#define OBCA_HIST_INF_PR 3
#define OBCA_HIST_THETA 4
#define OBCA_HIST_INF_DU 5
#define OBCA_HIST_COMPL 6
#define OBCA_HIST_MU 7
#define OBCA_HIST_ERR 8
#define OBCA_HIST_REG 9
#define OBCA_HIST_D_NORM 10
#define OBCA_HIST_ALPHA_PR 11
#define OBCA_HIST_ALPHA_DU 12
#define OBCA_HIST_LS_TRIALS 13
#define OBCA_HIST_FLAGS 14
#define OBCA_HIST_RHO 15
#define OBCA_HIST_F_MU_LOWERED 1   /* mu was lowered at this head */
#define OBCA_HIST_F_INERTIA 2      /* inertia correction: delta_w > 0 */
#define OBCA_HIST_F_TINY_STEP 4    /* tiny-step rule: step accepted without line search */
#define OBCA_HIST_F_RESET 8        /* line search failed, barrier parameter raised again (barrier reset) */
#define OBCA_HIST_F_ACCEPTABLE 16  /* the iterate passed IPOPT's acceptable-point test */

/* rows kept per instance for the following obca_solve calls; 0 (default) turns recording off.  Takes B * capacity *
 * OBCA_HIST_FIELDS doubles of device memory from the stream-ordered pool, released by obca_destroy or a later call.
 * The debug entry points (obca_debug_*) do not record. */
int obca_set_history(ObcaHandle* h, int32_t capacity);
/* the record of the last obca_solve: rows (B, capacity, OBCA_HIST_FIELDS) dev, may be NULL; count (B) dev int32 = heads
 * evaluated (may exceed capacity), may be NULL.  An error when recording is off. */
int obca_get_history(ObcaHandle* h, double* rows, int32_t* count, void* stream);

/* number of kernels this handle has launched so far (bench.py "gpu_launches") */
int64_t obca_launch_count(const ObcaHandle* h);

/* ---- introspection used by the parity tests (tests/ only) ------------------------------------ */
/* internal flat layout: fills out[0..n) with the offsets/sizes documented in obca_core.h (Lay) */
int obca_layout(const ObcaHandle* h, int64_t* out, int n);
/* raw internal vectors of instance b, copied to HOST buffers (NULL = skip):
 * x (nx), y (ny), zL (nx), zU (nx) */
int obca_debug_get_iterate(ObcaHandle* h, int b, double* x, double* y, double* zL, double* zU);
int obca_debug_set_iterate(ObcaHandle* h, int b, const double* x, const double* y, const double* zL, const double* zU);
/* evaluate at the stored iterate of instance b: c (ny), gl = grad f + J'y (nx), f -> host */
int obca_debug_eval(ObcaHandle* h, int b, double* c, double* gl, double* f);
/* Newton step at the stored iterate for barrier mu and regularisation delta_w: dx (nx), dy (ny) -> host;
 * returns 1 in *ok when the reduced Hessian was positive definite */
int obca_debug_step(ObcaHandle* h, int b, double mu, double delta_w, double* dx, double* dy, int32_t* ok);

/* K [dx; dy] at the stored iterate of instance b (collocation mode), K = [[W + Sigma + delta_w I, J'], [J, -delta_c]] applied
 * matrix-free by obca_refine.h: dx (nx), dy (ny) in -> r1 (nx), r2 (ny) out, all HOST buffers in the internal layout.
 * Sigma = zL / (x - xL) + zU / (xU - x) from the stored iterate. */
int obca_debug_kkt_apply(ObcaHandle* h, int b, double delta_w, const double* dx, const double* dy, double* r1, double* r2);

/* per-phase SM cycle counters summed over the resident CTAs (filled when the environment variable OBCA_PROFILE is set
 * at solve time; phase ids in obca_core.h) */
int obca_debug_profile(ObcaHandle* h, int64_t* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* OBCA_H_ */
