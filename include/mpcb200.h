/*
 * mpcb200.h -- C ABI of the B200-native batched receding-horizon OCP solver.
 *
 * This is the drop-in boundary for the ONE hot path of rst-tu-dortmund/mpc_local_planner:
 * everything below Controller::step() (reference: mpc_local_planner/include/mpc_local_planner/controller.h:61-104,
 * mpc_local_planner/src/controller.cpp:102-179), i.e. the OCP transcription (FiniteDifferencesGridSE2::createEdges,
 * src/optimal_control/finite_differences_grid_se2.cpp:36-152), the hypergraph derivative assembly and the
 * interior-point solve that the reference delegates to control_box_rst + Ipopt (src/controller.cpp:380-421).
 *
 * Plain C, plain pointers and sizes; no C++/torch types cross this boundary. All floating point is IEEE double.
 * All host arrays are row-major "[instance][k][component]" unless stated otherwise.
 * A handle owns one CUDA device's workspace; it is NOT thread-safe (same contract as Controller::step,
 * which is not re-entrant: src/controller.cpp:111-179 mutates the grid).  Functions return 0 on success and a
 * negative MPCB200_E_* code on failure; they never throw and never abort (reference convention: bool return,
 * no exception crosses step(), src/controller.cpp:114-123,172,178).
 */
#ifndef MPCB200_H_
#define MPCB200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define MPCB200_VERSION 100

/* ---- enums (ints in the struct so that ctypes/cgo bindings are trivial) -------------------------------- */

/* robot/type (src/controller.cpp:344-378) */
#define MPCB200_ROBOT_UNICYCLE 0          /* inc/systems/unicycle_robot.h:59-68 */
#define MPCB200_ROBOT_SIMPLE_CAR 1        /* inc/systems/simple_car.h:68-77  (rear wheel driving) */
#define MPCB200_ROBOT_SIMPLE_CAR_FRONT 2  /* inc/systems/simple_car.h:131-141 */
#define MPCB200_ROBOT_KIN_BICYCLE 3       /* inc/systems/kinematic_bicycle_model.h:65-77 */

/* grid/cost_integration_method (src/controller.cpp:318-333) */
#define MPCB200_COST_LEFT_SUM 0
#define MPCB200_COST_TRAPEZOIDAL 1
/* grid/collocation_method (src/controller.cpp:298-316) */
#define MPCB200_COLLOC_FORWARD 0   /* inc/optimal_control/fd_collocation_se2.h:54-69 (default, every shipped config) */
#define MPCB200_COLLOC_MIDPOINT 1  /* :91-108  f at the mean pose of the interval (heading by interpolate_angle) */
#define MPCB200_COLLOC_CRANK_NICOLSON 2 /* :130-147 -- not implemented: create() returns E_UNSUPPORTED (SURVEY App. C.1: the reference's code and its documentation disagree) */

/* planning/objective/type (src/controller.cpp:551-641) */
#define MPCB200_OBJ_MINIMUM_TIME 0            /* corbo::MinimumTime: J = (N-1)*dt */
#define MPCB200_OBJ_QUADRATIC_FORM 1          /* QuadraticFormCostSE2, src/optimal_control/quadratic_cost_se2.cpp:31-52 */
#define MPCB200_OBJ_MINIMUM_TIME_VIA_POINTS 2 /* src/optimal_control/min_time_via_points_cost.cpp:40-145 */

/* footprint_model/type (src/mpc_local_planner_ros.cpp:890-1028) */
#define MPCB200_FOOTPRINT_POINT 0
#define MPCB200_FOOTPRINT_CIRCULAR 1    /* params[0] = radius */
#define MPCB200_FOOTPRINT_TWO_CIRCLES 2 /* params = front_offset, front_radius, rear_offset, rear_radius */
#define MPCB200_FOOTPRINT_LINE 3        /* params = start.x, start.y, end.x, end.y (robot frame) */
#define MPCB200_FOOTPRINT_POLYGON 4     /* n_poly vertices in poly_xy (robot frame), closing edge implied */

/* obstacle types (teb_local_planner obstacles; SURVEY App. B.3) */
#define MPCB200_OBST_POINT 0  /* params: x, y */
#define MPCB200_OBST_CIRCLE 1 /* params: x, y, -, -, radius */
#define MPCB200_OBST_LINE 2   /* params: x0, y0, x1, y1 */

/* per-instance solver status written to status[] */
#define MPCB200_STATUS_CONVERGED 0       /* scaled KKT error <= tol */
#define MPCB200_STATUS_MAX_ITER 1        /* iteration cap hit (reference: EarlyTerminated => step() still returns true) */
#define MPCB200_STATUS_NUMERICAL_ERROR 2 /* inertia correction or line search failed */
#define MPCB200_STATUS_INVALID_INPUT 3   /* NaN/inf in the instance's inputs */

/* error codes */
#define MPCB200_OK 0
#define MPCB200_E_INVALID -1     /* bad argument / config */
#define MPCB200_E_UNSUPPORTED -2 /* feature of the reference that this build does not implement */
#define MPCB200_E_CUDA -3        /* CUDA runtime error (message in mpcb200_last_error) */
#define MPCB200_E_NOMEM -4
#define MPCB200_E_NODEVICE -5    /* no CUDA device: there is NO CPU fallback */

#define MPCB200_MAX_POLY 16
#define MPCB200_OBST_STRIDE 7    /* doubles per obstacle in mpcb200_obstacles.params */
#define MPCB200_INF 1e30         /* |bound| >= this means "no bound" (corbo CORBO_INF_DBL sentinel, SURVEY App. B.1) */

/*
 * Solver/OCP configuration shared by all instances of a handle.  Field names and defaults follow the reference's
 * ROS parameter keys (SURVEY App. D; src/controller.cpp:225-805).  mpcb200_default_config() fills the in-code
 * defaults of the reference.
 */
typedef struct mpcb200_config {
    /* robot (src/controller.cpp:344-378, 494-549, 733-800) */
    int robot_type;
    double wheelbase;      /* simple_car/wheelbase (0.5) */
    double length_rear;    /* kinematic_bicycle_vel_input/length_rear (1.0) */
    double length_front;   /* kinematic_bicycle_vel_input/length_front (1.0) */
    double u_lb[2];        /* control lower bounds: (-max_vel_x_backwards, -max_vel_theta | -max_steering_angle) */
    double u_ub[2];        /* control upper bounds */
    double du_lb[2];       /* control-rate lower bounds (-dec_lim_x, -acc_lim_theta|-max_steering_rate); <= -MPCB200_INF: off */
    double du_ub[2];       /* control-rate upper bounds; >= MPCB200_INF: off */
    /* grid (src/controller.cpp:225-342) */
    int n;                 /* grid/grid_size_ref: number of grid points N (x_0 .. x_{N-1}) */
    double dt_ref;         /* grid/dt_ref */
    int variable_dt;       /* grid/variable_grid/enable: dt is a decision variable (one shared dt) */
    double dt_lb, dt_ub;   /* grid/variable_grid/{min_dt,max_dt} */
    int xf_fixed[3];       /* grid/xf_fixed */
    int collocation;       /* grid/collocation_method */
    int warm_start;        /* grid/warm_start (fixed-dt grid only; the variable grid disables the shift,
                              inc/optimal_control/finite_differences_variable_grid_se2.h:85) */
    /* objective (src/controller.cpp:551-674) */
    int objective;
    double Q[9], R[4];     /* quadratic_form state/control weights, row-major full matrices */
    int terminal_cost;     /* planning/terminal_cost/type == "quadratic" */
    double Qf[9];
    double vp_position_weight;    /* minimum_time_via_points/position_weight */
    double vp_orientation_weight; /* .../orientation_weight (linear in the wrapped angle, SURVEY App. C.4) */
    int vp_ordered;               /* .../via_points_ordered */
    int vp_attraction_with_quadratic; /* EXTENSION (SURVEY 8d cfg 4 reading A): add the via-point attraction term to quadratic_form */
    /* collision avoidance (src/controller.cpp:711-729) */
    double min_obstacle_dist, force_inclusion_dist, cutoff_dist;
    int footprint_type;
    double footprint_params[4];
    int n_poly;
    double poly_xy[2 * MPCB200_MAX_POLY];
    int k_max_obstacles_per_stage; /* fixed row budget K per stage on the device (masked rows are exact no-ops) */
    /* solver (src/controller.cpp:380-421): the interior-point method replaces Ipopt */
    int max_iter;          /* solver/ipopt/iterations (100) */
    double tol;            /* scaled KKT error tolerance; "converged" <=> error <= tol */
    double mu_init;        /* initial barrier parameter; > 0: as given (Ipopt's mu_init, default there 0.1); 0 (default): chosen per
                              instance, |f(x_0)| / #rows clamped to [0.1, 1] (DESIGN.md, "initial barrier parameter") */
    int outer_iterations;  /* controller/outer_ocp_iterations */
    /* planning/objective/quadratic_form/integral_form (src/controller.cpp:593-594): the running cost enters as
       sum_k dt * l(x_k, u_k) (grid/cost_integration_method left_sum, finite_differences_grid_se2.cpp:66-70) or by the
       trapezoidal rule (`cost_integration` below).  Default 0 = every shipped configuration. */
    int quadratic_integral_form;
    /* planning/terminal_constraint (src/controller.cpp:676-709): type "l2_ball" = TerminalBallSE2, one inequality row on the
       final state, d' S d - gamma <= 0 with d = x_{N-1} - x_f (theta wrapped), final_state_conditions_se2.cpp:54-64;
       gamma is the configured `radius` passed through unchanged (controller.cpp:702-703).  Ignored when x_f is fully fixed. */
    /* Solver-side choice of the cold initial guess (not in the reference, which starts from the straight line start -> goal,
       full_discretization_grid_base_se2.cpp:192-239): among the 2n+1 laterally bumped lines
       p_k + 0.4 m * sin(pi k/(N-1)) n_perp, m = -n..n, the one that violates the obstacle clearances least is taken (the
       straight line itself whenever it is clear).  Only when no initial plan is supplied.  0 = always the straight line.
       Default 4 (DESIGN.md, "cold initial guess"). */
    int initial_guess_bumps;
    /* collision_avoidance/enable_dynamic_obstacles (src/controller.cpp:721-723): obstacles with a non-zero velocity are kept
       at every stage (stage_inequality_se2.cpp:99-106) and their rows use the position predicted at t = k dt with constant
       velocity (teb estimateSpatioTemporalDistance, stage_inequality_se2.cpp:177-189).  Default 0 (the reference's). */
    int enable_dynamic_obstacles;
    int terminal_ball;
    double terminal_ball_S[9];
    double terminal_ball_gamma;
    /* grid/cost_integration_method (src/controller.cpp:318-333), used by the integral form only:
       MPCB200_COST_LEFT_SUM (default)  sum_{k<=N-2} dt l(x_k, u_k)                        (finite_differences_grid_se2.cpp:66-70)
       MPCB200_COST_TRAPEZOIDAL         sum_{k<=N-2} dt/2 ( l(x_k, u_k) + l(x_{k+1}, u_k) ) (finite_differences_grid_se2.cpp:59-65;
       corbo's TrapezoidalIntegralCostEdge evaluates both ends with the control of the interval). */
    int cost_integration;
    /* planning/objective/quadratic_form/hybrid_cost_minimum_time (src/controller.cpp:595-620): adds the minimum-time term
       (N-1) dt to the quadratic control cost.  As in the reference it takes effect only with zero state weights Q and
       non-zero control weights R (and needs variable_dt); with any other weights the plain quadratic form is used. */
    int hybrid_cost_minimum_time;
    /* Cold initial guess exactly as the reference builds it (full_discretization_grid_base_se2.cpp:192-239: states on the
       straight line start -> goal or on the supplied plan, zero controls, dt = dt_ref): 1 switches the solver-side
       preprocessing off -- no choice among bumped lines (initial_guess_bumps is ignored), no repair of poses that violate
       obstacle rows, no control seeding.  Default 0: the preprocessing is ON, i.e. the default cold start is NOT the
       reference's; it is the one that lets 99.7 % instead of ~60 % of the BASELINE instances converge within the
       reference's 100 iterations (DESIGN.md "cold initial guess").  A locally convergent method inherits the homotopy class of
       its starting point, so the two modes may return different local optima of the same problem. */
    int reference_initial_guess;
} mpcb200_config;

/* Per-instance obstacle lists, fixed stride: instance b owns obstacles [b*max_per_instance, b*max_per_instance+count[b]).
 * max_per_instance <= 2048.  Lists of up to 64 slots are resident with the instance; longer lists (the raw costmap lists of
 * updateObstacleContainerWithCostmap) stay in these arrays on the device and the association (StageInequalitySE2::update,
 * stage_inequality_se2.cpp:73-147) copies what it selects for some stage into the 64 resident slots.  A selection that does not
 * fit any more is dropped and counted in MPCB200_SC_OBST_DROPPED (k_max_obstacles_per_stage x (n-2) <= 64 can never drop). */
typedef struct mpcb200_obstacles {
    int max_per_instance;
    const int* count;      /* [B] */
    const int* type;       /* [B*max_per_instance] MPCB200_OBST_* */
    const double* params;  /* [B*max_per_instance*MPCB200_OBST_STRIDE]: x0, y0, x1, y1, radius, vx, vy (velocity: dynamic obstacles) */
} mpcb200_obstacles;

/* Per-instance via-points (teb PoseSE2 list handed to Controller::configure, inc/controller.h:61-63). */
typedef struct mpcb200_viapoints {
    int max_per_instance;
    const int* count;      /* [B] */
    const double* poses;   /* [B*max_per_instance*3]: x, y, theta */
} mpcb200_viapoints;

typedef struct mpcb200_handle mpcb200_handle;

/* Fills *cfg with the reference's in-code defaults (SURVEY App. D): unicycle, N=20, dt_ref=0.3, minimum_time ... */
void mpcb200_default_config(mpcb200_config* cfg);

/*
 * Replaces Controller::configure (inc/controller.h:61-63, src/controller.cpp:58-100): validates the configuration,
 * selects `device`, allocates the device workspace for up to max_batch instances.
 */
int mpcb200_create(const mpcb200_config* cfg, int max_batch, int device, mpcb200_handle** out);

/*
 * Replaces Controller::step (inc/controller.h:65-67, src/controller.cpp:111-179) for a batch of B independent
 * instances.  Per instance: x0 = measured state (start pose), xf = goal pose, u_prev/u_prev_dt = previously applied
 * control and its age (StructuredOptimalControlProblem::setPreviousControlInput, src/mpc_local_planner_ros.cpp:384).
 *   x_init  optional [B][N][3] initial state guess (reference: _x_seq_init sampled at k*dt, src/controller.cpp:807-857);
 *           NULL => straight line start->goal with angle-aware linear interpolation (what the reference produces for
 *           a 2-pose plan).
 *   reinit  optional [B]: non-zero forces a cold re-initialisation of that instance (grid->clear(), src/controller.cpp:152-158);
 *           NULL => cold start on the first call after create/reset, warm start afterwards when cfg.warm_start.
 * Outputs (any may be NULL): u_seq [B][N][2] (last control duplicated, full_discretization_grid_base_se2.cpp:591-614),
 *   x_seq [B][N][3], dt_out [B], status [B], kkt_err [B] (final scaled KKT error), iters [B], solve_time_s [1]
 *   (device time of the whole batch, the analogue of OptimalControlResult.cpu_time).
 * Host pointers may be pageable or pinned; host<->device copies happen inside this call.
 */
int mpcb200_step_batch(mpcb200_handle* h, int B, const double* x0, const double* xf, const double* u_prev,
                       double u_prev_dt, const mpcb200_obstacles* obst, const mpcb200_viapoints* vp,
                       const double* x_init, const unsigned char* reinit, double* u_seq, double* x_seq,
                       double* dt_out, int* status, double* kkt_err, int* iters, double* solve_time_s);

/*
 * The same solves for a QUEUE of `total` instances (total may exceed max_batch by any factor): the handle's max_batch
 * workspaces form a pool of slots, and a slot whose instance has finished hands its result over and takes the next
 * instance of the queue while the other slots keep iterating (continuous batching).  The interior-point iterations of
 * different instances are independent, so every instance gets exactly the result mpcb200_step_batch would give it from a
 * cold start; what changes is the cost: a batch pays max-over-instances iterations, the pool pays the mean.
 * Arrays as in mpcb200_step_batch with B = total; always a cold start, no x_init / reinit; outer_iterations must be 1.
 * The queue has device arrays of its own: the resident batch (its inputs, its warm state and its iteration history) is left
 * as it was, and mpcb200_solve_resident / mpcb200_fetch_results afterwards see the batch of the last upload.
 */
int mpcb200_solve_stream(mpcb200_handle* h, int total, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                         const mpcb200_obstacles* obst, const mpcb200_viapoints* vp, double* u_seq, double* x_seq, double* dt_out,
                         int* status, double* kkt_err, int* iters, double* solve_time_s);

/* Replaces Controller::reset (inc/controller.h:104): which == NULL resets every instance, else those with which[b] != 0. */
int mpcb200_reset(mpcb200_handle* h, const unsigned char* which, int B);

/*
 * Horizon change of the whole batch: replaces FullDiscretizationGridBaseSE2::resampleTrajectory(n_new)
 * (src/optimal_control/full_discretization_grid_base_se2.cpp:440-524), the operation behind the grid adaptation of the
 * variable grid (FiniteDifferencesVariableGridSE2::adaptGridTimeBasedSingleStep,
 * src/optimal_control/finite_differences_variable_grid_se2.cpp:99-121: n + 1 when the optimised dt exceeds
 * dt_ref (1 + dt_hyst_ratio), n - 1 when it falls below dt_ref (1 - dt_hyst_ratio); the policy itself lives with the caller,
 * include/mpcb200_controller.hpp).  Every warm trajectory of the handle is resampled on the device to n_new grid points
 * over the same horizon time (dt becomes dt (n-1)/(n_new-1)); empty (reset / never solved) instances just take the new
 * horizon.  From the next mpcb200_step_batch on every per-instance array has n_new samples.  All instances of a handle
 * share the horizon: robots that adapt independently are grouped by n (one handle per group).
 * n_new must lie in [3, n the handle was created with] -- create the handle with config.n = grid/variable_grid/
 * grid_adaptation/max_grid_size and call mpcb200_resample(h, grid_size_ref) once before the first step.
 */
int mpcb200_resample(mpcb200_handle* h, int n_new);
/* current horizon and the capacity (config.n at create) */
int mpcb200_get_horizon(const mpcb200_handle* h, int* n, int* n_capacity);

/*
 * Costmap -> point obstacles for B robots: replaces MpcLocalPlannerROS::updateObstacleContainerWithCostmap
 * (src/mpc_local_planner_ros.cpp:474-499).  Every LETHAL cell (costmap_2d::LETHAL_OBSTACLE = 254) of the cells
 * mx = 0..size_x-2, my = 0..size_y-2 (the reference's loop bounds) becomes a point obstacle at the cell centre
 * (Costmap2D::mapToWorld: origin + (m + 0.5) resolution) unless it lies behind the robot (negative projection on the heading)
 * AND farther than behind_robot_dist (costmap_obstacles_behind_robot_dist).  Order = the reference's push_back order
 * (mx outer, my inner).  Outputs in the layout of mpcb200_obstacles with max_per_instance slots per robot:
 * count[b] = obstacles written = min(found[b], max_per_instance); found[b] = cells that qualified (found > count: the list was
 * cut); velocities 0.
 */
typedef struct mpcb200_costmaps {
    int size_x, size_y;          /* cells: Costmap2D::getSizeInCellsX / Y */
    double resolution;           /* metres per cell */
    const double* origin;        /* [B*2] world coordinates of the lower-left corner of cell (0,0): getOriginX / Y */
    const unsigned char* cost;   /* [B*size_y*size_x], cell (mx, my) at my*size_x + mx (Costmap2D::getIndex) */
} mpcb200_costmaps;
int mpcb200_costmap_obstacles(mpcb200_handle* h, int B, const mpcb200_costmaps* maps, const double* robot_pose /*[B*3]*/,
                              double behind_robot_dist, int max_per_instance, int* count /*[B]*/, int* found /*[B] or NULL*/,
                              int* type /*[B*max]*/, double* params /*[B*max*MPCB200_OBST_STRIDE]*/);

/* One planning cycle from the costmaps for B robots: updateObstacleContainerWithCostmap (mpc_local_planner_ros.cpp:474-499, robot
 * pose = x0) followed by Controller::step, as MpcLocalPlannerROS::computeVelocityCommands chains them (mpc_local_planner_ros.cpp:
 * 330-412).  The obstacle lists never leave the device: maps H2D -> extraction into the batch's obstacle arrays -> association
 * over the lists in global memory (up to 2048 per robot) -> solve.  obst_found[b] (optional) = cells that qualified; lists are cut
 * at max_per_instance.  Other arguments and results as mpcb200_step_batch. */
int mpcb200_step_batch_costmap(mpcb200_handle* h, int B, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                               const mpcb200_costmaps* maps, double behind_robot_dist, int max_per_instance, const mpcb200_viapoints* vp,
                               const double* x_init, const unsigned char* reinit, double* u_seq, double* x_seq, double* dt_out, int* status,
                               double* kkt_err, int* iters, int* obst_found, double* solve_time_s);
/*
 * Footprint-vs-costmap feasibility of the planned poses for B robots: replaces Controller::isPoseTrajectoryFeasible
 * (src/controller.cpp:859-917; caller src/mpc_local_planner_ros.cpp:414-428, which resets the planner on a rejection).
 * The footprint polygon (footprint_xy: n_footprint points in the robot frame = costmap_2d's footprint spec; fewer than 3 points
 * = "circular robot": only the centre cell is looked up) is laid over the robot's costmap at poses 0..look_ahead_idx of its
 * trajectory (look_ahead_idx < 0 or >= n: all poses = collision_check_no_poses -1) and, wherever two consecutive poses are
 * farther apart than inscribed_radius or turn by more than min_resolution_angular (collision_check_min_resolution_angular), at
 * evenly spaced poses in between.  feasible[b] = 0 iff some footprint cost is -1 (a LETHAL cell under an edge, or the centre
 * outside the map) -- exactly the reference's test (footprint vertices outside the map and unknown cells do not reject).
 *   x_seq  [B][n_poses][3] host trajectories, or NULL: the trajectories of the last solve, read on the device (n = config.n).
 * circumscribed_radius is accepted for signature parity (base_local_planner::CostmapModel::footprintCost ignores it too).
 */
int mpcb200_check_feasible(mpcb200_handle* h, int B, const mpcb200_costmaps* maps, const double* x_seq, int n_poses,
                           const double* footprint_xy, int n_footprint, double inscribed_radius, double circumscribed_radius,
                           double min_resolution_angular, int look_ahead_idx, unsigned char* feasible /*[B]*/);
/* device time (ms, CUDA events around the three kernels) of the last mpcb200_costmap_obstacles call */
double mpcb200_costmap_last_ms(const mpcb200_handle* h);

void mpcb200_destroy(mpcb200_handle* h);

/* Last error message of this handle (or of create() when h == NULL). Never NULL. */
const char* mpcb200_last_error(const mpcb200_handle* h);

/* ---- several devices of one node behind one handle (SURVEY 8e) ------------------------------------------------ */
/*
 * Instances are independent: the batch is cut into contiguous blocks, device r of the list solves instances
 * [r ceil(B/G), (r+1) ceil(B/G)) with its own workspace on its own stream (one host thread per device inside the call), and ONE
 * NCCL all-gather over NVLink / NVSwitch then leaves the packed optimal controls of the WHOLE batch on every device
 * (mpcb200_multi_device_controls: [G][ceil(B/G)][N-1][2] doubles, the slots behind B unused).  No other collective.  Per instance
 * the arithmetic is the single-device one: G-device results equal the 1-device results bit for bit.
 * NCCL is loaded at run time (dlopen "libnccl.so.2") when n_devices > 1; MPCB200_E_UNSUPPORTED if it cannot be loaded.
 */
typedef struct mpcb200_multi mpcb200_multi;
int mpcb200_create_multi(const mpcb200_config* cfg, int max_batch_total, const int* devices, int n_devices, mpcb200_multi** out);
/* same arguments as mpcb200_step_batch, for the whole batch; solve_time_s = the slowest device's device time */
int mpcb200_step_batch_multi(mpcb200_multi* m, int B, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                             const mpcb200_obstacles* obst, const mpcb200_viapoints* vp, const double* x_init, const unsigned char* reinit,
                             double* u_seq, double* x_seq, double* dt_out, int* status, double* kkt_err, int* iters, double* solve_time_s);
/* the gathered controls on device `rank` of the list (device pointer) and their size in doubles */
int mpcb200_multi_device_controls(mpcb200_multi* m, int rank, void** dev_ptr, long long* n_doubles);
/* copy of that buffer to the host (n_doubles doubles) */
int mpcb200_multi_fetch_controls(mpcb200_multi* m, int rank, double* host);
/* the single-device handle of device `rank` (reset, resample, options, statistics ...) */
mpcb200_handle* mpcb200_multi_handle(mpcb200_multi* m, int rank);
void mpcb200_destroy_multi(mpcb200_multi* m);
const char* mpcb200_multi_last_error(const mpcb200_multi* m);

/* ---- device-resident variant (inputs already in HBM; used by bench.py's kernel-only `value`) ----------- */

/*
 * Stage the inputs of a batch on the device once (same arguments as mpcb200_step_batch), then
 * mpcb200_solve_resident() re-runs init + association + solve from those resident inputs without any
 * host<->device traffic, and mpcb200_fetch_results() copies the results back.
 */
int mpcb200_upload_inputs(mpcb200_handle* h, int B, const double* x0, const double* xf, const double* u_prev,
                          double u_prev_dt, const mpcb200_obstacles* obst, const mpcb200_viapoints* vp,
                          const double* x_init);
int mpcb200_solve_resident(mpcb200_handle* h, int cold, double* solve_time_s);
int mpcb200_fetch_results(mpcb200_handle* h, double* u_seq, double* x_seq, double* dt_out, int* status,
                          double* kkt_err, int* iters);
/* Device pointer of the packed optimal controls [B][N-1][2] (for the NCCL all-gather of u*, SURVEY 8e) and its size. */
int mpcb200_device_controls(mpcb200_handle* h, void** dev_ptr, long long* n_doubles);
/* Device-to-device copy of the packed optimal controls into a caller-owned device buffer (e.g. the send buffer of the
   NCCL all-gather).  dst must hold B*(N-1)*2 doubles on the handle's device. */
int mpcb200_export_controls(mpcb200_handle* h, void* dst_dev);
/* Evict the L2 cache (writes a 320 MB scratch buffer); used between timed launches by the benchmark. */
int mpcb200_flush_l2(mpcb200_handle* h);

/* ---- kernel-level access: parity tests and the roofline measurement ------------------------------------ */

/* Workspace fields, each stored per instance as [component][k] (k = stage index 0..N-1, fastest). */
#define MPCB200_F_X 0      /* 3 x N   states */
#define MPCB200_F_U 1      /* 2 x N   controls (k = N-1 unused) */
#define MPCB200_F_NU 2     /* 3 x N   multipliers of the dynamics defects (k = N-1 unused) */
#define MPCB200_F_S 3      /* RS x N  slacks of the inequality rows, RS = 8 + K */
#define MPCB200_F_LAM 4    /* RS x N  multipliers of the inequality rows */
#define MPCB200_F_KKT 5    /* 42 x N  condensed KKT stage records (see DESIGN.md "KKT record") */
#define MPCB200_F_STEP 6   /* 8 x N   Newton step: dw (5), nu_plus (3) */
#define MPCB200_F_SCAL 7   /* 24      per-instance scalars (see MPCB200_SC_*) */
#define MPCB200_F_OBSIDX 8 /* K x N   associated obstacle per row slot as double: its RESIDENT slot (-1 = empty); = its list index for
                              lists of at most 64 obstacles */
#define MPCB200_F_OBSGIDX 9 /* 64      list index of each resident obstacle (lists of more than 64 obstacles), -1 = free slot */
#define MPCB200_KKT_WORDS 42
/* offsets inside one KKT stage record (DESIGN.md "KKT record"); stage k = 0..N-2, terminal data at k = N-1 */
#define MPCB200_K_H 0    /* 15: upper triangle (row-major) of the condensed 5x5 Hessian block of w_k = (x_k, u_k) */
#define MPCB200_K_G 15   /* 5 : condensed gradient */
#define MPCB200_K_A 20   /* 3 : dt * df/dtheta  (A_k = I + a e_theta^T) */
#define MPCB200_K_B 23   /* 6 : dt * df/du, row-major 3x2 */
#define MPCB200_K_E 29   /* 3 : defect e_k = x_k + dt f(x_k,u_k) - x_{k+1} */
#define MPCB200_K_C 32   /* 2 : diagonal of the cross block d2L/du_{k-1} du_k (control-rate rows) */
#define MPCB200_K_HB 34  /* 5 : border column d2L/dw_k d(dt) */
#define MPCB200_K_D 39   /* 3 : de_k/d(dt) = f(x_k,u_k) */
#define MPCB200_STEP_WORDS 8
#define MPCB200_SCAL_WORDS 32
/* indices into the SCAL field */
#define MPCB200_SC_DT 0
#define MPCB200_SC_MU 1
#define MPCB200_SC_RHO 2
#define MPCB200_SC_DELTA 3
#define MPCB200_SC_HTT 4
#define MPCB200_SC_GT 5
#define MPCB200_SC_DDT 6
#define MPCB200_SC_ERR0 7    /* scaled KKT error E_0 */
#define MPCB200_SC_ERRMU 8   /* barrier-problem error E_mu */
#define MPCB200_SC_ITER 9
#define MPCB200_SC_STATUS 10
#define MPCB200_SC_ALPHA 11
#define MPCB200_SC_OBJ 12
#define MPCB200_SC_INF 13    /* l1 infeasibility */
#define MPCB200_SC_DELTA_LAST 14
#define MPCB200_SC_NREG 15   /* number of inertia-correction refactorisations so far */
#define MPCB200_SC_BLOG 16   /* sum of log(slack) over active rows */
#define MPCB200_SC_GLDT 17   /* dL/d(dt) */
#define MPCB200_SC_NBT 18    /* line-search backtracks so far */
#define MPCB200_SC_COLD 19   /* 1 until the instance has been solved once (cold start pending) */
#define MPCB200_SC_VALID 22   /* 1 = the inputs of the instance are finite (else status INVALID_INPUT, never iterated) */
#define MPCB200_SC_OBST_DROPPED 23 /* long obstacle lists: selected obstacles that did not fit into the 64 resident slots */
#define MPCB200_SC_DEFER 21  /* 1 = the KKT phase spent its factorisation budget: null step, regularisation resumes next iteration */
#define MPCB200_SC_TINY 20   /* consecutive iterations with a step length below 1e-8 (2 => the instance is given up) */

int mpcb200_ws_count(const mpcb200_handle* h, int field);  /* number of components of a field (e.g. RS) */
int mpcb200_ws_read(mpcb200_handle* h, int field, int B, double* dst);        /* dst: [B][count][N] (SCAL: [B][MPCB200_SCAL_WORDS]) */
int mpcb200_ws_write(mpcb200_handle* h, int field, int B, const double* src);

/* phases of one solve, launchable one by one */
#define MPCB200_PHASE_INIT 0       /* cold initial guess + slack/multiplier initialisation */
#define MPCB200_PHASE_ASSOCIATE 1  /* obstacle / via-point association (StageInequalitySE2::update) */
#define MPCB200_PHASE_EVAL 2       /* stage functions + derivatives -> condensed KKT records, KKT error */
#define MPCB200_PHASE_KKT 3        /* block-tridiagonal Riccati factorisation + solve -> Newton step */
#define MPCB200_PHASE_LINESEARCH 4 /* step lengths, merit line search, iterate + barrier update */
#define MPCB200_NUM_PHASES 5
int mpcb200_run_phase(mpcb200_handle* h, int phase, int B);
/* Launch `phase` reps times back to back and report the mean device time per launch (CUDA events on the solver stream). */
int mpcb200_time_phase(mpcb200_handle* h, int phase, int B, int reps, int flush_l2, double* ms_per_launch);
/* Phased solve mode only: which phases a solve brackets with CUDA events for mpcb200_stats.ms (bit p = phase p).  Default: the
   KKT phase only (1 << MPCB200_PHASE_KKT) -- every bracket costs a few microseconds of stream time; 0x1f times all of them.
   (The fused solve kernel counts SM cycles per phase itself: mpcb200_stats.ms is then the mean time a CTA spent in the phase.) */
int mpcb200_set_timing(mpcb200_handle* h, unsigned phase_mask);
/* Run all work of this handle on the caller's CUDA stream (a cudaStream_t; NULL restores the handle's own stream), e.g. the
   stream the NCCL all-gather of the optimal controls is enqueued on.  The previous stream is drained first. */
int mpcb200_set_stream(mpcb200_handle* h, void* cuda_stream);
/* Execution options (never change results).  MPCB200_OPT_SOLVE_MODE: 0 (default) = one persistent kernel per solve -- a CTA owns
   an instance from the initial guess to convergence, all phases in shared memory; 1 = one kernel launch per phase, the host
   queues the iterations (the same device functions; per-phase CUDA-event timing, the KKT kernel measurable on its own). */
#define MPCB200_OPT_SOLVE_MODE 3
/* MPCB200_OPT_CTAS_PER_SM: cap on the CTAs of the solve kernel resident on one SM (0 = as many as fit; tuning / experiments). */
#define MPCB200_OPT_CTAS_PER_SM 4
/* MPCB200_OPT_SM_PHASE_SYNC: the CTAs of the solve kernel that share an SM enter each phase of the iteration together
   (instruction-cache locality; timing only).  -1 (default) = on when three or more CTAs fit on an SM, 0 = off, 1 = on with
   gates before evaluation, KKT and line search, 2 = on with gates before KKT and line search only. */
#define MPCB200_OPT_SM_PHASE_SYNC 5
/* MPCB200_OPT_ORDER_BY_HISTORY: 1 (default) = a batch solve takes its instances longest-first by the iteration counts the same
   slots needed in the previous batch solve of this handle (a batch costs its slowest instance; a robot that was hard in the last
   cycle tends to be hard in this one).  Order of execution only; 0 = index order. */
#define MPCB200_OPT_ORDER_BY_HISTORY 6
int mpcb200_set_option(mpcb200_handle* h, int option, int value);

/* Counters accumulated since the last mpcb200_stats_reset: kernels launched, device ms per phase. */
typedef struct mpcb200_stats {
    long long launches[MPCB200_NUM_PHASES];
    double ms[MPCB200_NUM_PHASES];
    long long launches_total;
    long long h2d_bytes, d2h_bytes;
    long long kkt_instances; /* number of (instance, iteration) pairs the KKT phase actually factorised */
    long long kkt_sweeps;    /* backward sweeps incl. inertia-correction refactorisations */
    double gate_ms;          /* mean time a CTA of the solve kernel waited for its SM neighbours (MPCB200_OPT_SM_PHASE_SYNC) */
} mpcb200_stats;
int mpcb200_stats_get(const mpcb200_handle* h, mpcb200_stats* out);
int mpcb200_stats_reset(mpcb200_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* MPCB200_H_ */
