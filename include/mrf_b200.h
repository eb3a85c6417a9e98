/* mrf_b200 -- C-ABI of the B200-native multi-robot-fabrics hot path.
 *
 * Drop-in boundary: these entry points are what a binding of the reference's planner call
 * surface calls instead of evaluating the CasADi functions.  The reference is pure Python; the
 * binding a maintainer adds is a ctypes stub (see INTEGRATION.md).  What each entry replaces
 * (paths relative to the reference repository root):
 *
 *   mrf_action_*          planner._funs._function / planner.compute_action(**kwargs)
 *                         examples/example_pandas_Jointspace.py:417-445,
 *                         multi_robot_fabrics/fabrics_planner/forward_planner_Cartesian.py:132-191
 *   mrf_rollout_*         ForwardFabricsPlanner.forward_multi_fabrics_symbolic + get_velocity_rollouts
 *                         + rollouts_numerical
 *                         multi_robot_fabrics/fabrics_planner/forward_planner_Jointspace.py:118-296,298-423
 *                         (with the RF-CV goal estimate of examples/example_pandas_Jointspace.py:346-348 and the
 *                         end-effector FK of :236-238,328-329 fused in)
 *   mrf_rollout_cart_*    FabricsRollouts.symbolic_forward_fabrics + rollouts_numerical + get_velocity_rollouts
 *                         multi_robot_fabrics/fabrics_planner/forward_planner_Cartesian.py:347-489,538-563
 *   mrf_rollout_cart_all_* the same for every robot of the handle in one launch: the per-robot FabricsRollouts calls of
 *                         examples/example_pandas_cartesian.py:361-418 (one rollouts_numerical per robot, each against
 *                         its own obstacle list)
 *   mrf_deadlock_*        deadlockprevention.deadlock_checking
 *                         multi_robot_fabrics/others_planner/deadlock_prevention.py:50-118
 *   mrf_kinematics_*      UtilsKinematics.necessary_kinematics fk/jac/jac_dot functions
 *                         multi_robot_fabrics/utils/utils.py:16-54 (as used at
 *                         examples/example_pandas_Jointspace.py:324-343)
 *   mrf_obstacles_*       define_symbolic_collision_link_poses sphere functions + compute_x_obsts_dyn_0 and the obstacle
 *                         assembly of the caller loop
 *                         multi_robot_fabrics/utils/utils.py:87-119, utils/utils_apply_fk.py:3-33,
 *                         examples/example_pandas_Jointspace.py:400-412
 *   mrf_point_action_*    point-mass planner compute_action (examples/example_pointmasses_static.py:102-129,191-199)
 *   mrf_point_episode_run_* the control loops of examples/example_pointmasses_static.py and _dynamic.py, many steps per call
 *   mrf_fsm_*             StateMachine.get_state_machine_panda + gripper action
 *                         multi_robot_fabrics/others_planner/state_machine.py:70-84,133-214
 *   mrf_episode_step_*    one iteration of the control loop examples/example_pandas_Jointspace.py:280-458 (coupled
 *                         joint-space rollouts) or examples/example_pandas_cartesian.py:295-462 (decoupled Cartesian rollouts,
 *                         MrfEpisode.rollout_model = 1)
 *   mrf_rollout_host_submit_* / _wait   get_velocity_rollouts for a stream of independent batches (sweeps)
 *
 * Conventions
 *  - Plain pointers and sizes; no exceptions cross the boundary.  Every function returns 0 on success or a
 *    negative MRF_E* code; mrf_last_error() gives the message of the calling thread's last failure.
 *  - "_dev" entries take DEVICE pointers owned by the caller, structure-of-arrays with the scenario index
 *    fastest (layouts below), and are asynchronous on the given cudaStream_t (passed as void*).
 *  - "_host" entries take HOST pointers in the reference's natural array-of-records order, copy to the device,
 *    run the same kernels and copy the results back (synchronous); page-locked rollout records are read by the kernel
 *    in place (see mrf_rollout_host_*).
 *  - There is no CPU fallback: without a CUDA device mrf_create fails with MRF_ENODEV.
 *  - A handle is not thread-safe; distinct handles are independent.
 */
#ifndef MRF_B200_H
#define MRF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRF_MAX_ROBOTS 4
#define MRF_DOF 7
#define MRF_NLINKS 8   /* panda_link1..8, examples/parameters_manipulators.py:25-26 */
#define MRF_REC 44     /* scalars per robot record */
#define MRF_OBST 10    /* scalars per obstacle sphere: x[3], xdot[3], xddot[3], radius */
#define MRF_GUARD_SLOTS 8   /* scratch slots of the mrf_rfcv_post_dev_f32 re-roll (concurrent post steps on different streams) */
#define MRF_MAX_STATIC 16   /* static spheres per robot in a coupled rollout (nr_obsts of the rollout planners) */
#define MRF_MAX_SPHERES_PER_LINK 8   /* n_obst_per_link, examples/configs/panda_config.yaml:8 (reference default 4) */
#define MRF_MAX_POINT_ROBOTS 8   /* point robots per scenario in mrf_point_episode_run_dev_* */

/* Per-robot record = the numeric arguments of one fabric action / of get_velocity_rollouts
 * (forward_planner_Jointspace.py:303-329), fixed order:
 *  [0..6] q  [7..13] qdot  [14..16] x_goal_0  [17] weight_goal_0  [18..20] x_goal_1  [21] weight_goal_1
 *  [22] x_goal_2  [23] weight_goal_2  [24..32] angle_goal_1 (row-major 3x3)  [33..36] constraint_0
 *  [37..42] radius_body_panda_link3..8  [43] reserved (0) */
enum { MRF_Q = 0, MRF_QD = 7, MRF_G0 = 14, MRF_W0 = 17, MRF_G1 = 18, MRF_W1 = 21, MRF_G2 = 22, MRF_W2 = 23,
       MRF_ANG = 24, MRF_CON = 33, MRF_RB = 37 };

enum { MRF_OK = 0, MRF_EINVAL = -1, MRF_ENODEV = -2, MRF_ECUDA = -3, MRF_ENOMEM = -4, MRF_EUNSUPPORTED = -5 };

/* Planner / rollout configuration (what the reference fixes at graph-construction time). */
typedef struct MrfConfig {
    int32_t struct_size;          /* sizeof(MrfConfig), ABI check */
    int32_t n_robots;             /* 1..MRF_MAX_ROBOTS */
    int32_t mode;                 /* 0 'acc', 1 'vel'  (planner.concretize(mode, time_step)) */
    int32_t static_or_dyn;        /* STATIC_OR_DYN_FABRICS (forward_planner_Jointspace.py:215-217) */
    int32_t has_collision_links;  /* 0: grasp planner, collision_links_nr=[] (example_pandas_Jointspace.py:160-166) */
    int32_t estimate_goal;        /* ESTIMATE_GOAL: 0 off, 1 Jacobian-column-0 "velocity" (example_pandas_Jointspace.py:
                                     236-238,346-348), 2 J*qdot (example_pandas_cartesian.py:355-357, utils.py:131) */
    int32_t estimate_robot;       /* robot whose goal is estimated (1 in the reference) */
    int32_t reserved0;
    double estimate_horizon;      /* 20 * 0.01 (example_pandas_Jointspace.py:347) */
    double dt;                    /* planner time_step == rollout dt (parameters_manipulators.py:8) */
    double eps;                   /* fabrics eps, 1e-6 */
    double jdot_sign;             /* fabrics DifferentialMap Jdot sign, -1 */
    double jdot_ref_sign;         /* utils.py:28 Jdot_sign, -1 (published sphere accelerations) */
    double exec_scale;            /* ExecutionLagrangian = exec_scale * qdot.qdot */
    double mount[MRF_MAX_ROBOTS][16];              /* row-major 4x4, example_pandas_Jointspace.py:108-118 */
    double limits[MRF_DOF][2];                     /* example_pandas_Jointspace.py:97-105 */
    double r_robots[MRF_MAX_ROBOTS][MRF_NLINKS];   /* sphere radii of each robot's links as seen by the others
                                                      (forward_planner_Jointspace.py:221) */
    /* deadlock heuristic constants, deadlock_prevention.py:20-27,64,66 */
    double dl_avg_vel_constant, dl_dist_constant, dl_goal_weight_follower, dl_goal_weight_leader;
    double dl_nr_goal_scale, dl_dist_endeff, dl_backoff;
    int32_t dl_time_wait, dl_time_gate;
    /* collision_links_nr of set_planner_panda (example_pandas_Jointspace.py:64,91-96,141-166) per robot: bit l-1 set <=>
     * panda_link l is a collision link.  As ego links only link3..8 carry leaves (link1/2 have a constant fk); as
     * obstacles of the other robots' rollouts every listed link is a sphere.  Default 0xFF (all eight links). */
    int32_t collision_link_mask[MRF_MAX_ROBOTS];
} MrfConfig;

typedef struct MrfHandle_* mrf_handle_t;

int mrf_version(void);
/* Message of the last failure ON THE CALLING THREAD (thread-local storage, not per handle: it also reports failures
 * of calls that have no handle yet, e.g. mrf_create). Valid until the same thread's next failing call. */
const char* mrf_last_error(void);
int mrf_config_default(MrfConfig* cfg, int n_robots);       /* the reference's 2/3-Panda set-up */
int mrf_create(const MrfConfig* cfg, int device, mrf_handle_t* out);
int mrf_destroy(mrf_handle_t h);
int mrf_device_count(void);

/* ------------------------------- device-pointer entries (SoA) ---------------------------------
 * B = number of scenarios, R = robots in the call, index b fastest:
 *   rec    [MRF_REC][R][B]
 *   obst   [S][MRF_OBST][R][B]          obstacle o of robot r in scenario b
 *   action [MRF_DOF][R][B]
 *   avg_vel[R][B]   x_ee [R][3][B]   goal_est [3][B] (x_goal_0 of robot `estimate_robot` as the rollout used it)
 *   qN, qdN [R][N][MRF_DOF][B]          (nullable)
 */
int mrf_action_dev_f64(mrf_handle_t h, int robot_first, int n_rob, const double* rec, int S, const double* obst,
                       double* action, int64_t B, void* stream);
int mrf_action_dev_f32(mrf_handle_t h, int robot_first, int n_rob, const float* rec, int S, const float* obst,
                       float* action, int64_t B, void* stream);

int mrf_rollout_dev_f64(mrf_handle_t h, const double* rec, int N, double* avg_vel, double* x_ee, double* goal_est,
                        double* qN, double* qdN, int64_t B, void* stream);
int mrf_rollout_dev_f32(mrf_handle_t h, const float* rec, int N, float* avg_vel, float* x_ee, float* goal_est,
                        float* qN, float* qdN, int64_t B, void* stream);

/* Cartesian (decoupled) rollout of robot `robot`: obstacles move with constant velocity, xddot = 0.
 *   rec [MRF_REC][B]  obst [S][MRF_OBST][B] (xddot ignored)  avg_vel [B]  qN,qdN [N][MRF_DOF][B] */
/* Coupled rollout whose planners also carry n_static STATIC spheres per robot -- x_obst_i / radius_obst_i of
 * define_rollout_planners(nr_obst = params.nr_obsts[i]) (example_pandas_Jointspace.py:172-193), the x_obsts /
 * radius_obsts arguments of get_velocity_rollouts (forward_planner_Jointspace.py:319-322): the same collision leaf with
 * a sphere at rest.   stat [n_static][4][R][B] = x, y, z, radius of sphere o of robot r; 0 <= n_static <= MRF_MAX_STATIC. */
int mrf_rollout_static_dev_f64(mrf_handle_t h, const double* rec, int N, int n_static, const double* stat, double* avg_vel,
                               double* x_ee, double* goal_est, double* qN, double* qdN, int64_t B, void* stream);
int mrf_rollout_static_dev_f32(mrf_handle_t h, const float* rec, int N, int n_static, const float* stat, float* avg_vel,
                               float* x_ee, float* goal_est, float* qN, float* qdN, int64_t B, void* stream);

int mrf_rollout_cart_dev_f64(mrf_handle_t h, int robot, const double* rec, int S, const double* obst, int N,
                             double* avg_vel, double* qN, double* qdN, int64_t B, void* stream);
int mrf_rollout_cart_dev_f32(mrf_handle_t h, int robot, const float* rec, int S, const float* obst, int N,
                             float* avg_vel, float* qN, float* qdN, int64_t B, void* stream);
/* Cartesian (decoupled) rollouts of EVERY robot of the handle in one launch, each robot against its own obstacle list
 * (the per-robot FabricsRollouts.rollouts_numerical / get_velocity_rollouts calls of
 * examples/example_pandas_cartesian.py:361-418; forward_planner_Cartesian.py:421-458 per robot).  Layouts of
 * mrf_action_dev_*:  rec [MRF_REC][R][B]  obst [S][MRF_OBST][R][B] (xddot ignored)  avg_vel [R][B]
 * qN, qdN [R][N][MRF_DOF][B] (nullable).  Robot r's results equal those of mrf_rollout_cart_dev_*(robot = r) on its slices. */
int mrf_rollout_cart_all_dev_f64(mrf_handle_t h, const double* rec, int S, const double* obst, int N, double* avg_vel,
                                 double* qN, double* qdN, int64_t B, void* stream);
int mrf_rollout_cart_all_dev_f32(mrf_handle_t h, const float* rec, int S, const float* obst, int N, float* avg_vel,
                                 float* qN, float* qdN, int64_t B, void* stream);

/* Link kinematics of the 8 collision links: x, v = J qdot, a = jdot_ref_sign * d(J qdot)/dq qdot.
 *   q, qdot [MRF_DOF][R][B];  x, v, a [MRF_NLINKS][3][R][B] (nullable) */
int mrf_kinematics_dev_f64(mrf_handle_t h, const double* q, const double* qdot, double* x, double* v, double* a,
                           int64_t B, void* stream);
int mrf_kinematics_dev_f32(mrf_handle_t h, const float* q, const float* qdot, float* x, float* v, float* a,
                           int64_t B, void* stream);

/* Obstacle staging for the executed action (replaces the per-step CasADi / environment calls of
 * examples/example_pandas_Jointspace.py:324-343,400-412 and multi_robot_fabrics/utils/utils_apply_fk.py:3-33 with the
 * sphere functions of multi_robot_fabrics/utils/utils.py:87-119): every robot's 8 * n_per_link collision spheres,
 * sphere s of link l at p_link + R_link * offsets[l][s] (offsets: HOST pointer, [8][n_per_link][3], link frame, see
 * create_simulation_manipulators.py:188-245), assembled into each ego robot's obstacle list (other robots ascending).
 *   vel_mode 0: every sphere carries its link ORIGIN's velocity J_link qdot (example_pandas_Jointspace.py:406-410)
 *   vel_mode 1: true sphere velocity J_sphere qdot (utils.py:109, utils_apply_fk.py:28)
 *   accelerations are 0, radius = r_robots[j][l]; STATIC_OR_DYN_FABRICS == 0 zeroes the velocities.
 *   q, qdot [MRF_DOF][R][B] -> obst [8 n (R-1)][MRF_OBST][R][B] (nullable), spheres_x, spheres_v [8 n][3][R][B] (nullable) */
int mrf_obstacles_dev_f64(mrf_handle_t h, int n_per_link, const double* offsets, int vel_mode, const double* q,
                          const double* qdot, double* obst, double* spheres_x, double* spheres_v, int64_t B, void* stream);
int mrf_obstacles_dev_f32(mrf_handle_t h, int n_per_link, const double* offsets, int vel_mode, const float* q,
                          const float* qdot, float* obst, float* spheres_x, float* spheres_v, int64_t B, void* stream);

/* Point-mass planner of BASELINE config C1 (examples/example_pointmasses_static.py:102-129,191-199 and
 * examples/example_pointmasses_dynamic.py:102-131,192-212): planner.compute_action for the 3-dof (x, y, theta) point
 * robot with Ss static spheres, Sd dynamic 2-D spheres and one 2-D goal, mode 'acc'.  Uses eps / jdot_sign / exec_scale
 * of the handle's MrfConfig.  Device layouts (b fastest):
 *   rec [10][B]: q[3], qdot[3], x_goal_0[2], weight_goal_0, radius_body_base_link
 *   stat [Ss][4][B]: x_obst[3], radius_obst       dyn [Sd][7][B]: x[2], xdot[2], xddot[2], radius      action [3][B]
 * Host layouts: rec [B][10], stat [B][Ss][4], dyn [B][Sd][7], action [B][3]. */
int mrf_point_action_dev_f64(mrf_handle_t h, const double* rec, int Ss, const double* stat, int Sd, const double* dyn,
                             double* action, int64_t B, void* stream);
int mrf_point_action_dev_f32(mrf_handle_t h, const float* rec, int Ss, const float* stat, int Sd, const float* dyn,
                             float* action, int64_t B, void* stream);
int mrf_point_action_host_f64(mrf_handle_t h, const double* rec, int Ss, const double* stat, int Sd, const double* dyn,
                              double* action, int64_t B);

/* Batched deadlock_checking step.  All arrays index b fastest; state arrays are updated in place.
 *   x_ee [R][3][B]  goals [R][3][B] (in/out)  weights [R][B] (in/out)
 *   exactly one of: avg_vel [R][B] (per-robot rollout averages; the kernel forms sum/R as
 *   example_pandas_Jointspace.py:375 does) or avg_sum [B] (the caller's scalar); the other NULL
 *   sm_state [R][B] (state-machine codes)  time_step [B]  time_deadlock_out [B] (in/out)
 *   st_int [4][B]: i_leader, i_follower, i_robots_dead[0], i_robots_dead[1]  (in/out; initial 0,1,0,1)
 *   st_goal [3][B]: goal_robot0 (in/out; initial 0)      flag [B] (out, nullable): `deadlock` raised this step */
int mrf_deadlock_dev_f64(mrf_handle_t h, const double* x_ee, double* goals, double* weights, const double* avg_vel,
                         const double* avg_sum, const int32_t* sm_state, const int32_t* time_step,
                         int32_t* time_deadlock_out, int32_t* st_int, double* st_goal, int32_t* flag, int64_t B,
                         void* stream);
int mrf_deadlock_dev_f32(mrf_handle_t h, const float* x_ee, float* goals, float* weights, const float* avg_vel,
                         const float* avg_sum, const int32_t* sm_state, const int32_t* time_step,
                         int32_t* time_deadlock_out, int32_t* st_int, float* st_goal, int32_t* flag, int64_t B,
                         void* stream);

/* The same step applied IN PLACE to the record tensor rec [MRF_REC][R][B] that mrf_rollout_dev / mrf_action_dev read: the
 * goals are rows MRF_G0..MRF_G0+2 and the weights row MRF_W0 -- the reference likewise mutates the caller's goal /
 * weight lists that compute_action then receives (example_pandas_Jointspace.py:379-380,423).  If goal_est [3][B] is
 * given and MrfConfig.estimate_goal is set, robot `estimate_robot`'s goal is first replaced by it (:346-348). */
int mrf_deadlock_rec_dev_f64(mrf_handle_t h, const double* x_ee, double* rec, const double* goal_est, const double* avg_vel,
                             const double* avg_sum, const int32_t* sm_state, const int32_t* time_step,
                             int32_t* time_deadlock_out, int32_t* st_int, double* st_goal, int32_t* flag, int64_t B,
                             void* stream);
int mrf_deadlock_rec_dev_f32(mrf_handle_t h, const float* x_ee, float* rec, const float* goal_est, const float* avg_vel,
                             const float* avg_sum, const int32_t* sm_state, const int32_t* time_step,
                             int32_t* time_deadlock_out, int32_t* st_int, float* st_goal, int32_t* flag, int64_t B,
                             void* stream);

/* RF-CV post step of a sweep: the deadlock heuristic in place on rec_work (as mrf_deadlock_rec_dev) with the per-scenario
 * results a sweep gathers written straight into result [R+1][B] (rows 0..R-1 = avg_vel, row R = deadlock flag as a
 * number; nullable).  rec = the records the rollout read (unchanged), rec_work = the tensor whose goal / weight rows the
 * heuristic overwrites (may be the same tensor if the caller does not reuse the records).
 *
 * FP32 ("deadlock flags identical", north star): the heuristic thresholds rollout outputs (deadlock_prevention.py:61-66:
 * vel_avg_tot < 0.16, end-effector distance < 0.35) and compares them with each other (:76 closest pair, :85 leader).
 * With risk [R][B] given (from mrf_rollout_risk_dev_f32), scenarios that have a candidate pair at all (states, time gate,
 * hands closer than the threshold plus the band) and whose FP32 values sit within a guard band of one of
 * those tests (the band widens with the stiffness indicator, see mrf_set_guard) or that are
 * non-finite are RE-ROLLED BY THE FP64 KERNEL from the same records inside this call, and the heuristic reads the FP64
 * values for them -- the flags then equal those of a float64 evaluation of the same inputs.  mrf_set_guard() tunes the
 * bands; mrf_guard_stats() reports how many scenarios were re-rolled.  risk == NULL: no re-roll (plain FP32 decision).
 * FP64: risk is ignored (nothing to guard).
 * slot (0..3; 4..7 belong to mrf_rfcv_host_submit_f32's pipeline) selects the scratch the re-roll uses: post steps that may run concurrently (different
 * streams) must use different slots; calls on one stream can share one.  out[2] of mrf_guard_stats refers to slot 0. */
int mrf_rfcv_post_dev_f32(mrf_handle_t h, const float* rec, int N, const float* x_ee, float* rec_work, const float* goal_est,
                          const float* avg_vel, const float* risk, const int32_t* sm_state, const int32_t* time_step,
                          int32_t* time_deadlock_out, int32_t* st_int, float* st_goal, int32_t* flag, float* result,
                          int64_t B, void* stream, int slot);
int mrf_rfcv_post_dev_f64(mrf_handle_t h, const double* rec, int N, const double* x_ee, double* rec_work,
                          const double* goal_est, const double* avg_vel, const double* risk, const int32_t* sm_state,
                          const int32_t* time_step, int32_t* time_deadlock_out, int32_t* st_int, double* st_goal,
                          int32_t* flag, double* result, int64_t B, void* stream, int slot);
/* mrf_rollout_dev without trajectories plus risk [R][B]: per robot the maximum over the horizon of the summed
 * collision-leaf metric (sphere leaf 0.02 w / (x^4 rho^2), plane leaf 0.2 s / x^2) -- large near contact, where the
 * explicit dt integration amplifies FP32 rounding.  Always the throughput kernel (no cooperative small-batch path). */
int mrf_rollout_risk_dev_f32(mrf_handle_t h, const float* rec, int N, float* avg_vel, float* x_ee, float* goal_est,
                             float* risk, int64_t B, void* stream);
int mrf_rollout_risk_dev_f64(mrf_handle_t h, const double* rec, int N, double* avg_vel, double* x_ee, double* goal_est,
                             double* risk, int64_t B, void* stream);
/* Guard bands of mrf_rfcv_post_dev_f32 (NULL / negative = keep).  A scenario with a candidate pair is re-rolled in FP64
 * when |vel_avg_tot - dl_avg_vel_constant| <= bands[t] + bands[3 + t] * vel_avg_tot, with the stiffness tier
 * t = (risk >= risk_edges[0]) + (risk >= risk_edges[1]); defaults bands = {2e-5, 4e-3, 4e-3, 0, 0.02, 0.4} (absolute,
 * relative), risk_edges = {40, 200}, calibrated against the FP64 kernel on 4 x 65536 random scenarios
 * (profiles/r2_guard_calibration.md) -- or when an end-effector distance is within band_dist (1e-5) of dl_dist_endeff / of
 * a competing distance, or when the FP32 result is non-finite.  cap = most scenarios re-rolled per call
 * (0 = max(256, B / 16)); the excess is counted as overflow and decided in FP32. */
int mrf_set_guard(mrf_handle_t h, const double* bands, const double* risk_edges, double band_dist, int64_t cap);
/* out[0] = scenarios re-rolled in FP64 so far, out[1] = overflow so far, out[2] = listed by the last call.  Synchronise
 * the streams the post steps ran on first. */
int mrf_guard_stats(mrf_handle_t h, int64_t* out);

/* Batched pick-and-place state machine step (SURVEY 8f rank 3): StateMachine.get_state_machine_panda and
 * get_gripper_action_panda, multi_robot_fabrics/others_planner/state_machine.py:70-84,133-214.
 *   nr_blocks: HOST pointer, blocks per robot [R]
 *   x_ee, goal_block, start_goal [R][3][B] (in);  q_grip [R][2][B] (in)
 *   goal, above [R][3][B] and weight [R][B] (in/out: get_goal_robot(), goal_above_block, get_weight_goal0())
 *   st [6][R][B] (in/out): state_machine_panda (initial 1), nr_blocks_success, nr_blocks_failed, time_gripping,
 *                          gripper closed (0/1), stop_time;   grip_action [R][2][B] (out, nullable) */
int mrf_fsm_dev_f64(mrf_handle_t h, const int32_t* nr_blocks, const double* x_ee, const double* q_grip,
                    const double* goal_block, const double* start_goal, double* goal, double* above, double* weight,
                    int32_t* st, double* grip_action, int64_t B, void* stream);
int mrf_fsm_dev_f32(mrf_handle_t h, const int32_t* nr_blocks, const float* x_ee, const float* q_grip,
                    const float* goal_block, const float* start_goal, float* goal, float* above, float* weight, int32_t* st,
                    float* grip_action, int64_t B, void* stream);

/* ------------------------------- host-pointer entries (AoS) -----------------------------------
 *   rec [B][R][MRF_REC]   obst [B][R][S][MRF_OBST]   action [B][R][MRF_DOF]
 *   avg_vel [B][R]  x_ee [B][R][3]  goal_est [B][3]  qN,qdN [B][R][N][MRF_DOF]  (nullable outputs skipped)
 *   mrf_rollout_host_*: when `rec` is page-locked (cudaHostAlloc / cudaHostRegister, 16-byte aligned), B >= 8192 and no
 *   trajectories are requested, the kernel reads the records in place over PCIe and writes page-locked results in
 *   place (one launch); pageable buffers take a chunk-pipelined staged path with identical results.  Environment:
 *   MRF_ZERO_COPY=0 forces the staged path, MRF_ZC_WINDOW=<tiles admitted to the bus at a time, default 32>. */
int mrf_action_host_f64(mrf_handle_t h, int robot_first, int n_rob, const double* rec, int S, const double* obst,
                        double* action, int64_t B);
int mrf_action_host_f32(mrf_handle_t h, int robot_first, int n_rob, const float* rec, int S, const float* obst,
                        float* action, int64_t B);
int mrf_rollout_host_f64(mrf_handle_t h, const double* rec, int N, double* avg_vel, double* x_ee, double* goal_est,
                         double* qN, double* qdN, int64_t B);
int mrf_rollout_host_f32(mrf_handle_t h, const float* rec, int N, float* avg_vel, float* x_ee, float* goal_est,
                         float* qN, float* qdN, int64_t B);
/*   rec [B][MRF_REC]  obst [B][S][MRF_OBST]  avg_vel [B]  qN,qdN [B][N][MRF_DOF] */
int mrf_rollout_cart_host_f64(mrf_handle_t h, int robot, const double* rec, int S, const double* obst, int N,
                              double* avg_vel, double* qN, double* qdN, int64_t B);
int mrf_rollout_cart_host_f32(mrf_handle_t h, int robot, const float* rec, int S, const float* obst, int N,
                              float* avg_vel, float* qN, float* qdN, int64_t B);
/* Sweeps of independent batches: a two-deep pipeline over the in-place path of mrf_rollout_host_*.  submit enqueues one
 * batch (all buffers page-locked; they must stay untouched until the matching wait) and returns; with two batches in
 * flight it first waits for the older one.  wait(all = 0) blocks until the oldest submitted batch has its results in
 * host memory, wait(all = 1) until every submitted batch has.  The PCIe reads of batch i+1 overlap the horizons of
 * batch i.  Same results as mrf_rollout_host_* (get_velocity_rollouts, forward_planner_Jointspace.py:298-336). */
int mrf_rollout_host_submit_f64(mrf_handle_t h, const double* rec, int N, double* avg_vel, double* x_ee, double* goal_est,
                                int64_t B);
int mrf_rollout_host_submit_f32(mrf_handle_t h, const float* rec, int N, float* avg_vel, float* x_ee, float* goal_est,
                                int64_t B);
/* Compact records for the same pipeline: rec_var [B][R][MRF_G1] holds only what changes from scenario to scenario (q,
 * qdot, x_goal_0, weight_goal_0 -- the per-step entries of the reference's inputs_action dict,
 * example_pandas_Jointspace.py:354-368); rec_shared [R][MRF_REC] (ordinary host memory, copied at submission) supplies the
 * remaining fields of every robot's record (x_goal_1/2, weights 1/2, angle_goal_1, constraint_0, body radii).  Less
 * than half the bytes cross PCIe; results are identical to submitting the expanded records. */
int mrf_rollout_host_submit_compact_f64(mrf_handle_t h, const double* rec_var, const double* rec_shared, int N,
                                        double* avg_vel, double* x_ee, double* goal_est, int64_t B);
int mrf_rollout_host_submit_compact_f32(mrf_handle_t h, const float* rec_var, const float* rec_shared, int N,
                                        float* avg_vel, float* x_ee, float* goal_est, int64_t B);
int mrf_rollout_host_wait(mrf_handle_t h, int all);

/* One RF-CV control step of a sweep END TO END from host memory, asynchronous like mrf_rollout_host_submit_* (same
 * two-deep pipeline, same mrf_rollout_host_wait): get_velocity_rollouts -> vel_avg_tot -> deadlock_checking
 * (example_pandas_Jointspace.py:354-385) for B scenarios.  The in-place rollout kernel reads the page-locked records
 * (rec_shared == NULL: rec [B][R][MRF_REC]; else compact rec [B][R][18] + rec_shared [R][MRF_REC]) over PCIe and keeps its
 * results on the device; the post step of mrf_rfcv_post_dev_f32 (FP64 guard re-roll -- the listed scenarios are read
 * from the same host records -- and the deadlock heuristic) follows on the same stream; only
 *   result    [R+1][B]  rows 0..R-1 = avg_vel per robot, row R = deadlock flag (page-locked, required)
 *   goals_out [4][R][B] x_goal_0 (3 rows) and weight_goal_0 of every robot AFTER the heuristic (page-locked, nullable)
 * travel back.  Stateless per batch: state-machine codes 0, the given time_step for every scenario, no deadlock history
 * (time_deadlock_out = 1000).  n_robots >= 2.  Its pipeline is FOUR deep (the post step of a batch runs while the
 * rollouts of the next two already occupy the GPU): a submission blocks until the one four calls earlier is complete, so a
 * caller cycling through four sets of buffers never overwrites data in flight; mrf_rollout_host_wait(h, 0) waits for the
 * oldest batch, (h, 1) for all. */
int mrf_rfcv_host_submit_f32(mrf_handle_t h, const float* rec, const float* rec_shared, int N, int32_t time_step,
                             float* result, float* goals_out, int64_t B);
/*   q, qdot [B][R][MRF_DOF]   x, v, a [B][R][MRF_NLINKS][3] */
int mrf_kinematics_host_f64(mrf_handle_t h, const double* q, const double* qdot, double* x, double* v, double* a,
                            int64_t B);

/*   x_ee, goals [B][R][3]  weights [B][R]  avg_sum [B]  sm_state [B][R]  time_step, time_deadlock_out, flag [B]
 *   st_int [B][4]  st_goal [B][3] */
int mrf_deadlock_host_f64(mrf_handle_t h, const double* x_ee, double* goals, double* weights, const double* avg_sum,
                          const int32_t* sm_state, const int32_t* time_step, int32_t* time_deadlock_out,
                          int32_t* st_int, double* st_goal, int32_t* flag, int64_t B);

/* One closed-loop control step of B independent scenarios, entirely on the device -- the loop body of
 * examples/example_pandas_Jointspace.py:280-458 with a kinematic environment (q += dt * clip(action), the urdfenvs 'vel'
 * mode, :454) and a reach task (state-machine code 0; success = every hand within `epsilon` of its goal, :35):
 *   clip qdot (:288) -> [rollout_fabrics: coupled rollouts with weight_goal_1 = w1_rollout (:352-376) -> RF-CV goal
 *   (:346-348) -> resolve_deadlocks: deadlock_checking (:379-385)] -> other robots' collision spheres, n_per_link per
 *   link, link-origin velocities (:400-412) -> executed action with weight_goal_1 = w1_action (:417-445) -> clip (:453),
 *   integrate, metrics (first step at which the task is reached, minimum sphere clearance :461-470, deadlock steps).
 * Seven kernel launches on `stream`; capture it in a CUDA graph and replay.  All pointers are device pointers of the
 * entry's precision (T) unless typed; b fastest.
 * rollout_model = 1 runs the loop body of examples/example_pandas_cartesian.py:295-462 instead
 * (rollouts: forward_planner_Cartesian.py:421-458): clip ->
 * hand FK and J qdot at the measured state (kin_scratch) -> RF-CV goal x_hand + estimate_horizon * J qdot of robot
 * `estimate_robot` written into its goal rows before the rollouts (:355-357; any nonzero MrfConfig.estimate_goal takes
 * this J qdot form here, 2 in MrfConfig terms) -> every robot's
 * sphere list with true sphere velocities (mrf_obstacles_dev vel_mode 1, :343-352) -> mrf_rollout_cart_all_dev with
 * weight_goal_1 = w1_rollout (20, :42) -> deadlock_checking on sum(avg_vel) / R (:405) -> the executed action as above
 * (link-origin velocities, vel_mode 0).  The rollouts use the planner with collision links in every state. */
typedef struct MrfEpisode {
    int32_t struct_size;        /* sizeof(MrfEpisode) */
    int32_t n_horizon;          /* rollout horizon (rollout_fabrics) */
    int32_t rollout_fabrics;    /* 0 = MRDF: no rollouts, no deadlock logic */
    int32_t resolve_deadlocks;
    int32_t n_per_link;         /* collision spheres per link seen by the executed action (and by the Cartesian rollouts) */
    int32_t rollout_model;      /* read when rollout_fabrics = 1.  0: coupled joint-space rollouts (ForwardFabricsPlanner,
                                   examples/example_pandas_Jointspace.py:352-376).  1: decoupled Cartesian rollouts
                                   (FabricsRollouts, examples/example_pandas_cartesian.py:343-418): each robot rolled out
                                   alone against the other robots' spheres moving at constant velocity; needs kin_scratch */
    double epsilon;             /* reach tolerance (0.05) */
    double w1_rollout, w1_action;   /* weight_goal_1: 10 in the rollouts (:43,364), 20 in the executed action (:427) */
    double clearance_radius_sum;    /* subtracted from sphere-centre distances (0.16) */
    double vel_limit[MRF_DOF];      /* :221 */
    const double* offsets;      /* HOST pointer [8][n_per_link][3], link-frame sphere offsets */
    void* rec;                  /* T [MRF_REC][R][B]: rows q, qdot are the live state; goal / weight rows are rewritten */
    void* goal0;                /* T [R][3][B] task goals (read-only for the reach task) */
    void* w0;                   /* T [R][B] task weight_goal_0 */
    void* avg_vel;              /* T [R][B]      (rollout_fabrics) */
    void* x_ee;                 /* T [R][3][B]   hand positions at the measured state */
    void* goal_est;             /* T [3][B]      (rollout_fabrics) */
    void* obst;                 /* T [8 n (R-1)][MRF_OBST][R][B] */
    void* spheres_x;            /* T [8 n][3][R][B] */
    void* action;               /* T [MRF_DOF][R][B] */
    void* kin_scratch;          /* T [3][8][3][R][B] (MRDF mode, pick-and-place, rollout_model = 1) */
    const int32_t* sm_state;    /* [R][B] state-machine codes (resolve_deadlocks) */
    int32_t* time_step;         /* [B] in/out, incremented */
    int32_t* time_deadlock_out; /* [B] in/out */
    int32_t* st_int;            /* [4][B] in/out, see mrf_deadlock_dev */
    void* st_goal;              /* T [3][B] in/out */
    int32_t* flag;              /* [B] out: deadlock raised this step */
    int32_t* done_at;           /* [B] in/out: first step index at which the task was reached (-1 = not yet) */
    int32_t* deadlock_steps;    /* [B] in/out: += flag */
    void* min_clearance;        /* T [B] in/out: running minimum */
    /* pick-and-place task (:289-312,417-448) instead of the reach task: each robot's state machine
     * (others_planner/state_machine.py:133-214, see mrf_fsm_dev) sets this step's goal0 / w0 (then in/out), gates the
     * deadlock logic, selects the obstacle-free grasp planner in state 2 and holds the arm in states 3 / 5; the finger
     * joints integrate its gripper velocity inside [0, 0.04]; blocks are kinematic (they do not fall, so the
     * state machine's "dropped" branch never fires); done_at = first step at which every robot reports state 10. */
    int32_t pick_and_place;
    int32_t n_blocks;           /* blocks per robot */
    const void* blocks;         /* T [n_blocks][R][3][B] rest positions of each robot's blocks (picked in order) */
    const void* start_goal;     /* T [R][3][B] */
    void* q_grip;               /* T [R][2][B] in/out finger joints (open = 0.04) */
    void* goal_block;           /* T [R][3][B] scratch: current block + 0.1 in z */
    void* fsm_above;            /* T [R][3][B] in/out */
    int32_t* fsm_st;            /* [6][R][B] in/out, rows as in mrf_fsm_dev_*; state initial 1 */
    void* grip_action;          /* T [R][2][B] out */
    int32_t* nonfinite_steps;   /* [B] in/out, nullable: control steps in which an executed action was non-finite (the arm
                                   then holds still for that step); FP32 near-contact divergence shows up here instead of
                                   vanishing into the success / clearance metrics */
} MrfEpisode;
int mrf_episode_step_dev_f64(mrf_handle_t h, const MrfEpisode* ep, int64_t B, void* stream);
int mrf_episode_step_dev_f32(mrf_handle_t h, const MrfEpisode* ep, int64_t B, void* stream);

/* Closed-loop point-mass episodes of B independent scenarios, n_steps control steps in ONE launch: the control loops of
 * examples/example_pointmasses_static.py (dynamic = 0) and examples/example_pointmasses_dynamic.py (dynamic = 1) with a
 * kinematic environment.  Per step, for every robot i of every scenario, all robots reading the state at the start of
 * the step (Jacobi order):
 *   1. metrics of the measured state: done_at = first time_step at which every robot is within `epsilon` of its goal in
 *      (x, y); running minima of the x-y robot-robot clearance |p_i - p_j| - (r_i + r_j) and of the robot-scene clearance
 *      |(x, y, 0.05) - c_o| - (r_o + r_i) (the distance the collision leaf sees).
 *   2. obstacles of robot i: the n_scene scene spheres, then the other robots ascending.  Static variant: robot j is a
 *      static sphere at its full joint position q_j = (x, y, theta), radius r_j -- the third component lands in the
 *      sphere's z, a quirk of the reference's static example kept as is (theta is only ever damped).  Dynamic variant:
 *      robot j is a 2-D sphere at q_j[0:2] with velocity qdot_j[0:2], acceleration 0, radius r_j.
 *   3. action: the planner of mrf_point_action_dev_* (mode 'acc', one 2-D goal, eps / jdot_sign / exec_scale of the
 *      handle's MrfConfig).  compute_action's |a| < 1e-6 zeroing is not applied (neither does mrf_episode_step_dev_*).
 *   4. environment: a non-finite action becomes 0 for the step, which is counted in nonfinite_steps; then
 *      qdot += dt a, q += dt qdot (semi-implicit Euler, dt = MrfConfig.dt, each product and sum rounded on its own).
 *      ASSUMPTION: urdfenvs integrates a commanded velocity through its velocity controller; this kinematic double
 *      integrator stands in for its acceleration mode.
 * No rollouts and no deadlock logic (the reference's point examples run neither).  Splitting an episode over several
 * calls (n_steps each) gives the same bits as one call.  Device pointers of the entry's precision T unless typed, b
 * fastest. */
typedef struct MrfPointEpisode {
    int32_t struct_size;        /* sizeof(MrfPointEpisode) */
    int32_t n_robots;           /* R, 2..MRF_MAX_POINT_ROBOTS */
    int32_t dynamic;            /* 0: other robots are static spheres (static example), 1: dynamic 2-D spheres */
    int32_t n_scene;            /* scene spheres per scenario, 0..MRF_MAX_STATIC */
    double epsilon;             /* reach tolerance in (x, y) */
    void* state;                /* T [6][R][B] in/out: q (x, y, theta), qdot */
    const void* goal;           /* T [R][2][B] */
    const void* weight;         /* T [R][B] weight_goal_0 */
    const void* radius;         /* T [R][B] radius_body_base_link */
    const void* scene;          /* T [n_scene][4][B] x, y, z, radius (nullable when n_scene = 0) */
    int32_t* time_step;         /* [B] in/out, += n_steps */
    int32_t* done_at;           /* [B] in/out (-1 = not yet) */
    int32_t* nonfinite_steps;   /* [B] in/out */
    void* min_clear_robots;     /* T [B] in/out: running minimum */
    void* min_clear_scene;      /* T [B] in/out: running minimum */
    void* traj;                 /* T [n_steps][3][R][B] out, nullable: q after each step of this call */
} MrfPointEpisode;
int mrf_point_episode_run_dev_f64(mrf_handle_t h, const MrfPointEpisode* ep, int64_t B, int32_t n_steps, void* stream);
int mrf_point_episode_run_dev_f32(mrf_handle_t h, const MrfPointEpisode* ep, int64_t B, int32_t n_steps, void* stream);

/* mrf_rollout_* picks between two kernels computing the same recurrence: the cooperative low-latency kernel (one CTA
 * per scenario, one warp per robot) for B <= max_batch, the throughput kernel (one thread per scenario and robot)
 * above.  Default 512; 0 disables the cooperative kernel. */
int mrf_set_coop_max_batch(mrf_handle_t h, int64_t max_batch);

/* Number of kernels this library has launched through handle h since creation (for bench accounting). */
int64_t mrf_launch_count(mrf_handle_t h);
/* Device time in ms of the last *_host_* call's kernel(s) (CUDA events on the handle's stream). */
double mrf_last_kernel_ms(mrf_handle_t h);

/* Measured FMA throughput (TFLOP/s, FMA = 2 flops) of the device's FP32 / FP64 pipes: the roofline denominator of
 * the compute-bound kernels (8 independent chains per thread, 8 CTAs of 256 threads per SM, best of 5). */
int mrf_fma_peak(mrf_handle_t h, int is_f64, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* MRF_B200_H */
