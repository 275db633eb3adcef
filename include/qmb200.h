/* qmb200 — C ABI of the B200-native batched MPC+WBC solver (drop-in for qm_control's per-tick numerical path).
 *
 * Every entry point replaces one reference interface; the thin C++ subclasses a maintainer adds on the
 * reference side (B200Wbc : qm::WbcBase, B200Mpc : ocs2::MPC_BASE) are shown in INTEGRATION.md.
 *
 * Conventions: plain pointers and sizes only; return 0 on success, negative on error (never throws);
 * qmb200_last_error() describes the last failure; the caller owns every buffer it passes; `_dev` variants
 * take device pointers and a cudaStream_t (as void*) and do not synchronise; one handle per GPU, calls on
 * one handle are serialised on its stream; batch = 1 works (plugin use).  All arithmetic is fp64
 * (ocs2::scalar_t).  Layouts are robot-major, fixed stride:
 *   state x[30]  = [h_lin/m(3), h_ang/m(3), base pos(3), base euler ZYX(3), joints(18: LF,LH,RF,RH,arm)]   task.info:150-189
 *   input u[30]  = [contact forces(12: LF,RF,LH,RH), joint velocities(18)]                                  task.info:252-286
 *   rbd[55]      = [euler ZYX(3), pos(3), joints(18), w_world(3), v_lin(3), joint vel(18), ee pos(3), ee quat xyzw(4)]
 *                                                                                  qm_estimation/src/StateEstimateBase.cpp:41-103
 *   cmd[54]      = [vdot(24), F(12), tau(18)]                                      qm_wbc/src/WbcBase.cpp:548-563
 *   mode         = 4-bit stance code LF=8 RF=4 LH=2 RH=1 (ocs2_legged_robot MotionPhaseDefinition)
 */
#ifndef QMB200_H
#define QMB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QMB200_NX 30
#define QMB200_NU 30
#define QMB200_RBD 55
#define QMB200_CMD 54
#define QMB200_TARGET 37   /* 30-dim state + end-effector pose [pos(3), quat xyzw(4)] (QMController.cpp:106-112) */
#define QMB200_EMAX 32     /* max events of one robot's mode schedule window */
#define QMB200_KMAX 4      /* max knots of one robot's target trajectory */

#define QMB200_WBC_HIERARCHICAL 0      /* qm::HierarchicalWbc      (qm_wbc/src/HierarchicalWbc.cpp:18-44)    */
#define QMB200_WBC_HIERARCHICAL_MPC 1  /* qm::HierarchicalMpcWbc   (qm_wbc/src/HierarchicalMpcWbc.cpp:18-34) */

/* per-robot status bits (the reference ignores solver status, HoQp.cpp:143; here it is reported).
 * Layout of a status word:  bits 0..7   WBC flags (QMB200_ST_ITER_CAP | _OVERFLOW | _NAN) — qmb200_wbc_update, qmb200_update, qmb200_tick
 *                           bits 8..15  MPC flags shifted left by 8 — only in the merged word qmb200_tick / qmb200_tick_dev return
 *                                       (qmb200_mpc_solve / qmb200_mpc_get_solution report the MPC flags unshifted in their own status array)
 *                           bit 16      QMB200_ST_SAFETY — qmb200_update / qmb200_control_law
 * Nothing else is ever OR-ed into a status word: the WBC's iteration counts live in qmb200_wbc_get_diagnostics. */
#define QMB200_ST_ITER_CAP 1
#define QMB200_ST_OVERFLOW 2      /* WBC: more rows than the working-set / level-0 buffers hold; MPC: node count > NMAX, event / target count out of range, swing phase not enclosed */
#define QMB200_ST_NAN 4
#define QMB200_ST_NOT_PD 8
#define QMB200_ST_NO_STEP 16      /* line search rejected every step size (solution = initial guess, as in SqpSolver::takeStep) */
#define QMB200_ST_CONVERGED 32    /* informational: SqpSolver::checkConvergence ended the SQP loop before sqp.sqpIteration (only when sqpIteration > 1) */
#define QMB200_ST_NEG_DT 64       /* an interval of the time grid has a non-positive duration: a pre-/post-event node within weakEpsilon (1e-6 s) of its neighbour but
                                     further than dt_min (1e-8 s), so getIntervalEnd - getIntervalStart < 0 [upstream ocs2_oc TimeDiscretization]; the stage cost is then
                                     weighted by a negative dt and the QP is not convex (comes with QMB200_ST_NOT_PD) */
#define QMB200_MPC_STATUS_SHIFT 8

typedef struct qmb200_handle qmb200_handle;

/* Replaces the constructor chain QMController::setupInterface/setupMpc/setupWbc
 * (qm_controllers/src/QMController.cpp:272-306,336-340) → QMInterface(taskFile, urdfFile, referenceFile)
 * (qm_interface/include/qm_interface/QMInterface.h:31-35). */
typedef struct {
  const char* task_file;        /* task.info */
  const char* urdf_file;        /* robot.urdf */
  const char* reference_file;   /* reference.info */
  const char* wbc_gains_file;   /* optional INFO file with a wbcGains{} block; NULL → defaults of qm_wbc/cfg/wbcWigeht.cfg:7-47 */
  int32_t batch;                /* robots per call on this GPU */
  int32_t device;               /* CUDA device ordinal */
  double time_horizon;          /* <= 0 → mpc.timeHorizon (task.info:140) */
  double dt;                    /* <= 0 → sqp.dt (task.info:78) */
  int32_t max_nodes;            /* <= 0 → ceil(horizon/dt) + 1 + 2*10 (room for 10 events inside the horizon) */
  int32_t wbc_variant;          /* QMB200_WBC_* */
} qmb200_config;

int qmb200_create(const qmb200_config* cfg, qmb200_handle** out);
void qmb200_destroy(qmb200_handle* h);
const char* qmb200_last_error(const qmb200_handle* h);   /* h may be NULL (error of a failed create) */

/* dimensions of this handle: batch, node capacity NMAX, event capacity, target-knot capacity */
int qmb200_get_dims(const qmb200_handle* h, int32_t* batch, int32_t* nmax, int32_t* emax, int32_t* kmax);
/* CentroidalModelInfo / settings as the reference exposes them (QMInterface.h:37-54): robotMass, initialState[30] (task.info:150-189),
 * defaultJointState[18] (reference.info:6-26), time horizon, dt */
int qmb200_get_model_info(const qmb200_handle* h, double* robot_mass, double* initial_state30, double* default_joint_state18, double* time_horizon, double* dt);
int qmb200_get_joint_name(const qmb200_handle* h, int32_t joint, char* out, int32_t capacity);

/* ---- WBC seam: qm::WbcBase::update(stateDesired, inputDesired, rbdStateMeasured, mode, period, time) → vector_t
 *      (qm_wbc/include/qm_wbc/WbcBase.h:31-32), batched.  Host-pointer version copies in/out on the handle's stream
 *      and returns after the result is in cmd/status. */
int qmb200_wbc_update(qmb200_handle* h, const double* x_des /*[B][30]*/, const double* u_des /*[B][30]*/, const double* rbd /*[B][55]*/,
                      const int32_t* mode /*[B]*/, const double* period /*[B]*/, const double* time /*[B]*/, double* cmd /*[B][54]*/, int32_t* status /*[B]*/);
int qmb200_wbc_update_dev(qmb200_handle* h, const double* x_des, const double* u_des, const double* rbd, const int32_t* mode, const double* period,
                          const double* time, double* cmd, int32_t* status, void* cuda_stream);
/* WbcBase::inputLast_ (WbcBase.cpp:42,212-213): set for all robots (NULL → zeros, the constructor state) / read back */
int qmb200_wbc_set_input_last(qmb200_handle* h, const double* input_last /*[B][30] or NULL*/);
int qmb200_wbc_get_input_last(qmb200_handle* h, double* input_last /*[B][30]*/);

/* WbcBase::dynamicCallback (qm_wbc/src/WbcBase.cpp:69-117, qm_wbc/cfg/wbcWigeht.cfg:7-47): the PD gains of the task formulators, replaceable at run time.
 * Takes effect for the next wbc_update / tick / update call on the handle's stream. */
typedef struct {
  double kp_swing, kd_swing, base_height_kp, base_height_kd, kp_base_linear, kd_base_linear, kp_base_angular, kd_base_angular;
  double kp_arm_joint[6], kd_arm_joint[6], kp_ee_linear[3], kd_ee_linear[3], kp_ee_angular[3], kd_ee_angular[3];
} qmb200_wbc_gains;
int qmb200_wbc_get_gains(const qmb200_handle* h, qmb200_wbc_gains* out);
int qmb200_wbc_set_gains(qmb200_handle* h, const qmb200_wbc_gains* gains);
/* Per-robot diagnostics of the last WBC update on this handle (the reference prints nothing: HoQp.cpp:143 drops qpOASES' return value):
 * diag[b] = it0 | it1 << 8 | it2 << 16 | nw << 24 — level-0 semismooth passes, active-set iterations of levels 1 and 2, final working-set size. */
int qmb200_wbc_get_diagnostics(qmb200_handle* h, int32_t* diag /*[B]*/);
/* Iteration caps of the WBC solver (defaults 30 / 80 ≙ nWSR = 100 of HoQp.cpp:141); a robot that hits one carries QMB200_ST_ITER_CAP.  <= 0 keeps the value. */
int qmb200_wbc_set_iteration_caps(qmb200_handle* h, int32_t level0_passes, int32_t active_set_iterations);

/* ---- MPC seam: ocs2::MPC_BASE::run → SqpSolver::run(t0, x0, t0+T), one SQP iteration (QMController.cpp:287-288,315-332),
 *      with the inputs the reference manager holds: mode schedule (SwitchedModelReferenceManager) and TargetTrajectories.
 *      The previous PrimalSolution (warm start, mpc.coldStart=false) lives in the handle. */
int qmb200_mpc_solve(qmb200_handle* h, const double* t0 /*[B]*/, const double* x0 /*[B][30]*/,
                     const int32_t* n_events /*[B]*/, const double* event_times /*[B][EMAX]*/, const int32_t* mode_sequence /*[B][EMAX+1]*/,
                     const int32_t* n_target /*[B]*/, const double* target_times /*[B][KMAX]*/, const double* target_states /*[B][KMAX][37]*/,
                     int32_t* n_nodes /*[B]*/, double* node_times /*[B][NMAX]*/, int32_t* node_events /*[B][NMAX]*/,
                     double* x_traj /*[B][NMAX][30]*/, double* u_traj /*[B][NMAX][30]*/, int32_t* status /*[B]*/, double* step_info /*[B][4] or NULL: alpha, cost, dyn SSE, eq SSE after the step*/);
int qmb200_mpc_solve_dev(qmb200_handle* h, const double* t0, const double* x0, const int32_t* n_events, const double* event_times, const int32_t* mode_sequence,
                         const int32_t* n_target, const double* target_times, const double* target_states, void* cuda_stream);
/* sqp.sqpIteration / costTol of the handle (task.info:28; the create-time values come from task.info): SqpSolver::runImpl runs up to that many
 * LQ → QP → line-search iterations per solve and leaves the loop early per robot on checkConvergence (step size, metrics, primal step) [upstream ocs2_sqp].
 * sqp_iterations <= 0 / cost_tol <= 0 keep the current value. */
int qmb200_mpc_set_iterations(qmb200_handle* h, int32_t sqp_iterations, double cost_tol);
/* drop the stored PrimalSolution: next solve starts from QMInitializer (qm_interface/src/initialization/QMInitializer.cpp:33-41) */
int qmb200_mpc_reset(qmb200_handle* h);
/* load a PrimalSolution as warm start (n_nodes[b] < 2 → cold start for robot b) */
int qmb200_mpc_set_solution(qmb200_handle* h, const int32_t* n_nodes, const double* node_times, const int32_t* node_events, const double* x_traj, const double* u_traj);
/* read the stored solution (device → host) */
int qmb200_mpc_get_solution(qmb200_handle* h, int32_t* n_nodes, double* node_times, int32_t* node_events, double* x_traj, double* u_traj, int32_t* status, double* step_info);

/* ---- MPC→WBC hand-off: MPC_MRT_Interface::evaluatePolicy(t, x, → optimizedState, optimizedInput, plannedMode) (QMController.cpp:141)
 *      on the stored solution and the mode schedule of the last solve. */
int qmb200_policy_eval(qmb200_handle* h, const double* t /*[B]*/, double* x_des /*[B][30]*/, double* u_des /*[B][30]*/, int32_t* mode /*[B]*/);
int qmb200_policy_eval_dev(qmb200_handle* h, const double* t, double* x_des, double* u_des, int32_t* mode, void* cuda_stream);

/* ---- feedback policy: useFeedbackPolicy of the ddp{} / sqp{} / ipm{} blocks (task.info:61,89,107).  When it is on, OCS2 stores the solve as an
 *      ocs2::LinearController u = uff(t) + K(t) x and MPC_MRT_Interface::evaluatePolicy(currentTime, currentState, ...) (QMController.cpp:141) reacts to the
 *      measured state between two MPC updates.  K_k = Px_k + Pu_k K~_k is the derivative of the QP's optimal input step at node k with respect to the state
 *      step (the projected Riccati gain mapped back to the full input), uff_k = u*_k - K_k x*_k on the stored solution; a pre-event node and the last node
 *      repeat the bias and gain of the node before them; bias and gain are interpolated separately on the node times.  Robots whose last solve carries
 *      QMB200_ST_NOT_PD, _NAN, _OVERFLOW or _NEG_DT keep the feed-forward policy (zero gain).  After qmb200_mpc_set_solution / qmb200_mpc_reset there is no
 *      controller until the next solve.  With the switch on, qmb200_tick evaluates at (t_eval, x0) and qmb200_update at (t_obs, x_obs); with it off every
 *      entry point evaluates the feed-forward policy, as before.  qmb200_create reads sqp.useFeedbackPolicy, qmb200_mpc_set_solver the chosen block's key. */
int qmb200_mpc_set_feedback_policy(qmb200_handle* h, int32_t on);
int qmb200_mpc_get_feedback_policy(const qmb200_handle* h, int32_t* on);
/* MPC_MRT_Interface::evaluatePolicy(currentTime, currentState, → optimizedState, optimizedInput, plannedMode): x_des and mode as qmb200_policy_eval; u_des of the
 * feedback policy at x (switch off: identical to qmb200_policy_eval, x is not read) */
int qmb200_policy_eval_state(qmb200_handle* h, const double* t /*[B]*/, const double* x /*[B][30]*/, double* x_des /*[B][30]*/, double* u_des /*[B][30]*/, int32_t* mode /*[B]*/);
int qmb200_policy_eval_state_dev(qmb200_handle* h, const double* t, const double* x, double* x_des, double* u_des, int32_t* mode, void* cuda_stream);
/* ocs2::LinearController of the last solve (timeStamp = the node times of qmb200_mpc_get_solution) for robots [b0, b0 + count): biasArray, gainArray (row = input,
 * column = state) per node, zero past the robot's node count; feedback[r] = 0 where the robot has the feed-forward controller (gain zero, bias = u*).
 * The host variant exports through a device scratch of at most 256 MB. */
int qmb200_mpc_get_controller(qmb200_handle* h, int32_t b0, int32_t count, double* bias /*[count][NMAX][30]*/, double* gain /*[count][NMAX][30][30]*/, int32_t* feedback /*[count]*/);
int qmb200_mpc_get_controller_dev(qmb200_handle* h, int32_t b0, int32_t count, double* bias, double* gain, int32_t* feedback, void* cuda_stream);

/* ---- value function: createValueFunction of the sqp{} / ipm{} blocks (OCS2 default false; the shipped task.info does not set it).  When it is on, the solve
 *      keeps what SqpSolver / IpmSolver::extractValueFunction keep after the QP of the robot's last iteration: per node k (node 0, event nodes and the terminal
 *      node included) dfdxx_k = P_k and dfdx_k = p_k - P_k xbar_k, where P_k, p_k are the Riccati cost-to-go of the state step dx_k in full state coordinates and
 *      xbar is that QP's linearization trajectory (the iterate before the step).  A robot that converged early keeps the value function of its last QP.
 *      getValueFunction(t, x) returns f = 0, dfdxx and dfdx interpolated linearly on the node times (the (index, alpha) of qmb200_policy_eval, clamped before the
 *      first and past the last node), then dfdx += dfdxx x.  valid[b] = 1 only when the last solve ran with the switch on, robot b's QP was factorised (no
 *      QMB200_ST_NOT_PD, _NAN, _OVERFLOW, _NEG_DT) and no qmb200_mpc_set_solution / qmb200_mpc_reset followed; elsewhere the outputs are zero.
 *      qmb200_create reads sqp.createValueFunction, qmb200_mpc_set_solver the chosen block's key; DDP turns the switch off (GaussNewtonDDP::getValueFunction has
 *      a different contract) and refuses it.  The records take NMAX * 3,968 B per robot, allocated when the switch is first turned on; if that allocation fails
 *      the call returns an error and the switch stays off.  With the switch off the solve is unchanged. */
int qmb200_mpc_set_value_function(qmb200_handle* h, int32_t on);
int qmb200_mpc_get_value_function(const qmb200_handle* h, int32_t* on);
int qmb200_value_function(qmb200_handle* h, const double* t /*[B]*/, const double* x /*[B][30]*/, double* dfdx /*[B][30]*/, double* dfdxx /*[B][30][30]*/, int32_t* valid /*[B]*/);
int qmb200_value_function_dev(qmb200_handle* h, const double* t, const double* x, double* dfdx, double* dfdxx, int32_t* valid, void* cuda_stream);

/* ---- one controller tick on the device: mpc_solve → policy_eval(t_eval) → wbc_update, torque buffer out.
 *      Host-pointer version: observation in, cmd out (the e2e path bench.py times). */
int qmb200_tick(qmb200_handle* h, const double* t0, const double* x0, const int32_t* n_events, const double* event_times, const int32_t* mode_sequence,
                const int32_t* n_target, const double* target_times, const double* target_states, const double* t_eval, const double* rbd,
                const double* period, double* cmd /*[B][54]*/, int32_t* status /*[B]*/);
int qmb200_tick_dev(qmb200_handle* h, const double* t0, const double* x0, const int32_t* n_events, const double* event_times, const int32_t* mode_sequence,
                    const int32_t* n_target, const double* target_times, const double* target_states, const double* t_eval, const double* rbd,
                    const double* period, double* cmd, int32_t* status, void* cuda_stream);

/* ---- observation: CentroidalModelRbdConversions::computeCentroidalStateFromRbdModel (QMController.cpp:238-241), host utility */
int qmb200_centroidal_state_from_rbd(const qmb200_handle* h, int32_t n, const double* rbd /*[n][55]*/, double* x /*[n][30]*/);

/* ---- gait front-end: GaitSchedule::getModeSchedule tiling of a ModeSequenceTemplate (QMInterface.cpp:455-480, gait.info) for one robot:
 *      STANCE until t_start, then the template repeated; window [lo, hi]; returns the number of events written (<= EMAX) or negative. */
int qmb200_gait_schedule(const char* gait_file, const char* gait_name, double t_start, double lo, double hi,
                         double* event_times /*[EMAX]*/, int32_t* mode_sequence /*[EMAX+1]*/);

/* ---- stateful gait front-end: ocs2::legged_robot::GaitSchedule as QMInterface::loadGaitSchedule builds it (QMInterface.cpp:455-480) and
 *      GaitReceiver / SwitchedModelReferenceManager drive it [upstream ocs2_legged_robot, recalled]: the schedule starts as
 *      reference.info:initialModeSchedule with defaultModeSequenceTemplate as the active template; a gait command
 *      (GaitJoyPublisher.cpp:35-60 → a gait.info template) is inserted at the end of the current horizon after phaseTransitionStanceTime
 *      of stance (task.info:9); every solve asks for the window [t0 - T, tf + T] (trim + tile).  Host object, one per robot. */
typedef struct qmb200_gait qmb200_gait;
int qmb200_gait_create(const char* task_file, const char* reference_file, qmb200_gait** out);
void qmb200_gait_destroy(qmb200_gait* g);
/* GaitSchedule::insertModeSequenceTemplate(template, startTime, finalTime); GaitReceiver passes (finalTime of the solve, timeHorizon) */
int qmb200_gait_insert_template(qmb200_gait* g, const char* gait_file, const char* gait_name, double start_time, double final_time);
/* GaitSchedule::getModeSchedule(lowerBoundTime, upperBoundTime): returns the number of events written (<= EMAX) or negative */
int qmb200_gait_get_mode_schedule(qmb200_gait* g, double lower_bound_time, double upper_bound_time, double* event_times /*[EMAX]*/, int32_t* mode_sequence /*[EMAX+1]*/);

/* ---- controller side of the path (SURVEY.md section 8f): the steps of QMController::update around evaluatePolicy / WbcBase::update and the
 *      publisher that feeds the solver, batched on the device.  The caller owns the per-robot controller state these functions read and
 *      write (the members of QMController / QmTargetTrajectoriesInteractiveMarker they mirror); `_dev` variants take device pointers. */
#define QMB200_TARGET_CMD_VEL 0      /* cmdVelToTargetTrajectories      (QmTargetTrajectoriesPublisher_node.cpp:73-113): cmd = vx, vy, vz, yaw rate */
#define QMB200_TARGET_EE_CMD_VEL 1   /* EeCmdVelToTargetTrajectories    (:118-165): cmd = vx, vy, vz of the end effector */
#define QMB200_TARGET_EE_GOAL 2      /* EEgoalPoseToTargetTrajectories  (:172-208) + processFeedback (QmTargetTrajectoriesPublisher.cpp:94-109): cmd = pos(3), quat xyzw(4) */
#define QMB200_JOINT_CMD 5           /* HybridJointHandle::setCommand(posDes, velDes, kp, kd, ff) (HybridJointInterface.h:55-61) */
#define QMB200_ST_SAFETY 0x10000     /* SafetyChecker::check failed (SafetyChecker.h:22-35): the reference stops the controller */
#define QMB200_ST_HW_RING_FULL 2     /* qmb200_hw_write: more than 32 commands inside the delay window (the oldest was dropped) */

/* QMController::updateStateEstimation tail (QMController.cpp:236-243): t_obs += period; x_obs = computeCentroidalStateFromRbdModel(rbd) with
 * the yaw unwrapped against the previous x_obs[9] (angles::shortest_angular_distance). */
int qmb200_observation_update(qmb200_handle* h, const double* rbd /*[B][55]*/, const double* period /*[B]*/, double* t_obs /*[B] in-out*/, double* x_obs /*[B][30] in-out*/);
int qmb200_observation_update_dev(qmb200_handle* h, const double* rbd, const double* period, double* t_obs, double* x_obs, void* cuda_stream);

/* TargetTrajectories from a command (QmTargetTrajectoriesPublisher_node.cpp:44-208) in the layout qmb200_mpc_solve takes; constants from
 * reference.info (comHeight, defaultJointState, target*Velocity) and task.info (mpc.timeHorizon).  last_ee_target mirrors lastEeTarget_
 * (initial value qmb200_initial_ee_target: QmTargetTrajectoriesPublisher.h:55-57). */
int qmb200_target_trajectories(qmb200_handle* h, int32_t kind, const double* cmd /*[B][7]*/, const double* t_obs /*[B]*/, const double* x_obs /*[B][30]*/, const double* ee_state /*[B][7] pos, quat xyzw*/,
                               double* last_ee_target /*[B][7] in-out*/, int32_t* n_target /*[B]*/, double* target_times /*[B][KMAX]*/, double* target_states /*[B][KMAX][37]*/);
int qmb200_target_trajectories_dev(qmb200_handle* h, int32_t kind, const double* cmd, const double* t_obs, const double* x_obs, const double* ee_state, double* last_ee_target,
                                   int32_t* n_target, double* target_times, double* target_states, void* cuda_stream);
void qmb200_initial_ee_target(double* last_ee_target7);

/* SafetyChecker::check + QMController::updateControlLaw (QMController.cpp:159-165,177-190) or, for a handle created with
 * QMB200_WBC_HIERARCHICAL_MPC, QMMpcController::updateControlLaw (:427-445).  joint_cmd entries the reference does not write in a given call
 * (legs before t = 10 s; the position-controlled arm of QMMpcController) keep their previous value, as the joint handles do. */
int qmb200_control_law(qmb200_handle* h, const double* x_des /*[B][30]*/, const double* u_des /*[B][30]*/, const double* wbc_cmd /*[B][54]*/, const double* t_obs /*[B]*/, const double* x_obs /*[B][30]*/,
                       double* joint_cmd /*[B][18][5] in-out*/, double* arm_pos_cmd /*[B][6] in-out*/, double* last_time /*[B] in-out*/, int32_t* status /*[B]*/);
int qmb200_control_law_dev(qmb200_handle* h, const double* x_des, const double* u_des, const double* wbc_cmd, const double* t_obs, const double* x_obs, double* joint_cmd, double* arm_pos_cmd,
                           double* last_time, int32_t* status, void* cuda_stream);
/* dynamic_reconfigure kp_arm_wbc / kd_arm_wbc (QMController.cpp:357-362; defaults 0.0 / 0.5, qm_controllers/cfg/weight.cfg:7-8) */
int qmb200_set_arm_gains(qmb200_handle* h, double kp_arm_wbc, double kd_arm_wbc);

/* Plant stand-in, QMHWSim::writeSim (qm_gazebo/src/QMHWSim.cpp:98-116): the commands pass a per-robot delay FIFO (kept in the handle) and
 * the joint effort is kp (posDes - q) + kd (velDes - qd) + ff.  time == period clears the FIFO (simulation reset). */
int qmb200_hw_write(qmb200_handle* h, const double* time /*[B]*/, const double* period /*[B]*/, const double* joint_cmd /*[B][18][5]*/, const double* joint_pos /*[B][18]*/, const double* joint_vel /*[B][18]*/,
                    double* effort /*[B][18]*/, int32_t* status /*[B]*/);
int qmb200_hw_write_dev(qmb200_handle* h, const double* time, const double* period, const double* joint_cmd, const double* joint_pos, const double* joint_vel, double* effort, int32_t* status, void* cuda_stream);
/* gazebo/delay (qm_gazebo/config/default.yaml:2; QMHWSim.cpp:33-35 defaults to 0); clears the FIFO */
int qmb200_hw_set_delay(qmb200_handle* h, double delay);

/* The whole QMController::update (QMController.cpp:128-175) on the stored policy: observation update → evaluatePolicy(t_obs) → WbcBase::update
 * (period, t_obs) → safety check + control law.  cmd = the WBC 54-vector, status = WBC status | QMB200_ST_SAFETY. */
int qmb200_update(qmb200_handle* h, const double* rbd /*[B][55]*/, const double* period /*[B]*/, double* t_obs /*[B] in-out*/, double* x_obs /*[B][30] in-out*/, double* joint_cmd /*[B][18][5] in-out*/,
                  double* arm_pos_cmd /*[B][6] in-out*/, double* last_time /*[B] in-out*/, double* cmd /*[B][54]*/, int32_t* status /*[B]*/);
int qmb200_update_dev(qmb200_handle* h, const double* rbd, const double* period, double* t_obs, double* x_obs, double* joint_cmd, double* arm_pos_cmd, double* last_time, double* cmd, int32_t* status, void* cuda_stream);

/* ---- tick pipeline: qmb200_tick / qmb200_tick_dev cut the batch into `chunks` (1..8) robot ranges and run each range's
 *      MPC solve → evaluatePolicy → WbcBase::update chain on its own CUDA stream (forked from / joined into the caller's stream), so
 *      kernels with different bottlenecks overlap on the SMs.  Robots are independent (the reference runs one controller per robot,
 *      QMController.cpp:128-148), so results do not depend on the setting.  Default: 1. */
int qmb200_set_pipeline(qmb200_handle* h, int chunks);

/* measurement support (bench.py): per-kernel device times of the tick [setup, lq, riccati, linesearch, policy_eval, wbc] in ms (mean per call),
 * and the measured fp64 FMA throughput of this GPU */
int qmb200_set_profiling(qmb200_handle* h, int on);
int qmb200_collect_kernel_times(qmb200_handle* h);
int qmb200_get_kernel_times(qmb200_handle* h, double* ms6);
/* the part of ms6[1] (LQ approximation) spent in the thread-per-node flow kernel (kinematics, flow maps, constraint rows); the rest is the warp-per-node projection kernel */
int qmb200_get_flow_kernel_time(qmb200_handle* h, double* ms);
int qmb200_measure_fp64_peak(qmb200_handle* h, double* tflops);

/* diagnostics: the QP step (dx, du) of the last solve and per-robot scalars [armijo, baseline cost, dyn SSE, eq SSE, |dx|, |du|, -, -] */
int qmb200_debug_get_step(qmb200_handle* h, double* dx /*[B][NMAX][30]*/, double* du /*[B][NMAX][30]*/, double* robot /*[B][8]*/);
/* ---- solver variants (SURVEY 8f-3).  QMInterface loads four solver blocks (QMInterface.cpp:69-73: ddp{}, sqp{}, ipm{}, rollout{}); QMController::setupMpc runs
 *      SqpMpc (QMController.cpp:287-288), the handle's default.  The other two blocks select, on the same OCP, LQ model (K2) and backward pass (K3):
 *      IPM  ocs2 IpmSolver with ipm{} (task.info:95-125).  The OCP of qm_interface has no inequality constraint terms (soft constraints + state-input
 *           equalities only, QMInterface.cpp:79-142), so the interior-point iteration carries no barrier / slack / dual variables and its primal step is the
 *           Newton step of the equality-constrained problem - the SQP step; what changes are the iteration count and the filter line-search thresholds
 *           (ipmIteration, deltaTol, g_max = 10, g_min).
 *      DDP  ocs2 GaussNewtonDDP with ddp{} (task.info:33-71) in its discrete-time form (ddp.algorithm ILQR; the file's SLQ integrates a continuous-time Riccati
 *           equation and ODE45 rollouts, which cannot be pinned without a reference run): nominal single-shooting rollout from the measured state, LQ
 *           approximation along it, the discrete Riccati backward pass, rollout line search of the affine controller on merit = cost + penalty * sqrt(ISE of
 *           the state-input equalities) over step lengths maxStepLength * 0.5^j >= minStepLength. */
#define QMB200_SOLVER_SQP 0
#define QMB200_SOLVER_IPM 1
#define QMB200_SOLVER_DDP 2
int qmb200_mpc_set_solver(qmb200_handle* h, int32_t solver);
int qmb200_mpc_get_solver(const qmb200_handle* h, int32_t* solver, int32_t* iterations, double* delta_tol, double* g_max, double* g_min);

/* ---- multi-GPU (SURVEY 8e): robots are independent, rank g owns a contiguous robot range, the only exchange per tick is ONE all-gather of the torque rows.
 *      NCCL is driven from this library (opened with dlopen at the first call: no link-time dependency).  Bootstrap: rank 0 calls qmb200_comm_get_unique_id and
 *      ships the 128 bytes to the other ranks by any means; every rank then calls qmb200_comm_init on its handle (collective, like ncclCommInitRank). */
#define QMB200_COMM_ID_BYTES 128
int qmb200_comm_get_unique_id(void* id128);
int qmb200_comm_init(qmb200_handle* h, int32_t nranks, int32_t rank, const void* id128);
int qmb200_comm_destroy(qmb200_handle* h);                                   /* also done by qmb200_destroy */
int qmb200_comm_info(const qmb200_handle* h, int32_t* nranks, int32_t* rank, int32_t* nccl_version);
/* torque_all[r * B + i][0:18] = torque rows (cmd[.][36:54]) of rank r's robot i, on every rank: one pack kernel + one ncclAllGather on `cuda_stream` (NULL: the
 * handle's stream).  nccl_comm: an ncclComm_t of the caller, or NULL for the handle's communicator (no communicator at all: single rank, plain copy).
 * perm (device, optional): the batch was submitted in gait-binned order, perm[p] = original local index of the robot at position p; the gathered buffer is in
 * ORIGINAL order.  All ranks must hold the same batch size. */
int qmb200_allgather_torque(qmb200_handle* h, void* nccl_comm, const double* cmd_local /*[B][54] device*/, const int32_t* perm /*[B] device or NULL*/,
                            double* torque_all /*[nranks * B][18] device*/, void* cuda_stream);
/* Host helper for mixed-gait batches (BASELINE configs[4]): permutation that sorts the robots by contact phase (stance code at t0, events in the window, time to the
 * next event); perm[p] = original index of the robot at position p. */
int qmb200_gait_bin_permutation(int32_t n, const double* t0, const int32_t* n_events, const double* event_times /*[n][EMAX]*/, const int32_t* modes /*[n][EMAX+1]*/, int32_t* perm /*[n]*/);

/* Host-only (no CUDA device needed): run the constructor chain's parsers (QMInterface::setupModel / setupOptimalControlProblem inputs: task.info, robot.urdf,
 * reference.info, optional gains file — batch / device of cfg are ignored) and copy the resulting model + settings constants (the block replicated to every GPU)
 * into out.  Returns the block size in bytes (also when out is NULL or capacity is too small: nothing is copied then), negative on a parse error
 * (qmb200_last_error(NULL)).  Used to check that two sets of input files define the same problem, bit for bit. */
int64_t qmb200_debug_model_blob(const qmb200_config* cfg, void* out, int64_t capacity);

/* number of kernels this library launched since create (bench.py's gpu_launches) */
int64_t qmb200_launch_count(const qmb200_handle* h);
/* stream the handle launches on (cudaStream_t as void*) */
void* qmb200_stream(const qmb200_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* QMB200_H */
