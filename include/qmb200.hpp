// qmb200.hpp — header-only C++17 host side above the C ABI (include/qmb200.h), mirroring the classes of qm_control that sit on the hot path:
// same names, argument meaning and error behaviour, so that code written against the reference reads the same.  No ROS / OCS2 / Eigen
// types: ocs2::vector_t becomes std::vector<double>; batched overloads take plain arrays.  There is no CPU fallback: constructing a solver
// without a CUDA device throws.
//
//   qm::QMInterface            qm_interface/include/qm_interface/QMInterface.h:28-104   (file triple; throws std::invalid_argument on missing files, QMInterface.cpp:45,53,61)
//   qm::WbcBase                qm_wbc/include/qm_wbc/WbcBase.h:24-118                   (update(stateDesired, inputDesired, rbdStateMeasured, mode, period, time) → vector_t[54])
//   qm::HierarchicalWbc        qm_wbc/include/qm_wbc/HierarchicalWbc.h, src/HierarchicalWbc.cpp:18-44
//   qm::HierarchicalMpcWbc     qm_wbc/src/HierarchicalMpcWbc.cpp:18-34
//   qm::SqpMpc                 the ocs2::SqpMpc + MPC_MRT_Interface pair QMController::setupMpc / setupMrt build (QMController.cpp:286-312)
//   qm::QMController           qm_controllers/include/qm_controllers/QMController.h:37-118 — numerical body of starting() / update() / advanceMpc()
#pragma once
#include <cstdint>
#include <fstream>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "qmb200.h"

namespace qm {

using scalar_t = double;
using vector_t = std::vector<double>;

class QMInterface {
 public:
  QMInterface(const std::string& taskFile, const std::string& urdfFile, const std::string& referenceFile) : taskFile_(taskFile), urdfFile_(urdfFile), referenceFile_(referenceFile) {
    if (!exists(taskFile)) throw std::invalid_argument("[QMInterface] Task file not found: " + taskFile);                  // QMInterface.cpp:45
    if (!exists(urdfFile)) throw std::invalid_argument("[QMInterface] URDF file not found: " + urdfFile);                  // :53
    if (!exists(referenceFile)) throw std::invalid_argument("[QMInterface] targetCommand file not found: " + referenceFile);   // :61
  }
  const std::string& taskFile() const { return taskFile_; }
  const std::string& urdfFile() const { return urdfFile_; }
  const std::string& referenceFile() const { return referenceFile_; }

 private:
  static bool exists(const std::string& p) { std::ifstream f(p); return f.good(); }
  std::string taskFile_, urdfFile_, referenceFile_;
};

// RAII owner of one qmb200_handle (one per GPU); shared by the WBC, the MPC and the controller mirrors.
class Solver {
 public:
  Solver(const QMInterface& interface, int batch = 1, int device = 0, int wbcVariant = QMB200_WBC_HIERARCHICAL, double timeHorizon = 0.0, double dt = 0.0, const std::string& wbcGainsFile = "") {
    qmb200_config cfg{}; cfg.task_file = interface.taskFile().c_str(); cfg.urdf_file = interface.urdfFile().c_str(); cfg.reference_file = interface.referenceFile().c_str();
    cfg.wbc_gains_file = wbcGainsFile.empty() ? nullptr : wbcGainsFile.c_str(); cfg.batch = batch; cfg.device = device; cfg.time_horizon = timeHorizon; cfg.dt = dt; cfg.max_nodes = 0; cfg.wbc_variant = wbcVariant;
    const int rc = qmb200_create(&cfg, &h_);
    if (rc == -2) throw std::invalid_argument(std::string("[qmb200] ") + qmb200_last_error(nullptr));    // unreadable / inconsistent input files
    if (rc != 0) throw std::runtime_error(std::string("[qmb200] ") + qmb200_last_error(nullptr));         // no CUDA device, out of memory, ...
    qmb200_get_dims(h_, &batch_, &nmax_, nullptr, nullptr);
  }
  ~Solver() { qmb200_destroy(h_); }
  Solver(const Solver&) = delete;
  Solver& operator=(const Solver&) = delete;
  qmb200_handle* get() const { return h_; }
  int batch() const { return batch_; }
  int maxNodes() const { return nmax_; }
  void check(int rc, const char* what) const { if (rc != 0) throw std::runtime_error(std::string(what) + ": " + qmb200_last_error(h_)); }

 private:
  qmb200_handle* h_ = nullptr; int32_t batch_ = 0, nmax_ = 0;
};

class WbcBase {
 public:
  explicit WbcBase(std::shared_ptr<Solver> solver) : solver_(std::move(solver)) {}
  virtual ~WbcBase() = default;
  virtual void loadTasksSetting(const std::string& /*taskFile*/, bool /*verbose*/) {}   // limits and friction are read at construction (WbcBase.cpp:565-596)

  // WbcBase.h:31-32, one robot (the handle must have batch 1): returns [vdot(24); F(12); tau(18)] (WbcBase.cpp:548-563).  Like the reference it never
  // reports a solver failure through the return value (HoQp.cpp:143); lastStatus() exposes the status word.
  virtual vector_t update(const vector_t& stateDesired, const vector_t& inputDesired, const vector_t& rbdStateMeasured, size_t mode, scalar_t period, scalar_t time) {
    if (solver_->batch() != 1) throw std::runtime_error("WbcBase::update(vector_t ...): the handle was created with batch != 1, use the array overload");
    if (stateDesired.size() != QMB200_NX || inputDesired.size() != QMB200_NU || rbdStateMeasured.size() != QMB200_RBD) throw std::runtime_error("WbcBase::update: wrong vector size");
    vector_t cmd(QMB200_CMD); const int32_t m = static_cast<int32_t>(mode);
    solver_->check(qmb200_wbc_update(solver_->get(), stateDesired.data(), inputDesired.data(), rbdStateMeasured.data(), &m, &period, &time, cmd.data(), &status_), "WbcBase::update");
    return cmd;
  }
  // batched: arrays over the handle's robots ([B][30], [B][30], [B][55], [B], [B], [B] → [B][54], [B])
  void update(const double* stateDesired, const double* inputDesired, const double* rbdStateMeasured, const int32_t* mode, const double* period, const double* time, double* cmd, int32_t* status) {
    solver_->check(qmb200_wbc_update(solver_->get(), stateDesired, inputDesired, rbdStateMeasured, mode, period, time, cmd, status), "WbcBase::update");
  }
  int32_t lastStatus() const { return status_; }
  // WbcBase::dynamicCallback (WbcBase.cpp:69-117)
  qmb200_wbc_gains gains() const { qmb200_wbc_gains g{}; solver_->check(qmb200_wbc_get_gains(solver_->get(), &g), "WbcBase::gains"); return g; }
  void dynamicCallback(const qmb200_wbc_gains& config) { solver_->check(qmb200_wbc_set_gains(solver_->get(), &config), "WbcBase::dynamicCallback"); }

 protected:
  std::shared_ptr<Solver> solver_; int32_t status_ = 0;
};

class HierarchicalWbc : public WbcBase {
 public:
  explicit HierarchicalWbc(const QMInterface& interface, int batch = 1, int device = 0) : WbcBase(std::make_shared<Solver>(interface, batch, device, QMB200_WBC_HIERARCHICAL)) {}
  explicit HierarchicalWbc(std::shared_ptr<Solver> solver) : WbcBase(std::move(solver)) {}
};
class HierarchicalMpcWbc : public WbcBase {
 public:
  explicit HierarchicalMpcWbc(const QMInterface& interface, int batch = 1, int device = 0) : WbcBase(std::make_shared<Solver>(interface, batch, device, QMB200_WBC_HIERARCHICAL_MPC)) {}
  explicit HierarchicalMpcWbc(std::shared_ptr<Solver> solver) : WbcBase(std::move(solver)) {}
};

// ocs2::ModeSchedule / ocs2::TargetTrajectories in the solver's flat layout (one robot)
struct ModeSchedule { std::vector<double> eventTimes; std::vector<int32_t> modeSequence; };          // modeSequence.size() == eventTimes.size() + 1
struct TargetTrajectories { std::vector<double> timeTrajectory; std::vector<vector_t> stateTrajectory; };   // states of 37 = 30 + EE pose
// ocs2::LinearController of one robot: u(t, x) = bias(t) + gain(t) x, piecewise linear in t on timeStamp (gainArray[k]: 30 x 30 row-major, row = input).
// feedback == false: the feed-forward controller (no solve since the last set_solution / reset, or the last QP had no defined gain).
struct LinearController { std::vector<double> timeStamp; std::vector<vector_t> biasArray, gainArray; bool feedback = false; };
// ocs2::ScalarFunctionQuadraticApproximation of the value function at (t, x): f (0, as SqpSolver::getValueFunction leaves it), dfdx (30), dfdxx (30 x 30 row-major)
struct ValueFunction { scalar_t f = 0.0; vector_t dfdx, dfdxx; };
struct PrimalSolution { std::vector<double> timeTrajectory; std::vector<int32_t> postEventAnnotation; std::vector<vector_t> stateTrajectory, inputTrajectory; int32_t status = 0; double stepSize = 0.0; };

// SqpMpc + MPC_MRT_Interface for one robot (QMController.cpp:286-312): run() = MPC_BASE::run (sqp.sqpIteration SQP iterations, warm started), evaluatePolicy()
class SqpMpc {
 public:
  explicit SqpMpc(std::shared_ptr<Solver> solver) : solver_(std::move(solver)) { if (solver_->batch() != 1) throw std::runtime_error("SqpMpc: the single-robot mirror needs a batch-1 handle"); }
  void reset() { solver_->check(qmb200_mpc_reset(solver_->get()), "SqpMpc::reset"); }
  // the other solver blocks QMInterface loads (QMInterface.cpp:69-73): ocs2::IpmMpc with ipm{} / ocs2::GaussNewtonDDP_MPC with ddp{} on the same OCP (qmb200.h: QMB200_SOLVER_*)
  void setSolver(int32_t solver) { solver_->check(qmb200_mpc_set_solver(solver_->get(), solver), "SqpMpc::setSolver"); }
  PrimalSolution run(scalar_t initTime, const vector_t& initState, const ModeSchedule& modeSchedule, const TargetTrajectories& targets) {
    if (initState.size() != QMB200_NX) throw std::runtime_error("SqpMpc::run: wrong state size");
    const int32_t ne = static_cast<int32_t>(modeSchedule.eventTimes.size()), nk = static_cast<int32_t>(targets.timeTrajectory.size());
    if (ne > QMB200_EMAX || modeSchedule.modeSequence.size() != modeSchedule.eventTimes.size() + 1) throw std::runtime_error("SqpMpc::run: bad mode schedule");
    if (nk < 1 || nk > QMB200_KMAX || targets.stateTrajectory.size() != targets.timeTrajectory.size()) throw std::runtime_error("SqpMpc::run: bad target trajectories");
    double ev[QMB200_EMAX] = {0}; int32_t md[QMB200_EMAX + 1];
    for (int i = 0; i <= QMB200_EMAX; ++i) md[i] = 15;
    for (int i = 0; i < ne; ++i) ev[i] = modeSchedule.eventTimes[i];
    for (int i = 0; i <= ne; ++i) md[i] = modeSchedule.modeSequence[i];
    double tk[QMB200_KMAX] = {0}; std::vector<double> ts(QMB200_KMAX * QMB200_TARGET, 0.0);
    for (int k = 0; k < nk; ++k) { tk[k] = targets.timeTrajectory[k]; if (targets.stateTrajectory[k].size() != QMB200_TARGET) throw std::runtime_error("SqpMpc::run: target state must have 37 entries"); for (int i = 0; i < QMB200_TARGET; ++i) ts[k * QMB200_TARGET + i] = targets.stateTrajectory[k][i]; }
    const int nmax = solver_->maxNodes(); int32_t n = 0, status = 0; std::vector<double> t(nmax), x(nmax * QMB200_NX), u(nmax * QMB200_NU); std::vector<int32_t> e(nmax); double info[4];
    solver_->check(qmb200_mpc_solve(solver_->get(), &initTime, initState.data(), &ne, ev, md, &nk, tk, ts.data(), &n, t.data(), e.data(), x.data(), u.data(), &status, info), "SqpMpc::run");
    PrimalSolution sol; sol.status = status; sol.stepSize = info[0];
    for (int k = 0; k < n; ++k) { sol.timeTrajectory.push_back(t[k]); sol.postEventAnnotation.push_back(e[k]); sol.stateTrajectory.emplace_back(x.begin() + k * QMB200_NX, x.begin() + (k + 1) * QMB200_NX); sol.inputTrajectory.emplace_back(u.begin() + k * QMB200_NU, u.begin() + (k + 1) * QMB200_NU); }
    return sol;
  }
  // MPC_MRT_Interface::evaluatePolicy(currentTime, currentState, → optimizedState, optimizedInput, plannedMode) (QMController.cpp:141; feed-forward policy)
  void evaluatePolicy(scalar_t currentTime, vector_t& optimizedState, vector_t& optimizedInput, size_t& plannedMode) {
    optimizedState.resize(QMB200_NX); optimizedInput.resize(QMB200_NU); int32_t mode = 0;
    solver_->check(qmb200_policy_eval(solver_->get(), &currentTime, optimizedState.data(), optimizedInput.data(), &mode), "SqpMpc::evaluatePolicy"); plannedMode = static_cast<size_t>(mode);
  }
  // the reference's signature: with setFeedbackPolicy(true) the input reacts to currentState (u = uff(t) + K(t) x), otherwise the overload above
  void evaluatePolicy(scalar_t currentTime, const vector_t& currentState, vector_t& optimizedState, vector_t& optimizedInput, size_t& plannedMode) {
    if (currentState.size() != QMB200_NX) throw std::runtime_error("SqpMpc::evaluatePolicy: wrong state size");
    optimizedState.resize(QMB200_NX); optimizedInput.resize(QMB200_NU); int32_t mode = 0;
    solver_->check(qmb200_policy_eval_state(solver_->get(), &currentTime, currentState.data(), optimizedState.data(), optimizedInput.data(), &mode), "SqpMpc::evaluatePolicy"); plannedMode = static_cast<size_t>(mode);
  }
  // useFeedbackPolicy of the solver block (task.info:61,89,107); setSolver() re-reads the chosen block's value
  void setFeedbackPolicy(bool on) { solver_->check(qmb200_mpc_set_feedback_policy(solver_->get(), on ? 1 : 0), "SqpMpc::setFeedbackPolicy"); }
  // createValueFunction of the solver block; setSolver() re-reads the chosen block's value (DDP: off, and turning it on throws)
  void setValueFunction(bool on) { solver_->check(qmb200_mpc_set_value_function(solver_->get(), on ? 1 : 0), "SqpMpc::setValueFunction"); }
  // SqpSolver::getValueFunction(time, state) (MPC_MRT_Interface::getValueFunction); throws std::runtime_error when there is none, as OCS2 does when
  // valueFunction_ is empty (switch off at the last solve, set_solution / reset since, or the last QP was not factorised)
  ValueFunction getValueFunction(scalar_t time, const vector_t& state) {
    if (state.size() != QMB200_NX) throw std::runtime_error("SqpMpc::getValueFunction: wrong state size");
    ValueFunction v; v.dfdx.resize(QMB200_NX); v.dfdxx.resize((size_t)QMB200_NX * QMB200_NX); int32_t valid = 0;
    solver_->check(qmb200_value_function(solver_->get(), &time, state.data(), v.dfdx.data(), v.dfdxx.data(), &valid), "SqpMpc::getValueFunction");
    if (!valid) throw std::runtime_error("SqpMpc::getValueFunction: no value function (createValueFunction off at the last solve, no solve since set_solution / reset, or the QP was not factorised)");
    return v;
  }
  // PrimalSolution::controllerPtr_ as a LinearController (MPC_MRT_Interface::getPolicy)
  LinearController getLinearController() {
    const int nmax = solver_->maxNodes(); int32_t n = 0, fb = 0; std::vector<double> t(nmax), bias((size_t)nmax * QMB200_NU), gain((size_t)nmax * QMB200_NU * QMB200_NX);
    solver_->check(qmb200_mpc_get_solution(solver_->get(), &n, t.data(), nullptr, nullptr, nullptr, nullptr, nullptr), "SqpMpc::getLinearController");
    solver_->check(qmb200_mpc_get_controller(solver_->get(), 0, 1, bias.data(), gain.data(), &fb), "SqpMpc::getLinearController");
    LinearController c; c.feedback = fb != 0;
    for (int k = 0; k < n; ++k) { c.timeStamp.push_back(t[k]); c.biasArray.emplace_back(bias.begin() + (size_t)k * QMB200_NU, bias.begin() + (size_t)(k + 1) * QMB200_NU);
      c.gainArray.emplace_back(gain.begin() + (size_t)k * QMB200_NU * QMB200_NX, gain.begin() + (size_t)(k + 1) * QMB200_NU * QMB200_NX); }
    return c;
  }

 private:
  std::shared_ptr<Solver> solver_;
};

// Numerical body of QMController (one robot): starting() / advanceMpc() / update(); the ROS handles stay with the caller, which applies jointCommand()
// to its HybridJointHandles.  QMMpcController = the same with a HierarchicalMpcWbc handle.
class QMController {
 public:
  struct HybridJointCommand { double posDes, velDes, kp, kd, ff; };
  explicit QMController(const QMInterface& interface, int device = 0, bool mpcArmVariant = false)
      : solver_(std::make_shared<Solver>(interface, 1, device, mpcArmVariant ? QMB200_WBC_HIERARCHICAL_MPC : QMB200_WBC_HIERARCHICAL)), mpc_(solver_), state_(QMB200_NX, 0.0), jointCmd_(18 * QMB200_JOINT_CMD, 0.0), armPosCmd_(6, 0.0) {}
  // QMController::starting (QMController.cpp:98-126): first observation from the measured state
  void starting(const vector_t& measuredRbdState, scalar_t time) {
    if (measuredRbdState.size() != QMB200_RBD) throw std::runtime_error("QMController::starting: rbd state must have 55 entries");
    solver_->check(qmb200_centroidal_state_from_rbd(solver_->get(), 1, measuredRbdState.data(), state_.data()), "QMController::starting"); time_ = time; lastTime_ = time; mpc_.reset();
  }
  // mpcMrtInterface_->advanceMpc() (QMController.cpp:315-332) on the current observation
  PrimalSolution advanceMpc(const ModeSchedule& modeSchedule, const TargetTrajectories& targets) { return mpc_.run(time_, state_, modeSchedule, targets); }
  // QMController::update (QMController.cpp:128-175): returns false when the safety check fails (the reference calls stopRequest)
  bool update(const vector_t& measuredRbdState, scalar_t period, vector_t& wbcOutput) {
    if (measuredRbdState.size() != QMB200_RBD) throw std::runtime_error("QMController::update: rbd state must have 55 entries");
    wbcOutput.resize(QMB200_CMD); int32_t status = 0;
    solver_->check(qmb200_update(solver_->get(), measuredRbdState.data(), &period, &time_, state_.data(), jointCmd_.data(), armPosCmd_.data(), &lastTime_, wbcOutput.data(), &status), "QMController::update");
    status_ = status; return (status & QMB200_ST_SAFETY) == 0;
  }
  HybridJointCommand jointCommand(int j) const { const double* c = jointCmd_.data() + QMB200_JOINT_CMD * j; return {c[0], c[1], c[2], c[3], c[4]}; }
  double armPositionCommand(int j) const { return armPosCmd_[j]; }
  scalar_t observationTime() const { return time_; }
  const vector_t& observationState() const { return state_; }
  int32_t lastStatus() const { return status_; }
  void dynamicCallback(double kp_arm_wbc, double kd_arm_wbc) { solver_->check(qmb200_set_arm_gains(solver_->get(), kp_arm_wbc, kd_arm_wbc), "QMController::dynamicCallback"); }   // QMController.cpp:357-362
  Solver& solver() { return *solver_; }

 private:
  std::shared_ptr<Solver> solver_; SqpMpc mpc_; scalar_t time_ = 0.0, lastTime_ = 0.0; vector_t state_, jointCmd_, armPosCmd_; int32_t status_ = 0;
};

}  // namespace qm
