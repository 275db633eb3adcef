// C-ABI of libqmb200 (include/qmb200.h).  Host logic only: argument checks, device buffers, stream ordering,
// kernel launches.  No CPU fallback: every compute entry point launches the sm_100a kernels or fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/qmb200.h"
#include "host/qm_config.h"
#include "kernels/mpc_api.cuh"
#include "kernels/ctrl_api.cuh"

namespace qmb {
void launch_wbc_update(const DevModel* mdl, int B, const double* x_des, const double* u_des, const double* rbd, const int32_t* mode, const double* period, const double* time,
                       double* input_last, int variant, double* cmd, int32_t* status, cudaStream_t stream, int b0 = 0, int b1 = -1, int32_t* diag = nullptr);
int wbc_configure_device();   // per-device kernel attributes (opt-in shared memory): wbc_kernel.cu / mpc_kernels.cu
int mpc_configure_device();
}

using namespace qmb;

static thread_local std::string g_create_error;

struct qmb200_handle {
  HostModel hm;
  DevModel* d_model = nullptr;
  int B = 0, nmax = 0, variant = 0, device = 0;
  cudaStream_t stream = nullptr;
  std::string err, task_file;   // task_file: qmb200_mpc_set_solver re-reads the sqp{} / ipm{} / ddp{} block
  int64_t launches = 0;
  // staging for the host-pointer API
  double *d_xdes = nullptr, *d_udes = nullptr, *d_rbd = nullptr, *d_period = nullptr, *d_time = nullptr, *d_cmd = nullptr, *d_input_last = nullptr, *d_teval = nullptr, *d_xeval = nullptr;
  int32_t *d_mode = nullptr, *d_status = nullptr, *d_wbc_diag = nullptr;   // d_wbc_diag: per-robot WBC iteration counts (qmb200_wbc_get_diagnostics), kept out of the status word
  MpcBuffers mpc;   // device buffers of the MPC path (kernels/mpc_api.cuh)
  std::vector<void*> allocs;
  bool profiling = false; cudaEvent_t ev[8] = {nullptr};   // [0..4] MPC kernels, [5..6] policy / wbc brackets, [7] flow kernel | LQ kernel
  double kernel_ms[7] = {0, 0, 0, 0, 0, 0, 0}; int64_t kernel_calls = 0; bool ev_pending = false;   // kernel_ms[6]: the flow kernel's share of [1]
  // tick pipeline: the batch is cut into `chunks` robot ranges, each running its MPC → policy → WBC chain on its own stream, so that
  // kernels with different bottlenecks (LQ: instruction latency, Riccati: shared-memory bandwidth, WBC) share the SMs
  static constexpr int MAX_CHUNKS = 8;
  // controller-side constants and staging (capi_ctrl.inc)
  TargetParams target_prm{}; ControlLawParams law_prm{0, 0.0, 0.5};
  bool c_ready = false; double *c_tobs = nullptr, *c_xobs = nullptr, *c_jcmd = nullptr, *c_armpos = nullptr, *c_lasttime = nullptr, *c_cmd7 = nullptr, *c_ee = nullptr, *c_lastee = nullptr,
                               *c_jpos = nullptr, *c_jvel = nullptr, *c_effort = nullptr, *c_ttimes = nullptr, *c_tstates = nullptr; int32_t *c_status = nullptr, *c_ntarget = nullptr;
  double hw_delay = 0.0; double *hw_ring_cmd = nullptr, *hw_ring_stamp = nullptr; int32_t* hw_ring_state = nullptr;   // QMHWSim command-delay FIFO
  void* comm = nullptr; int comm_ranks = 0, comm_rank = 0; double* d_send = nullptr;   // NCCL communicator of this handle (capi_comm.inc) and the packed torque rows
  int chunks = 1; cudaStream_t cs[MAX_CHUNKS] = {nullptr}; cudaEvent_t fork_ev = nullptr, join_ev[MAX_CHUNKS] = {nullptr};
  // useFeedbackPolicy of the active solver block; has_controller: the stage records / projected gains belong to the stored solution (a solve ran since the
  // last set_solution / reset).  Policy evaluation is feedback only when both hold.
  bool feedback_policy = false, has_controller = false;
  double *d_ctrl_bias = nullptr, *d_ctrl_gain = nullptr; int32_t* d_ctrl_fb = nullptr; int ctrl_rows = 0;   // bounded scratch of qmb200_mpc_get_controller
  bool feedback_on() const { return feedback_policy && has_controller; }
  // createValueFunction of the active solver block (never on with DDP); has_value_function: the last solve ran with it on and no set_solution / reset
  // followed, so mpc.vf holds that solve's records.  qmb200_value_function reports a robot valid when this holds and its last QP was factorised.
  bool value_function = false, has_value_function = false;
  double *d_vf_dfdx = nullptr, *d_vf_dfdxx = nullptr; int32_t* d_vf_valid = nullptr;   // staging of qmb200_value_function
};

namespace {
template <class T> bool dalloc(qmb200_handle* h, T** p, size_t count) {
  void* q = nullptr; cudaError_t e = cudaMalloc(&q, count * sizeof(T));
  if (e != cudaSuccess) { h->err = std::string("cudaMalloc failed: ") + cudaGetErrorString(e); return false; }
  cudaMemsetAsync(q, 0, count * sizeof(T), h->stream); h->allocs.push_back(q); *p = static_cast<T*>(q); return true;   // zeroed in stream order with the handle's work (lazy allocators synchronise once, see ctrl_alloc)
}
int fail(qmb200_handle* h, const std::string& msg) { if (h) h->err = msg; else g_create_error = msg; return -1; }
#define QMB_CUDA(h, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(h, std::string(#call) + ": " + cudaGetErrorString(e_)); } while (0)
}  // namespace

extern "C" {

int qmb200_create(const qmb200_config* cfg, qmb200_handle** out) {
  if (!cfg || !out) return fail(nullptr, "qmb200_create: null argument");
  if (!cfg->task_file || !cfg->urdf_file || !cfg->reference_file) return fail(nullptr, "qmb200_create: task/urdf/reference file required");
  if (cfg->batch < 1) return fail(nullptr, "qmb200_create: batch must be >= 1");
  qmb200_handle* h = new qmb200_handle();
  try {
    h->hm = build_host_model(cfg->task_file, cfg->urdf_file, cfg->reference_file, cfg->wbc_gains_file ? cfg->wbc_gains_file : "");
    // constants of the target publisher node (QmTargetTrajectoriesPublisher_node.cpp:225-229)
    InfoFile ref(cfg->reference_file), task(cfg->task_file);
    h->target_prm.com_height = ref.number("comHeight"); h->target_prm.target_displacement_velocity = ref.number("targetDisplacementVelocity");
    h->target_prm.target_rotation_velocity = ref.number("targetRotationVelocity"); h->target_prm.time_to_target = task.number("mpc.timeHorizon");
    for (int j = 0; j < NJ; ++j) h->target_prm.default_joint_state[j] = h->hm.default_joint_state[j];
    h->feedback_policy = task.boolean("sqp.useFeedbackPolicy", false);   // the handle starts with SqpMpc (QMController.cpp:287-288)
    h->value_function = task.boolean("sqp.createValueFunction", false);
  } catch (const std::exception& e) { g_create_error = e.what(); delete h; return -2; }
  if (cfg->time_horizon > 0) h->hm.dev.time_horizon = cfg->time_horizon;
  if (cfg->dt > 0) h->hm.dev.dt = cfg->dt;
  h->task_file = cfg->task_file;
  h->B = cfg->batch; h->variant = cfg->wbc_variant; h->device = cfg->device; h->law_prm.variant = cfg->wbc_variant == QMB200_WBC_HIERARCHICAL_MPC ? 1 : 0;
  const int nint = (int)std::ceil(h->hm.dev.time_horizon / h->hm.dev.dt - 1e-9);
  h->nmax = cfg->max_nodes > 0 ? cfg->max_nodes : nint + 1 + 20;
  int ndev = 0; cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) { g_create_error = std::string("qmb200_create: no CUDA device (") + cudaGetErrorString(e) + ") — this library has no CPU fallback"; delete h; return -3; }
  if (cudaSetDevice(cfg->device) != cudaSuccess) { g_create_error = "qmb200_create: cudaSetDevice failed"; delete h; return -3; }
  cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  // kernel attributes are per device: set them for THIS handle's device (a process may hold handles on several GPUs)
  if (wbc_configure_device() != 0 || mpc_configure_device() != 0) { g_create_error = std::string("qmb200_create: cudaFuncSetAttribute failed: ") + cudaGetErrorString(cudaGetLastError()); qmb200_destroy(h); return -3; }
  const size_t B = (size_t)h->B;
  bool ok = dalloc(h, &h->d_model, 1) && dalloc(h, &h->d_xdes, B * NX) && dalloc(h, &h->d_udes, B * NU) && dalloc(h, &h->d_rbd, B * QMB200_RBD) && dalloc(h, &h->d_period, B) &&
            dalloc(h, &h->d_time, B) && dalloc(h, &h->d_cmd, B * QMB200_CMD) && dalloc(h, &h->d_input_last, B * NU) && dalloc(h, &h->d_mode, B) && dalloc(h, &h->d_status, B) && dalloc(h, &h->d_teval, B) && dalloc(h, &h->d_xeval, B * NX) && dalloc(h, &h->d_wbc_diag, B);
  if (ok) { std::string merr; ok = mpc_alloc(h->mpc, h->B, h->nmax, merr, h->allocs, h->stream); if (!ok) h->err = merr; }
  if (ok && h->value_function) ok = dalloc(h, &h->mpc.vf, B * h->nmax * VF_DBL);   // 3,968 B per robot and node
  if (!ok) { g_create_error = h->err; qmb200_destroy(h); return -4; }
  cudaMemcpyAsync(h->d_model, &h->hm.dev, sizeof(DevModel), cudaMemcpyHostToDevice, h->stream);
  if (cudaStreamSynchronize(h->stream) != cudaSuccess) { g_create_error = std::string("qmb200_create: ") + cudaGetErrorString(cudaGetLastError()); qmb200_destroy(h); return -4; }   // buffers zeroed, constants resident before any (user-stream) launch
  *out = h; return 0;
}

void qmb200_destroy(qmb200_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  qmb200_comm_destroy(h);
  if (h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
  for (int c = 0; c < qmb200_handle::MAX_CHUNKS; ++c) { if (h->cs[c]) { cudaStreamSynchronize(h->cs[c]); cudaStreamDestroy(h->cs[c]); } if (h->join_ev[c]) cudaEventDestroy(h->join_ev[c]); }
  if (h->fork_ev) cudaEventDestroy(h->fork_ev);
  for (void* p : h->allocs) cudaFree(p);
  delete h;
}

const char* qmb200_last_error(const qmb200_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int64_t qmb200_debug_model_blob(const qmb200_config* cfg, void* out, int64_t capacity) {
  if (!cfg || !cfg->task_file || !cfg->urdf_file || !cfg->reference_file) { g_create_error = "qmb200_debug_model_blob: task/urdf/reference file required"; return -1; }
  try {
    HostModel hm = build_host_model(cfg->task_file, cfg->urdf_file, cfg->reference_file, cfg->wbc_gains_file ? cfg->wbc_gains_file : "");
    if (cfg->time_horizon > 0) hm.dev.time_horizon = cfg->time_horizon; if (cfg->dt > 0) hm.dev.dt = cfg->dt;
    if (out && capacity >= (int64_t)sizeof(DevModel)) std::memcpy(out, &hm.dev, sizeof(DevModel));
    return (int64_t)sizeof(DevModel);
  } catch (const std::exception& e) { g_create_error = e.what(); return -2; }
}

int qmb200_get_dims(const qmb200_handle* h, int32_t* batch, int32_t* nmax, int32_t* emax, int32_t* kmax) {
  if (!h) return -1; if (batch) *batch = h->B; if (nmax) *nmax = h->nmax; if (emax) *emax = QMB200_EMAX; if (kmax) *kmax = QMB200_KMAX; return 0;
}
int qmb200_get_model_info(const qmb200_handle* h, double* robot_mass, double* initial_state30, double* default_joint_state18, double* time_horizon, double* dt) {
  if (!h) return -1;
  if (robot_mass) *robot_mass = h->hm.dev.total_mass;
  if (initial_state30) std::memcpy(initial_state30, h->hm.initial_state, sizeof(double) * NX);
  if (default_joint_state18) std::memcpy(default_joint_state18, h->hm.default_joint_state, sizeof(double) * NJ);
  if (time_horizon) *time_horizon = h->hm.dev.time_horizon; if (dt) *dt = h->hm.dev.dt; return 0;
}
int qmb200_get_joint_name(const qmb200_handle* h, int32_t joint, char* out, int32_t capacity) {
  if (!h || joint < 0 || joint >= NJ || !out || capacity < 1) return -1; std::snprintf(out, capacity, "%s", h->hm.joint_names[joint].c_str()); return 0;
}
int64_t qmb200_launch_count(const qmb200_handle* h) { return h ? h->launches : 0; }
void* qmb200_stream(const qmb200_handle* h) { return h ? (void*)h->stream : nullptr; }

// ------------------------------------------------------------------ WBC
int qmb200_wbc_update_dev(qmb200_handle* h, const double* x_des, const double* u_des, const double* rbd, const int32_t* mode, const double* period, const double* time,
                          double* cmd, int32_t* status, void* cuda_stream) {
  if (!h) return -1; if (!x_des || !u_des || !rbd || !mode || !period || !time || !cmd || !status) return fail(h, "qmb200_wbc_update_dev: null buffer");
  QMB_CUDA(h, cudaSetDevice(h->device));
  launch_wbc_update(h->d_model, h->B, x_des, u_des, rbd, mode, period, time, h->d_input_last, h->variant, cmd, status, cuda_stream ? (cudaStream_t)cuda_stream : h->stream, 0, -1, h->d_wbc_diag);
  h->launches += 1;
  QMB_CUDA(h, cudaGetLastError());
  return 0;
}

int qmb200_wbc_update(qmb200_handle* h, const double* x_des, const double* u_des, const double* rbd, const int32_t* mode, const double* period, const double* time, double* cmd, int32_t* status) {
  if (!h) return -1; if (!x_des || !u_des || !rbd || !mode || !period || !time || !cmd || !status) return fail(h, "qmb200_wbc_update: null buffer");
  QMB_CUDA(h, cudaSetDevice(h->device));
  const size_t B = (size_t)h->B; cudaStream_t s = h->stream;
  QMB_CUDA(h, cudaMemcpyAsync(h->d_xdes, x_des, B * NX * 8, cudaMemcpyHostToDevice, s)); QMB_CUDA(h, cudaMemcpyAsync(h->d_udes, u_des, B * NU * 8, cudaMemcpyHostToDevice, s));
  QMB_CUDA(h, cudaMemcpyAsync(h->d_rbd, rbd, B * QMB200_RBD * 8, cudaMemcpyHostToDevice, s)); QMB_CUDA(h, cudaMemcpyAsync(h->d_mode, mode, B * 4, cudaMemcpyHostToDevice, s));
  QMB_CUDA(h, cudaMemcpyAsync(h->d_period, period, B * 8, cudaMemcpyHostToDevice, s)); QMB_CUDA(h, cudaMemcpyAsync(h->d_time, time, B * 8, cudaMemcpyHostToDevice, s));
  int rc = qmb200_wbc_update_dev(h, h->d_xdes, h->d_udes, h->d_rbd, h->d_mode, h->d_period, h->d_time, h->d_cmd, h->d_status, s); if (rc) return rc;
  QMB_CUDA(h, cudaMemcpyAsync(cmd, h->d_cmd, B * QMB200_CMD * 8, cudaMemcpyDeviceToHost, s)); QMB_CUDA(h, cudaMemcpyAsync(status, h->d_status, B * 4, cudaMemcpyDeviceToHost, s));
  QMB_CUDA(h, cudaStreamSynchronize(s));
  return 0;
}
int qmb200_wbc_set_input_last(qmb200_handle* h, const double* input_last) {
  if (!h) return -1; QMB_CUDA(h, cudaSetDevice(h->device));
  if (input_last) QMB_CUDA(h, cudaMemcpyAsync(h->d_input_last, input_last, (size_t)h->B * NU * 8, cudaMemcpyHostToDevice, h->stream)); else QMB_CUDA(h, cudaMemsetAsync(h->d_input_last, 0, (size_t)h->B * NU * 8, h->stream));
  QMB_CUDA(h, cudaStreamSynchronize(h->stream)); return 0;
}
int qmb200_wbc_get_input_last(qmb200_handle* h, double* input_last) {
  if (!h || !input_last) return -1; QMB_CUDA(h, cudaSetDevice(h->device));
  QMB_CUDA(h, cudaMemcpyAsync(input_last, h->d_input_last, (size_t)h->B * NU * 8, cudaMemcpyDeviceToHost, h->stream)); QMB_CUDA(h, cudaStreamSynchronize(h->stream)); return 0;
}

int qmb200_wbc_get_gains(const qmb200_handle* h, qmb200_wbc_gains* g) {
  if (!h || !g) return -1; const DevModel& d = h->hm.dev;
  g->kp_swing = d.kp_swing; g->kd_swing = d.kd_swing; g->base_height_kp = d.base_height_kp; g->base_height_kd = d.base_height_kd; g->kp_base_linear = d.base_linear_kp; g->kd_base_linear = d.base_linear_kd;
  g->kp_base_angular = d.base_angular_kp; g->kd_base_angular = d.base_angular_kd;
  for (int i = 0; i < 6; ++i) { g->kp_arm_joint[i] = d.arm_joint_kp[i]; g->kd_arm_joint[i] = d.arm_joint_kd[i]; }
  for (int i = 0; i < 3; ++i) { g->kp_ee_linear[i] = d.ee_linear_kp[i]; g->kd_ee_linear[i] = d.ee_linear_kd[i]; g->kp_ee_angular[i] = d.ee_angular_kp[i]; g->kd_ee_angular[i] = d.ee_angular_kd[i]; }
  return 0;
}
int qmb200_wbc_set_gains(qmb200_handle* h, const qmb200_wbc_gains* g) {
  if (!h) return -1; if (!g) return fail(h, "qmb200_wbc_set_gains: null gains");
  QMB_CUDA(h, cudaSetDevice(h->device)); DevModel& d = h->hm.dev;
  d.kp_swing = g->kp_swing; d.kd_swing = g->kd_swing; d.base_height_kp = g->base_height_kp; d.base_height_kd = g->base_height_kd; d.base_linear_kp = g->kp_base_linear; d.base_linear_kd = g->kd_base_linear;
  d.base_angular_kp = g->kp_base_angular; d.base_angular_kd = g->kd_base_angular;
  for (int i = 0; i < 6; ++i) { d.arm_joint_kp[i] = g->kp_arm_joint[i]; d.arm_joint_kd[i] = g->kd_arm_joint[i]; }
  for (int i = 0; i < 3; ++i) { d.ee_linear_kp[i] = g->kp_ee_linear[i]; d.ee_linear_kd[i] = g->kd_ee_linear[i]; d.ee_angular_kp[i] = g->kp_ee_angular[i]; d.ee_angular_kd[i] = g->kd_ee_angular[i]; }
  // stream-ordered update of the replicated constants: kernels already queued keep the old gains, later ones see the new
  QMB_CUDA(h, cudaMemcpyAsync(h->d_model, &h->hm.dev, sizeof(DevModel), cudaMemcpyHostToDevice, h->stream)); QMB_CUDA(h, cudaStreamSynchronize(h->stream)); return 0;
}

// Per-robot WBC diagnostics of the last update on this handle: it0 | it1 << 8 | it2 << 16 | nw << 24 (level-0 semismooth passes, active-set iterations of
// levels 1 and 2, final working-set size).  They used to ride in the status word, where they collided with the MPC / safety bits.
int qmb200_wbc_get_diagnostics(qmb200_handle* h, int32_t* diag) {
  if (!h || !diag) return -1; QMB_CUDA(h, cudaSetDevice(h->device));
  QMB_CUDA(h, cudaMemcpyAsync(diag, h->d_wbc_diag, (size_t)h->B * 4, cudaMemcpyDeviceToHost, h->stream)); QMB_CUDA(h, cudaStreamSynchronize(h->stream)); return 0;
}
// Iteration caps of the WBC solver (defaults 30 / 80; robots that hit a cap carry QMB200_ST_ITER_CAP).  <= 0 keeps the current value.
int qmb200_wbc_set_iteration_caps(qmb200_handle* h, int32_t level0_passes, int32_t active_set_iterations) {
  if (!h) return -1; QMB_CUDA(h, cudaSetDevice(h->device));
  if (level0_passes > 0) h->hm.dev.wbc_iter_cap0 = level0_passes; if (active_set_iterations > 0) h->hm.dev.wbc_iter_cap = active_set_iterations;
  QMB_CUDA(h, cudaMemcpyAsync(h->d_model, &h->hm.dev, sizeof(DevModel), cudaMemcpyHostToDevice, h->stream)); QMB_CUDA(h, cudaStreamSynchronize(h->stream)); return 0;
}

}  // extern "C"

#include "capi_mpc.inc"
#include "capi_ctrl.inc"
#include "capi_comm.inc"
