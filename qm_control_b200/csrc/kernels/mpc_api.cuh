// Host-visible interface of the MPC kernels: device buffers of one handle and the launchers.
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "dev_common.cuh"

namespace qmb {

constexpr int EMAX = 32, KMAX = 4, TARGET_DIM = 37;
// Per-node projected LQ stage as the LQ kernel (K2) hands it to the Riccati kernel (K3): the STRUCTURED record (11,872 B instead of the 32,576 B of the dense
// round-1 record).  The projected problem is stored in the model's sparsity, and every dense piece has the row pitch of the shared-memory matrix it lands in, so
// that K3 fetches a node with bulk copies (cp.async.bulk → SASS UBLKCP, signalled on mbarriers: one each for the A~ rows, the B~ rows and the tail, one per row of Q~) instead of ~1700 16-byte cp.async:
//   A~ = I + [rows 3:12 dense] + [leg-joint rows 12:24: dtw * Px on the 12 support columns of the leg]      B~ = [rows 0:3: dtw/m at free force columns]
//   + [rows 3:12 dense] + [joint rows: dtw at the own free column, dtw * Pu2 in the eliminated pivot row of a swing leg]
//   R~ is block diagonal over input triples (<= 3 entries per row), S~ has <= 8 non-zero rows (free joints of swing legs) of 12 support entries.
constexpr int LDX = 36, LDB = 28, LDG = 34, LDH = 24;   // shared-memory pitches of the 30-, 18-column matrices of K3 (see mpc_kernels.cu)
constexpr int ST_AR = 0;                 // 9 x LDX : rows 3:12 of A~ ; column 30 = b~[3:12] ; columns 31.. zero
constexpr int ST_BR = ST_AR + 9 * LDX;   // 9 x LDB : rows 3:12 of B~ ; columns 18.. zero
constexpr int ST_Q = ST_BR + 9 * LDB;    // Q~ (symmetric): LOWER triangle, row r = r + 1 entries padded to an even count (rows stay 16-byte aligned: one bulk copy
                                         //   per row into the pitch-LDX buffer); q~ travels in the tail      (terminal node: the final cost)
constexpr int Q_PACKED = 480;            //   sum over r < 30 of 2 * ((r + 2) / 2)
__host__ __device__ constexpr int q_row_offset(int r) { return (r & 1) ? 2 * ((r >> 1) + 1) * ((r >> 1) + 1) : 2 * (r >> 1) * ((r >> 1) + 1); }
__host__ __device__ constexpr int q_row_padded(int r) { return (r + 2) & ~1; }
static_assert(q_row_offset(29) + q_row_padded(29) == Q_PACKED && q_row_offset(1) == 2 && q_row_offset(2) == 4 && q_row_offset(3) == 8, "packed lower triangle with even rows");
constexpr int ST_TAIL = ST_Q + Q_PACKED; // the small pieces, one contiguous block:
constexpr int T_PXJ = 0;                 //   12 x 12: Px rows of the 12 leg-joint velocity inputs on their support columns (zero rows for free joints)
constexpr int T_b = 144, T_q = 174, T_r = 204;   // b~ (30), q~ (30), r~ (18)
constexpr int T_RT = 222;                //   18 x 3 : R~[a][column of input 3*(fa/3) + jc] (arm inputs: [a][0] = diagonal); rows a >= m: identity padding
constexpr int T_SJ = 276;                //   8 x 12 : S~ rows of the free joints of swing legs (slot = 2 * foot + position among the leg's two free joints)
constexpr int T_PU2 = 372, T_PED = 380;  //   Pu2 (4 feet x 2), P_e of the dependent inputs (16)
constexpr int T_MISC = 396;              //   dtw = dt (w1 + w2), cost, dynamics SSE, equality SSE of the node
constexpr int T_INT = 400;               //   int32[56]: type (0 intermediate, 1 event, 2 terminal), m, ndep, dep[16], free[18], pivot[4] (joint eliminated in a swing leg, -1 stance),
                                         //   pcol[4][2] (projected columns of a swing leg's two free joints, -1 stance)
constexpr int TAIL_DBL = 428, STAGE_DBL = ST_TAIL + TAIL_DBL;
constexpr int SI_TYPE = 0, SI_M = 1, SI_NDEP = 2, SI_DEP = 3, SI_FREE = 19, SI_PIV = 37, SI_PCOL = 41;
static_assert(STAGE_DBL == 1484 && (ST_BR % 2 == 0) && (ST_Q % 2 == 0) && (ST_TAIL % 2 == 0) && (TAIL_DBL % 2 == 0), "16-byte aligned pieces");
constexpr int GAIN_DBL = 18 * LDG;       // feedback K (m x 30) with the pitch of its shared-memory target, feedforward k in column 30
constexpr int ROBOT_DBL = 8;                 // armijo, base cost, base dyn SSE, base eq SSE, |dx|, |du|
// Value function record of one node (createValueFunction): dfdxx = P_k as a packed lower triangle (entry (r, c), c <= r, at r (r + 1) / 2 + c), then
// dfdx = p_k - P_k xbar_k (xbar: the linearization trajectory of the QP), padded to an even count
constexpr int VF_P = 465, VF_DBL = 496;
static_assert(VF_P == 30 * 31 / 2 && VF_DBL >= VF_P + 30 && VF_DBL % 2 == 0, "value function record");

// PrimalSolution of every robot: node count, node times, event annotation (0 none, 1 pre-event, 2 post-event), x, u
struct MpcSolutionDev { int32_t* n_nodes = nullptr; double* t = nullptr; int32_t* event = nullptr; double* x = nullptr; double* u = nullptr; };

struct MpcBuffers {
  int B = 0, nmax = 0, cur = 0;
  // inputs of the last solve (kept for policy evaluation: mode schedule)
  double *t0 = nullptr, *x0 = nullptr, *event_times = nullptr, *target_times = nullptr, *target_states = nullptr;
  int32_t *n_events = nullptr, *modes = nullptr, *n_target = nullptr;
  MpcSolutionDev sol[2];
  double *ddp_trial = nullptr;  // DDP line search: cost and equality SSE of every step length, [B][32][2]
  double *node_rec = nullptr;   // K2a -> K2b: per node the flow-map / constraint / end-effector record (ne::NodeRec, 492 doubles)
  double *stage = nullptr, *gains = nullptr, *dx = nullptr, *du = nullptr, *robot = nullptr, *step_info = nullptr;
  double *vf = nullptr;         // [B][nmax][VF_DBL] value function of the last QP (createValueFunction), allocated by the handle on first use
  int32_t *stage_i = nullptr, *status = nullptr;
};
bool mpc_alloc(MpcBuffers& m, int B, int nmax, std::string& err, std::vector<void*>& allocs, cudaStream_t stream);
int mpc_configure_device();   // per-device opt-in shared memory of the MPC kernels (qmb200_create, after cudaSetDevice)

struct MpcProblemDev { const double* t0; const double* x0; const int32_t* n_events; const double* event_times; const int32_t* modes; const int32_t* n_target; const double* target_times; const double* target_states; };

// One SQP iteration for robots [b0, b1) (4 kernels on `stream`): reads m.sol[m.cur], writes m.sol[1 - m.cur]; the caller
// flips m.cur after queueing every range.  Returns the number of kernels launched.
// `ev` (optional, 8 events): [0..4] recorded before K1 and after each of K1, K2 (flow + LQ), K3, K4 for per-kernel timing; [7] between the flow kernel and the LQ kernel.
// `value_fn`: K3 also stores every node's value function into m.vf (which must be allocated); the launch count does not change.
int mpc_solve_launch(const DevModel* mdl, const DevModel& host_mdl, MpcBuffers& m, const MpcProblemDev& p, int b0, int b1, cudaStream_t stream, cudaEvent_t* ev = nullptr, bool value_fn = false);
// fp64 FMA throughput microbenchmark (roofline denominator for the compute-bound kernels); returns TFLOP/s
double measure_fp64_peak(cudaStream_t stream);
// evaluatePolicy on m.sol[m.cur]; returns kernels launched
int mpc_policy_eval_launch(const MpcBuffers& m, const double* t, double* x_des, double* u_des, int32_t* mode, cudaStream_t stream, int b0 = 0, int b1 = -1);
// evaluatePolicy(t, x): with `feedback` the LinearController of the last solve (stage record + projected gains, u = uff(t) + K(t) x), otherwise exactly
// mpc_policy_eval_launch (x is not read).  One launch either way; returns kernels launched
int mpc_policy_launch(const DevModel* mdl, const MpcBuffers& m, bool feedback, const double* t, const double* x, double* x_des, double* u_des, int32_t* mode, cudaStream_t stream, int b0 = 0, int b1 = -1);
// dense LinearController of robots [b0, b0 + count): bias [count][nmax][30], gain [count][nmax][30][30] (row = input), feedback flag [count]; `valid` false (no
// solve since the last set_solution / reset) exports the feed-forward controller
int mpc_controller_export_launch(const DevModel* mdl, const MpcBuffers& m, bool valid, int b0, int count, double* bias, double* gain, int32_t* feedback, cudaStream_t stream);
// getValueFunction(t, x) of every robot: dfdxx [B][30][30] (full, symmetric) and dfdx [B][30] of the stored records interpolated on the node times as
// mpc_policy_eval_launch interpolates, plus dfdxx x; valid[b] = `valid` and robot b's last QP was factorised.  Zero outputs where valid[b] = 0.  Returns kernels launched
int mpc_value_function_launch(const MpcBuffers& m, bool valid, const double* t, const double* x, double* dfdx, double* dfdxx, int32_t* valid_out, cudaStream_t stream);
// input fix-up after loading a solution from the host (inputs at pre-event / last nodes)
int mpc_fixup_launch(const MpcBuffers& m, cudaStream_t stream);

}  // namespace qmb
