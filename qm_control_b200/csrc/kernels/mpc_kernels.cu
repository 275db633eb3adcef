// Batched one-iteration multiple-shooting SQP (the MPC tick of qm_control):
//   SqpSolver::runImpl as QMController configures it (qm_controllers/src/QMController.cpp:287-288, task.info:75-92)
//   [upstream ocs2_sqp / ocs2_oc multiple_shooting, recalled — SURVEY.md App. A.5]:
//     K1 mpc_setup_kernel      timeDiscretizationWithEvents + initializeStateInputTrajectories (QMInitializer.cpp:33-41 when cold)
//     K2 setupQuadraticSubproblem in two kernels: mpc_flow_kernel (one THREAD per node: kinematics, both RK2 flow maps with Jacobian blocks, constraint rows,
//        end-effector error) -> 3.9 KB node record -> mpc_lq_kernel (one warp per node: cost quadratic model, projection, RK2 sensitivities, structured stage record)
//     K3 mpc_riccati_kernel    OCP-QP (HPIPM without inequality rows = Riccati backward/forward sweep) + armijo metric: one CTA per robot (the recursion is
//        sequential in time), every 30x30 block in shared memory, products on fp64 tensor-core tiles, records fetched by TMA bulk copies
//     K4 mpc_linesearch_kernel takeStep: filter line search, trajectory update: one CTA per robot, one thread per node
//     mpc_rollout_kernel       DDP variant: single-shooting rollouts, one thread per robot (and step length)
#include <cstdlib>
#include "mpc_api.cuh"
#include "mpc_device.cuh"
#include "node_eval.cuh"
#include "wlinalg.cuh"

namespace qmb {

#ifndef QMB_LQ_WARPS
#define QMB_LQ_WARPS 4
#endif
#ifndef QMB_LQ_MINB
#define QMB_LQ_MINB 4
#endif
constexpr int LQ_WARPS = QMB_LQ_WARPS, LS_WARPS = 4, SETUP_WARPS = 4;
enum { MST_ITER_CAP = 1, MST_OVERFLOW = 2, MST_NAN = 4, MST_NOT_PD = 8, MST_NO_STEP = 16, MST_CONVERGED = 32, MST_NEG_DT = 64 };   // NEG_DT: an interval with non-positive duration (include/qmb200.h)   // CONVERGED: checkConvergence stopped the SQP loop before sqpIteration

__device__ __forceinline__ double interval_start(double t, int ev) { return ev == 2 ? t + WEAK_EPS : t; }
__device__ __forceinline__ double interval_end(double t, int ev) { return ev == 1 ? t - WEAK_EPS : t; }
// caller-provided counts are clamped on every use (the _dev entry points take arbitrary device arrays); K1 flags an out-of-range count with MST_OVERFLOW
__device__ __forceinline__ int clamp_events(int ne) { return ne < 0 ? 0 : (ne > EMAX ? EMAX : ne); }
__device__ __forceinline__ int clamp_targets(int nk) { return nk < 1 ? 1 : (nk > KMAX ? KMAX : nk); }
__device__ __forceinline__ int flag_mask(int mode) { int m = 0; for (int i = 0; i < 4; ++i) if (contact_flag(mode, i)) m |= 1 << i; return m; }

// =====================================================================================================
// K1: time grid + initial guess
// per-warp shared-memory staging of K1 (nmax entries each): previous grid, new grid, and for every interval of the new grid where its values come from
struct SetupIdx { int iu, ix; double au, ax; };
__host__ __device__ inline size_t setup_smem_per_warp(int nmax) { return (size_t)nmax * (8 + 8 + 4 + sizeof(SetupIdx) + 4) + 8 * EMAX + 64; }
__global__ void __launch_bounds__(32 * SETUP_WARPS) mpc_setup_kernel(const DevModel* __restrict__ mdl, int b0, int B, int nmax, MpcProblemDev p, MpcSolutionDev prev, MpcSolutionDev next, int32_t* __restrict__ status) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31; const int b = b0 + blockIdx.x * SETUP_WARPS + warp; if (b >= B) return;
  extern __shared__ __align__(16) unsigned char s_setup[];
  unsigned char* base = s_setup + (size_t)warp * ((setup_smem_per_warp(nmax) + 15) & ~(size_t)15);
  double* spt = reinterpret_cast<double*>(base); double* sgt = spt + nmax; SetupIdx* sidx = reinterpret_cast<SetupIdx*>(sgt + nmax); double* sev = reinterpret_cast<double*>(sidx + nmax);
  int32_t* sge = reinterpret_cast<int32_t*>(sev + EMAX); int32_t* sflag = sge + nmax; unsigned char* smodes = reinterpret_cast<unsigned char*>(sflag + nmax);
  const double t0 = p.t0[b], tf = t0 + mdl->time_horizon, dt = mdl->dt; const int ne = clamp_events(p.n_events[b]); int st = 0;
  if (ne != p.n_events[b] || clamp_targets(p.n_target[b]) != p.n_target[b]) st |= MST_OVERFLOW;
  { const double* gev = p.event_times + (size_t)b * EMAX; const int32_t* gmodes = p.modes + (size_t)b * (EMAX + 1); sev[lane] = (lane < ne) ? gev[lane] : 0.0; smodes[lane] = (unsigned char)((lane <= ne) ? gmodes[lane] : 15); if (lane == 0) smodes[EMAX] = (unsigned char)((EMAX <= ne) ? gmodes[EMAX] : 15); }
  __syncwarp();
  const double* ev = sev; const unsigned char* modes = smodes;
  // ---- timeDiscretizationWithEvents [upstream ocs2_oc/oc_data/TimeDiscretization.cpp]: sequential by nature, kept in registers / shared memory ----
  int n = 0;
  if (lane == 0) {
    const double dt_min = 10.0 * 1e-9; /* 10 * ocs2 numeric_traits::limitEpsilon [upstream] */ double last_t = t0; int last_e = 0; sgt[0] = t0; sge[0] = 0; n = 1; int next_ev = lower_bound_idx(ev, ne, t0);
    while (last_t < tf) {
      double nt = last_t + dt; int nev = 0; bool is_event = false;
      if (next_ev < ne && nt >= ev[next_ev]) { nt = ev[next_ev]; is_event = true; nev = 1; ++next_ev; }
      if (nt >= tf) { is_event = false; nt = tf; nev = 0; }
      if (nt > last_t + dt_min) { if (n >= nmax) { st |= MST_OVERFLOW; break; } sgt[n] = nt; sge[n] = nev; ++n; last_t = nt; last_e = nev; } else if (last_e != 2) { sgt[n - 1] = nt; sge[n - 1] = nev; last_t = nt; last_e = nev; } else if (nt >= tf) break;
      if (is_event) { if (n >= nmax) { st |= MST_OVERFLOW; break; } sgt[n] = nt; sge[n] = 2; ++n; last_t = nt; last_e = 2; }
    }
    next.n_nodes[b] = n;
  }
  n = __shfl_sync(FULL, n, 0); st |= __shfl_sync(FULL, st, 0);
  __syncwarp();
  double* gt = next.t + (size_t)b * nmax; int32_t* ge = next.event + (size_t)b * nmax;
  for (int i = lane; i < n; i += 32) { gt[i] = sgt[i]; ge[i] = sge[i]; }
  // ---- initializeStateInputTrajectories [upstream ocs2_oc/multiple_shooting/Initialization.cpp] ----
  const int np = prev.n_nodes ? prev.n_nodes[b] : 0; const bool has_prev = np >= 2;
  { const double* gpt = prev.t + (size_t)b * nmax; for (int i = lane; i < np && i < nmax; i += 32) spt[i] = gpt[i]; __syncwarp(); }
  const double* pt = spt; const double* __restrict__ px = prev.x + (size_t)b * nmax * NX; const double* __restrict__ pu = prev.u + (size_t)b * nmax * NU;
  const double state_till = has_prev ? pt[np - 1] : t0, input_till = has_prev ? pt[np - 2] : t0;
  double* __restrict__ gx = next.x + (size_t)b * nmax * NX; double* __restrict__ gu = next.u + (size_t)b * nmax * NU;
  // where every interval takes its values from (lane = interval: the binary searches over the previous grid run 32 at a time):
  //   flag 2 pre-event node (no input, state carried), 1 warm start (interpolation of the previous solution), 0 QMInitializer (weight-compensating input, state held)
  for (int k = lane; k < n - 1; k += 32) {
    int flag = 2; SetupIdx ix{0, 0, 1.0, 1.0};
    if (sge[k] != 1) {
      const double t = interval_start(sgt[k], sge[k]), tn = interval_end(sgt[k + 1], sge[k + 1]);
      if (!has_prev || t > input_till || tn > state_till) { flag = 0; ix.iu = mode_at_time(ev, modes, ne, t); }   // QMInitializer::compute: the mode selects the weight-compensating input
      else { flag = 1; time_segment(pt, np, t, ix.iu, ix.au); time_segment(pt, np, tn, ix.ix, ix.ax); }
    }
    sflag[k] = flag; sidx[k] = ix;
  }
  __syncwarp();
  auto lerp = [&](const double* __restrict__ traj, int idx, double a) { return (lane < NX) ? a * traj[(size_t)idx * NX + lane] + (1.0 - a) * traj[(size_t)(idx + 1 < np ? idx + 1 : idx) * NX + lane] : 0.0; };
  double xk;
  { const double ti = interval_start(sgt[0], sge[0]); if (has_prev && ti < state_till) { int idx; double a; time_segment(pt, np, ti, idx, a); xk = lerp(px, idx, a); } else xk = (lane < NX ? p.x0[(size_t)b * NX + lane] : 0.0); }
  if (lane < NX) gx[lane] = xk;
  // sequential only through the carried state; the loads of an interval do not depend on the previous one, so four intervals are in flight
#pragma unroll 4
  for (int k = 0; k < n - 1; ++k) {
    const int flag = sflag[k]; const SetupIdx ix = sidx[k]; double uk = 0.0;
    if (flag == 1) { uk = lerp(pu, ix.iu, ix.au); xk = lerp(px, ix.ix, ix.ax); }
    else if (flag == 0) { const int mode = ix.iu; int nst = 0; for (int i = 0; i < 4; ++i) nst += contact_flag(mode, i); if (lane < 12 && (lane % 3) == 2 && contact_flag(mode, lane / 3)) uk = mdl->total_mass * 9.81 / nst; }
    if (lane < NX) { gu[(size_t)k * NU + lane] = uk; gx[(size_t)(k + 1) * NX + lane] = xk; }
  }
  if (lane < NX && n >= 1) gu[(size_t)(n - 1) * NU + lane] = 0.0;
  if (lane == 0) status[b] = st;
}

// =====================================================================================================
// K2: linear-quadratic approximation + projection of one node (one warp per node).
// Everything is kept in the model's natural sparsity: the continuous Jacobians have 9 non-trivial rows, the velocity
// constraint of a foot touches 12 state columns (h, euler angles, own leg joints) and its own 3 joint-velocity inputs,
// the input weight couples joint velocities only inside a leg.  The projection is therefore assembled per leg
// (3x12 blocks) and written straight into the dense stage record the Riccati kernel consumes.
struct LqLate { double BrdF[9 * 12], BrdJ[3 * NJ], bvec[NX]; };                // produced by the RK2 combination, after the cost / projection blocks have consumed rec.foot and rec.ee
struct alignas(16) LqSmem {   // 16-byte vector loads of the record: every warp's slice starts 16-byte aligned
  ne::NodeRec rec;                                                             // the node's record from the flow kernel (K2a); LqLate overlays rec.foot[] once the cost / projection / Jacobian expansion have consumed it
  QuadWs quad; LegWs leg[4];
  double x[NX], u[NU];                                                         // (x, u) of the node in the layout stage_cost_quad reads (x then u)
  double A1r[9 * NX], Ar[9 * NX];                                              // rows 3:12 of df/dx at the two RK2 stages; A1r becomes A_d - I in place.  Until expand_flow fills it, Ar holds the robot's mode schedule
  double Pe_full[NU], rs[NU];
  int dep_idx[MAXDEP], free_idx[MU], col_of_input[NU];
};
static_assert(9 * NX * 8 >= EMAX * 8 + EMAX + 8, "the mode schedule (event times + modes) is staged in the Ar buffer until the flow Jacobians are expanded");
static_assert(sizeof(LqLate) <= 4 * sizeof(ne::FootBlk) && offsetof(ne::NodeRec, foot) == 0, "LqLate overlays the foot blocks of the record");
static_assert(sizeof(LqSmem) % 16 == 0 && offsetof(LqSmem, rec) == 0, "aligned record slice");
static_assert((sizeof(LqSmem) * LQ_WARPS + 1024) * QMB_LQ_MINB <= 232448, "projection kernel: QMB_LQ_MINB CTAs of LQ_WARPS warps per SM (13.8 KB per node: four CTAs of four warps = 16 nodes in flight)");

// =====================================================================================================
// K2a: flow kernel - one THREAD per node (node_eval.cuh).  Kinematics of the five chains, both RK2 stages of the flow map with their Jacobian blocks, the
// foot-velocity rows with their Jacobians and the end-effector error with its Jacobian: 492 doubles per node, handed to K2b through HBM (written once, read once,
// both fully coalesced: the warp transposes 32 thread-private records through shared memory, K2b's warp reads its node's record as one contiguous run).
#ifndef QMB_FL_MINB
#define QMB_FL_MINB 2
#endif
constexpr int FL_WARPS = 4, FL_TILE = 64;   // widest block of the record: a foot (63 doubles)
constexpr int FL_SMEM = FL_WARPS * 32 * (FL_TILE + 1) * 8;
__global__ void __launch_bounds__(32 * FL_WARPS, QMB_FL_MINB) mpc_flow_kernel(const DevModel* __restrict__ mdl, int b0, int B, int nmax, MpcProblemDev p, MpcSolutionDev sol, double* __restrict__ rec, const int32_t* __restrict__ status) {
  // Each block of the record is produced straight into the lane's row of the warp's transposition tile (shared memory: the record never lives in thread-local
  // memory - with 57 k resident threads a 4 KB stack frame is 230 MB, more than the L2) and leaves as one contiguous run per node and store instruction.
  extern __shared__ __align__(16) unsigned char smem_raw[]; double (*tile)[32][FL_TILE + 1] = reinterpret_cast<double (*)[32][FL_TILE + 1]>(smem_raw);   // [FL_WARPS][32][FL_TILE + 1]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31; const long long gid = (long long)blockIdx.x * (32 * FL_WARPS) + tid;
  const int b = b0 + (int)(gid / nmax), k = (int)(gid % nmax);
  const int n = (b < B) ? sol.n_nodes[b] : 0;
  bool work = b < B && k < n && !(status[b] & MST_CONVERGED);
  const bool terminal = work && (k == n - 1);
  if (work && !terminal && sol.event[(size_t)b * nmax + k] == 1) work = false;   // event node: identity jump map, nothing to evaluate
  const unsigned active = __ballot_sync(FULL, work); if (!active) return;
  double* row = &tile[warp][lane][0]; double* gbase = rec + ((size_t)b0 * nmax + (size_t)(gid - lane)) * ne::NODE_REC_DBL;   // node index = robot * nmax + k, as K2b reads it
  auto flush = [&](int off, int cnt) {   // rows of the tile -> records: 32 (or 64) consecutive doubles of one node per store instruction
    __syncwarp();
#pragma unroll 4
    for (int rw = 0; rw < 32; ++rw) if ((active >> rw) & 1u) { double* g = gbase + (size_t)rw * ne::NODE_REC_DBL + off; if (lane < cnt) g[lane] = tile[warp][rw][lane]; if (lane + 32 < cnt) g[lane + 32] = tile[warp][rw][lane + 32]; }
    __syncwarp(); };
  double x[NX], u[NU]; ne::BaseKin bk; ne::FlowAcc acc; double t = 0.0, dt = 0.0;
  if (work) {
    const double* gt = sol.t + (size_t)b * nmax; const int32_t* ge = sol.event + (size_t)b * nmax;
    const double* xk = sol.x + ((size_t)b * nmax + k) * NX; const double* uk = sol.u + ((size_t)b * nmax + k) * NU;
#pragma unroll
    for (int i = 0; i < NX; ++i) { x[i] = xk[i]; u[i] = terminal ? 0.0 : uk[i]; }
    t = interval_start(gt[k], ge[k]); dt = terminal ? 0.0 : interval_end(gt[k + 1], ge[k + 1]) - t;
    ne::base_eval<true>(mdl, x, bk); ne::flow_acc_init(acc);
  }
#pragma unroll 1
  for (int i = 0; i < 4; ++i) {   // foot blocks: kinematics of the leg, foot-velocity rows
    if (work) { ne::FootBlk* fb = reinterpret_cast<ne::FootBlk*>(row); double al[9];
      ne::foot_eval<true>(mdl, x, u, bk, i, acc, fb->d, fb->pf, fb->Jl, al, fb->JxF);
      if (!terminal) ne::foot_velocity_1<true>(mdl, x, u, bk, i, fb->d, fb->Jl, al, fb->e, fb->C); }
    flush(i * ne::FOOT_DBL, ne::FOOT_DBL);
  }
  double f1[12];
  if (work) { ne::FlowBlk* fl = reinterpret_cast<ne::FlowBlk*>(row); ne::flow_finish<true>(mdl, x, bk, acc, fl->f, fl);
#pragma unroll
    for (int i = 0; i < 12; ++i) f1[i] = fl->f[i]; }
  flush(4 * ne::FOOT_DBL, ne::FLOW_DBL);
  { ne::EeRec ee;   // end-effector error and its Jacobian: 78 doubles, two flushes
    if (work) { const int nk = clamp_targets(p.n_target[b]); const ne::TargetSeg sg = ne::target_segment(p.target_times + (size_t)b * KMAX, p.target_states + (size_t)b * KMAX * TARGET_DIM, nk, t);
      double pref[3], qref[4]; ne::target_pose(sg, nk, pref, qref); ne::ee_eval<true>(mdl, x, bk, pref, qref, ee.e, ee.Je);
#pragma unroll
      for (int j = 0; j < 39; ++j) row[j] = reinterpret_cast<const double*>(&ee)[j]; }
    flush(4 * ne::FOOT_DBL + ne::FLOW_DBL, 39);
    if (work) {
#pragma unroll
      for (int j = 0; j < 39; ++j) row[j] = reinterpret_cast<const double*>(&ee)[39 + j]; }
    flush(4 * ne::FOOT_DBL + ne::FLOW_DBL + 39, 39); }
  const bool stage2 = work && !terminal;
  if (stage2) {   // second RK2 stage at x + c dt k1 (rows 12:30 of the flow map are the joint-velocity inputs)
    const double cdt = mdl->rk_c * dt;
#pragma unroll
    for (int i = 0; i < NX; ++i) x[i] += cdt * (i < 12 ? f1[i < 12 ? i : 0] : u[i]);
    ne::base_eval<true>(mdl, x, bk); ne::flow_acc_init(acc);
#pragma unroll 1
    for (int i = 0; i < 4; ++i) { ne::Foot2Blk* f2 = reinterpret_cast<ne::Foot2Blk*>(row) + i; ne::foot_eval<true>(mdl, x, u, bk, i, acc, f2->d, nullptr, nullptr, nullptr, f2->JxF); }
  }
  flush(4 * ne::FOOT_DBL + ne::FLOW_DBL + ne::EE_DBL, 4 * ne::FOOT2_DBL);
  if (stage2) { ne::FlowBlk* fl = reinterpret_cast<ne::FlowBlk*>(row); ne::flow_finish<true>(mdl, x, bk, acc, fl->f, fl); }
  flush(4 * ne::FOOT_DBL + ne::FLOW_DBL + ne::EE_DBL + 4 * ne::FOOT2_DBL, ne::FLOW_DBL);
}

// =====================================================================================================
// K2b: cost quadratic model, equality constraints, projection, RK2 sensitivities and the structured stage record of one node (one warp per node), on the
// record of the flow kernel.
// (A CTA-wide re-alignment of the warps at phase boundaries - instruction-cache sharing - was measured and dropped: 21.88 ms with, 21.42 ms without, profiles/r02_ab_k3.jsonl.)
// rows 3:12 of df/dx (9 x 30, two thirds zeros) from the Jacobian blocks of a flow record: fill, then lane = column writes
// its own non-zeros (the fill and the column writes are separated by a warp barrier)
__device__ __forceinline__ void expand_flow(const ne::FlowBlk& fb, const double* jxf0, int fstride /*doubles between two feet*/, double* Ar, int lfp, int lane) {
  for (int e = lane; e < 9 * NX; e += 32) Ar[e] = 0.0;
  __syncwarp();
  if (lane < 24) {
    const int col = lane;
    if (col < 3) Ar[(3 + col) * NX + col] = 1.0;                                                         // d pdot / d h_lin = I
    else if (col < 6) { for (int a = 0; a < 3; ++a) { Ar[(3 + a) * NX + col] = fb.Mpc[3 * a + col - 3]; Ar[(6 + a) * NX + col] = fb.Mtw[3 * a + col - 3]; } }   // d / d h_ang
    else if (col >= 9 && col < 12) { for (int a = 0; a < 3; ++a) { Ar[a * NX + col] = fb.hth[col - 9][a]; Ar[(3 + a) * NX + col] = fb.vp[col - 9][a]; Ar[(6 + a) * NX + col] = fb.vt[col - 9][a]; } }   // d / d theta
    else if (col >= 12) { const int j12 = col - 12; const double* jf = jxf0 + foot_of_leg_joint(lfp, j12) * fstride + 3 * (j12 % 3); for (int a = 0; a < 3; ++a) Ar[a * NX + col] = jf[a]; }   // d hdot_ang / d q_leg = (J_j x F) / m
  }
  __syncwarp();
}
__global__ void __launch_bounds__(32 * LQ_WARPS, QMB_LQ_MINB) mpc_lq_kernel(const DevModel* __restrict__ mdl, int b0, int B, int nmax, MpcProblemDev p, MpcSolutionDev sol, const double* __restrict__ rec, double* __restrict__ stage, int32_t* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31; const long long gid = (long long)blockIdx.x * LQ_WARPS + warp;
  const int b = b0 + (int)(gid / nmax), k = (int)(gid % nmax);
  if (b >= B) return;
  // Everything the node needs from HBM is requested up front and independently (addresses depend on (b, k) only; every buffer covers all B * nmax nodes): the
  // record of the flow kernel, (x, u, x_next), the grid entries.  Only then is the node classified - a padding node wastes a few sectors, a regular node sees
  // one memory round trip instead of four dependent ones (node count -> event flag -> state -> record).
  LqSmem& sm = reinterpret_cast<LqSmem*>(smem_raw)[warp]; LqLate& lt = *reinterpret_cast<LqLate*>(&sm.rec.foot[0]);
  const size_t node = (size_t)b * nmax + k; const bool has_next = k + 1 < nmax;
  const double2* rg = reinterpret_cast<const double2*>(rec + node * ne::NODE_REC_DBL); double2 rr[(ne::NODE_REC_DBL / 2 + 31) / 32];
#pragma unroll
  for (int q = 0; q < (ne::NODE_REC_DBL / 2 + 31) / 32; ++q) { const int e = lane + 32 * q; rr[q] = (e < ne::NODE_REC_DBL / 2) ? __ldg(rg + e) : make_double2(0.0, 0.0); }
  const double* xk = sol.x + node * NX; const double* uk = sol.u + node * NU;
  const double xv = (lane < NX) ? xk[lane] : 0.0, uv = (lane < NU) ? uk[lane] : 0.0, xnv = (lane < NX && has_next) ? xk[NX + lane] : 0.0;
  const double* gt = sol.t + (size_t)b * nmax; const int32_t* ge = sol.event + (size_t)b * nmax;
  const double tk = gt[k], tk1 = has_next ? gt[k + 1] : 0.0; const int ek = ge[k], ek1 = has_next ? ge[k + 1] : 0;
  const int ne = clamp_events(p.n_events[b]); double* s_ev = sm.Ar; unsigned char* s_modes = reinterpret_cast<unsigned char*>(sm.Ar + EMAX); const double* ev = s_ev; const unsigned char* modes = s_modes;   // staged once per node: the binary searches and the swing-interval scans hit shared memory
  { const double* gev = p.event_times + (size_t)b * EMAX; const int32_t* gmodes = p.modes + (size_t)b * (EMAX + 1); s_ev[lane] = (lane < ne) ? gev[lane] : 0.0; s_modes[lane] = (unsigned char)((lane <= ne) ? gmodes[lane] : 15); if (lane == 0) s_modes[EMAX] = (unsigned char)((EMAX <= ne) ? gmodes[EMAX] : 15); }
  const int n = sol.n_nodes[b];
  const bool work = k < n && !(status[b] & MST_CONVERGED);   // MST_CONVERGED: SqpSolver::runImpl left the iteration loop for this robot
  if (!work) return;
  double* sg = stage + node * STAGE_DBL;
  const bool terminal = (k == n - 1);
  if (lane < NX) { sm.x[lane] = xv; sm.u[lane] = terminal ? 0.0 : uv; }   // the next node's state (defect) stays in the lane's register
  __syncwarp();
  if (!terminal && ek == 1) {   // event node: identity jump map, no input, no cost (setupEventNode)
    double* tl = sg + ST_TAIL; int32_t* si = reinterpret_cast<int32_t*>(tl + T_INT);
    double d = 0.0; if (lane < NX) { d = xv - xnv; tl[T_b + lane] = d; }
    const double ss = warp_sum(d * d);
    if (lane == 0) { si[SI_TYPE] = 1; si[SI_M] = 0; si[SI_NDEP] = 0; tl[T_MISC] = 0.0; tl[T_MISC + 1] = 0.0; tl[T_MISC + 2] = ss; tl[T_MISC + 3] = 0.0; }
    return;
  }
  { double2* rs = reinterpret_cast<double2*>(&sm.rec);   // the node's record: one contiguous 3.9 KB run, 16 bytes per lane and load
#pragma unroll
    for (int q = 0; q < (ne::NODE_REC_DBL / 2 + 31) / 32; ++q) { const int e = lane + 32 * q; if (e < ne::NODE_REC_DBL / 2) rs[e] = rr[q]; } }
  __syncwarp();
  const int lfp = pack_leg_foot(mdl);
  const int nk = clamp_targets(p.n_target[b]); const double* tt = p.target_times + (size_t)b * KMAX; const double* ts = p.target_states + (size_t)b * KMAX * TARGET_DIM;
  const double t = interval_start(tk, ek);
  const double dt = terminal ? 0.0 : interval_end(tk1, ek1) - t;
  const int mode = mode_at_time(ev, modes, ne, t); const int fm = terminal ? 0 : flag_mask(mode);
  if (!terminal && !(dt > 0.0) && lane == 0) atomicOr(&status[b], MST_NEG_DT);   // getIntervalDuration <= 0: an event within weakEpsilon of a grid node (QMB200_ST_NEG_DT)
  double cost_val = 0.0, eq_ss = 0.0; int ndep = 0, m = 0; double b1v[3] = {0.0, 0.0, 0.0}, b2v[3] = {0.0, 0.0, 0.0};
  {
  // ---- cost quadratic model at (x, u) (the end-effector error and its Jacobian come with the record) ----
  struct XU { double x[NX], u[NU]; }; static_assert(offsetof(LqSmem, u) == offsetof(LqSmem, x) + NX * 8, "x then u");
  cost_val = stage_cost_quad(mdl, reinterpret_cast<const XU*>(sm.x), &sm.rec.ee, &sm.quad, target_xnom(tt, ts, nk, t, lane), fm, terminal, lane);
  if (terminal) {   // setupTerminalNode: finalEndEffector soft constraint only (QMInterface.cpp:104)
    double* tl = sg + ST_TAIL; int32_t* si = reinterpret_cast<int32_t*>(tl + T_INT);
    for (int r = 0; r < NX; ++r) { const int a = ee_pos(r); if (lane < q_row_padded(r)) { const int cc = (lane <= r) ? ee_pos(lane) : -1; sg[ST_Q + q_row_offset(r) + lane] = (a >= 0 && cc >= 0) ? sm.quad.E[a * 12 + cc] : 0.0; } }   // final cost: packed lower triangle
    if (lane < NX) tl[T_q + lane] = sm.quad.qf[lane];                                                                                                       // and its gradient
    if (lane == 0) { si[SI_TYPE] = 2; si[SI_M] = 0; si[SI_NDEP] = 0; tl[T_MISC] = 0.0; tl[T_MISC + 1] = cost_val; tl[T_MISC + 2] = 0.0; tl[T_MISC + 3] = 0.0; }
    return;
  }
  int nd_before = 0; for (int i = 0; i < 4; ++i) if (i < lane) nd_before += ((fm >> i) & 1) ? 3 : 4;
  ndep = 0; for (int i = 0; i < 4; ++i) ndep += ((fm >> i) & 1) ? 3 : 4;
  m = NU - ndep;
  if (lane < NU) sm.Pe_full[lane] = 0.0;
  bool swing_ok = true; int pivot = -1;
  if (lane < 4) {   // lane = foot (contact order); its leg's first joint = foot_leg
    const int i = lane; const int first = mdl->foot_leg[i]; LegWs& L = sm.leg[i]; L.first = first; L.stance = (fm >> i) & 1;
    if (L.stance) { for (int j = 0; j < 3; ++j) { sm.dep_idx[nd_before + j] = 12 + first + j; L.dep[j] = 1; } L.pivot = -1; for (int a = 0; a < 3; ++a) eq_ss += sm.rec.foot[i].e[a] * sm.rec.foot[i].e[a]; }
    else {
      double zp, zv; swing_ok = swing_reference(mdl, ev, modes, ne, i, t, zp, zv);
      double ez = sm.rec.foot[i].e[2] - zv; if (mdl->position_error_gain != 0.0) ez += mdl->position_error_gain * (sm.rec.foot[i].pf[2] - zp);
      sm.rec.foot[i].e[2] = ez;
      for (int a = 0; a < 3; ++a) { sm.dep_idx[nd_before + a] = 3 * i + a; eq_ss += sm.u[3 * i + a] * sm.u[3 * i + a]; }
      eq_ss += ez * ez;
      double best = -1.0; for (int j = 0; j < 3; ++j) { const double a = fabs(sm.rec.foot[i].Jl[3 * j + 2]); if (a > best) { best = a; pivot = j; } }   // pivot: largest |d v_z / d qdot_j|
      sm.dep_idx[nd_before + 3] = 12 + first + pivot; L.pivot = pivot; for (int j = 0; j < 3; ++j) L.dep[j] = (j == pivot);
    }
  }
  eq_ss = warp_sum(eq_ss);
  if (!__all_sync(FULL, swing_ok)) { if (lane == 0) atomicOr(&status[b], MST_OVERFLOW); }
  __syncwarp();
  // free / dependent partition of the 30 inputs
  bool is_dep = false; if (lane < NU) for (int d = 0; d < ndep; ++d) is_dep |= (sm.dep_idx[d] == lane);
  const unsigned free_mask = __ballot_sync(FULL, lane < NU && !is_dep);
  if (lane < NU) { const int rank = __popc(free_mask & ((1u << lane) - 1u)); sm.col_of_input[lane] = is_dep ? -1 : rank; if (!is_dep) sm.free_idx[rank] = lane; }
  __syncwarp();
  // ---- per-leg projection blocks (structured elimination; the projected optimum does not depend on the null-space basis) ----
  if (lane < 4) {
    const int i = lane; LegWs& L = sm.leg[i]; const int first = L.first;
    for (int a = 0; a < 3; ++a) for (int c = 0; c < 3; ++c) L.Rl[3 * a + c] = quad_R(mdl, &sm.quad, 12 + first + a, 12 + first + c);
    for (int j = 0; j < 3; ++j) { L.free_col[j] = sm.col_of_input[12 + first + j]; L.Pe[j] = 0.0; for (int c = 0; c < 12; ++c) L.Px[j][c] = 0.0; }
    L.Pu2[0] = L.Pu2[1] = 0.0;
    if (L.stance) {   // zero velocity: Jl dqd = -(C dx + e)  →  dqd = -Jl^{-1} (C dx + e)
      double Jm[9], Ji[9]; for (int a = 0; a < 3; ++a) for (int j = 0; j < 3; ++j) Jm[3 * a + j] = sm.rec.foot[i].Jl[3 * j + a]; inv3(Jm, Ji);
      for (int j = 0; j < 3; ++j) { double pe = 0.0; for (int a = 0; a < 3; ++a) pe -= Ji[3 * j + a] * sm.rec.foot[i].e[a]; L.Pe[j] = pe; sm.Pe_full[12 + first + j] = pe;
        for (int c = 0; c < 12; ++c) { double sv = 0.0; for (int a = 0; a < 3; ++a) sv -= Ji[3 * j + a] * sm.rec.foot[i].C[a][c]; L.Px[j][c] = sv; } }
    } else {          // zero force: dF = -F ; normal velocity: pivot joint eliminated
      for (int a = 0; a < 3; ++a) sm.Pe_full[3 * i + a] = -sm.u[3 * i + a];
      const double piv = sm.rec.foot[i].Jl[3 * pivot + 2], nip = -1.0 / piv;
      L.Pe[pivot] = sm.rec.foot[i].e[2] * nip; sm.Pe_full[12 + first + pivot] = L.Pe[pivot];
      for (int c = 0; c < 12; ++c) L.Px[pivot][c] = sm.rec.foot[i].C[2][c] * nip;
      int nf = 0; for (int j = 0; j < 3; ++j) if (j != pivot) L.Pu2[nf++] = sm.rec.foot[i].Jl[3 * j + 2] * nip;
    }
    // rs = r + R Pe on the leg's joint inputs (the product Rl Px is formed where it is used: Q~ needs Px' (Rl Px), one 3-vector per row)
    for (int a = 0; a < 3; ++a) { double sv = sm.quad.rf[12 + first + a]; for (int j = 0; j < 3; ++j) sv += L.Rl[3 * a + j] * L.Pe[j]; L.rs[a] = sv; }
  }
  __syncwarp();
  // rs of every input: r + R Pe (R couples joint velocities only inside a leg; forces and arm inputs only with themselves)
  if (lane < NU) {
    double sv = sm.quad.rf[lane];
    if (lane < 12) { const int f = lane / 3; for (int a = 0; a < 3; ++a) sv += quad_R(mdl, &sm.quad, lane, 3 * f + a) * sm.Pe_full[3 * f + a]; }
    else if (lane < 24) { const int i = foot_of_leg_joint(lfp, lane - 12); sv = sm.leg[i].rs[(lane - 12) % 3]; }
    sm.rs[lane] = sv;
  }
  // continuous-time Jacobians of the two RK2 stages from the record's blocks
  const double imr = 1.0 / mdl->total_mass;
  expand_flow(sm.rec.s1, sm.rec.foot[0].JxF, ne::FOOT_DBL, sm.A1r, lfp, lane); expand_flow(sm.rec.s2, sm.rec.foot2[0].JxF, ne::FOOT2_DBL, sm.Ar, lfp, lane);
  // force block of rows 3:6 of df/du at both stages, column c = lane < 12 (foot i = c / 3, axis a = c % 3): cross(d_i, e_a)[r] / m - three entries per stage, kept in registers
  // (the foot blocks of the record are about to be overlaid by the RK2 combination's outputs)
  if (lane < 12) { const int i = lane / 3, a = lane - 3 * i; const double* d1 = sm.rec.foot[i].d; const double* d2 = sm.rec.foot2[i].d;
#pragma unroll
    for (int r = 0; r < 3; ++r) if (r != a) { const double sgn = ((a - r + 3) % 3 == 1) ? -imr : imr; b1v[r] = sgn * d1[3 - r - a]; b2v[r] = sgn * d2[3 - r - a]; } }
  __syncwarp();
  }
  const double w1 = mdl->rk_w1, w2 = mdl->rk_w2, cdt = mdl->rk_c * dt, mass = mdl->total_mass, dtw = dt * (w1 + w2), imass = 1.0 / mass;
  double bb = 0.0; if (lane < NX) { const double fa = lane < 12 ? sm.rec.s1.f[lane < 12 ? lane : 0] : sm.u[lane], fb = lane < 12 ? sm.rec.s2.f[lane < 12 ? lane : 0] : sm.u[lane];   // rows 12:30 of the flow map: the joint-velocity inputs
    bb = xv + dt * (w1 * fa + w2 * fb) - xnv; lt.bvec[lane] = bb; }   // defect
  const double dyn_ss = warp_sum(bb * bb);
  // A_d - I (rows 3:12) = dt (w1 A1 + w2 (A2 + c dt A2 A1)) ; B_d rows 3:12 = dt (w1 B1 + w2 (B2 + c dt A2 B1)): force columns (9x12), joint columns only in the h_ang rows (3x18)
  if (lane < NX) {   // lane = column c: needs column c of A1 only, so A1r can be overwritten in place
    const int c = lane; double a1[9], out[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) a1[q] = sm.A1r[q * NX + c];
#pragma unroll
    for (int r = 0; r < 9; ++r) { const double* a2 = sm.Ar + r * NX; double aa = 0.0;
#pragma unroll
      for (int q = 0; q < 9; ++q) aa = fma(a2[3 + q], a1[q], aa);
      out[r] = dt * (w1 * a1[r] + w2 * (a2[c] + cdt * aa));
      if (c < 12) { double b1 = 0.0, b2 = 0.0; if (r < 3) { b1 = b1v[r < 3 ? r : 0]; b2 = b2v[r < 3 ? r : 0]; } double ab = a2[c % 3] * imass;
#pragma unroll
        for (int q = 0; q < 3; ++q) ab += a2[3 + q] * b1v[q]; lt.BrdF[r * 12 + c] = dt * (w1 * b1 + w2 * (b2 + cdt * ab)); }
      else if (r < 3) lt.BrdJ[r * NJ + c - 12] = dt * w2 * cdt * a2[c]; }
#pragma unroll
    for (int r = 0; r < 9; ++r) sm.A1r[r * NX + c] = out[r];
  }
  __syncwarp();
  // ---- projected dynamics: b~ = b + B_d Pe (lane = state row) ; rows 3:12 of A~ = A_d + B_d Px (the h_ang rows pick up the dependent joint velocities) ----
  double* tl = sg + ST_TAIL; int32_t* si = reinterpret_cast<int32_t*>(tl + T_INT);
  if (lane < NX) {
    const int r = lane; double bt = lt.bvec[r];
    if (r >= 3 && r < 6) {       // + sum_legs BrdJ[r][joint] * Px_joint (accumulated in the shared-memory row, own thread)
      double* arow = sm.A1r + (r - 3) * NX; double acc[12];
#pragma unroll
      for (int i = 0; i < 4; ++i) { const LegWs& L = sm.leg[i];
#pragma unroll
        for (int c = 0; c < 12; ++c) acc[c] = 0.0;
        for (int j = 0; j < 3; ++j) if (L.dep[j]) { const double coef = lt.BrdJ[(r - 3) * NJ + L.first + j]; bt += coef * L.Pe[j];
#pragma unroll
          for (int c = 0; c < 12; ++c) acc[c] = fma(coef, L.Px[j][c], acc[c]); }
#pragma unroll
        for (int c = 0; c < 12; ++c) arow[sup_col(c, L.first)] += acc[c];
      }
    }
    if (r >= 12 && r < 24) {     // dependent joint-velocity rows: I + dtw * Px
      const int i = foot_of_leg_joint(lfp, r - 12); const LegWs& L = sm.leg[i]; const int j = (r - 12) % 3;
      if (L.dep[j]) bt += dtw * L.Pe[j];
    }
    if (r < 3) for (int f = 0; f < 4; ++f) bt += (dtw * imass) * sm.Pe_full[3 * f + r];
    if (r >= 3 && r < 12) for (int f = 0; f < 4; ++f) if (!sm.leg[f].stance) for (int a = 0; a < 3; ++a) bt += lt.BrdF[(r - 3) * 12 + 3 * f + a] * sm.Pe_full[3 * f + a];
    tl[T_b + r] = bt;
    if (r >= 3 && r < 12) sg[ST_AR + (r - 3) * LDX + NX] = bt;   // b~[3:12] also rides in column 30 of the dense A~ rows (K3's vector recursion)
  }
  if (lane >= 3 && lane < 12) sm.A1r[(lane - 3) * NX + lane] += 1.0;   // A1r rows become rows 3:12 of A~ themselves (own row of each lane: no hazard with the h_ang update above)
  __syncwarp();
  // rows 3:12 of A~ with K3's shared-memory pitch (one 240-byte run per store instruction), zero padding columns 31..35
#pragma unroll
  for (int r = 0; r < 9; ++r) { if (lane < NX) sg[ST_AR + r * LDX + lane] = sm.A1r[r * NX + lane]; else if (lane == 31) sg[ST_AR + r * LDX + 31] = 0.0; }
  for (int e = lane; e < 36; e += 32) sg[ST_AR + (e >> 2) * LDX + 32 + (e & 3)] = 0.0;
  // Px rows of the 12 leg-joint velocity inputs on their support columns: K3 rebuilds rows 12:24 of A~ (I + dtw Px) and the dependent inputs of the rollout from them
  for (int e = lane; e < 144; e += 32) { const int j12 = e / 12, c = e - 12 * j12; const LegWs& L = sm.leg[foot_of_leg_joint(lfp, j12)]; const int j = j12 % 3; tl[T_PXJ + e] = L.dep[j] ? L.Px[j][c] : 0.0; }
  // rows 3:12 of B~ (force columns; joint columns reach the h_ang rows only), pitch LDB, zero padding; the remaining rows of B~ are structured (see mpc_api.cuh)
  for (int e = lane; e < 9 * LDB; e += 32) {
    const int rr = e / LDB, a = e - rr * LDB; const int r = 3 + rr; double v = 0.0;
    if (a < m) { const int fa = sm.free_idx[a];
      if (fa < 12) v = lt.BrdF[rr * 12 + fa];
      else if (r < 6) { v = lt.BrdJ[rr * NJ + fa - 12];
        if (fa < 24) { const LegWs& L = sm.leg[foot_of_leg_joint(lfp, fa - 12)]; if (!L.stance) { const int jf = (fa - 12) % 3; v += lt.BrdJ[rr * NJ + L.first + L.pivot] * L.Pu2[jf > L.pivot ? jf - 1 : jf]; } } }
    }
    sg[ST_BR + e] = v;
  }
  // ---- projected cost (changeOfInputVariables [upstream]); quadratic model scaled by dt ----
  if (lane < NX) {   // q~ = q + Px' rs ; Q~ = Q + Px' R Px : per leg a 12x12 block on its support columns
    const int r = lane; double acc[NX];
    if (mdl->q_is_diag) { const double qrr = mdl->Qdiag[r];
#pragma unroll
      for (int c = 0; c < NX; ++c) acc[c] = (c == r) ? qrr : 0.0; }
    else {
#pragma unroll
      for (int c = 0; c < NX; ++c) acc[c] = mdl->Q[r * NX + c]; }
    double qv = sm.quad.qf[r];
    const int ea = ee_pos(r);
    if (ea >= 0) {
#pragma unroll
      for (int c = 0; c < 6; ++c) { acc[6 + c] += sm.quad.E[ea * 12 + c]; acc[24 + c] += sm.quad.E[ea * 12 + 6 + c]; }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const LegWs& L = sm.leg[i]; const int first = L.first;   // first is 0,3,6,9 in some foot order: resolve the static column block by comparing
      const int pr = (r < 6) ? r : ((r >= 9 && r < 12) ? r - 3 : ((r >= 12 + first && r < 15 + first) ? 9 + r - 12 - first : -1));
      if (pr >= 0) {
        double blk[12];
#pragma unroll
        for (int c = 0; c < 12; ++c) blk[c] = 0.0;
        double w3[3] = {0.0, 0.0, 0.0};   // row pr of Px' Rl ; then blk = w3' Px  (= row pr of Px' Rl Px)
        for (int j = 0; j < 3; ++j) if (L.dep[j]) { const double pj = L.Px[j][pr]; qv = fma(pj, L.rs[j], qv);
#pragma unroll
          for (int a = 0; a < 3; ++a) w3[a] = fma(pj, L.Rl[3 * j + a], w3[a]); }
        for (int a = 0; a < 3; ++a) if (L.dep[a]) { const double wa = w3[a];
#pragma unroll
          for (int c = 0; c < 12; ++c) blk[c] = fma(wa, L.Px[a][c], blk[c]); }
#pragma unroll
        for (int c = 0; c < 6; ++c) acc[c] += blk[c];
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[9 + c] += blk[6 + c];
        // leg-specific columns 12+first+c: first ∈ {0,3,6,9}
#pragma unroll
        for (int l = 0; l < 4; ++l) if (first == 3 * l) {
#pragma unroll
          for (int c = 0; c < 3; ++c) acc[12 + 3 * l + c] += blk[9 + c]; }
      }
    }
    // Q~ is symmetric and leaves as its packed lower triangle: lane r holds row r = column r, so for every c the lanes r <= c store the run Q~[c][0..c] of
    // packed row c - one contiguous piece per store instruction; q~ goes to the tail
    const double dq = sm.quad.qdiag[r];
#pragma unroll
    for (int c = 0; c < NX; ++c) if (r <= c) sg[ST_Q + q_row_offset(c) + r] = dt * (acc[c] + ((c == r) ? dq : 0.0));
    if (!(r & 1)) sg[ST_Q + q_row_offset(r) + r + 1] = 0.0;   // even rows carry one padding entry
    tl[T_q + r] = dt * qv;
  }
  for (int e = lane; e < 8 * 12; e += 32) tl[T_SJ + e] = 0.0;
  __syncwarp();
  if (lane < MU) {   // r~ = Pu' rs ; S~ = Pu' (R Px) (non-zero only for the free joints of swing legs) ; R~ = Pu' R Pu (block diagonal over the input triples)
    const int a = lane; double rt[3] = {0.0, 0.0, 0.0}; double rtil = 0.0;
    if (a < m) {
      const int fa = sm.free_idx[a]; double rv = sm.rs[fa]; int li = -1, jf = -1;
      if (fa >= 12 && fa < 24) { li = foot_of_leg_joint(lfp, fa - 12); jf = (fa - 12) % 3; }
      const bool swing_joint = li >= 0 && !sm.leg[li].stance;
      if (swing_joint) {   // free joint of a swing leg: coupled to the pivot through R_leg and Pu
        const LegWs& L = sm.leg[li]; const int pv = L.pivot; const int jfi = jf > pv ? jf - 1 : jf; const double pu = L.Pu2[jfi];
        rv += pu * L.rs[pv];
        const double coef = L.Rl[3 * jf + pv]; double* Srow = tl + T_SJ + (2 * li + jfi) * 12;
        const double cf = dt * (coef + pu * L.Rl[3 * pv + pv]);   // only the pivot row of Px is non-zero in a swing leg: (Rl Px)[pv] = Rl[pv][pv] Px[pv]
        for (int c = 0; c < 12; ++c) Srow[c] = cf * L.Px[pv][c];
      }
      rtil = dt * rv;
      // R is block diagonal (3x3 blocks over force / leg-joint triples, diagonal over the arm): only the free inputs of fa's own block contribute to row a
      if (fa >= 24) rt[0] = dt * quad_R(mdl, &sm.quad, fa, fa);
      else { const int bi = fa / 3;
        for (int jc = 0; jc < 3; ++jc) { const int fc = 3 * bi + jc; if (sm.col_of_input[fc] < 0) continue;
          double v = quad_R(mdl, &sm.quad, fa, fc);
          if (swing_joint) { const LegWs& L = sm.leg[li]; const int pv = L.pivot; const double pa = L.Pu2[jf > pv ? jf - 1 : jf], pc = L.Pu2[jc > pv ? jc - 1 : jc];
            v += pa * L.Rl[3 * pv + jc] + L.Rl[3 * jf + pv] * pc + pa * L.Rl[3 * pv + pv] * pc; }
          rt[jc] = dt * v; } }
    }
    tl[T_r + a] = rtil; tl[T_RT + 3 * a] = rt[0]; tl[T_RT + 3 * a + 1] = rt[1]; tl[T_RT + 3 * a + 2] = rt[2];
  }
  if (lane < 4) { const LegWs& L = sm.leg[lane]; tl[T_PU2 + 2 * lane] = L.Pu2[0]; tl[T_PU2 + 2 * lane + 1] = L.Pu2[1]; si[SI_PIV + lane] = L.stance ? -1 : L.pivot;
    // projected columns of the leg's two free joints (swing legs): the rollout needs them for the eliminated pivot joint
    int nf = 0; for (int jj = 0; jj < 3; ++jj) if (!L.stance && jj != L.pivot) si[SI_PCOL + 2 * lane + nf++] = L.free_col[jj]; if (L.stance) { si[SI_PCOL + 2 * lane] = -1; si[SI_PCOL + 2 * lane + 1] = -1; } }
  if (lane < MAXDEP) { const int d = lane; double pe = 0.0; int di = -1; if (d < ndep) { di = sm.dep_idx[d]; pe = sm.Pe_full[di]; } tl[T_PED + d] = pe; si[SI_DEP + d] = di; }
  if (lane < MU) si[SI_FREE + lane] = (lane < m) ? sm.free_idx[lane] : -1;
  if (lane == 0) { si[SI_TYPE] = 0; si[SI_M] = m; si[SI_NDEP] = ndep; tl[T_MISC] = dtw; tl[T_MISC + 1] = dt * cost_val; tl[T_MISC + 2] = dt * dyn_ss; tl[T_MISC + 3] = dt * eq_ss; }
}

// =====================================================================================================
// K3: Riccati backward sweep + forward rollout of the projected LQ problem.
// One CTA (4 warps) per robot.  Every product of the backward sweep is a set of 8x8x4 fp64 tensor-core tiles (DMMA) on dense 30x30 / 30x18 matrices in shared
// memory; the Cholesky + triangular solves are warp-specialised with the factor in registers.  The structured stage record of K2 (mpc_api.cuh) reaches shared
// memory through the TMA engine: per node four bulk copies (cp.async.bulk: rows 3:12 of A~ and of B~, the Q~ block, the 3.4 KB tail) signalled on mbarriers,
// issued by one thread one node ahead; the sparse remainder of A~ / B~ (identity, dtw * Px on support columns, dtw at free columns) is rebuilt in place from the
// tail while the previous node's phase 4 runs.  -DQMB_TMA=0 replaces the bulk copies by 16-byte cp.async spread over the CTA (same record, same schedule; the A/B
// measurement is in profiles/).  The projected input dimension is padded to MU = 18 (identity rows in R~, zero rows in S~ / B~), so nothing depends on the mode.
#ifndef QMB_TMA
#define QMB_TMA 1
#endif
constexpr int RIC_THREADS = 128, RIC_NTYPE = 512;
// Leading dimensions (mpc_api.cuh).  MMA operands are fetched as X[(k0 + t) * ld + c0 + g] (t = lane % 4, g = lane / 4): 2 * ld = 8 (mod 32) or
// 24 (mod 32) puts the four k-rows of a half-warp on disjoint bank octets, i.e. every fragment load is conflict free.
struct RicSmem {
  double P[NX * LDX];                       // value function: Hessian in columns 0..29, gradient p in column 30; receives Q~ (C operand of phase 3) in between
  double A[NX * LDX];                       // A~ (column 30: b~)
  double W[NX * LDX];                       // W = P'A (column 30: p + P b~)
  double Bm[NX * LDB], PB[NX * LDB];        // B~ ; P'B~, later Y = L^{-1}[G | h] (18 x LDX)
  double G[MU * LDG];                       // G = S~ + B~'W (column 30: h = r~ + B~'(p + P b~))
  double H[MU * LDH];                       // H = R~ + B~'P B~
  double Lt[MU * MU];                       // Cholesky factor of H, transposed: Lt[c][a] = L[a][c] (strict lower part; pivots live as reciprocals in dut)
  alignas(16) double tail[TAIL_DBL];        // backward sweep: the node's small pieces (Px rows, b~, q~, r~, R~ / S~ entries, index lists)
  double dx[32], dut[32], tmp[32];
  double red[RIC_THREADS / 32][4];
  alignas(8) unsigned long long bar[4];     // mbarriers: 0 = A~/B~ rows (forward: buffer set 0), 1 = tail, 2 = Q~, 3 = forward buffer set 1
  int flag; int pad_;
  signed char srow[MU + 2], sfirst[MU + 2]; // projected input a: S~ slot (2 * foot + position) and first joint of its leg when a is a free joint of a swing leg, else -1
  unsigned char ntype[RIC_NTYPE];           // node types of the whole horizon, loaded once: the sweep's control flow never waits on a global load
};
static_assert(sizeof(RicSmem) <= 57344 - 64, "Riccati kernel must keep four CTAs per SM");

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* b, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(b)), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* b, unsigned bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(b)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void mbar_wait(unsigned long long* b, unsigned parity) {
  asm volatile("{\n .reg .pred p;\n WAIT_LOOP:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra WAIT_DONE;\n bra WAIT_LOOP;\n WAIT_DONE:\n}\n" ::"r"(smem_u32(b)), "r"(parity) : "memory");
}
// one contiguous run global -> shared through the TMA engine (bytes: multiple of 16, both addresses 16-byte aligned); completion is signalled on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
// A "copy group": with QMB_TMA one elected thread arms the mbarrier and issues the bulk copies; without it every thread copies its share with cp.async and the
// group is closed by cp.async.wait_all + a CTA barrier at the point where the TMA path waits on the mbarrier.
struct CopyGroup {
  unsigned long long* bar; unsigned phase;
  __device__ __forceinline__ void begin(unsigned bytes, int tid) { if (QMB_TMA && tid == 0) mbar_expect_tx(bar, bytes); }
  __device__ __forceinline__ void copy(void* dst, const void* src, unsigned bytes, int tid, int nthr = RIC_THREADS, int t0 = 0) {
    if (QMB_TMA) { if (tid == 0) bulk_g2s(dst, src, bytes, bar); }
    else { const int me = tid - t0; if (me >= 0 && me < nthr) for (unsigned o = 16u * me; o < bytes; o += 16u * nthr) cp_async16((char*)dst + o, (const char*)src + o); }
  }
  // returns after the group's bytes are visible to the calling thread (TMA) / to the whole CTA (cp.async path: includes a barrier, so every thread must call it)
  __device__ __forceinline__ void wait() { if (QMB_TMA) mbar_wait(bar, phase & 1u); else { cp_async_wait_all(); __syncthreads(); } ++phase; }
  __device__ __forceinline__ void skip() { ++phase; }
};

// ---- fp64 tensor-core tiles (DMMA.8x8x4, mma.sync m8n8k4 f64: measured 37 TFLOP/s on B200, the same rate as the DFMA pipe at 1/8 of
// the issue slots and ~1/3 of the shared-memory operand traffic of a 4x4 register tile).  C(8x8) += A(8x4) B(4x8) with
// A[i][k] = X[k][i0 + i], B[k][j] = Y[k][j0 + j]: lane (g = lane / 4, t = lane % 4) holds A[g][t], B[t][g], C[g][2t], C[g][2t + 1].
__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
// c[m][n] += (+-) X[0:K, i0 + 8m ..]' Y[0:K, j0 + 8n ..] for an MT x NT block of 8x8 tiles; K need not be a multiple of 4 (tail lanes feed zeros)
template <int K, int MT, int NT, bool NEG>
__device__ __forceinline__ void warp_mma(const double* __restrict__ X, int ldx, int i0, const double* __restrict__ Y, int ldy, int j0, double (&c)[MT][NT][2], int g, int t) {
#pragma unroll
  for (int ks = 0; ks < (K + 3) / 4; ++ks) {
    const int kr = 4 * ks + t; const bool ok = (4 * ks + 3 < K) || (kr < K);
    double a[MT], bf[NT];
#pragma unroll
    for (int m = 0; m < MT; ++m) { const double v = ok ? X[kr * ldx + i0 + 8 * m + g] : 0.0; a[m] = NEG ? -v : v; }
#pragma unroll
    for (int n = 0; n < NT; ++n) bf[n] = ok ? Y[kr * ldy + j0 + 8 * n + g] : 0.0;
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
      for (int n = 0; n < NT; ++n) dmma884(c[m][n], a[m], bf[n]);
  }
}
template <int MT, int NT>
__device__ __forceinline__ void cfrag_load(const double* M, int ld, int i0, int j0, int rows, double (&c)[MT][NT][2], int g, int t) {
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int n = 0; n < NT; ++n) { const int ri = i0 + 8 * m + g;
      if (ri < rows) { const double2 v = *reinterpret_cast<const double2*>(M + ri * ld + j0 + 8 * n + 2 * t); c[m][n][0] = v.x; c[m][n][1] = v.y; } else { c[m][n][0] = 0.0; c[m][n][1] = 0.0; } }
}
template <int MT, int NT>
__device__ __forceinline__ void cfrag_store(double* M, int ld, int i0, int j0, int rows, const double (&c)[MT][NT][2], int g, int t) {
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int n = 0; n < NT; ++n) { const int ri = i0 + 8 * m + g; if (ri < rows) *reinterpret_cast<double2*>(M + ri * ld + j0 + 8 * n + 2 * t) = make_double2(c[m][n][0], c[m][n][1]); }
}
// support position (0..11) of state column j for the leg whose first joint is `first`, -1 outside the support (inverse of sup_col)
__device__ __forceinline__ int sup_pos(int j, int first) { return j < 6 ? j : ((j >= 9 && j < 12) ? j - 3 : (((unsigned)(j - 12 - first) < 3u) ? 9 + j - 12 - first : -1)); }

// kValueFn (createValueFunction): every node's cost-to-go of dx_k is also stored as a VF_DBL record (mpc_api.cuh) in `vf`, re-centred on the linearization
// trajectory sol.x (which K4 overwrites only after this kernel): dfdxx_k = P_k, dfdx_k = p_k - P_k xbar_k.  P_{k+1} is complete and read-only at the top of
// iteration k (both node types) until phase 3 / the event update rewrite column 30, so node k+1 is stored there; node 0 after the sweep.  The false
// instantiation is the kernel without the stores.
template <bool kValueFn>
__global__ void __launch_bounds__(RIC_THREADS, 4) mpc_riccati_kernel(const DevModel* __restrict__ mdl, int b0, int B, int nmax, MpcProblemDev p, MpcSolutionDev sol, const double* __restrict__ stage,
                                                                  double* __restrict__ gains, double* __restrict__ dxo, double* __restrict__ duo, double* __restrict__ robot, int32_t* __restrict__ status,
                                                                  double* __restrict__ vf) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RicSmem& sm = *reinterpret_cast<RicSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, ti = tid >> 2, jb = tid & 3; const int b = b0 + blockIdx.x;
  if (status[b] & MST_CONVERGED) return;
  const int n = sol.n_nodes[b]; const int N = n - 1;
  const double* sgb = stage + (size_t)b * nmax * STAGE_DBL; double* gb = gains + (size_t)b * nmax * GAIN_DBL;
  const int lfp = pack_leg_foot(mdl); const double imass = 1.0 / mdl->total_mass;
  for (int e = tid; e < (int)(sizeof(RicSmem) / 8); e += RIC_THREADS) reinterpret_cast<double*>(&sm)[e] = 0.0;   // zero everything once (padding columns, static zero rows)
  __syncthreads();
  if (tid < NX && (tid < 3 || tid >= 24)) sm.A[tid * LDX + tid] = 1.0;   // identity rows of A~ that no node ever changes
  if (tid == 0) { for (int i = 0; i < 4; ++i) mbar_init(&sm.bar[i], 1); asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");           // the zero fill (generic proxy) is ordered before the first bulk copy (async proxy) by this fence + the barrier below
  const bool types_in_smem = n <= RIC_NTYPE;
  auto rec_type = [&](int k) -> int { return reinterpret_cast<const int32_t*>(sgb + (size_t)k * STAGE_DBL + ST_TAIL + T_INT)[SI_TYPE]; };
  if (types_in_smem) for (int k = tid; k < n; k += RIC_THREADS) sm.ntype[k] = (unsigned char)rec_type(k);   // published by the barrier below
  auto node_type = [&](int k) -> int { return types_in_smem ? (int)sm.ntype[k] : rec_type(k); };
  CopyGroup gAB{&sm.bar[0], 0u}, gT{&sm.bar[1], 0u}, gQ{&sm.bar[2], 0u}, gF1{&sm.bar[3], 0u};
  auto issue_ab = [&](int k) { const double* sg = sgb + (size_t)k * STAGE_DBL; gAB.begin((9 * LDX + 9 * LDB) * 8, tid);
    gAB.copy(sm.A + 3 * LDX, sg + ST_AR, 9 * LDX * 8, tid); gAB.copy(sm.Bm + 3 * LDB, sg + ST_BR, 9 * LDB * 8, tid); };     // rows 3:12 of A~ (with b~ in column 30) and of B~
  auto issue_tail = [&](int k) { gT.begin(TAIL_DBL * 8, tid); gT.copy(sm.tail, sgb + (size_t)k * STAGE_DBL + ST_TAIL, TAIL_DBL * 8, tid); };
  // Q~ (packed lower triangle, one 3.8 KB run) lands in the B~ buffer, which is idle between phase 2 and the next node's fetch; only the three helper warps of
  // node k wait for it, and they have slack (the factorisation warp is the critical path of phase 3)
  auto issue_q = [&](int k) { gQ.begin(Q_PACKED * 8, tid); gQ.copy(sm.Bm, sgb + (size_t)k * STAGE_DBL + ST_Q, Q_PACKED * 8, tid); };
  // rebuild the structured part of A~ / B~ of the node whose tail sits in sm.tail (all threads; A~ rows 3:12 and B~ rows 3:12 arrive by copy)
  auto expand = [&]() {
    const double* tl = sm.tail; const int32_t* si = reinterpret_cast<const int32_t*>(tl + T_INT); const double dtw = tl[T_MISC];
    for (int e = tid; e < 144; e += RIC_THREADS) { const int j12 = e / 12, c = e - 12 * j12; const int col = sup_col(c, 3 * (j12 / 3));   // rows 12:24: I + dtw * Px on the leg's support columns
      sm.A[(12 + j12) * LDX + col] = ((col == 12 + j12) ? 1.0 : 0.0) + dtw * tl[T_PXJ + e]; }
    if (tid < NX && (tid < 3 || tid >= 12)) sm.A[tid * LDX + NX] = tl[T_b + tid];                                                    // b~ (rows 3:12 came with the dense rows)
    for (int e = tid; e < 21 * MU; e += RIC_THREADS) {   // B~ rows 0:3 and 12:30, every element evaluated (no zero fill + scatter: no ordering between threads needed)
      const int rr = e / MU, a = e - rr * MU; const int r = rr < 3 ? rr : rr + 9; const int fa = si[SI_FREE + a]; double v = 0.0;
      if (fa >= 0) {
        if (r < 3) { if (fa < 12 && fa - 3 * (fa / 3) == r) v = dtw * imass; }                                                       // h_lin rows: F / m
        else if (fa == r) v = dtw;                                                                                                  // joint position rows: own joint velocity
        else if (fa >= 12 && fa < 24) { const int j = fa - 12, lg = j / 3, foot = (lfp >> (2 * lg)) & 3; const int pv = si[SI_PIV + foot];   // eliminated pivot joint of a swing leg
          if (pv >= 0 && r == 12 + 3 * lg + pv) { const int jf = j - 3 * lg; v = dtw * tl[T_PU2 + 2 * foot + (jf > pv ? jf - 1 : jf)]; } }
      }
      sm.Bm[r * LDB + a] = v;
    }
    if (tid < MU) { const int fa = si[SI_FREE + tid]; int slot = -1, first = 0;
      if (fa >= 12 && fa < 24) { const int j = fa - 12, lg = j / 3, foot = (lfp >> (2 * lg)) & 3; const int pv = si[SI_PIV + foot]; if (pv >= 0) { const int jf = j - 3 * lg; slot = 2 * foot + (jf > pv ? jf - 1 : jf); first = 3 * lg; } }
      sm.srow[tid] = (signed char)slot; sm.sfirst[tid] = (signed char)first; }
  };
  // value function record of node kk from sm.P (all threads; sm.P must hold P_kk, p_kk and stay unchanged until the caller's next barrier).  Packed entry e
  // is (r, e - r (r + 1) / 2) with r = floor((sqrt(8e + 1) - 1) / 2): 8e + 1 < 2^24 is exact in fp32 and the correctly rounded square root of a non-square
  // 8e + 1 stays below the next integer.  dfdx: 4 threads per row as the rollout's K dx
  auto store_vf = [&](int kk) {
    double* out = vf + ((size_t)b * nmax + kk) * VF_DBL;
    for (int e = tid; e < VF_P; e += RIC_THREADS) { const int r = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f); out[e] = sm.P[r * LDX + e - (r * (r + 1) >> 1)]; }
    const double* xb = sol.x + ((size_t)b * nmax + kk) * NX; double s = 0.0;
    if (ti < NX) {
#pragma unroll
      for (int v = 0; v < 8; ++v) { const int c = jb * 8 + v; if (c < NX) s = fma(sm.P[ti * LDX + c], xb[c], s); } }
    s += __shfl_xor_sync(FULL, s, 1); s += __shfl_xor_sync(FULL, s, 2);
    if (ti < NX && jb == 0) out[VF_P + ti] = sm.P[ti * LDX + NX] - s;
  };
  // terminal value function and baseline performance
  for (int e = tid; e < NX * NX; e += RIC_THREADS) { const int r = e / NX, c = e - r * NX; sm.P[r * LDX + c] = sgb[(size_t)N * STAGE_DBL + ST_Q + q_row_offset(r > c ? r : c) + (r > c ? c : r)]; }
  if (tid < NX) sm.P[tid * LDX + NX] = sgb[(size_t)N * STAGE_DBL + ST_TAIL + T_q + tid];
  double perf0 = 0, perf1 = 0, perf2 = 0;
  for (int k = tid; k < n; k += RIC_THREADS) { const double* pf = sgb + (size_t)k * STAGE_DBL + ST_TAIL + T_MISC + 1; perf0 += pf[0]; perf1 += pf[1]; perf2 += pf[2]; }
  if (tid < NX) { const double d = p.x0[(size_t)b * NX + tid] - sol.x[(size_t)b * nmax * NX + tid]; sm.dx[tid] = d; perf1 += d * d; }
  perf0 = warp_sum(perf0); perf1 = warp_sum(perf1); perf2 = warp_sum(perf2);
  if (lane == 0) { sm.red[warp][0] = perf0; sm.red[warp][1] = perf1; sm.red[warp][2] = perf2; }
  __syncthreads();
  double perf[3]; for (int i = 0; i < 3; ++i) perf[i] = sm.red[0][i] + sm.red[1][i] + sm.red[2][i] + sm.red[3][i];
  if (N >= 1) { issue_tail(N - 1); if (node_type(N - 1) != 1) issue_ab(N - 1); gT.wait(); if (node_type(N - 1) != 1) expand(); }
  int st = 0;
  // backward sweep: every product is a set of 8x8 DMMA tiles spread over the four warps.  The vector recursion rides in column 30 of
  // the matrices (b~, p + P b~, h, q~, p), so no separate matrix-vector products are needed.
  const int g = lane >> 2, t = lane & 3;
  for (int k = N - 1; k >= 0; --k) {
    const int type = node_type(k); const int tnext = k > 0 ? node_type(k - 1) : 1;
    if (type == 1) {                                // event node: A = I, no input: p += P b   (b~ of the node is in the tail, which expand-time waited for)
      __syncthreads();                              // P of node k+1 is complete
      if (kValueFn) store_vf(k + 1);
      if (tid < NX) { double sv = sm.P[tid * LDX + NX]; for (int j = 0; j < NX; ++j) sv = fma(sm.P[tid * LDX + j], sm.tail[T_b + j], sv); sm.tmp[tid] = sv; }
      __syncthreads();
      if (tid < NX) sm.P[tid * LDX + NX] = sm.tmp[tid];
      if (k > 0) { issue_tail(k - 1); if (tnext != 1) issue_ab(k - 1); gT.wait(); if (tnext != 1) expand(); }
      continue;
    }
    gAB.wait(); if (QMB_TMA) __syncthreads();     // rows 3:12 of A~, B~ have landed; the rebuilt rows and P of node k+1 are visible to everybody
    if (kValueFn) store_vf(k + 1);
    // ---- phase 1: W = P'A (32x32: warp = 16x16 block; column 30: p + P b~) ; PB = P'B~ (32x24: warp = row tile) ----
    // Rows 24:30 of A~ (arm joint positions) are identity rows with b~ in column 30, rows 24:30 of B~ carry dtw at the arm's own projected columns (the last six
    // free inputs): their contributions to every product of the sweep are copies / scaled copies of rows of P, W, PB and enter through the C fragments, so the
    // tensor-core contraction runs over k = 0..23 only (6 instead of 8 k-steps in phases 1-3: 130 of 606 DMMA per node less).
    const double dtw_k = sm.tail[T_MISC]; const int acol0 = reinterpret_cast<const int32_t*>(sm.tail + T_INT)[SI_M] - 6;   // projected column of arm joint 24
    { const int i0 = 16 * (warp >> 1), j0 = 16 * (warp & 1);
      double c[2][2][2] = {};
      if (warp & 1) {   // right-hand block: n-tile 1 holds columns 24..31; lane t owns columns 24 + 2t, 25 + 2t (t = 3: column 30 = p + P b~, column 31 = padding)
#pragma unroll
        for (int m = 0; m < 2; ++m) { const int ri = i0 + 8 * m + g; if (ri < NX) {
            if (t < 3) { c[m][1][0] = sm.P[(24 + 2 * t) * LDX + ri]; c[m][1][1] = sm.P[(25 + 2 * t) * LDX + ri]; }
            else { double sv = sm.P[ri * LDX + NX];
#pragma unroll
              for (int kk = 24; kk < NX; ++kk) sv = fma(sm.P[kk * LDX + ri], sm.A[kk * LDX + NX], sv);
              c[m][1][0] = sv; } } } }
      warp_mma<24, 2, 2, false>(sm.P, LDX, i0, sm.A, LDX, j0, c, g, t);
      cfrag_store<2, 2>(sm.W, LDX, i0, j0, NX, c, g, t);
      double d[1][3][2];
#pragma unroll
      for (int nn = 0; nn < 3; ++nn)
#pragma unroll
        for (int e = 0; e < 2; ++e) { const int a = 8 * nn + 2 * t + e - acol0, ri = 8 * warp + g; d[0][nn][e] = ((unsigned)a < 6u && ri < NX) ? dtw_k * sm.P[(24 + a) * LDX + ri] : 0.0; }
      warp_mma<24, 1, 3, false>(sm.P, LDX, 8 * warp, sm.Bm, LDB, 0, d, g, t);
      cfrag_store<1, 3>(sm.PB, LDB, 8 * warp, 0, NX, d, g, t); }
    __syncthreads();                                 // W, PB visible; P is dead until phase 3
    if (tid < NX) sm.P[tid * LDX + NX] = sm.tail[T_q + tid];   // q~ waits in column 30 of the dead buffer (the tail is replaced after phase 2)
    // ---- phase 2: G = S~ + B~'W (24x32: warp = column tile; column 30: h = r~ + B~'(p + P b~)) ; H = R~ + B~'PB (24x24: warps 0-2).  S~, r~ and R~ are
    //      not stored densely: the C fragments are initialised from the structured entries of the tail ----
    { const double* tl = sm.tail; const int32_t* si = reinterpret_cast<const int32_t*>(tl + T_INT); const int mm = si[SI_M];
      double c[3][1][2];
#pragma unroll
      for (int mt = 0; mt < 3; ++mt) { const int a = 8 * mt + g; const bool rowok = a < MU; const int slot = rowok ? sm.srow[a] : -1, first = rowok ? sm.sfirst[a] : 0;
#pragma unroll
        for (int e = 0; e < 2; ++e) { const int j = 8 * warp + 2 * t + e; double v = 0.0;
          if (rowok) { if (j == NX) v = tl[T_r + a]; else if (slot >= 0 && j < NX) { const int ps = sup_pos(j, first); if (ps >= 0) v = tl[T_SJ + slot * 12 + ps]; }
            if ((unsigned)(a - acol0) < 6u) v = fma(dtw_k, sm.W[(24 + a - acol0) * LDX + j], v); }   // arm rows of B~: dtw * W[24 + ., :]
          c[mt][0][e] = v; } }
      warp_mma<24, 3, 1, false>(sm.Bm, LDB, 0, sm.W, LDX, 8 * warp, c, g, t); cfrag_store<3, 1>(sm.G, LDG, 0, 8 * warp, MU, c, g, t);
      if (warp < 3) { double d[3][1][2];
#pragma unroll
        for (int mt = 0; mt < 3; ++mt) { const int a = 8 * mt + g; const int fa = (a < MU) ? si[SI_FREE + a] : -1;
#pragma unroll
          for (int e = 0; e < 2; ++e) { const int cc = 8 * warp + 2 * t + e; double v = 0.0;
            if (a < MU && cc < MU) { if (a >= mm) v = (a == cc) ? 1.0 : 0.0;                                  // identity padding of the projected input
              else if (fa >= 24) v = (a == cc) ? tl[T_RT + 3 * a] : 0.0;                                      // arm: diagonal
              else { const int fc = si[SI_FREE + cc]; if (fc >= 0 && fc / 3 == fa / 3) v = tl[T_RT + 3 * a + fc - 3 * (fc / 3)]; }   // own input triple
              if ((unsigned)(a - acol0) < 6u) v = fma(dtw_k, sm.PB[(24 + a - acol0) * LDB + cc], v); }                                 // arm rows of B~: dtw * PB[24 + ., :]
            d[mt][0][e] = v; } }
        warp_mma<24, 3, 1, false>(sm.Bm, LDB, 0, sm.PB, LDB, 8 * warp, d, g, t); cfrag_store<3, 1>(sm.H, LDH, 0, 8 * warp, MU, d, g, t); } }
    __syncthreads();
    issue_q(k);                                      // B~ is idle now: Q~ of this node streams into it
    if (k > 0) issue_tail(k - 1);                   // the tail buffer is free: next node's small pieces stream in during phase 3
    // ---- phase 3: one warp factors H and solves for Y and the gains ; the other three compute P <- Q~ + A~'W (column 30: q~ + A~'(p + P b~)).
    // The serial role rotates over the warps (= over the SM sub-partitions): co-resident CTAs would otherwise queue their serial sections on one scheduler.
    const int sw = (k + b) & 3;
    if (!QMB_TMA) gQ.wait();                        // cp.async path: the wait contains a CTA barrier, so all four warps take it
    if (warp == sw) {
      if (QMB_TMA) gQ.skip();
      // (a) Cholesky of H with the factor in registers (lane = row, read from the upper triangle: column access is bank-conflict free;
      //     pivot and column broadcasts by shuffle) fused with the forward substitution Y = L^{-1}[G | h] (lane = column of [G | h]):
      //     the broadcast L[c][j] that updates row c of the factor is exactly the multiplier of the right-looking substitution step,
      //     so Y costs one more FMA per shuffle and no extra dependent chain.  Lanes >= MU carry zeros in the factor role.
      double hr[MU], y[MU]; double dinv = 0.0; bool ok = true; double* Yb = sm.PB;   // PB is free after phase 2; Y uses leading dimension LDX
#pragma unroll
      for (int c = 0; c < MU; ++c) { hr[c] = (lane < MU) ? sm.H[c * LDH + lane] : 0.0; y[c] = sm.G[c * LDG + lane]; }
#pragma unroll
      for (int j = 0; j < MU; ++j) {
        const double djj = __shfl_sync(FULL, hr[j], j); if (!(djj > 0.0)) ok = false;
        const double inv = rsqrt(djj); const double lij = hr[j] * inv;
        if (lane == j) dinv = inv;
        if (lane < MU) sm.Lt[j * MU + lane] = lij;
        y[j] *= inv; Yb[j * LDX + lane] = y[j];
#pragma unroll
        for (int c = j + 1; c < MU; ++c) { const double lcj = __shfl_sync(FULL, lij, c); hr[c] = fma(-lij, lcj, hr[c]); y[c] = fma(-lcj, y[j], y[c]); }
      }
      if (lane < MU) sm.dut[lane] = dinv;
      if (!ok && lane == 0) sm.flag = 1;
      __syncwarp();
      // (b) back substitution K = -L^{-T} Y, lane = column: factor entries are warp-uniform broadcasts, the running column lives in registers.
      //     The gains leave with the pitch of their shared-memory target in the rollout (K rows of LDG doubles, feed-forward k in column 30).
      double* gk = gb + (size_t)k * GAIN_DBL;
#pragma unroll
      for (int a = MU - 1; a >= 0; --a) {  // L' z = y, right-looking over row a of L'
        asm volatile("" ::: "memory");
        y[a] *= sm.dut[a];
        gk[a * LDG + lane] = -y[a];
#pragma unroll
        for (int c = 0; c < a; ++c) y[c] = fma(-sm.Lt[c * MU + a], y[a], y[c]);
      }
    } else {
      if (QMB_TMA) gQ.wait();                                                  // Q~ (packed lower triangle) is in the B~ buffer, q~ in column 30 of P
      const int hi = (warp - sw - 1) & 3;                                      // helper index 0..2: 8x8 tiles hi, hi+3, ... of the 4x4 tile grid
      // (tried: all tiles' A~'W first and the wait for Q~ afterwards - 12 more live registers, 17.2 -> 17.7 ms, profiles/r02_ab_k3_rejected.json)
      for (int tile = hi; tile < 16; tile += 3) { const int i0 = 8 * (tile >> 2), j0 = 8 * (tile & 3);
        double c[1][1][2]; const int ri = i0 + g;   // C operand = Q~ (packed lower triangle in the B~ buffer) | q~ (column 30 of P)
#pragma unroll
        for (int e = 0; e < 2; ++e) { const int cj = j0 + 2 * t + e; double v = (ri < NX && cj <= NX) ? (cj == NX ? sm.P[ri * LDX + NX] : (cj <= ri ? sm.Bm[q_row_offset(ri) + cj] : sm.Bm[q_row_offset(cj) + ri])) : 0.0;
          if (ri >= 24 && ri < NX && cj <= NX) v += sm.W[ri * LDX + cj];   // identity rows 24:30 of A~: row ri of A~'W is row ri of W
          c[0][0][e] = v; }
        warp_mma<24, 1, 1, false>(sm.A, LDX, i0, sm.W, LDX, j0, c, g, t); cfrag_store<1, 1>(sm.P, LDX, i0, j0, NX, c, g, t); }
    }
    __syncthreads();
    if (sm.flag) { st |= MST_NOT_PD; if (k > 0) gT.wait(); break; }            // (an in-flight copy must land before the CTA may exit)
    if (k > 0) { if (tnext != 1) issue_ab(k - 1); gT.wait(); if (tnext != 1) expand(); }   // A~/B~ buffers are free: fetch and rebuild the next node while phase 4 runs
    // ---- phase 4: P -= Y'Y, column 30: p -= Y' yh (warp = 16x16 block; the top-of-loop barrier closes this phase) ----
    { const double* Yb = sm.PB; const int i0 = 16 * (warp >> 1), j0 = 16 * (warp & 1);
      double c[2][2][2]; cfrag_load<2, 2>(sm.P, LDX, i0, j0, NX, c, g, t); warp_mma<MU, 2, 2, true>(Yb, LDX, i0, Yb, LDX, j0, c, g, t); cfrag_store<2, 2>(sm.P, LDX, i0, j0, NX, c, g, t); }
  }
  __syncthreads();
  if (kValueFn && !(st & MST_NOT_PD)) store_vf(0);   // the rollout's first copies land in buffer set 0; sm.P (set 1) is rewritten after its first barrier
  // ---- forward rollout: du~ = K dx + k ; dx+ = A~ dx + B~ du~ + b~ ; du = Px dx + Pu du~ + Pe ; armijo = sum q~'dx + r~'du~.  Works on the structured
  //      record directly (no dense A~ / B~): per node four copies - gains, rows 3:12 of A~ and B~, tail - into one of two buffer sets ----
  double armijo = 0.0, dxn2 = 0.0, dun2 = 0.0;
  if (!(st & MST_NOT_PD)) {
    // buffer set 0: {G, A[0:9 rows], Bm[0:9 rows], A + 9 rows} ; set 1: {W, P, PB, P + 9 rows}
    auto issue_fwd = [&](int k) {
      if (k >= N) return; const int o = k & 1; CopyGroup& cg = o ? gF1 : gAB; const double* sg = sgb + (size_t)k * STAGE_DBL; const bool ev = node_type(k) == 1;
      cg.begin((ev ? 0 : (GAIN_DBL + 9 * LDX + 9 * LDB) * 8) + TAIL_DBL * 8, tid);
      cg.copy((o ? sm.P : sm.A) + 9 * LDX, sg + ST_TAIL, TAIL_DBL * 8, tid);
      if (!ev) { cg.copy(o ? sm.W : sm.G, gb + (size_t)k * GAIN_DBL, GAIN_DBL * 8, tid); cg.copy(o ? sm.P : sm.A, sg + ST_AR, 9 * LDX * 8, tid); cg.copy(o ? sm.PB : sm.Bm, sg + ST_BR, 9 * LDB * 8, tid); } };
    issue_fwd(0);
    for (int k = 0; k < N; ++k) {
      const int o = k & 1; const double* Kb = o ? sm.W : sm.G; const double* ARb = o ? sm.P : sm.A; const double* BRb = o ? sm.PB : sm.Bm; const double* tl = (o ? sm.P : sm.A) + 9 * LDX;
      double* dxk = dxo + ((size_t)b * nmax + k) * NX; double* duk = duo + ((size_t)b * nmax + k) * NU;
      // dx is double buffered (sm.dx / sm.tmp): the next state is written into the other buffer, and the barrier at the top of the next
      // iteration publishes it - two barriers per node instead of four
      const double* dxc = (k & 1) ? sm.tmp : sm.dx; double* dxn = (k & 1) ? sm.dx : sm.tmp;
      if (o) gF1.wait(); else gAB.wait();
      if (QMB_TMA) __syncthreads();              // record k has landed; dx(k) (written by other threads in the previous iteration) is visible; nobody reads buffer set (k+1)&1 any more
      issue_fwd(k + 1);
      const int32_t* si = reinterpret_cast<const int32_t*>(tl + T_INT); const int type = si[SI_TYPE], ndep = si[SI_NDEP], mm = si[SI_M]; const double dtw = tl[T_MISC];
      if (tid < NX) { const double dxi = dxc[tid]; dxk[tid] = dxi; dxn2 += dxi * dxi; }
      if (type == 1) { if (tid < NX) { duk[tid] = 0.0; dxn[tid] = dxc[tid] + tl[T_b + tid]; } continue; }
      { double s = 0.0;   // du~ = K dx + k: 4 threads per row (all lanes take part in the quad reduction); columns 30 / 31 of K meet dx[30] = dx[31] = 0
        if (ti < MU) { const double* kr = Kb + ti * LDG + jb * 8; const double* dx = dxc + jb * 8;
#pragma unroll
          for (int v = 0; v < 8; ++v) s = fma(kr[v], dx[v], s); }
        s += __shfl_xor_sync(FULL, s, 1); s += __shfl_xor_sync(FULL, s, 2); if (ti < MU && jb == 0) sm.dut[ti] = s + Kb[ti * LDG + NX]; }
      __syncthreads();
      { // dependent inputs du_d = Px_d dx + Pu_d du~ + Pe_d, 8 threads per input (MAXDEP * 8 = all 128 threads); a dependent joint also owns its row of the dynamics:
        // dx+[joint] = dx[joint] + dtw * (Px dx + Pu du~) + b~[joint]
        static_assert(MAXDEP * 8 == RIC_THREADS, "one 8-thread group per dependent input");
        const int d = tid >> 3, q8 = tid & 7; double s = 0.0; const int di = (d < ndep) ? si[SI_DEP + d] : -1;
        if (di >= 12) { const int j = di - 12, lg = j / 3, first = 3 * lg; const double* px = tl + T_PXJ + j * 12;
          s = px[q8] * dxc[sup_col(q8, first)]; if (q8 < 4) s = fma(px[q8 + 8], dxc[sup_col(q8 + 8, first)], s);
          if (q8 >= 4 && q8 < 6) { const int foot = (lfp >> (2 * lg)) & 3; const int col = si[SI_PCOL + 2 * foot + q8 - 4]; if (si[SI_PIV + foot] >= 0 && col >= 0) s = fma(tl[T_PU2 + 2 * foot + q8 - 4], sm.dut[col], s); } }
        s += __shfl_xor_sync(FULL, s, 1); s += __shfl_xor_sync(FULL, s, 2); s += __shfl_xor_sync(FULL, s, 4);
        if (di >= 0 && q8 == 0) { const double full = s + tl[T_PED + d]; duk[di] = full; dun2 += full * full; if (di >= 12) dxn[di] = dxc[di] + dtw * s + tl[T_b + di]; } }
      if (tid < NX) armijo += tl[T_q + tid] * dxc[tid];
      if (tid < MU) { const double dut = sm.dut[tid]; armijo += tl[T_r + tid] * dut; const int fi = si[SI_FREE + tid];
        if (fi >= 0) { duk[fi] = dut; dun2 += dut * dut; if (fi >= 12) dxn[fi] = dxc[fi] + dtw * dut + tl[T_b + fi]; } }   // free joint: dx+ = dx + dtw du + b~
      if (warp == 1 && lane < 3) { double acc = 0.0; for (int a = 0; a < mm; ++a) { const int fa = si[SI_FREE + a]; if (fa < 12 && fa - 3 * (fa / 3) == lane) acc += sm.dut[a]; }   // h_lin rows: forces / m
        dxn[lane] = dxc[lane] + dtw * imass * acc + tl[T_b + lane]; }
      if (warp >= 2) { const int rr = (tid - 64) >> 2; double s = 0.0;   // dense rows 3:12: A~ row . dx + B~ row . du~  (4 threads per row; column 30 of the A~ row is b~ and meets dx[30] = 0)
        if (rr < 9) { const double* ar = ARb + rr * LDX + jb * 8; const double* dx = dxc + jb * 8;
#pragma unroll
          for (int v = 0; v < 8; ++v) s = fma(ar[v], dx[v], s);
          if (jb < 3) { const double* br = BRb + rr * LDB + jb * 8; const double* du = sm.dut + jb * 8;
#pragma unroll
            for (int v = 0; v < 8; ++v) s = fma(br[v], du[v], s); } }
        s += __shfl_xor_sync(FULL, s, 1); s += __shfl_xor_sync(FULL, s, 2); if (rr < 9 && jb == 0) dxn[3 + rr] = s + tl[T_b + 3 + rr]; }
    }
    __syncthreads();
    if (tid < NX) { const double dxi = ((N & 1) ? sm.tmp : sm.dx)[tid]; dxo[((size_t)b * nmax + N) * NX + tid] = dxi; duo[((size_t)b * nmax + N) * NU + tid] = 0.0; dxn2 += dxi * dxi; armijo += sgb[(size_t)N * STAGE_DBL + ST_TAIL + T_q + tid] * dxi; }
  }
  armijo = warp_sum(armijo); dxn2 = warp_sum(dxn2); dun2 = warp_sum(dun2);
  __syncthreads();
  if (lane == 0) { sm.red[warp][0] = armijo; sm.red[warp][1] = dxn2; sm.red[warp][2] = dun2; }
  __syncthreads();
  if (tid == 0) { double a = 0, x2 = 0, u2 = 0; for (int w = 0; w < RIC_THREADS / 32; ++w) { a += sm.red[w][0]; x2 += sm.red[w][1]; u2 += sm.red[w][2]; }
    double* rb = robot + (size_t)b * ROBOT_DBL; rb[0] = a; rb[1] = perf[0]; rb[2] = perf[1]; rb[3] = perf[2]; rb[4] = sqrt(x2); rb[5] = sqrt(u2); if (st) atomicOr(&status[b], st); }
}

// =====================================================================================================
// K4: filter line search (one CTA per robot; warps stride over nodes) + trajectory update + input fix-up
// One THREAD per node (node_eval.cuh): the trial point's kinematics, flow maps, cost and constraint residuals are chains of scalar work with 3..9 useful lanes in
// the warp-per-node form (7.2 ms at 8192 robots); here every lane carries a node, nothing lives in shared memory, and the per-robot sums are a block reduction.
__device__ __forceinline__ void fixup_inputs(MpcSolutionDev sol, int b, int nmax, int n, int tid, int nthreads) {
  // toPrimalSolution [upstream]: input at a pre-event node repeats the previous one; last input repeated
  const int32_t* ge = sol.event + (size_t)b * nmax; double* gu = sol.u + (size_t)b * nmax * NU;
  // thread i owns component i at every node: the copies chain through k inside one thread, so no barrier is needed (the caller synchronises before the call)
  for (int i = tid; i < NU; i += nthreads) for (int k = 1; k < n; ++k) if ((k == n - 1) || (ge[k] == 1)) gu[(size_t)k * NU + i] = gu[(size_t)(k - 1) * NU + i];
}

#ifndef QMB_LS_MINB
#define QMB_LS_MINB 4
#endif
__global__ void __launch_bounds__(32 * LS_WARPS, QMB_LS_MINB) mpc_linesearch_kernel(const DevModel* __restrict__ mdl, int b0, int B, int nmax, MpcProblemDev p, MpcSolutionDev sol, const double* __restrict__ dxo, const double* __restrict__ duo,
                                                                     const double* __restrict__ robot, int32_t* __restrict__ status, double* __restrict__ step_info, int iteration) {
  __shared__ double red[LS_WARPS][3]; __shared__ int decision; __shared__ double s_ev[EMAX]; __shared__ unsigned char s_modes[EMAX + 8];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31; const int b = b0 + blockIdx.x; if (b >= B) return;
  if (status[b] & MST_CONVERGED) return;
  const int n = sol.n_nodes[b]; const int N = n - 1;
  const double* gt = sol.t + (size_t)b * nmax; const int32_t* ge = sol.event + (size_t)b * nmax;
  double* gx = sol.x + (size_t)b * nmax * NX; double* gu = sol.u + (size_t)b * nmax * NU; const double* gdx = dxo + (size_t)b * nmax * NX; const double* gdu = duo + (size_t)b * nmax * NU;
  const int ne = clamp_events(p.n_events[b]); const double* ev = s_ev; const unsigned char* modes = s_modes;
  if (tid < 32) { const double* gev = p.event_times + (size_t)b * EMAX; const int32_t* gmodes = p.modes + (size_t)b * (EMAX + 1); s_ev[lane] = (lane < ne) ? gev[lane] : 0.0; s_modes[lane] = (unsigned char)((lane <= ne) ? gmodes[lane] : 15); if (lane == 0) s_modes[EMAX] = (unsigned char)((EMAX <= ne) ? gmodes[EMAX] : 15); }
  __syncthreads();
  const int nk = clamp_targets(p.n_target[b]); const double* tt = p.target_times + (size_t)b * KMAX; const double* ts = p.target_states + (size_t)b * KMAX * TARGET_DIM;
  const double* rb = robot + (size_t)b * ROBOT_DBL; const double armijo = rb[0], base_cost = rb[1], base_viol = sqrt(rb[2] + rb[3]), dxn = rb[4], dun = rb[5];
  const bool failed = (status[b] & MST_NOT_PD) != 0;
  double alpha = 1.0; bool accepted = false; double sc = base_cost, sd = rb[2], se = rb[3];
  const double w1 = mdl->rk_w1, w2 = mdl->rk_w2;
  while (!failed) {
    double cost = 0.0, dyn = 0.0, eq = 0.0;
    for (int k = tid; k <= N; k += 32 * LS_WARPS) {
      double xa[NX], ua[NU]; const bool terminal = (k == N);
#pragma unroll
      for (int i = 0; i < NX; ++i) { xa[i] = gx[(size_t)k * NX + i] + alpha * gdx[(size_t)k * NX + i]; ua[i] = terminal ? 0.0 : gu[(size_t)k * NU + i] + alpha * gdu[(size_t)k * NU + i]; }
      if (k == 0) { double s = 0.0; for (int i = 0; i < NX; ++i) { const double d = p.x0[(size_t)b * NX + i] - xa[i]; s = fma(d, d, s); } dyn += s; }
      if (!terminal && ge[k] == 1) { double s = 0.0; for (int i = 0; i < NX; ++i) { const double d = xa[i] - (gx[(size_t)(k + 1) * NX + i] + alpha * gdx[(size_t)(k + 1) * NX + i]); s = fma(d, d, s); } dyn += s; continue; }
      const double t = interval_start(gt[k], ge[k]);
      const double dt = terminal ? 1.0 : interval_end(gt[k + 1], ge[k + 1]) - t; const int mode = mode_at_time(ev, modes, ne, t); const int fm = terminal ? 0 : flag_mask(mode);
      ne::BaseKin bk; ne::FlowAcc acc; double f1[12];
      ne::base_eval<false>(mdl, xa, bk); ne::flow_acc_init(acc);
      { double fe[4][3], pf[4][3];
#pragma unroll 1
        for (int i = 0; i < 4; ++i) { double d[3], Jl[9]; ne::foot_eval<false>(mdl, xa, ua, bk, i, acc, d, pf[i], Jl, nullptr, nullptr); if (!terminal) ne::foot_velocity_1<false>(mdl, xa, ua, bk, i, d, Jl, nullptr, fe[i], nullptr); }
        if (!terminal) eq += dt * ne::equality_ss(mdl, ua, fe, pf, fm, ev, modes, ne, t, nullptr); }
      ne::flow_finish<false>(mdl, xa, bk, acc, f1, nullptr);
      { const ne::TargetSeg sg = ne::target_segment(tt, ts, nk, t); double pref[3], qref[4], ee[6]; ne::target_pose(sg, nk, pref, qref); ne::ee_eval<false>(mdl, xa, bk, pref, qref, ee, nullptr);
        cost += dt * ne::cost_value(mdl, xa, ua, sg, ee, fm, terminal); }
      if (terminal) continue;
      const double cdt = mdl->rk_c * dt;   // second stage in place (the trial state is re-read from L2 for the defect)
#pragma unroll
      for (int i = 0; i < NX; ++i) xa[i] += cdt * (i < 12 ? f1[i < 12 ? i : 0] : ua[i]);
      double f2[12]; ne::base_eval<false>(mdl, xa, bk); ne::flow_acc_init(acc);
#pragma unroll 1
      for (int i = 0; i < 4; ++i) { double d[3]; ne::foot_eval<false>(mdl, xa, ua, bk, i, acc, d, nullptr, nullptr, nullptr, nullptr); }
      ne::flow_finish<false>(mdl, xa, bk, acc, f2, nullptr);
      double s = 0.0;
#pragma unroll
      for (int i = 0; i < NX; ++i) { const double fa = (i < 12) ? f1[i < 12 ? i : 0] : ua[i], fb = (i < 12) ? f2[i < 12 ? i : 0] : ua[i];   // rows 12:30 of the flow map are the joint-velocity inputs
        const double x0i = gx[(size_t)k * NX + i] + alpha * gdx[(size_t)k * NX + i];
        const double d = x0i + dt * (w1 * fa + w2 * fb) - (gx[(size_t)(k + 1) * NX + i] + alpha * gdx[(size_t)(k + 1) * NX + i]); s = fma(d, d, s); }
      dyn += dt * s;
    }
    cost = warp_sum(cost); dyn = warp_sum(dyn); eq = warp_sum(eq);
    if (lane == 0) { red[warp][0] = cost; red[warp][1] = dyn; red[warp][2] = eq; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double c = 0, dd = 0, e = 0; for (int w = 0; w < LS_WARPS; ++w) { c += red[w][0]; dd += red[w][1]; e += red[w][2]; }
      // FilterLinesearch::acceptStep [upstream ocs2_oc/search_strategy/FilterLinesearch.cpp]
      const double sv = sqrt(dd + e), am = alpha * armijo; bool acc;
      if (sv > mdl->g_max) acc = sv < (1.0 - mdl->gamma_c) * base_viol;
      else if (sv < mdl->g_min && base_viol < mdl->g_min && am < 0.0) acc = c < base_cost + mdl->armijo_factor * am;
      else acc = (c < base_cost - mdl->gamma_c * base_viol) || (sv < (1.0 - mdl->gamma_c) * base_viol);
      red[0][0] = c; red[0][1] = dd; red[0][2] = e;
      int dec = 0; if (acc) dec = 1; else { const double an = alpha * mdl->alpha_decay; if ((an * dxn < mdl->delta_tol && an * dun < mdl->delta_tol) || an < mdl->alpha_min) dec = 2; }
      decision = dec;
    }
    __syncthreads();
    const int dec = decision; sc = red[0][0]; sd = red[0][1]; se = red[0][2];
    __syncthreads();
    if (dec == 1) { accepted = true; break; }
    if (dec == 2) break;
    alpha *= mdl->alpha_decay;
  }
  if (accepted) {
    // x += alpha dx, u += alpha du: four independent elements per thread and round (the loads of a round are issued before its stores)
    const int tot = n * NX, totu = N * NU, nt = blockDim.x;
    for (int e0 = threadIdx.x; e0 < tot; e0 += 4 * nt) {
      double vx[4], vu[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) { const int e = e0 + q * nt; vx[q] = (e < tot) ? gx[e] + alpha * gdx[e] : 0.0; vu[q] = (e < totu) ? gu[e] + alpha * gdu[e] : 0.0; }
#pragma unroll
      for (int q = 0; q < 4; ++q) { const int e = e0 + q * nt; if (e < tot) gx[e] = vx[q]; if (e < totu) gu[e] = vu[q]; }
    }
  } else { alpha = 0.0; sc = base_cost; sd = rb[2]; se = rb[3]; }
  __syncthreads();
  fixup_inputs(sol, b, nmax, n, threadIdx.x, blockDim.x);
  if (threadIdx.x == 0) {
    int flags = accepted ? 0 : MST_NO_STEP;
    if (iteration + 1 < mdl->sqp_iterations) {   // SqpSolver::checkConvergence [upstream ocs2_sqp, recalled]: STEPSIZE, METRICS, PRIMAL (ITERATIONS = the host loop bound)
      const bool stepsize = alpha < mdl->alpha_min;                                                       // a rejected step reports stepSize 0
      const bool metrics = fabs(sc - base_cost) < mdl->cost_tol && sqrt(sd + se) < mdl->g_min;
      const bool primal = alpha * dxn < mdl->delta_tol && alpha * dun < mdl->delta_tol;
      if (stepsize || metrics || primal) flags |= MST_CONVERGED;
    }
    if (flags) atomicOr(&status[b], flags);
    double* si = step_info + (size_t)b * 4; si[0] = alpha; si[1] = sc; si[2] = sd; si[3] = se; }
}

// =====================================================================================================
// DDP variant (ddp{} of task.info:33-71, qmb200_mpc_set_solver): single-shooting rollouts.  One warp per robot, sequential in time.
//   mode 0  nominal rollout: x_0 = measured state, x_{k+1} = RK2(x_k, u_nom,k) - the trajectory the LQ approximation is built along (no dynamics defect)
//   mode 1  line search [upstream ocs2_ddp LineSearchStrategy, recalled]: for alpha = maxStep * contraction^j >= minStep roll out the updated affine controller
//           u = u_nom + alpha du_ff + K (x - x_nom) - evaluated from the structured stage record and the projected gains exactly as K3's linear rollout does,
//           du = Px dx + Pu (K~ dx + alpha k~) + alpha Pe - and accept the first alpha with merit = cost + penalty * sqrt(equality SSE) below the nominal merit.
// The reference integrates these rollouts with ODE45 (rollout{}, task.info:128-136) and, for algorithm SLQ, sweeps a continuous-time Riccati equation; this is the
// discrete-time form on the solver's own grid (ddp.algorithm ILQR): same LQ model, same backward pass as the SQP path (K2 / K3).
// Thread-parallel form (node_eval.cuh): a rollout is sequential in time, so one THREAD carries one rollout - the nominal rollout one per robot, the line search
// one per (robot, step length): all step lengths of ddp.lineSearch run side by side (what OCS2 does with its thread pool) and the first accepted one in descending
// order wins, so the result is the sequential search's.  The accepted step is then re-rolled in place by one thread per robot (mode 2).
constexpr int RO_THREADS = 128, RO_MAXTRIALS = 32;
// one RK2 step of the flow map from (x, u); with PERF also the node's cost (unscaled by dt) and equality SSE at (x, u).  x is replaced by the next state.
template <bool PERF, class MT>
__device__ __forceinline__ void rollout_step(const DevModel* __restrict__ mdl, double* x, const double* u, double t, double dt, int fm, const double* ev, const MT* modes, int ne, const double* tt, const double* ts, int nk, double& cost, double& eq) {
  ne::BaseKin bk; ne::FlowAcc acc; double f1[12], x2[NX]; ne::base_eval<false>(mdl, x, bk); ne::flow_acc_init(acc);
  if (PERF) { double fe[4][3], pf[4][3];
#pragma unroll 1
    for (int i = 0; i < 4; ++i) { double d[3], Jl[9]; ne::foot_eval<false>(mdl, x, u, bk, i, acc, d, pf[i], Jl, nullptr, nullptr); ne::foot_velocity_1<false>(mdl, x, u, bk, i, d, Jl, nullptr, fe[i], nullptr); }
    eq += dt * ne::equality_ss(mdl, u, fe, pf, fm, ev, modes, ne, t, nullptr);
    const ne::TargetSeg sg = ne::target_segment(tt, ts, nk, t); double pref[3], qref[4], ee[6]; ne::target_pose(sg, nk, pref, qref); ne::ee_eval<false>(mdl, x, bk, pref, qref, ee, nullptr);
    cost += dt * ne::cost_value(mdl, x, u, sg, ee, fm, false);
  } else {
#pragma unroll 1
    for (int i = 0; i < 4; ++i) { double d[3]; ne::foot_eval<false>(mdl, x, u, bk, i, acc, d, nullptr, nullptr, nullptr, nullptr); } }
  ne::flow_finish<false>(mdl, x, bk, acc, f1, nullptr);
  const double cdt = mdl->rk_c * dt, w1 = mdl->rk_w1, w2 = mdl->rk_w2;
#pragma unroll
  for (int i = 0; i < NX; ++i) x2[i] = x[i] + cdt * (i < 12 ? f1[i < 12 ? i : 0] : u[i]);
  double f2[12]; ne::base_eval<false>(mdl, x2, bk); ne::flow_acc_init(acc);
#pragma unroll 1
  for (int i = 0; i < 4; ++i) { double d[3]; ne::foot_eval<false>(mdl, x2, u, bk, i, acc, d, nullptr, nullptr, nullptr, nullptr); }
  ne::flow_finish<false>(mdl, x2, bk, acc, f2, nullptr);
#pragma unroll
  for (int i = 0; i < NX; ++i) x[i] += dt * (w1 * (i < 12 ? f1[i < 12 ? i : 0] : u[i]) + w2 * (i < 12 ? f2[i < 12 ? i : 0] : u[i]));
}
// input of the updated affine controller at node k: u = u_nom + Px dx + Pu (K~ dx + alpha k~) + alpha Pe, from the structured stage record and the projected gains
__device__ __forceinline__ void rollout_input(const double* __restrict__ tl, const double* __restrict__ Kg, const double* __restrict__ unom, const double* dxv, double alpha, int lfp, double* un) {
  const int32_t* si = reinterpret_cast<const int32_t*>(tl + T_INT); const int ndep = si[SI_NDEP]; double dut[MU];
  for (int a = 0; a < MU; ++a) { const double* kr = Kg + a * LDG; double s0 = 0.0, s1 = 0.0;   // du~ = K~ dx + alpha k~ (rows of padded inputs are zero)
#pragma unroll 5
    for (int j = 0; j < NX; j += 2) { s0 = fma(kr[j], dxv[j], s0); s1 = fma(kr[j + 1], dxv[j + 1], s1); }
    dut[a] = s0 + s1 + alpha * kr[NX]; }
  for (int c = 0; c < NU; ++c) un[c] = unom[c];
  for (int a = 0; a < MU; ++a) { const int fa = si[SI_FREE + a]; if (fa >= 0) un[fa] += dut[a]; }
  for (int d = 0; d < ndep; ++d) { const int di = si[SI_DEP + d]; double du = alpha * tl[T_PED + d];
    if (di >= 12) { const int j = di - 12, lg = j / 3, first = 3 * lg; const double* px = tl + T_PXJ + j * 12;
      for (int c = 0; c < 12; ++c) du = fma(px[c], dxv[sup_col(c, first)], du);
      const int foot = (lfp >> (2 * lg)) & 3; if (si[SI_PIV + foot] >= 0) for (int q2 = 0; q2 < 2; ++q2) { const int col = si[SI_PCOL + 2 * foot + q2]; if (col >= 0) du = fma(tl[T_PU2 + 2 * foot + q2], dut[col], du); } }
    un[di] += du; }
}
// mode 0: nominal rollout (thread = robot).  mode 2: decision on the trial merits + in-place rollout of the accepted step (thread = robot).
#ifndef QMB_RO_MINB
#define QMB_RO_MINB 2
#endif
__global__ void __launch_bounds__(RO_THREADS, QMB_RO_MINB) mpc_rollout_kernel(const DevModel* __restrict__ mdl, int b0, int B, int nmax, MpcProblemDev p, MpcSolutionDev sol, const double* __restrict__ stage, const double* __restrict__ gains,
                                                                   double* __restrict__ trial, const double* __restrict__ robot, int32_t* __restrict__ status, double* __restrict__ step_info, int mode_ls, int n_trials, int tr_pitch, int iteration) {
  const long long gid = (long long)blockIdx.x * RO_THREADS + threadIdx.x;
  const int b = b0 + (int)gid; if (b >= B) return;
  if (status[b] & MST_CONVERGED) return;
  const int n = sol.n_nodes[b]; const int N = n - 1;
  const double* gt = sol.t + (size_t)b * nmax; const int32_t* ge = sol.event + (size_t)b * nmax;
  double* gx = sol.x + (size_t)b * nmax * NX; double* gu = sol.u + (size_t)b * nmax * NU;
  const int ne = clamp_events(p.n_events[b]); const double* ev = p.event_times + (size_t)b * EMAX; const int32_t* modes = p.modes + (size_t)b * (EMAX + 1);
  const int lfp = pack_leg_foot(mdl);
  const int nk = clamp_targets(p.n_target[b]); const double* tt = p.target_times + (size_t)b * KMAX; const double* ts = p.target_states + (size_t)b * KMAX * TARGET_DIM;
  double xa[NX], cost = 0.0, eq = 0.0;
  if (mode_ls == 0) {
#pragma unroll
    for (int i = 0; i < NX; ++i) { xa[i] = p.x0[(size_t)b * NX + i]; gx[i] = xa[i]; }
    for (int k = 0; k < N; ++k) {
      if (ge[k] != 1) { const double t = interval_start(gt[k], ge[k]); const double dt = interval_end(gt[k + 1], ge[k + 1]) - t; double u[NU];
#pragma unroll
        for (int i = 0; i < NU; ++i) u[i] = gu[(size_t)k * NU + i];
        rollout_step<false>(mdl, xa, u, t, dt, 0, ev, modes, ne, tt, ts, nk, cost, eq); }
#pragma unroll
      for (int i = 0; i < NX; ++i) gx[(size_t)(k + 1) * NX + i] = xa[i];
    }
    return;
  }
  const double* rb = robot + (size_t)b * ROBOT_DBL; const double base_cost = rb[1], base_eq = rb[3]; const double pen = mdl->ddp_penalty;
  const double merit0 = base_cost + pen * sqrt(base_eq); const bool failed = (status[b] & MST_NOT_PD) != 0;
  double* tb = trial + (size_t)b * RO_MAXTRIALS * 2;
  double alpha = mdl->ddp_max_step; bool accepted = false; double sc = base_cost, se = base_eq;
  {   // mode 2: the first step length (descending) whose merit passes the armijo test [upstream ocs2_ddp LineSearchStrategy, recalled]
    if (!failed) for (int j = 0; j < n_trials; ++j) { const double c = tb[2 * j], e = tb[2 * j + 1], merit = c + pen * sqrt(e);
        if (merit < merit0 - mdl->ddp_armijo * alpha * fabs(merit0)) { accepted = true; sc = c; se = e; break; } alpha *= mdl->ddp_contraction; }
  }
  if (accepted) {
    const double* sgb = stage + (size_t)b * nmax * STAGE_DBL; const double* gb = gains + (size_t)b * nmax * GAIN_DBL;
    double xnom[NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) { xa[i] = p.x0[(size_t)b * NX + i]; xnom[i] = gx[i]; }
#pragma unroll
    for (int i = 0; i < NX; ++i) gx[i] = xa[i];
    for (int k = 0; k < N; ++k) {
      if (ge[k] == 1) {   // event node: identity jump map, no input
        for (int i = 0; i < NU; ++i) gu[(size_t)k * NU + i] = 0.0;
      } else {
        const double* tl = sgb + (size_t)k * STAGE_DBL + ST_TAIL; double dxv[NX], un[NU];
#pragma unroll
        for (int i = 0; i < NX; ++i) dxv[i] = xa[i] - xnom[i];
        rollout_input(tl, gb + (size_t)k * GAIN_DBL, gu + (size_t)k * NU, dxv, alpha, lfp, un);
        for (int i = 0; i < NU; ++i) gu[(size_t)k * NU + i] = un[i];
        const double t = interval_start(gt[k], ge[k]); const double dt = interval_end(gt[k + 1], ge[k + 1]) - t; const int fm = flag_mask(mode_at_time(ev, modes, ne, t));
        rollout_step<false>(mdl, xa, un, t, dt, fm, ev, modes, ne, tt, ts, nk, cost, eq);
      }
      // the nominal state of the next node is read before the new one replaces it (in-place commit)
#pragma unroll
      for (int i = 0; i < NX; ++i) { xnom[i] = gx[(size_t)(k + 1) * NX + i]; gx[(size_t)(k + 1) * NX + i] = xa[i]; }
    }
  }
  if (!accepted) { alpha = 0.0; sc = base_cost; se = base_eq; }
  // toPrimalSolution [upstream]: input at a pre-event node repeats the previous one; last input repeated
  for (int k = 1; k < n; ++k) { if ((k == n - 1) || (ge[k] == 1)) for (int i = 0; i < NU; ++i) gu[(size_t)k * NU + i] = gu[(size_t)(k - 1) * NU + i]; }
  { int flags = accepted ? 0 : MST_NO_STEP; if (!accepted && iteration + 1 < mdl->sqp_iterations) flags |= MST_CONVERGED; if (flags) atomicOr(&status[b], flags);
    double* si = step_info + (size_t)b * 4; si[0] = alpha; si[1] = sc; si[2] = 0.0; si[3] = se; }
}

// The trial rollouts of the line search: thread = (robot, step length), the step lengths of a robot on adjacent lanes; cost and equality SSE of every step length go to
// `trial` [B][RO_MAXTRIALS][2].  The CTA walks the horizon in lock step and stages the feedback gains of its robots' current node in shared memory (one coalesced
// copy per node instead of 18 x 31 scattered loads per thread: those loads were 45 % of the samples of the unstaged kernel).
constexpr int RO_RPC_MAX = 16;   // robots per CTA: 16 x 4.9 KB of gains
__global__ void __launch_bounds__(RO_THREADS, QMB_RO_MINB) mpc_rollout_trials_kernel(const DevModel* __restrict__ mdl, int b0, int B, int nmax, MpcProblemDev p, MpcSolutionDev sol, const double* __restrict__ stage, const double* __restrict__ gains,
                                                                          double* __restrict__ trial, const double* __restrict__ robot, const int32_t* __restrict__ status, int n_trials, int tr_pitch, int rpc) {
  extern __shared__ __align__(16) unsigned char smem_raw[]; double* sK = reinterpret_cast<double*>(smem_raw);   // [rpc][GAIN_DBL]
  __shared__ int s_kmax;
  const int tid = threadIdx.x, nthr = blockDim.x, r = tid / tr_pitch, tr = tid - r * tr_pitch; const int bfirst = b0 + blockIdx.x * rpc, b = bfirst + r;
  const bool active = b < B && tr < n_trials && !(status[b] & (MST_CONVERGED | MST_NOT_PD));
  const int N = active ? sol.n_nodes[b] - 1 : 0;
  if (tid == 0) s_kmax = 0;
  __syncthreads();
  if (active) atomicMax(&s_kmax, N);
  __syncthreads();
  const int kmax = s_kmax; if (kmax <= 0) return;   // CTA-uniform
  const size_t bb = active ? (size_t)b : 0;
  const double* gt = sol.t + bb * nmax; const int32_t* ge = sol.event + bb * nmax; const double* gx = sol.x + bb * nmax * NX; const double* gu = sol.u + bb * nmax * NU;
  const int ne = clamp_events(p.n_events[bb]); const double* ev = p.event_times + bb * EMAX; const int32_t* modes = p.modes + bb * (EMAX + 1);
  const int lfp = pack_leg_foot(mdl);
  const int nk = clamp_targets(p.n_target[bb]); const double* tt = p.target_times + bb * KMAX; const double* ts = p.target_states + bb * KMAX * TARGET_DIM;
  const double* sgb = stage + bb * nmax * STAGE_DBL;
  double alpha = mdl->ddp_max_step; for (int j = 0; j < tr; ++j) alpha *= mdl->ddp_contraction;
  double xa[NX], xnom[NX], cost = 0.0, eq = 0.0;
#pragma unroll
  for (int i = 0; i < NX; ++i) { xa[i] = p.x0[bb * NX + i]; xnom[i] = gx[i]; }
  for (int k = 0; k < kmax; ++k) {
    __syncthreads();                                                   // the readers of node k - 1 are done
    for (int e = tid; e < rpc * GAIN_DBL; e += nthr) { const int rr = e / GAIN_DBL; const int br = bfirst + rr; sK[e] = (br < B) ? gains[((size_t)br * nmax + k) * GAIN_DBL + (e - rr * GAIN_DBL)] : 0.0; }
    __syncthreads();
    if (active && k < N) {
      if (ge[k] != 1) {   // (event node: identity jump map, no input)
        const double* tl = sgb + (size_t)k * STAGE_DBL + ST_TAIL; double dxv[NX], un[NU];
#pragma unroll
        for (int i = 0; i < NX; ++i) dxv[i] = xa[i] - xnom[i];
        rollout_input(tl, sK + r * GAIN_DBL, gu + (size_t)k * NU, dxv, alpha, lfp, un);
        const double t = interval_start(gt[k], ge[k]); const double dt = interval_end(gt[k + 1], ge[k + 1]) - t; const int fm = flag_mask(mode_at_time(ev, modes, ne, t));
        rollout_step<true>(mdl, xa, un, t, dt, fm, ev, modes, ne, tt, ts, nk, cost, eq);
      }
#pragma unroll
      for (int i = 0; i < NX; ++i) xnom[i] = gx[(size_t)(k + 1) * NX + i];
    }
  }
  if (active) {   // final cost at x_N
    const double t = interval_start(gt[N], ge[N]); ne::BaseKin bk; ne::base_eval<false>(mdl, xa, bk); double u0[NU]; for (int i = 0; i < NU; ++i) u0[i] = 0.0;
    const ne::TargetSeg sg = ne::target_segment(tt, ts, nk, t); double pref[3], qref[4], ee[6]; ne::target_pose(sg, nk, pref, qref); ne::ee_eval<false>(mdl, xa, bk, pref, qref, ee, nullptr);
    cost += ne::cost_value(mdl, xa, u0, sg, ee, 0, true);
    double* tb = trial + (size_t)b * RO_MAXTRIALS * 2; tb[2 * tr] = cost; tb[2 * tr + 1] = eq; }
}

__global__ void mpc_fixup_kernel(int B, int nmax, MpcSolutionDev sol) { const int b = blockIdx.x; if (b >= B) return; const int n = sol.n_nodes[b]; if (n >= 2) fixup_inputs(sol, b, nmax, n, threadIdx.x, blockDim.x); }

// =====================================================================================================
// MPC_MRT_Interface::evaluatePolicy with a feed-forward policy (QMController.cpp:141): linear interpolation of the stored solution, modeAtTime
__global__ void mpc_policy_eval_kernel(int b0, int B, int nmax, MpcSolutionDev sol, const int32_t* __restrict__ n_events, const double* __restrict__ event_times, const int32_t* __restrict__ modes,
                                       const double* __restrict__ tq, double* __restrict__ x_des, double* __restrict__ u_des, int32_t* __restrict__ mode_out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31; const int b = b0 + blockIdx.x * (blockDim.x >> 5) + warp; if (b >= B) return;
  const int n = sol.n_nodes[b]; const double* gt = sol.t + (size_t)b * nmax; const double t = tq[b];
  int idx; double a; time_segment(gt, n, t, idx, a); const int i2 = (idx + 1 < n) ? idx + 1 : idx;
  const double* gx = sol.x + (size_t)b * nmax * NX; const double* gu = sol.u + (size_t)b * nmax * NU;
  if (lane < NX) { x_des[(size_t)b * NX + lane] = a * gx[(size_t)idx * NX + lane] + (1.0 - a) * gx[(size_t)i2 * NX + lane]; u_des[(size_t)b * NU + lane] = a * gu[(size_t)idx * NU + lane] + (1.0 - a) * gu[(size_t)i2 * NU + lane]; }
  if (lane == 0) mode_out[b] = mode_at_time(event_times + (size_t)b * EMAX, modes + (size_t)b * (EMAX + 1), clamp_events(n_events[b]), t);
}

// =====================================================================================================
// Feedback policy (useFeedbackPolicy of the ddp / sqp / ipm blocks): the LinearController u = uff(t) + K(t) x of the last solve
// [upstream ocs2_oc multiple_shooting::toPrimalSolution with feedback, recalled]:
//   K_k = Px_k + Pu_k K~_k (remapProjectedGain), uff_k = u*_k - K_k x*_k on the solution after the step; a pre-event node and the last node repeat the bias and
//   gain of the node before them.  The controller is never materialised: the solve's stage record and projected gains stay untouched until the next solve, and
//   rollout_input() with alpha = 0 evaluates u*_s + (Px_s + Pu_s K~_s)(x - x*_s) = uff_s + K_s x from them.
// Robots whose last QP has no defined K~ (not positive definite, NaN, overflow, non-positive interval) keep the feed-forward policy.
constexpr int MST_NO_FEEDBACK = MST_OVERFLOW | MST_NAN | MST_NOT_PD | MST_NEG_DT;
// node whose bias and gain node k of an n-node solution uses, -1 when there is none (zero gain, bias = u*_k)
__device__ __forceinline__ int controller_node(const int32_t* __restrict__ ge, int n, int k) {
  int s = k; while (s > 0 && (s == n - 1 || ge[s] == 1)) --s;
  return (s >= n - 1 || ge[s] == 1) ? -1 : s;
}
// One warp per robot: the two bracketing nodes' projected gains (4.9 KB each) and record tails (3.4 KB each) are staged in shared memory with coalesced loads,
// then lanes 0 / 1 evaluate one node each with rollout_input() on the staged copy, and the lanes of the inputs blend the two with alpha.
constexpr int PF_WARPS = 2;
struct PolicySmem { double K[2][GAIN_DBL]; double tail[2][TAIL_DBL]; double dx[2][NX]; double u[2][NU]; };
__global__ void __launch_bounds__(32 * PF_WARPS) mpc_policy_feedback_kernel(const DevModel* __restrict__ mdl, int b0, int B, int nmax, MpcSolutionDev sol, const double* __restrict__ stage,
                                                                           const double* __restrict__ gains, const int32_t* __restrict__ status, const int32_t* __restrict__ n_events,
                                                                           const double* __restrict__ event_times, const int32_t* __restrict__ modes, const double* __restrict__ tq,
                                                                           const double* __restrict__ xq, double* __restrict__ x_des, double* __restrict__ u_des, int32_t* __restrict__ mode_out) {
  __shared__ PolicySmem s_pol[PF_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31; const int b = b0 + blockIdx.x * PF_WARPS + warp; if (b >= B) return;
  PolicySmem& sm = s_pol[warp];
  const int n = sol.n_nodes[b]; const double* gt = sol.t + (size_t)b * nmax; const int32_t* ge = sol.event + (size_t)b * nmax; const double t = tq[b];
  int idx; double a; time_segment(gt, n, t, idx, a); const int i2 = (idx + 1 < n) ? idx + 1 : idx;
  const double* gx = sol.x + (size_t)b * nmax * NX; const double* gu = sol.u + (size_t)b * nmax * NU;
  if (lane < NX) x_des[(size_t)b * NX + lane] = a * gx[(size_t)idx * NX + lane] + (1.0 - a) * gx[(size_t)i2 * NX + lane];
  if (lane == 0) mode_out[b] = mode_at_time(event_times + (size_t)b * EMAX, modes + (size_t)b * (EMAX + 1), clamp_events(n_events[b]), t);
  if (status[b] & MST_NO_FEEDBACK) {   // the feed-forward arithmetic of mpc_policy_eval_kernel
    if (lane < NU) u_des[(size_t)b * NU + lane] = a * gu[(size_t)idx * NU + lane] + (1.0 - a) * gu[(size_t)i2 * NU + lane];
    return;
  }
  const int src0 = controller_node(ge, n, idx), src1 = controller_node(ge, n, i2);
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int s = j ? src1 : src0; if (s < 0) continue;   // warp-uniform
    const size_t node = (size_t)b * nmax + s; const double* kg = gains + node * GAIN_DBL; const double* tl = stage + node * STAGE_DBL + ST_TAIL;
    for (int e = lane; e < GAIN_DBL; e += 32) sm.K[j][e] = kg[e];
    for (int e = lane; e < TAIL_DBL; e += 32) sm.tail[j][e] = tl[e];
    if (lane < NX) sm.dx[j][lane] = xq[(size_t)b * NX + lane] - gx[(size_t)s * NX + lane];
  }
  __syncwarp();
  if (lane < 2) {
    const int s = lane ? src1 : src0;
    if (s >= 0) rollout_input(sm.tail[lane], sm.K[lane], gu + (size_t)s * NU, sm.dx[lane], 0.0, pack_leg_foot(mdl), sm.u[lane]);
    else { const int k = lane ? i2 : idx; for (int c = 0; c < NU; ++c) sm.u[lane][c] = gu[(size_t)k * NU + c]; }
  }
  __syncwarp();
  if (lane < NU) u_des[(size_t)b * NU + lane] = a * sm.u[0][lane] + (1.0 - a) * sm.u[1][lane];
}

// Dense LinearController of robots [b0, b0 + count): one warp per (robot, node).  Lane j < 30 evaluates column j of K_k as rollout_input() of the unit vector e_j
// around a zero nominal input, lane 30 the bias u*_s + K_s (0 - x*_s).  Robots without a controller (or with `valid` false) get a zero gain and bias = u*_k.
__global__ void __launch_bounds__(32) mpc_controller_export_kernel(const DevModel* __restrict__ mdl, int b0, int nmax, MpcSolutionDev sol, const double* __restrict__ stage, const double* __restrict__ gains,
                                                                  const int32_t* __restrict__ status, int valid, double* __restrict__ bias, double* __restrict__ gain, int32_t* __restrict__ feedback) {
  const int r = blockIdx.x, k = blockIdx.y, lane = threadIdx.x; const int b = b0 + r;
  const int n = sol.n_nodes[b]; const bool fb = valid && !(status[b] & MST_NO_FEEDBACK);
  if (k == 0 && lane == 0) feedback[r] = fb ? 1 : 0;
  const int32_t* ge = sol.event + (size_t)b * nmax; const double* gx = sol.x + (size_t)b * nmax * NX; const double* gu = sol.u + (size_t)b * nmax * NU;
  double* bo = bias + ((size_t)r * nmax + k) * NU; double* go = gain + ((size_t)r * nmax + k) * NU * NX;
  const int s = (fb && k < n) ? controller_node(ge, n, k) : -1;
  if (s < 0) {
    for (int e = lane; e < NU * NX; e += 32) go[e] = 0.0;
    if (lane < NU) bo[lane] = (k < n) ? gu[(size_t)k * NU + lane] : 0.0;
    return;
  }
  if (lane > NX) return;
  const size_t node = (size_t)b * nmax + s; double dxv[NX], zero[NU], un[NU];
  for (int i = 0; i < NX; ++i) { dxv[i] = (lane < NX) ? (i == lane ? 1.0 : 0.0) : -gx[(size_t)s * NX + i]; zero[i] = 0.0; }
  rollout_input(stage + node * STAGE_DBL + ST_TAIL, gains + node * GAIN_DBL, lane < NX ? zero : gu + (size_t)s * NU, dxv, 0.0, pack_leg_foot(mdl), un);
  if (lane < NX) { for (int i = 0; i < NU; ++i) go[(size_t)i * NX + lane] = un[i]; }
  else { for (int i = 0; i < NU; ++i) bo[i] = un[i]; }
}

// =====================================================================================================
// Value function (createValueFunction of the sqp / ipm blocks): SqpSolver::getValueFunction(t, x) [upstream ocs2_sqp, recalled] - f = 0, dfdxx and dfdx of
// the stored records interpolated linearly on the node times (the (index, alpha) of mpc_policy_eval_kernel, clamped outside the horizon), then
// dfdx += dfdxx x.  One warp per robot: the two bracketing records (7.9 KB) are staged with coalesced loads and blended in place, so the dense dfdxx
// written out and the one multiplying x are the same numbers; lane r < 30 forms row r of dfdxx x.
constexpr int VF_WARPS = 4;
struct VfSmem { double v[2][VF_DBL]; double x[NX]; };
__global__ void __launch_bounds__(32 * VF_WARPS) mpc_value_function_kernel(int B, int nmax, MpcSolutionDev sol, const double* __restrict__ vf, const int32_t* __restrict__ status, int valid,
                                                                           const double* __restrict__ tq, const double* __restrict__ xq, double* __restrict__ dfdx, double* __restrict__ dfdxx,
                                                                           int32_t* __restrict__ valid_out) {
  __shared__ VfSmem s_vf[VF_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31; const int b = blockIdx.x * VF_WARPS + warp; if (b >= B) return;
  VfSmem& sm = s_vf[warp]; double* Po = dfdxx + (size_t)b * NX * NX; double* go = dfdx + (size_t)b * NX;
  const int n = sol.n_nodes[b]; const bool ok = valid && n >= 1 && !(status[b] & MST_NO_FEEDBACK);
  if (lane == 0) valid_out[b] = ok ? 1 : 0;
  if (!ok) { for (int e = lane; e < NX * NX; e += 32) Po[e] = 0.0; if (lane < NX) go[lane] = 0.0; return; }
  int idx; double a; time_segment(sol.t + (size_t)b * nmax, n, tq[b], idx, a); const int i2 = (idx + 1 < n) ? idx + 1 : idx;
  const double* r0 = vf + ((size_t)b * nmax + idx) * VF_DBL; const double* r1 = vf + ((size_t)b * nmax + i2) * VF_DBL;
  for (int e = lane; e < VF_P + NX; e += 32) { sm.v[0][e] = r0[e]; sm.v[1][e] = r1[e]; }
  if (lane < NX) sm.x[lane] = xq[(size_t)b * NX + lane];
  __syncwarp();
  for (int e = lane; e < VF_P + NX; e += 32) sm.v[0][e] = a * sm.v[0][e] + (1.0 - a) * sm.v[1][e];
  __syncwarp();
  const double* V = sm.v[0];
  for (int e = lane; e < NX * NX; e += 32) { const int r = e / NX, c = e - r * NX; Po[e] = (c <= r) ? V[(r * (r + 1) >> 1) + c] : V[(c * (c + 1) >> 1) + r]; }
  if (lane < NX) { double s = V[VF_P + lane];
    for (int c = 0; c < NX; ++c) s = fma((c <= lane) ? V[(lane * (lane + 1) >> 1) + c] : V[(c * (c + 1) >> 1) + lane], sm.x[c], s);
    go[lane] = s; }
}

// =====================================================================================================
bool mpc_alloc(MpcBuffers& m, int B, int nmax, std::string& err, std::vector<void*>& allocs, cudaStream_t stream) {
  m.B = B; m.nmax = nmax; m.cur = 0;
  if (SETUP_WARPS * ((setup_smem_per_warp(nmax) + 15) & ~(size_t)15) > 200 * 1024) { err = "max_nodes too large for the grid staging of the setup kernel (limit ~1000 nodes)"; return false; }
  auto A = [&](auto** p, size_t count) { void* q = nullptr; const size_t bytes = count * sizeof(**p); cudaError_t e = cudaMalloc(&q, bytes); if (e != cudaSuccess) { err = std::string("cudaMalloc (MPC buffers) failed: ") + cudaGetErrorString(e); return false; } cudaMemsetAsync(q, 0, bytes, stream); allocs.push_back(q); *p = static_cast<std::remove_reference_t<decltype(**p)>*>(q); return true; };
  const size_t Bn = (size_t)B * nmax;
  bool ok = A(&m.t0, B) && A(&m.x0, (size_t)B * NX) && A(&m.n_events, B) && A(&m.event_times, (size_t)B * EMAX) && A(&m.modes, (size_t)B * (EMAX + 1)) && A(&m.n_target, B) && A(&m.target_times, (size_t)B * KMAX) && A(&m.target_states, (size_t)B * KMAX * TARGET_DIM);
  for (int s = 0; s < 2 && ok; ++s) ok = A(&m.sol[s].n_nodes, B) && A(&m.sol[s].t, Bn) && A(&m.sol[s].event, Bn) && A(&m.sol[s].x, Bn * NX) && A(&m.sol[s].u, Bn * NU);
  ok = ok && A(&m.stage, Bn * STAGE_DBL) && A(&m.gains, Bn * GAIN_DBL) && A(&m.dx, Bn * NX) && A(&m.du, Bn * NU) && A(&m.node_rec, Bn * ne::NODE_REC_DBL) && A(&m.ddp_trial, (size_t)B * RO_MAXTRIALS * 2) && A(&m.robot, (size_t)B * ROBOT_DBL) && A(&m.status, B) && A(&m.step_info, (size_t)B * 4);
  return ok;
}

int mpc_configure_device() {
  cudaError_t e = cudaFuncSetAttribute(mpc_setup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);   // 48 B per node and warp: opt-in beyond nmax ~ 250
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpc_flow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FL_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpc_rollout_trials_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RO_RPC_MAX * GAIN_DBL * 8);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpc_lq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(LqSmem) * LQ_WARPS));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpc_riccati_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RicSmem));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mpc_riccati_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RicSmem));
  return (int)e;
}

int mpc_solve_launch(const DevModel* mdl, const DevModel& hm, MpcBuffers& m, const MpcProblemDev& p, int b0, int b1, cudaStream_t stream, cudaEvent_t* ev, bool value_fn) {
  const int nb = b1 - b0, nmax = m.nmax; if (nb <= 0) return 0;
  MpcSolutionDev prev = m.sol[m.cur], next = m.sol[1 - m.cur];   // the caller flips m.cur once all ranges are queued
  if (ev) cudaEventRecord(ev[0], stream);
  mpc_setup_kernel<<<(nb + SETUP_WARPS - 1) / SETUP_WARPS, 32 * SETUP_WARPS, SETUP_WARPS * ((setup_smem_per_warp(nmax) + 15) & ~(size_t)15), stream>>>(mdl, b0, b1, nmax, p, prev, next, m.status);
  if (ev) cudaEventRecord(ev[1], stream);
  const long long nodes = (long long)nb * nmax; const int iters = hm.sqp_iterations < 1 ? 1 : hm.sqp_iterations; int launched = 1;
  const bool ddp = hm.solver == 2; int n_trials = 0, tr_pitch = 1;
  if (ddp) { for (double a = hm.ddp_max_step; a >= hm.ddp_min_step && n_trials < RO_MAXTRIALS; a *= hm.ddp_contraction) ++n_trials; while (tr_pitch < n_trials) tr_pitch *= 2; }   // step lengths of ddp.lineSearch; lanes of a warp: trials of the same robot side by side
  const int ro_grid = (nb + RO_THREADS - 1) / RO_THREADS; const int ro_rpc = (RO_THREADS / tr_pitch < RO_RPC_MAX) ? RO_THREADS / tr_pitch : RO_RPC_MAX;   // robots per CTA of the trial kernel
  if (ddp) { mpc_rollout_kernel<<<ro_grid, RO_THREADS, 0, stream>>>(mdl, b0, b1, nmax, p, next, m.stage, m.gains, m.ddp_trial, m.robot, m.status, m.step_info, 0, 1, 1, 0); ++launched; }   // nominal rollout from the measured state
  // SqpSolver::runImpl: for (iter < sqpIteration) { LQ approximation; QP; line search; checkConvergence }.  Robots whose convergence test fired
  // carry MST_CONVERGED and skip the remaining iterations inside the kernels (the per-kernel events time the last iteration's launches).
  for (int it = 0; it < iters; ++it) {
    mpc_flow_kernel<<<(unsigned)((nodes + 32 * FL_WARPS - 1) / (32 * FL_WARPS)), 32 * FL_WARPS, FL_SMEM, stream>>>(mdl, b0, b1, nmax, p, next, m.node_rec, m.status);
    if (ev && it == iters - 1) cudaEventRecord(ev[7], stream);
    mpc_lq_kernel<<<(unsigned)((nodes + LQ_WARPS - 1) / LQ_WARPS), 32 * LQ_WARPS, sizeof(LqSmem) * LQ_WARPS, stream>>>(mdl, b0, b1, nmax, p, next, m.node_rec, m.stage, m.status);
    if (ev && it == iters - 1) cudaEventRecord(ev[2], stream);
    if (value_fn && m.vf) mpc_riccati_kernel<true><<<nb, RIC_THREADS, sizeof(RicSmem), stream>>>(mdl, b0, b1, nmax, p, next, m.stage, m.gains, m.dx, m.du, m.robot, m.status, m.vf);
    else mpc_riccati_kernel<false><<<nb, RIC_THREADS, sizeof(RicSmem), stream>>>(mdl, b0, b1, nmax, p, next, m.stage, m.gains, m.dx, m.du, m.robot, m.status, nullptr);
    if (ev && it == iters - 1) cudaEventRecord(ev[3], stream);
    if (ddp) { mpc_rollout_trials_kernel<<<(nb + ro_rpc - 1) / ro_rpc, ro_rpc * tr_pitch, (size_t)ro_rpc * GAIN_DBL * 8, stream>>>(mdl, b0, b1, nmax, p, next, m.stage, m.gains, m.ddp_trial, m.robot, m.status, n_trials, tr_pitch, ro_rpc);   // all step lengths side by side
      mpc_rollout_kernel<<<ro_grid, RO_THREADS, 0, stream>>>(mdl, b0, b1, nmax, p, next, m.stage, m.gains, m.ddp_trial, m.robot, m.status, m.step_info, 2, n_trials, tr_pitch, it); ++launched; }   // decision + in-place rollout of the accepted step
    else mpc_linesearch_kernel<<<nb, 32 * LS_WARPS, 0, stream>>>(mdl, b0, b1, nmax, p, next, m.dx, m.du, m.robot, m.status, m.step_info, it);
    launched += 4;
  }
  if (ev) cudaEventRecord(ev[4], stream);
  return launched;
}

int mpc_policy_eval_launch(const MpcBuffers& m, const double* t, double* x_des, double* u_des, int32_t* mode, cudaStream_t stream, int b0, int b1) {
  if (b1 < 0) b1 = m.B; if (b1 <= b0) return 0;
  mpc_policy_eval_kernel<<<(b1 - b0 + 3) / 4, 128, 0, stream>>>(b0, b1, m.nmax, m.sol[m.cur], m.n_events, m.event_times, m.modes, t, x_des, u_des, mode);
  return 1;
}
int mpc_policy_launch(const DevModel* mdl, const MpcBuffers& m, bool feedback, const double* t, const double* x, double* x_des, double* u_des, int32_t* mode, cudaStream_t stream, int b0, int b1) {
  if (!feedback) return mpc_policy_eval_launch(m, t, x_des, u_des, mode, stream, b0, b1);
  if (b1 < 0) b1 = m.B; if (b1 <= b0) return 0;
  mpc_policy_feedback_kernel<<<(b1 - b0 + PF_WARPS - 1) / PF_WARPS, 32 * PF_WARPS, 0, stream>>>(mdl, b0, b1, m.nmax, m.sol[m.cur], m.stage, m.gains, m.status, m.n_events, m.event_times, m.modes, t, x, x_des, u_des, mode);
  return 1;
}
int mpc_controller_export_launch(const DevModel* mdl, const MpcBuffers& m, bool valid, int b0, int count, double* bias, double* gain, int32_t* feedback, cudaStream_t stream) {
  if (count <= 0) return 0;
  mpc_controller_export_kernel<<<dim3(count, m.nmax), 32, 0, stream>>>(mdl, b0, m.nmax, m.sol[m.cur], m.stage, m.gains, m.status, valid ? 1 : 0, bias, gain, feedback);
  return 1;
}
int mpc_value_function_launch(const MpcBuffers& m, bool valid, const double* t, const double* x, double* dfdx, double* dfdxx, int32_t* valid_out, cudaStream_t stream) {
  mpc_value_function_kernel<<<(m.B + VF_WARPS - 1) / VF_WARPS, 32 * VF_WARPS, 0, stream>>>(m.B, m.nmax, m.sol[m.cur], m.vf, m.status, (valid && m.vf) ? 1 : 0, t, x, dfdx, dfdxx, valid_out);
  return 1;
}
int mpc_fixup_launch(const MpcBuffers& m, cudaStream_t stream) { mpc_fixup_kernel<<<m.B, 32, 0, stream>>>(m.B, m.nmax, m.sol[m.cur]); return 1; }

// ---- fp64 FMA throughput probe: 8 independent chains per thread, enough CTAs to fill every SM ----
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) { x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b); x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b); }
  if (x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7 == 12345.678) out[0] = x0;
}
double measure_fp64_peak(cudaStream_t stream) {
  double* d = nullptr; cudaMalloc(&d, 8); cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  int dev = 0, sms = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int blocks = sms * 8, iters = 1 << 15; double best = 0.0;
  fp64_peak_kernel<<<blocks, 256, 0, stream>>>(d, 1024, 0.999999, 1e-9);
  for (int rep = 0; rep < 3; ++rep) {
    cudaEventRecord(e0, stream); fp64_peak_kernel<<<blocks, 256, 0, stream>>>(d, iters, 0.999999, 1e-9); cudaEventRecord(e1, stream); cudaEventSynchronize(e1);
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1); const double tf = 2.0 * 8.0 * iters * 256.0 * blocks / (ms * 1e-3) / 1e12; if (tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d); return best;
}

}  // namespace qmb
