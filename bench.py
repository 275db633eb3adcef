#!/usr/bin/env python3
"""bench.py — MPC+WBC iterations/s of the batched solver on B200 (BASELINE.json metric).

One "step" = one controller tick for every robot of the batch: MPC solve (one multiple-shooting SQP iteration over the
horizon: LQ approximation + projection + Riccati + filter line search), policy evaluation, WBC update (3-level HoQp) →
54-vector; with N>1 GPUs one all-gather of the torque buffer.  Workload = BASELINE.json configs[3] shape on ONE GPU:
trot gait schedule, horizon 1.0 s / dt 0.01 (100 intervals + event nodes), batch 8192 robots PER GPU (weak scaling),
synthetic 24-DoF states (SURVEY §8d), fp64.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference] [--dump-outputs DIR]

`value`   device-resident: inputs already in HBM, CUDA events on the launch stream, max over ranks.
`e2e`     the same tick through the C-ABI host call qmb200_tick with pinned HOST buffers (H2D of the observation,
          schedule and targets, D2H of the 54-vector inside the timed region).
`--impl reference` times the CPU restatement of the reference path (oracle/, all host threads) on a bounded sample.
`--dump-outputs DIR` writes what the last timed step returned as DIR/<name>.npy (see dump_outputs).  The inputs are seeded
          per robot, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PIPELINE_CHUNKS = 1         # qmb200_set_pipeline: measured neutral on B200 (grids drain in launch order), so the bench runs one chain
UNIT_BATCH = 8192           # one "iteration" of the metric = one tick of an 8192-robot batch
DT, HORIZON, CONFIG = 0.01, 1.0, 4
METRIC = "mpc_wbc_iters_per_s"
UNIT = "iter/s (one iter = MPC+WBC tick of an 8192-robot batch, horizon 100)"


def algorithmic_bytes(n_intervals):
    """Per robot-iteration (SURVEY §8d): warm start + solution, feedback hand-off, observation/targets/WBC I/O; split per kernel (DESIGN.md §roofline)."""
    N = n_intervals
    return dict(lq=8 * (60 * N + 30) + 1352, riccati=2 * 8 * N * (30 * 30 + 30) + 8 * (60 * N + 30), linesearch=3 * 8 * (60 * N + 30), wbc=1856, setup=8 * (60 * N + 30) + 496, policy_eval=480,
                total=15840 * N + 4184)


def riccati_counted():
    """COUNTED tensor-core work of the backward sweep: ncu sm__inst_executed_pipe_tensor_subpipe_dmma.sum of one capture at 1024 robots x 100 regular nodes, and the
    tensor sub-pipe activity of the same capture (profiles/r03_riccati_dmma.json, written by tools/dmma_json.py from the ncu csv; round 2: 606 DMMA per node, 37.9 %)."""
    path = os.path.join(ROOT, "profiles", "r03_riccati_dmma.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except Exception:
            pass
    return {"dmma_per_node": 606.0, "tensor_pipe_active_pct": 37.88, "source": "profiles/r02c_riccati_dmma.csv"}


def riccati_flops(n_intervals):
    """DMMA.8x8x4 warp instructions per node x 512 flop.  The scalar work (Cholesky, substitutions, rollout) is not counted."""
    return riccati_counted()["dmma_per_node"] * 512.0 * n_intervals


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True); self.index = index; self.rows = []; self.stop_flag = False; self.proc = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        try:
            if self.proc:
                self.proc.terminate()
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def usable_cores():
    """Host threads this process may really use: scheduler affinity capped by the cgroup CPU quota (os.cpu_count() ignores both - round 1's CPU arm ran
    128 threads on whatever share of the box the container had, and its value moved 5x between two boxes)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0]); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    quota = q / per
            break
        except Exception:
            continue
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n, {"affinity": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None, "os_cpu_count": os.cpu_count(), "cgroup_quota_cpus": quota}


CPU_SAMPLE = 256            # robots of the bounded CPU sample (BASELINE.md section 2: >= 256)
REF_DESIGN_POINT = "reference design point (config, not a measurement): <= 10 ms per MPC iteration on 3 solver threads at 100 Hz, N ~ 67 (task.info:77,146)"


def cpu_ticks(o, prob, wbc, nmax, cores, ticks, warm):
    """`warm` untimed + `ticks` timed warm-started controller ticks of the whole sample on `cores` threads; returns seconds per timed tick (list)."""
    n = prob["t0"].shape[0]; prev = None; il = np.zeros((n, 30)); out = []; prob = dict(prob)
    for s in range(warm + ticks):
        t = time.perf_counter()
        prev = o.tick_batch(prob, nmax, prob["t0"] + 0.002, wbc["rbd"], wbc["period"], il if prev is None else prev["input_last"], prev=prev, nthreads=cores)
        el = time.perf_counter() - t; prob = dict(prob); prob["t0"] = prob["t0"] + DT
        if s >= warm:
            out.append(el)
    return out


def cpu_measure(cores, ticks, warm, n=CPU_SAMPLE):
    """CPU restatement of the reference path (oracle/), one robot per task on a std::thread pool over the usable host cores: bounded sample of the
    bench workload, measured TWICE (spread reported), plus the single-thread cost of one robot-tick."""
    from qm_control_b200 import synthetic
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _oracle import Oracle
    nmax = int(round(HORIZON / DT)) + 21
    prob, wbc = synthetic.make_batch(np.arange(n), config=CONFIG, horizon=HORIZON); wbc = {k: v[:n] for k, v in wbc.items()}
    o = Oracle(); o.mpc_set(dt=DT, horizon=HORIZON)
    runs = [cpu_ticks(o, prob, wbc, nmax, cores, ticks, warm) for _ in range(2)]
    per_run = [float(np.mean(r)) for r in runs]; sec = float(np.mean(per_run)); spread = abs(per_run[0] - per_run[1]) / sec
    one = {k: v[:4] for k, v in prob.items()}; w1 = {k: v[:4] for k, v in wbc.items()}
    t1 = cpu_ticks(o, one, w1, nmax, 1, 1, 1)[0] / 4.0           # one thread, 4 robots back to back, warm-started tick
    value = (n / UNIT_BATCH) / sec
    info = {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_step": sec * 1e3,
            "sample": "%d robots per step (bounded sample of the 8192-robot batch: value = sample/8192 per measured second), trot, N=100, warm-started ticks, %d host threads, 2 runs x %d ticks" % (n, cores, ticks),
            "runs_ms_per_step": [p * 1e3 for p in per_run], "run_to_run_spread": spread, "single_thread_ms_per_robot_tick": t1 * 1e3,
            "parallel_efficiency": (t1 * n / cores) / sec, "context": REF_DESIGN_POINT,
            "note": "CPU restatement of the reference path (oracle/, forward-mode-AD Jacobians, literal HoQp): the reference's OCS2 + Pinocchio + qpOASES stack cannot be built offline; a reported baseline, not the optimisation target"}
    return info


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores, how = usable_cores()
    info = cpu_measure(cores, ticks=max(1, args.steps), warm=max(1, min(args.warmup, 1)))
    info["core_count_source"] = how
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": info["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": info["ms_per_step"],
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": "MPC+WBC tick, trot gait, horizon 1.0 s / dt 0.01, CPU restatement of the reference path (OCS2/Pinocchio/qpOASES cannot be built offline)", "same_config_as_b200_arm": "same workload, bounded sample of %d of its 8192 robots per step" % CPU_SAMPLE},
                      "cpu_baseline": info, "e2e": {"value": info["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


DUMP_LIMIT = 64 << 20      # bytes --dump-outputs may write in all


def dump_outputs(path, arrays):
    """Each array as <path>/<name>.npy in float64 (int32 status words convert exactly).  When they would exceed DUMP_LIMIT, every array keeps the same
    fraction of its rows (robots), drawn with a fixed seed so that equal row counts keep equal rows, and <name>_rows.npy lists the rows kept."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        frac = (DUMP_LIMIT - 4096) / (total + 8 * sum(a.shape[0] for a in arrays.values()))   # the row lists and .npy headers count too
        for k in list(arrays):
            n = arrays[k].shape[0]; rows = np.sort(np.random.default_rng(0).choice(n, max(1, int(n * frac)), replace=False))
            arrays[k] = arrays[k][rows]; arrays[k + "_rows"] = rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


KEYS = ("t0", "x0", "n_events", "event_times", "modes", "n_target", "target_times", "target_states")
ST_NAMES = {1: "iter_cap", 2: "overflow", 4: "nan", 8: "not_pd", 16: "no_step", 32: "converged", 64: "neg_dt"}


class TickLoop:
    """One handle + device-resident inputs for `batch` robots of a synthetic config; step() = one MPC+WBC tick (+ the all-gather of the torque rows when world > 1),
    everything issued through the C-ABI on one CUDA stream."""

    def __init__(self, q, torch, dev, local, stream, batch, ids, config, world, rank, chunks=1, binned=False):
        from qm_control_b200 import parallel, synthetic
        self.torch = torch; self.world = world; self.B = batch; self.stream = stream
        self.solver = q.Solver(batch=batch, device=local, dt=DT, time_horizon=HORIZON); self.solver.set_pipeline(chunks)
        parallel.init_comm(self.solver, rank, world)
        prob, wbc = synthetic.make_batch(ids, config=config, horizon=HORIZON)
        self.perm_d = None
        if binned:   # gait-binned submission order (SURVEY 8e): the gathered torque buffer is un-permuted by the pack kernel
            perm = self.solver.gait_bin_permutation(prob); prob = {k: v[perm] for k, v in prob.items()}; wbc = {k: v[perm] for k, v in wbc.items()}
            self.perm_d = torch.from_numpy(perm).to(dev)
        self.prob, self.wbc = prob, wbc
        self.pdev = {k: torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in KEYS}
        self.rbd_d = torch.from_numpy(np.ascontiguousarray(wbc["rbd"])).to(dev); self.per_d = torch.from_numpy(np.ascontiguousarray(wbc["period"])).to(dev)
        self.te_d = torch.from_numpy(prob["t0"] + 0.002).to(dev)
        self.cmd_d = torch.zeros((batch, 54), dtype=torch.float64, device=dev); self.st_d = torch.zeros(batch, dtype=torch.int32, device=dev)
        self.all_d = torch.zeros((batch * world, 18), dtype=torch.float64, device=dev)
        self.ev = None

    def step(self, time_gather=False):
        s = self.solver
        s.tick_dev(self.pdev, self.te_d, self.rbd_d, self.per_d, self.cmd_d, self.st_d, stream=self.stream)
        if self.world > 1 or self.perm_d is not None:
            if time_gather:
                a = self.torch.cuda.Event(enable_timing=True); b = self.torch.cuda.Event(enable_timing=True); a.record()
            s.allgather_torque(self.cmd_d, self.all_d, self.perm_d, stream=self.stream)
            if time_gather:
                b.record(); self.ev = (a, b)
        self.pdev["t0"] += DT; self.te_d.add_(DT)   # the observation time advances one MPC period per tick

    def timed(self, steps, warmup, dev, dist=None):
        torch = self.torch
        for _ in range(warmup):
            self.step()
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        l0 = self.solver.launch_count; e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev); e0.record()
        for i in range(steps):
            self.step(time_gather=(i == steps - 1))
        e1.record(); torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        ag = self.ev[0].elapsed_time(self.ev[1]) if self.ev else 0.0
        return e0.elapsed_time(e1) / steps, self.solver.launch_count - l0, ag

    def outputs(self):
        """What the last step handed its caller: the 54-vector and status word per robot, and the gathered torque rows when step() gathers them."""
        out = {"cmd": self.cmd_d.cpu().numpy(), "status": self.st_d.cpu().numpy()}
        if self.world > 1 or self.perm_d is not None:
            out["torque_all"] = self.all_d.cpu().numpy()
        return out

    def flagged(self):
        st = self.st_d.cpu().numpy(); mpc = (st >> 8) & 0xFF; wbcs = st & 0xFF; out = {}
        for bit, name in ST_NAMES.items():
            if name in ("no_step", "converged"):
                continue
            n = int(np.count_nonzero(mpc & bit)); m = int(np.count_nonzero(wbcs & bit)) if bit <= 4 else 0
            if n:
                out["mpc_" + name] = n
            if m:
                out["wbc_" + name] = m
        return out


def side_workload(args, q, torch, dev, local, stream):
    """Bench lines of BASELINE configs[1] (MPC only, B = 1024, stance), configs[2] (WBC only, B = 4096, L2 flushed between launches) and configs[4]'s per-GPU
    share (mixed gaits, B = 2048) on one GPU.  Same JSON contract as the main line, value in robot-iterations of THAT workload per second."""
    from qm_control_b200 import synthetic
    peaks, peak_src = measured_peaks(); n_int = int(round(HORIZON / DT)); W = args.workload
    if W == "mixed":
        B = args.batch if args.batch != UNIT_BATCH else 2048; loop = TickLoop(q, torch, dev, local, stream, B, np.arange(3 * B, 4 * B), 5, 1, 0)
        ms, launches, _ = loop.timed(args.steps, args.warmup, dev); ab = algorithmic_bytes(n_int)["total"]; outputs = loop.outputs
        out = {"workload": "configs[4] per-GPU share: mixed stance / trot / flying-trot batch, full MPC+WBC tick", "batch": B, "flagged": loop.flagged()}
    elif W == "mpc":
        B = args.batch if args.batch != UNIT_BATCH else 1024; solver = q.Solver(batch=B, device=local, dt=DT, time_horizon=HORIZON)
        prob, _ = synthetic.make_batch(np.arange(B), config=2, horizon=HORIZON); pdev = {k: torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in KEYS}
        def step():
            solver.mpc_solve_dev(pdev, stream=stream); pdev["t0"] += DT
        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize(dev); l0 = solver.launch_count; e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record()
        for _ in range(args.steps):
            step()
        e1.record(); torch.cuda.synchronize(dev); ms = e0.elapsed_time(e1) / args.steps; launches = solver.launch_count - l0; ab = 15840 * n_int + 2328; outputs = solver.mpc_get_solution
        out = {"workload": "configs[1]: batched MPC only (one SQP iteration), state 30 / input 30, horizon 100, stance", "batch": B, "l2": "stage buffer %.1f GB >> 126 MB L2" % (B * solver.nmax * 1484 * 8 / 1e9)}
    else:
        B = args.batch if args.batch != UNIT_BATCH else 4096; solver = q.Solver(batch=B, device=local)
        prob, wbc = synthetic.make_batch(np.arange(B), config=3); x_des, u_des, mode = synthetic.nominal_wbc_inputs(prob, solver.robot_mass)
        u_des = u_des + synthetic.uniform(77, np.arange(B), 1, 30, -1.0, 1.0) * np.r_[np.full(12, 5.0), np.full(18, 0.2)]
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        xd, ud, rb, md, pe, tm = t(x_des), t(u_des), t(wbc["rbd"]), t(mode.astype(np.int32)), t(wbc["period"]), t(np.full(B, 12.0)); cmd = torch.zeros((B, 54), dtype=torch.float64, device=dev); st = torch.zeros(B, dtype=torch.int32, device=dev)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev); pairs = []
        for i in range(args.warmup + args.steps):
            flush.fill_(i & 0xFF)                                           # write 256 MB: nothing of the previous launch survives in the 126 MB L2
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True); a.record()
            solver.wbc_update_dev(xd, ud, rb, md, pe, tm, cmd, st, stream=stream); b.record()
            if i >= args.warmup:
                pairs.append((a, b))
        torch.cuda.synchronize(dev); ms = float(np.mean([a.elapsed_time(b) for a, b in pairs])); launches = args.steps; ab = 1856
        outputs = lambda: {"cmd": cmd.cpu().numpy(), "status": st.cpu().numpy()}
        out = {"workload": "configs[2]: batched WBC only (3-level HoQp, 36 decision variables, 54 outputs), stance", "batch": B, "l2": "256 MB written between launches (L2 flush), timed per launch with CUDA events", "flagged_robots": int(np.count_nonzero(st.cpu().numpy()))}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs())
    ach = ab * B / (ms * 1e-3) / 1e9
    print(json.dumps({"metric": "robot_iters_per_s", "value": B / (ms * 1e-3), "unit": "robot-iterations/s of the named workload", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": out, "gpu_launches": int(launches),
                      "roofline": {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None, "algorithmic_bytes_per_robot": ab, "peak_source": peak_src,
                                   "note": "latency / fp64-issue bound path (DESIGN.md section 4); the HBM fraction is what BASELINE.json asks for"}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1); ap.add_argument("--steps", type=int, default=10); ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=UNIT_BATCH); ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="tick", choices=["tick", "mpc", "wbc", "mixed"], help="tick = the BASELINE metric (default); mpc / wbc / mixed = configs[1] / [2] / [4] side lines on one GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true"); ap.add_argument("--no-e2e", action="store_true"); ap.add_argument("--no-extras", action="store_true", help="skip the strong-scaling and configs[4] records")
    ap.add_argument("--solver", default="sqp", choices=["sqp", "ipm", "ddp"], help="MPC solver variant (qmb200_mpc_set_solver); the BASELINE metric is quoted on sqp, the controller's solver")
    ap.add_argument("--chunks", type=int, default=PIPELINE_CHUNKS, help="robot ranges run as concurrent stream chains inside one tick")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world); return
    import torch
    import qm_control_b200 as q
    from qm_control_b200 import parallel
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    rank, world, local = parallel.init_distributed()
    torch.cuda.set_device(local); dev = torch.device("cuda", local)
    side = torch.cuda.Stream(dev); torch.cuda.set_stream(side)   # a non-default stream: its handle is what the C-ABI launches on, and torch events bracket it
    stream = side.cuda_stream; dist = torch.distributed if world > 1 else None
    if args.workload != "tick":
        if rank == 0:
            side_workload(args, q, torch, dev, local, stream)
        return
    B = args.batch; n_int = int(round(HORIZON / DT))
    loop = TickLoop(q, torch, dev, local, stream, B, np.arange(rank * B, (rank + 1) * B), CONFIG, world, rank, chunks=args.chunks); solver = loop.solver
    if args.solver != "sqp":
        solver.mpc_set_solver(args.solver)
    for _ in range(args.warmup):
        loop.step()
    sampler = ClockSampler(local); sampler.start(); time.sleep(0.15)
    ms_local, launches, ag_ms = loop.timed(args.steps, 0, dev, dist)
    clocks = sampler.finish()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loop.outputs())
    ms = parallel.max_over_ranks(ms_local, dev); ag_ms = parallel.max_over_ranks(ag_ms, dev)
    value = (B * world / UNIT_BATCH) / (ms * 1e-3)
    flagged = loop.flagged()

    # per-kernel device times (separate profiled ticks; CUDA events inside the library on the same stream)
    ktimes = {}
    try:
        solver.set_profiling(True)
        for _ in range(3):
            loop.step(); torch.cuda.synchronize(dev); solver.collect_kernel_times()
        ktimes = solver.kernel_times(); solver.set_profiling(False)
    except Exception as e:   # measurement support only
        ktimes = {"error": str(e)}
    peaks, peak_src = measured_peaks(); ab = algorithmic_bytes(n_int)
    roof = None
    if ktimes and "error" not in ktimes:
        dom = max(("lq", "riccati", "linesearch", "wbc"), key=lambda k: ktimes[k])
        achieved = ab[dom] * B / (ktimes[dom] * 1e-3) / 1e9
        fp64_peak = None
        try:
            fp64_peak = solver.measure_fp64_peak()
        except Exception:
            pass
        # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture per kernel (profiles/traffic_r02.json, bytes per robot at the
        # captured batch; every kernel's traffic is linear in the batch), scaled to this launch
        per_kernel = {}; tj = {}
        for name in ("traffic_r03.json", "traffic_r02.json", "traffic_r01.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath):
                try:
                    tj = json.load(open(tpath)); tj["_file"] = name; break
                except Exception:
                    tj = {}
        for kname in ("lq", "riccati", "linesearch", "wbc"):
            tr = tj.get(kname, {}).get("dram_bytes_per_robot")
            per_kernel[kname] = {"ms": ktimes[kname], "algorithmic_GBps": ab[kname] * B / (ktimes[kname] * 1e-3) / 1e9, "traffic_bytes_per_launch": (tr * B) if tr else None,
                                 "dram_GBps": (tr * B / (ktimes[kname] * 1e-3) / 1e9) if tr else None}
        roof = {"bound": "hbm", "kernel": "mpc_%s_kernel" % dom if dom != "wbc" else "wbc_update_kernel", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                "traffic": per_kernel[dom]["traffic_bytes_per_launch"], "traffic_source": tj.get("_file"),
                "peak_source": peak_src, "kernel_ms": ktimes, "per_kernel": per_kernel, "algorithmic_bytes_per_robot": ab[dom],
                "whole_tick": {"achieved": ab["total"] * B / (ms_local * 1e-3) / 1e9, "frac": ab["total"] * B / (ms_local * 1e-3) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes_per_robot": ab["total"]},
                "fp64": {"kernel": "mpc_riccati_kernel", "achieved_tflops": riccati_flops(n_int) * B / (ktimes["riccati"] * 1e-3) / 1e12 if ktimes.get("riccati") else None, "peak_tflops": fp64_peak, "peak_source": "measured in-process (FMA microbenchmark)",
                         "frac": (riccati_flops(n_int) * B / (ktimes["riccati"] * 1e-3) / 1e12 / fp64_peak) if (fp64_peak and ktimes.get("riccati")) else None,
                         "flops_source": "counted: ncu DMMA instruction count x 512 (%s); tensor (DMMA) sub-pipe activity of the same capture" % riccati_counted().get("source"), "tensor_pipe_active_pct": riccati_counted().get("tensor_pipe_active_pct"), "dmma_per_node": riccati_counted().get("dmma_per_node"),
                         "note": "the path is fp64 latency/issue bound, not HBM bound (SURVEY 8d: ~48 FLOP/B against a ~6 FLOP/B fp64 ridge); the Riccati products run on the fp64 tensor cores (DMMA.8x8x4, same 37 TFLOP/s peak as the DFMA pipe, tools/microbench/dmma_peak.cu); the HBM fraction is reported because BASELINE.json asks for it"}}

    # strong scaling as BASELINE.json states configs[3] / [4]: the TOTAL batch is fixed and split over the ranks
    extras = {}
    if not args.no_extras:
        try:
            Bs = UNIT_BATCH // world; sl = TickLoop(q, torch, dev, local, stream, Bs, np.arange(rank * Bs, (rank + 1) * Bs), CONFIG, world, rank) if world > 1 else None
            if sl is not None:
                sm_, _, sag = sl.timed(max(3, args.steps // 2), 2, dev, dist); sm_ = parallel.max_over_ranks(sm_, dev); sag = parallel.max_over_ranks(sag, dev)
                extras["strong_config3"] = {"global_batch": UNIT_BATCH, "batch_per_gpu": Bs, "ms_per_step": sm_, "value": 1.0 / (sm_ * 1e-3), "unit": UNIT, "allgather_ms": sag,
                                            "waves": {"riccati_ctas_per_sm_slot": Bs / (148 * 4.0), "wbc_ctas_per_sm": -(-Bs // 8) / 148.0}}
                del sl
            else:
                extras["strong_config3"] = {"global_batch": UNIT_BATCH, "batch_per_gpu": UNIT_BATCH, "ms_per_step": ms, "value": value, "unit": UNIT, "allgather_ms": ag_ms, "note": "one GPU: identical to the main line"} if B == UNIT_BATCH else None
            B5 = 2 * UNIT_BATCH // world; rec = {}
            for binned in (False, True):
                ml = TickLoop(q, torch, dev, local, stream, B5, np.arange(rank * B5, (rank + 1) * B5), 5, world, rank, binned=binned)
                m5, _, a5 = ml.timed(max(3, args.steps // 2), 2, dev, dist); m5 = parallel.max_over_ranks(m5, dev)
                rec["gait_binned" if binned else "submission_order"] = {"ms_per_step": m5, "value": 2.0 / (m5 * 1e-3), "allgather_ms": parallel.max_over_ranks(a5, dev), "flagged": ml.flagged()}
                del ml; torch.cuda.empty_cache()
            rec.update({"global_batch": 2 * UNIT_BATCH, "batch_per_gpu": B5, "unit": UNIT, "workload": "configs[4]: mixed stance / trot / flying-trot batch, 16384 robots in total",
                        "note": "no warp ever holds two robots (K3: CTA per robot; WBC / K2: warp per robot / node), so gait binning removes no divergence; what it evens out is the per-CTA tail (robots of one contact phase cost the same): ~3 % on B200"})
            extras["config5_mixed"] = rec
        except Exception as e:   # the extra records must never take the main line down
            extras["error"] = repr(e)

    # end-to-end through the host C-ABI call with pinned host buffers
    e2e = None
    if not args.no_e2e:
        solver.mpc_reset(); solver.wbc_set_input_last(None); prob, wbc = loop.prob, loop.wbc
        pin = {k: torch.from_numpy(np.ascontiguousarray(prob[k])).pin_memory() for k in KEYS}
        hp = {k: v.numpy() for k, v in pin.items()}
        te_h = torch.from_numpy((prob["t0"] + 0.002).copy()).pin_memory().numpy(); rbd_h = torch.from_numpy(wbc["rbd"]).pin_memory().numpy(); per_h = torch.from_numpy(wbc["period"]).pin_memory().numpy()
        h2d = sum(v.nbytes for v in hp.values()) + te_h.nbytes + rbd_h.nbytes + per_h.nbytes; d2h = B * 54 * 8 + B * 4
        for s in range(args.warmup):
            solver.tick(hp, te_h, rbd_h, per_h); hp["t0"] += DT; te_h += DT
        if world > 1:
            torch.distributed.barrier()
        t = time.perf_counter()
        for s in range(args.steps):
            cmd_h, st_h = solver.tick(hp, te_h, rbd_h, per_h); hp["t0"] += DT; te_h += DT
            if world > 1:
                loop.cmd_d.copy_(torch.from_numpy(cmd_h)); solver.allgather_torque(loop.cmd_d, loop.all_d, None, stream=stream); torch.cuda.synchronize(dev)
        el = (time.perf_counter() - t) / args.steps
        el = parallel.max_over_ranks(el, dev)
        e2e = {"value": (B * world / UNIT_BATCH) / el, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": el * 1e3}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cores, how = usable_cores(); cpu = cpu_measure(cores, ticks=2, warm=1); cpu["core_count_source"] = how
        except Exception as e:
            cpu = {"error": str(e)}
    if rank == 0:
        nr, _, nccl_v = solver.comm_info()
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": {"workload": "full MPC+WBC tick (BASELINE configs[3] shape): trot gait schedule, horizon 1.0 s / dt 0.01 (100 intervals + event nodes), 24-DoF quadruped-manipulator, one SQP iteration + 3-level HoQp",
                          "batch_per_gpu": B, "mpc_solver": args.solver, "pipeline_chunks": args.chunks, "global_batch": B * world, "robot_ticks_per_s": B * world / (ms * 1e-3),
                          "parallelism": "dp%d (robots sharded, one NCCL all-gather of the torque rows per tick issued by the C++ host: qmb200_allgather_torque)" % world, "allgather_ms": ag_ms, "nccl_version": nccl_v,
                          "l2": "per-tick working set (LQ stage buffer %.1f GB) >> 126 MB L2; no flush needed" % (B * solver.nmax * 1484 * 8 / 1e9),
                          "robots_flagged": flagged, "robots_flagged_note": "mpc_neg_dt / mpc_not_pd: synthetic robot 1758's schedule puts an event 0.68 us after a grid node, which gives the interval a NEGATIVE duration in upstream's own time discretisation (weakEpsilon shift > gap > dt_min): a non-convex QP every exact solver rejects; root-caused in tests/test_neg_interval_cpu.py"},
               "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e}
        out.update(extras)
        print(json.dumps(out))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
