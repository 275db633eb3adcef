"""Cost of the feedback policy (useFeedbackPolicy) on the bench workload: 8192 trot robots (BASELINE configs[4]: dt 0.01, horizon 1 s), warm-started ticks.

  tick            qmb200_tick_dev with the switch off and on, alternated in the same process (the solve is the same code, so the difference is the policy kernel)
  policy          qmb200_policy_eval_dev vs qmb200_policy_eval_state_dev (switch on) after a solve, CUDA events over many calls
  export          qmb200_mpc_get_controller_dev for 1024 robots (dense bias + 30x30 gains of every node)

Writes one JSON file (--out) with the card name, power limit and clocks read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DT, HORIZON, CONFIG, B = 0.01, 1.0, 4, 8192
KEYS = ("t0", "x0", "n_events", "event_times", "modes", "n_target", "target_times", "target_states")


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    return dict(zip(q.split(","), [v.strip() for v in out[0].split(",")])) if out else {}


def main():
    ap = argparse.ArgumentParser(); ap.add_argument("--out", required=True); ap.add_argument("--ticks", type=int, default=20); ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--calls", type=int, default=200); a = ap.parse_args()
    import torch
    import qm_control_b200 as q
    from qm_control_b200 import interface as qi, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("bench_feedback_policy: no CUDA device")
    dev = torch.device("cuda:0"); info = gpu_info()
    s = q.Solver(batch=B, dt=DT, time_horizon=HORIZON); stream = s.stream
    prob, wbc = synthetic.make_batch(np.arange(B), config=CONFIG, horizon=HORIZON)
    pdev = {k: torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in KEYS}
    rbd = torch.from_numpy(np.ascontiguousarray(wbc["rbd"])).to(dev); per = torch.from_numpy(np.ascontiguousarray(wbc["period"])).to(dev)
    te = torch.from_numpy(prob["t0"] + 0.002).to(dev); cmd = torch.zeros((B, 54), dtype=torch.float64, device=dev); st = torch.zeros(B, dtype=torch.int32, device=dev)
    ext = torch.cuda.ExternalStream(stream)

    def ticks(n):
        with torch.cuda.stream(ext):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(ext)
            for _ in range(n):
                s.tick_dev(pdev, te, rbd, per, cmd, st, stream=stream); pdev["t0"] += DT; te.add_(DT)
            e1.record(ext); e1.synchronize()
        return e0.elapsed_time(e1) / n

    ticks(a.ticks)                                                                  # warm-up: cold start, then warm-started ticks
    res = {"off": [], "on": []}; launches = {}
    for r in range(a.repeats):
        for mode in ("off", "on") if r % 2 == 0 else ("on", "off"):
            s.mpc_set_feedback_policy(mode == "on"); l0 = s.launch_count; res[mode].append(ticks(a.ticks)); launches[mode] = (s.launch_count - l0) / a.ticks
    # policy evaluation after the last (warm) solve
    s.mpc_set_feedback_policy(True)
    xq = pdev["x0"] + 0.001; xd = torch.zeros((B, 30), dtype=torch.float64, device=dev); ud = torch.zeros_like(xd); md = torch.zeros(B, dtype=torch.int32, device=dev)

    def policy(state):
        with torch.cuda.stream(ext):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(ext)
            for _ in range(a.calls):
                if state:
                    s.policy_eval_state_dev(te, xq, xd, ud, md, stream=stream)
                else:
                    s.lib.qmb200_policy_eval_dev(s.h, qi._p(te), qi._p(xd), qi._p(ud), qi._p(md), qi.C.c_void_p(stream))
            e1.record(ext); e1.synchronize()
        return e0.elapsed_time(e1) / a.calls * 1e3

    policy(False); policy(True); pol = {"policy_eval": [], "policy_eval_state": []}
    for r in range(a.repeats):
        pol["policy_eval"].append(policy(False)); pol["policy_eval_state"].append(policy(True))
    fb = s.mpc_get_controller()["feedback"]
    # dense export of 1024 robots
    R = 1024; bias = torch.zeros((R, s.nmax, 30), dtype=torch.float64, device=dev); gain = torch.zeros((R, s.nmax, 30, 30), dtype=torch.float64, device=dev); flag = torch.zeros(R, dtype=torch.int32, device=dev)
    exp = []
    for r in range(a.repeats + 1):
        with torch.cuda.stream(ext):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(ext)
            s.mpc_get_controller_dev(0, R, bias, gain, flag, stream=stream); e1.record(ext); e1.synchronize()
        exp.append(e0.elapsed_time(e1))
    stat = lambda v: dict(mean=float(np.mean(v)), min=float(np.min(v)), max=float(np.max(v)), samples=[float(x) for x in v])
    out = dict(gpu=info, workload=dict(batch=B, dt=DT, horizon=HORIZON, config=CONFIG, nmax=s.nmax, ticks_per_sample=a.ticks, repeats=a.repeats, policy_calls=a.calls),
               tick_ms=dict(off=stat(res["off"]), on=stat(res["on"]), launches_per_tick=launches),
               policy_us=dict(policy_eval=stat(pol["policy_eval"]), policy_eval_state=stat(pol["policy_eval_state"])),
               robots_with_feedback=int(fb.sum()), export_1024_robots_ms=stat(exp[1:]),
               export_bytes=int(R * s.nmax * 30 * 31 * 8))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "tick_ms", "policy_us", "export_1024_robots_ms", "robots_with_feedback")}, default=str)[:3000])


if __name__ == "__main__":
    main()
