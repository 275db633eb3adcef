"""Cost of the value function (createValueFunction) on the bench workload: 8192 trot robots (BASELINE configs[4]: dt 0.01, horizon 1 s), warm-started ticks.

  tick            qmb200_tick_dev with the switch off and on, alternated in the same process (the difference is K3's stores of the records)
  k3              the Riccati kernel's time (ms6[2] of qmb200_get_kernel_times) with the switch off and on, alternated, per-kernel events on
  value_function  qmb200_value_function_dev for the whole batch after a solve, CUDA events over many calls

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
    from qm_control_b200 import synthetic
    if not torch.cuda.is_available():
        raise SystemExit("bench_value_function: no CUDA device")
    dev = torch.device("cuda:0"); info = gpu_info()
    s = q.Solver(batch=B, dt=DT, time_horizon=HORIZON); stream = s.stream
    prob, wbc = synthetic.make_batch(np.arange(B), config=CONFIG, horizon=HORIZON)
    pdev = {k: torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in KEYS}
    rbd = torch.from_numpy(np.ascontiguousarray(wbc["rbd"])).to(dev); per = torch.from_numpy(np.ascontiguousarray(wbc["period"])).to(dev)
    te = torch.from_numpy(prob["t0"] + 0.002).to(dev); cmd = torch.zeros((B, 54), dtype=torch.float64, device=dev); st = torch.zeros(B, dtype=torch.int32, device=dev)
    ext = torch.cuda.ExternalStream(stream)

    def ticks(n, collect=False):
        with torch.cuda.stream(ext):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(ext)
            for _ in range(n):
                s.tick_dev(pdev, te, rbd, per, cmd, st, stream=stream); pdev["t0"] += DT; te.add_(DT)
                if collect:
                    s.collect_kernel_times()
            e1.record(ext); e1.synchronize()
        return e0.elapsed_time(e1) / n

    s.mpc_set_value_function(True); ticks(a.ticks); s.mpc_set_value_function(False); ticks(a.ticks)   # warm-up: cold start, then warm-started ticks, both kernels
    res = {"off": [], "on": []}; k3 = {"off": [], "on": []}; launches = {}
    for r in range(a.repeats):
        for mode in ("off", "on") if r % 2 == 0 else ("on", "off"):
            s.mpc_set_value_function(mode == "on"); l0 = s.launch_count; res[mode].append(ticks(a.ticks)); launches[mode] = (s.launch_count - l0) / a.ticks
    for r in range(a.repeats):                                                      # per-kernel events in runs of their own (they serialise the tick)
        for mode in ("off", "on") if r % 2 == 0 else ("on", "off"):
            s.mpc_set_value_function(mode == "on"); s.set_profiling(True); ticks(a.ticks, collect=True); k3[mode].append(float(s.kernel_times()["riccati"])); s.set_profiling(False)
    # evaluation after the last (warm) solve with the switch on
    s.mpc_set_value_function(True); ticks(1)
    xq = pdev["x0"] + 0.001; g = torch.zeros((B, 30), dtype=torch.float64, device=dev); H = torch.zeros((B, 30, 30), dtype=torch.float64, device=dev)
    ok = torch.zeros(B, dtype=torch.int32, device=dev)

    def evaluate():
        with torch.cuda.stream(ext):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record(ext)
            for _ in range(a.calls):
                s.value_function_dev(te, xq, g, H, ok, stream=stream)
            e1.record(ext); e1.synchronize()
        return e0.elapsed_time(e1) / a.calls * 1e3

    evaluate(); ev = [evaluate() for _ in range(a.repeats)]
    stat = lambda v: dict(mean=float(np.mean(v)), min=float(np.min(v)), max=float(np.max(v)), samples=[float(x) for x in v])
    record_bytes = B * s.nmax * 496 * 8
    out = dict(gpu=info, workload=dict(batch=B, dt=DT, horizon=HORIZON, config=CONFIG, nmax=s.nmax, ticks_per_sample=a.ticks, repeats=a.repeats, calls=a.calls),
               tick_ms=dict(off=stat(res["off"]), on=stat(res["on"]), launches_per_tick=launches),
               k3_ms=dict(off=stat(k3["off"]), on=stat(k3["on"])),
               value_function_us=stat(ev), robots_valid=int(ok.sum().item()),
               bytes_allocated=dict(records=int(record_bytes), host_call_staging=int(B * (30 + 900) * 8 + B * 4)))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "tick_ms", "k3_ms", "value_function_us", "robots_valid")}, default=str)[:3000])


if __name__ == "__main__":
    main()
