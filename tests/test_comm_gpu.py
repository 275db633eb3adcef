"""The multi-GPU data path of the C-ABI (include/qmb200.h: qmb200_comm_*, qmb200_allgather_torque, qmb200_gait_bin_permutation).
One GPU: pack + un-permute; two GPUs (skipped on a one-GPU box): the real NCCL all-gather issued by the C++ host, each rank a process (torchrun-style env)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_gait_binning_and_unpermuted_gather_on_one_gpu():
    import torch
    import qm_control_b200 as q
    from qm_control_b200 import synthetic
    B = 96; dev = torch.device("cuda", 0); s = q.Solver(batch=B, dt=0.015); prob, wbc = synthetic.make_batch(np.arange(B), config=5)
    perm = s.gait_bin_permutation(prob); assert sorted(perm.tolist()) == list(range(B))
    ne = prob["n_events"]; mode0 = np.array([prob["modes"][b, np.searchsorted(prob["event_times"][b, :ne[b]], prob["t0"][b], side="left")] for b in range(B)])
    assert np.all(np.diff(mode0[perm]) >= 0) and len(set(mode0)) >= 3                      # robots in the same contact phase are adjacent
    cmd0, st0 = s.tick(prob, prob["t0"] + 0.002, wbc["rbd"], wbc["period"])
    s2 = q.Solver(batch=B, dt=0.015); pb = {k: v[perm] for k, v in prob.items()}
    cmd1, st1 = s2.tick(pb, pb["t0"] + 0.002, wbc["rbd"][perm], wbc["period"][perm])
    assert np.array_equal(cmd1, cmd0[perm])                                                  # a robot's result does not depend on its position
    cmd_d = torch.from_numpy(cmd1).to(dev); all_d = torch.zeros((B, 18), dtype=torch.float64, device=dev)
    s2.allgather_torque(cmd_d, all_d, torch.from_numpy(perm).to(dev)); torch.cuda.synchronize()
    assert np.array_equal(all_d.cpu().numpy(), cmd0[:, 36:])                                 # gathered buffer in ORIGINAL order
    s2.allgather_torque(cmd_d, all_d, None); torch.cuda.synchronize(); assert np.array_equal(all_d.cpu().numpy(), cmd1[:, 36:])
    assert s2.comm_info()[0] == 1


WORKER = r"""
import os, sys, numpy as np, torch
sys.path.insert(0, os.environ["QMB_ROOT"])
import qm_control_b200 as q
from qm_control_b200 import parallel, synthetic
rank, world, local = parallel.init_distributed(); torch.cuda.set_device(local); dev = torch.device("cuda", local)
B = 64; s = q.Solver(batch=B, device=local, dt=0.015); parallel.init_comm(s, rank, world); assert s.comm_info()[:2] == (world, rank)
ids = np.arange(rank * B, (rank + 1) * B); prob, wbc = synthetic.make_batch(ids, config=4)
cmd, st = s.tick(prob, prob["t0"] + 0.002, wbc["rbd"], wbc["period"])
cmd_d = torch.from_numpy(cmd).to(dev); all_d = torch.zeros((B * world, 18), dtype=torch.float64, device=dev)
s.allgather_torque(cmd_d, all_d); torch.cuda.synchronize()
ref = q.Solver(batch=B * world, device=local, dt=0.015); pa, wa = synthetic.make_batch(np.arange(B * world), config=4)
cmd_all, _ = ref.tick(pa, pa["t0"] + 0.002, wa["rbd"], wa["period"])
assert np.array_equal(all_d.cpu().numpy(), cmd_all[:, 36:]), "gathered torques differ from the single-GPU batch"
print("rank %d ok, nccl %d" % (rank, s.comm_info()[2]))
torch.distributed.destroy_process_group()
"""


def test_two_rank_nccl_allgather(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    w = tmp_path / "worker.py"; w.write_text(WORKER)
    env = dict(os.environ, QMB_ROOT=ROOT)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29533", str(w)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count(" ok") == 2
