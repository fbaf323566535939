#!/usr/bin/env python3
"""Small deterministic workload for compute-sanitizer (memcheck / racecheck / synccheck) runs of the kernels that exchange
data through shared memory between CTA barriers -- the whole-horizon rollout kernel and the per-step policy kernel -- and
of the sliced host-buffer path.  Ragged batch sizes; the two rollout paths must agree bit for bit.

    compute-sanitizer --tool racecheck python tools/sanitize_rollout.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("FOOTSIES_B200_HOST_CHUNK_ENVS", "256")
import numpy as np
import torch

from footsies_gym_b200 import FootsiesEnv
from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector

dev = torch.device("cuda:0")
horizon = int(os.environ.get("SAN_HORIZON", "12"))
for hidden, n in ((64, 200), (32, 333), (128, 70)):
    torch.manual_seed(hidden)
    pol = MLPPolicy(hidden).to(dev)
    outs = []
    for mode in ("step", "horizon"):
        env = FootsiesEnv(num_envs=n, device=dev, seed=3)
        col = RolloutCollector(env, pol, horizon=horizon, use_cuda_graph=False, fused=mode, seed=5)
        col.collect()
        outs.append({k: v.clone() for k, v in col.collect().items()})
        torch.cuda.synchronize()
        env.close()
    for k in outs[0]:
        assert torch.equal(outs[0][k], outs[1][k]), (hidden, n, k)
    print("rollout ok", hidden, n, flush=True)
rng = np.random.default_rng(0)
env = FootsiesEnv(num_envs=1000, device=dev, seed=1)
env.reset_host()
for t in range(10):
    env.step_host(rng.integers(0, 8, size=1000, dtype=np.uint8))
env.close()
print("host path ok")
print("sanitize_rollout done")
