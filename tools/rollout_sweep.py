#!/usr/bin/env python3
"""Whole-horizon rollout kernel (fg_rollout_mlp) against batch size and hidden size (developer tool).
usage: python tools/rollout_sweep.py            # sweep
       python tools/rollout_sweep.py --one N H  # one configuration in this process"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def one(n, hidden, reps=5, self_play=False, mode="horizon"):
    import torch
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
    dev = torch.device("cuda:0")
    env = FootsiesEnv(num_envs=n, device=dev, seed=0, opponent="self_play" if self_play else None)
    pol = MLPPolicy(hidden).to(dev)
    col = RolloutCollector(env, pol, horizon=128, fused=mode, opponent_policy=pol if self_play else None,
                           mirror_opponent=self_play)
    col.collect(); col.collect(); torch.cuda.synchronize()
    f0 = env.episode_stats()["env_frames"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        col.collect()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    fr = (env.episode_stats()["env_frames"] - f0) / reps
    print(f"n={n} hidden={hidden} self_play={self_play} mode={mode}: {ms * 1e3 / 128:.2f} us per step, "
          f"{fr / (ms * 1e-3):.3e} env-frames/s", flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--one":
        one(int(sys.argv[2]), int(sys.argv[3]))
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "--self-play":
        for n in (16384, 1048576):
            for mode in ("horizon", "step"):
                one(n, 64, self_play=True, mode=mode)
        sys.exit(0)
    for n, hidden in ((16384, 64), (131072, 64), (1048576, 64), (16384, 32), (16384, 128)):
        subprocess.run([sys.executable, os.path.abspath(__file__), "--one", str(n), str(hidden)])
