#!/usr/bin/env python3
"""Cost of delayed observations (FootsiesEnv frame_delay) on the whole-horizon rollout path, microseconds per policy step
of RolloutCollector.collect(), hidden 64.

    python tools/delay_rollout_bench.py [--sizes 16384 131072 1048576] [--delays 0 1 4 8] [--horizon 128] [--rounds 5]

For every size, against the in-game bot ("bot") and in self-play with one network on both sides ("self"), delay 0 is the
existing kernel (fg_rollout_mlp*) and every other delay the frame_delay kernel (fg_rollout_mlp_delayed), whose queue
moves about 80 more bytes per battle and step.  At the smallest size the eager per-step path with delay 4
(fused="step": fg_policy_mlp_sample + fg_step + fg_delay_ring_step + a copy per step, no CUDA graph) is timed next to
them.  Cases are ALTERNATED: every round times each case once (CUDA events around --reps back-to-back collect() calls
after --warmup untimed ones), so drift of the shared host and of the clocks hits all of them alike; the median over rounds
is reported with the spread.  Every case has its own env of the same size and seed.  Prints the GPU name and power limit
first.
"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from footsies_gym_b200 import FootsiesEnv
from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable ({e})"
    return name, q


def make(opp, delay, fused, n, horizon, dev, pol):
    env = FootsiesEnv(num_envs=n, device=dev, seed=0, frame_delay=delay, opponent="bot" if opp == "bot" else "self_play")
    kw = {} if opp == "bot" else dict(opponent_policy=pol, mirror_opponent=True)
    col = RolloutCollector(env, pol, horizon=horizon, seed=1, fused=fused, **kw)
    assert col.mode == fused, (opp, delay, fused, col.mode)
    return col


def time_collect(col, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        col.collect()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) * 1000.0 / (reps * col.horizon)      # us per policy step


def bench(n, delays, horizon, rounds, reps, warmup, eager):
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    pol = MLPPolicy(64).to(dev)
    cases = [(opp, d, "horizon") for opp in ("bot", "self") for d in delays]
    if eager:
        cases += [(opp, 4, "step") for opp in ("bot", "self")]
    cols = {c: make(c[0], c[1], c[2], n, horizon, dev, pol) for c in cases}
    for c, col in cols.items():
        for _ in range(warmup):
            col.collect()
    torch.cuda.synchronize()
    samples = {c: [] for c in cases}
    for _ in range(rounds):
        for c in cases:
            samples[c].append(time_collect(cols[c], reps if c[2] == "horizon" else 1))
    print(f"\n== {n} battles, H = 64, horizon {horizon}, {rounds} alternated rounds x {reps} collects "
          f"(eager: 1 collect) ==")
    print(f"{'opponent':8s} {'delay':>5s} {'path':8s} {'median us/step':>15s} {'min':>9s} {'max':>9s} {'vs delay 0':>11s}")
    for c in cases:
        med = statistics.median(samples[c])
        base = statistics.median(samples[(c[0], delays[0], "horizon")])
        print(f"{c[0]:8s} {c[1]:5d} {c[2]:8s} {med:15.2f} {min(samples[c]):9.2f} {max(samples[c]):9.2f} "
              f"{100.0 * (med / base - 1):+10.2f}%")
    del cols
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[16384, 131072, 1048576])
    ap.add_argument("--delays", type=int, nargs="+", default=[0, 1, 4, 8], help="the first one is the baseline")
    ap.add_argument("--horizon", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=0, help="collects per timed sample (0: about 0.1 s of work)")
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("delay_rollout_bench needs a CUDA device: there is nothing to measure without one")
    name, q = gpu_info()
    print(f"GPU: {name}  (nvidia-smi name, power.limit, clocks.max.sm: {q})")
    for k, n in enumerate(a.sizes):
        reps = a.reps or max(2, min(200, int(100e3 / max(1.0, n / 16384 * 4.5 * a.horizon))))
        bench(n, a.delays, a.horizon, a.rounds, reps, a.warmup, eager=k == 0)


if __name__ == "__main__":
    main()
