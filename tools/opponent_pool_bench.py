#!/usr/bin/env python3
"""Self-play rollout cost of an opponent pool: fg_rollout_mlp with one P2 network against fg_rollout_mlp_pool with pools of
1, 4 and 16 networks (equal shares), whole-horizon launches through RolloutCollector, microseconds per policy step.

    python tools/opponent_pool_bench.py [--config 16384:64 131072:64 1048576:64 16384:128] [--horizon 128] [--rounds 7]
                                        [--variants single pool1 pool4 pool16 pool3+bot bot vsbot]

The only work a pool adds is a scan of at most 16 range ends per CTA and one statistics add per CTA, so the expected
difference is nil.  The in-game bot as a member (fg_rollout_mlp_pool_bot): pool3+bot = 3 networks + the bot, a quarter of
the battles each; bot = a pool of just the bot; vsbot = fg_rollout_mlp against the bot (an opponent="bot" env).  The
bot's CTAs skip the second network, so adding it should make a pool cheaper, never dearer.  Variants are ALTERNATED: every round times each variant once (CUDA events around --reps back-to-back
collect() calls after --warmup untimed ones per variant), so drift of the shared host and the clocks hits all of them
alike; the median over rounds is reported with the spread.  Every variant has its own env of the same size and seed.  A
collector's buffers (about 90 bytes per battle and step) fit the 126 MB L2 at 16 384 battles x 128 steps, not from
131 072 battles up.  Prints the GPU name and power limit first.
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

VARIANTS = ("single", "pool1", "pool4", "pool16")
BOT_VARIANTS = ("pool3+bot", "bot", "vsbot")


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable ({e})"
    return name, q


def make(variant, n, hidden, horizon, dev, p1, members):
    env = FootsiesEnv(num_envs=n, device=dev, seed=0, opponent="bot" if variant == "vsbot" else "self_play")
    if variant == "vsbot":
        return RolloutCollector(env, p1, horizon=horizon, seed=1)
    if variant == "single":
        return RolloutCollector(env, p1, horizon=horizon, seed=1, opponent_policy=members[0], mirror_opponent=True)
    pool = {"pool3+bot": members[:3] + ["bot"], "bot": ["bot"]}.get(variant) or members[:int(variant[4:])]
    return RolloutCollector(env, p1, horizon=horizon, seed=1, opponent_pool=pool, mirror_opponent=True)


def time_collect(col, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        col.collect()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) * 1000.0 / (reps * col.horizon)      # us per policy step


def bench(n, hidden, horizon, rounds, reps, warmup, variants=VARIANTS):
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    p1 = MLPPolicy(hidden).to(dev)
    members = [MLPPolicy(hidden).to(dev) for _ in range(16)]
    cols = {v: make(v, n, hidden, horizon, dev, p1, members) for v in variants}
    for v, c in cols.items():
        assert c.mode == "horizon", v
        for _ in range(warmup):
            c.collect()
    torch.cuda.synchronize()
    samples = {v: [] for v in variants}
    for _ in range(rounds):
        for v in variants:
            samples[v].append(time_collect(cols[v], reps))
    base = statistics.median(samples[variants[0]])
    print(f"\n== {n} battles, H = {hidden}, horizon {horizon}, {rounds} alternated rounds x {reps} collects ==")
    print(f"{'variant':9s} {'median us/step':>15s} {'min':>9s} {'max':>9s} {'vs ' + variants[0]:>10s}")
    rows = []
    for v in variants:
        med = statistics.median(samples[v])
        print(f"{v:9s} {med:15.2f} {min(samples[v]):9.2f} {max(samples[v]):9.2f} {100.0 * (med / base - 1):+9.2f}%")
        rows.append((v, med, min(samples[v]), max(samples[v])))
    # per-member counters are consistent with the handle's (a cheap sanity check at every measured size)
    for v, c in cols.items():
        if c.opponent_pool is not None:
            st = c.opponent_pool_stats().sum(0).cpu().tolist()
            es = c.env.episode_stats()
            assert st == [es["episodes"], es["p1_wins"], es["p2_wins"], es["double_ko"]], (v, st, es)
    del cols
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", nargs="+", default=["16384:64", "131072:64", "1048576:64", "16384:128"],
                    help="battles:hidden")
    ap.add_argument("--horizon", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=0, help="collects per timed sample (0: about 0.1 s of work)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--variants", nargs="+", default=list(VARIANTS), choices=VARIANTS + BOT_VARIANTS,
                    help="the first one is the baseline of the last column")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("opponent_pool_bench needs a CUDA device: there is nothing to measure without one")
    name, q = gpu_info()
    print(f"GPU: {name}  (nvidia-smi name, power.limit, clocks.max.sm: {q})")
    for cfg in a.config:
        n, hidden = (int(x) for x in cfg.split(":"))
        reps = a.reps or max(2, min(200, int(100e3 / max(1.0, n / 16384 * 4.5 * a.horizon))))
        bench(n, hidden, a.horizon, a.rounds, reps, a.warmup, a.variants)


if __name__ == "__main__":
    main()
