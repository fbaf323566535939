#!/usr/bin/env python3
"""PPO against the in-game bot, entirely on the GPU (BASELINE.json configs[4] in use).

    python examples/ppo_footsies.py [--envs 16384] [--horizon 128] [--iters 40] [--frame-skip 1] [--self-play]
                                    [--pool K --snapshot-every S]
    torchrun --nproc-per-node 8 examples/ppo_footsies.py          # one process per GPU, gradients all-reduced

Rollouts come from footsies_gym_b200.rollout.RolloutCollector: the fused policy kernel samples actions from the
observation tensor the step kernel wrote, the step kernel writes the next observation / reward / done flag straight
into the rollout buffers, one launch per horizon (fg_rollout_mlp keeps the battles in registers for all 128 steps).  The
collector also evaluates the value MLP over every observation of the horizon (fg_value_mlp, one launch) and computes GAE
advantages and returns (fg_gae, one launch).  The update is ordinary torch (clipped PPO); the policy's and the value
network's parameters are updated in place, so the next rollout reads the new weights.
Prints the win rate against the bot per iteration (from the kernel's own episode statistics).
With --self-play the training rollouts are played against the same network on the mirrored observation (still one
launch per horizon) and the win rate against the in-game bot comes from a separate evaluation rollout per iteration.
With --self-play --pool K the opponent is a pool of K networks sharing the battles equally (fg_rollout_mlp_pool, still
one launch per horizon): member 0 is the live policy, the other K - 1 slots hold frozen snapshots of it, refreshed one
slot at a time in round-robin order every S iterations (all start as the initial policy).  Each iteration also prints the
win rate against every member, from the kernel's per-member counters (all-reduced over the ranks, which use the same
shares).
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch
import torch.distributed as dist

from footsies_gym_b200.distributed import env_rank_world, make_sharded_env
from footsies_gym_b200.rollout import MLPPolicy, MLPValue, RolloutCollector


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384, help="envs per GPU")
    ap.add_argument("--horizon", type=int, default=128)
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--frame-skip", type=int, default=1)
    ap.add_argument("--epochs", type=int, default=2)
    ap.add_argument("--minibatches", type=int, default=8)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--gamma", type=float, default=0.995)
    ap.add_argument("--lam", type=float, default=0.95)
    ap.add_argument("--clip", type=float, default=0.2)
    ap.add_argument("--entropy", type=float, default=0.01)
    ap.add_argument("--self-play", action="store_true", help="train against the same network playing the mirrored side")
    ap.add_argument("--pool", type=int, default=0, help="with --self-play: play against a pool of this many networks "
                    "(the live policy + K - 1 snapshots)")
    ap.add_argument("--snapshot-every", type=int, default=5, help="iterations between two snapshots into the pool")
    a = ap.parse_args()
    if a.pool and not a.self_play:
        ap.error("--pool needs --self-play")
    if a.pool < 0 or a.pool > 16 or a.snapshot_every < 1:
        ap.error("--pool must be in 1 .. 16 and --snapshot-every positive")

    rank, local_rank, world = env_rank_world()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)

    env = make_sharded_env(a.envs * world, frame_skip=a.frame_skip, seed=0, opponent="self_play" if a.self_play else None)
    policy = MLPPolicy(64).to(dev)
    value = MLPValue(64).to(dev)
    params = list(policy.parameters()) + list(value.parameters())
    if world > 1:
        for p in params:
            dist.broadcast(p.data, 0)
    opt = torch.optim.Adam(params, lr=a.lr)
    pool = None
    if a.pool:
        pool = [policy] + [MLPPolicy(64).to(dev) for _ in range(a.pool - 1)]
        for m in pool[1:]:
            m.load_state_dict(policy.state_dict())
            m.requires_grad_(False)
    col = RolloutCollector(env, policy, horizon=a.horizon, use_cuda_graph=True, seed=rank,
                           opponent_policy=policy if a.self_play and not a.pool else None, mirror_opponent=a.self_play,
                           opponent_pool=pool, value=value, gamma=a.gamma, gae_lambda=a.lam)
    next_slot = 1
    eval_env = eval_col = None
    if a.self_play:                       # the yardstick stays the in-game bot
        eval_env = make_sharded_env(a.envs * world, frame_skip=a.frame_skip, seed=1)
        eval_col = RolloutCollector(eval_env, policy, horizon=a.horizon, seed=1000 + rank)
    n, h = env.num_envs, a.horizon
    stat_env = eval_env if a.self_play else env
    prev = stat_env.episode_stats()
    prev_pool = col.opponent_pool_stats() if pool else None
    t_roll = t_upd = 0.0
    for it in range(a.iters):
        t0 = time.perf_counter()
        out = col.collect()
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        obs, act, logp_old = out["obs"], out["actions"].long(), out["logp"]
        rew = out["rewards"]
        # GAE came with the rollout: an env that terminated at step t restarts by itself (the step after is the reset,
        # reward 0), so the bootstrap is cut at the terminal step
        ret = out["returns"]
        with torch.no_grad():
            adv = out["advantages"]
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        flat = lambda x: x.reshape(h * n, *x.shape[2:])     # noqa: E731
        fo, fa, fl, fadv, fret = flat(obs), flat(act), flat(logp_old), flat(adv), flat(ret)
        for _ in range(a.epochs):
            perm = torch.randperm(h * n, device=dev)
            for mb in perm.chunk(a.minibatches):
                logits = policy(fo[mb])
                lp_all = torch.log_softmax(logits, -1)
                lp = lp_all.gather(1, fa[mb, None]).squeeze(1)
                ratio = (lp - fl[mb]).exp()
                pg = -torch.min(ratio * fadv[mb], ratio.clamp(1 - a.clip, 1 + a.clip) * fadv[mb]).mean()
                vl = 0.5 * (value(fo[mb]) - fret[mb]).pow(2).mean()
                ent = -(lp_all.exp() * lp_all).sum(-1).mean()
                loss = pg + 0.5 * vl - a.entropy * ent
                opt.zero_grad(set_to_none=True)
                loss.backward()
                if world > 1:
                    for p in params:
                        dist.all_reduce(p.grad, op=dist.ReduceOp.AVG)
                torch.nn.utils.clip_grad_norm_(params, 0.5)
                opt.step()
        torch.cuda.synchronize(dev)
        t2 = time.perf_counter()
        t_roll += t1 - t0
        t_upd += t2 - t1
        frames = env.episode_stats()["env_frames"] - (0 if it == 0 else frames_seen)
        frames_seen = env.episode_stats()["env_frames"]
        if world > 1:
            ft = torch.tensor([frames], dtype=torch.int64, device=dev)
            dist.all_reduce(ft)
            frames = int(ft.item())
        if a.self_play:
            eval_col.collect()
        st = stat_env.all_reduce_stats()
        ep = st["episodes"] - prev["episodes"]
        wins = st["p1_wins"] - prev["p1_wins"]
        prev = st
        pool_msg = ""
        if pool:
            cur = col.opponent_pool_stats()
            d = cur - prev_pool                              # [K, 4] this iteration: episodes, P1 wins, P2 wins, double KOs
            prev_pool = cur
            if world > 1:
                dist.all_reduce(d)
            d = d.cpu()
            pool_msg = "  win rate vs pool [" + " ".join(f"{int(w) / max(int(e), 1):.2f}" for e, w in d[:, :2].tolist()) + "]"
            if (it + 1) % a.snapshot_every == 0 and a.pool > 1:
                pool[next_slot].load_state_dict(policy.state_dict())     # played from the next collect() on
                next_slot = next_slot % (a.pool - 1) + 1
        if rank == 0:
            print(f"iter {it:3d}  episodes {ep:8d}  win rate vs bot {wins / max(ep, 1):.3f}  mean reward/step {float(rew.mean()):+.4f}  "
                  f"rollout {frames / (t1 - t0) / 1e6:8.1f} M env-frames/s  update {t2 - t1:.2f} s{pool_msg}", flush=True)
    if rank == 0:
        print(f"total: rollouts {t_roll:.1f} s, updates {t_upd:.1f} s")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
