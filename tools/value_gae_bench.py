#!/usr/bin/env python3
"""Critic side of a PPO iteration on one GPU: value pass (fg_value_mlp) and GAE (fg_gae) against the torch code they
replace, alone and inside RolloutCollector.collect(), plus the PPO example's whole iteration before / after.

    python tools/value_gae_bench.py [--envs 16384 1048576] [--horizon 128] [--hidden 64]

Times are CUDA-event times over warmed shapes (every timed shape runs --warmup times first); the example iteration is a
host clock around work that ends in a device synchronise.  Prints the GPU name and power limit first.
"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from footsies_gym_b200 import FootsiesEnv
from footsies_gym_b200.rollout import MLPPolicy, MLPValue, RolloutCollector, compute_gae

MACS_PER_ROW = 3 * (8 * 64 + 64 * 64 + 64 * 8)   # H = 64: 3 split products x (layer 1 + layer 2 + padded head n-tile)
MUFU_PER_ROW = 2 * 2 * 64                         # 128 tanh, two MUFU (ex2, rcp) each
GAE_BYTES_PER_ELEM = 4 + 1 + 4 + 4 + 4            # reward, done, value in; advantage, return out


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable ({e})"
    return name, q


def cuda_time(fn, reps, warmup):
    """Mean ms per call between two CUDA events around `reps` back-to-back calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / reps


def example_gae_loop(rew, done, v, gamma, lam):
    """examples/ppo_footsies.py's GAE before fg_gae (done as float)."""
    h, n = rew.shape
    adv = torch.zeros_like(rew)
    last = torch.zeros(n, device=rew.device)
    for t in range(h - 1, -1, -1):
        nonterm = 1.0 - done[t]
        delta = rew[t] + gamma * v[t + 1] * nonterm - v[t]
        last = delta + gamma * lam * nonterm * last
        adv[t] = last
    return adv, adv + v[:h]


def torch_values(value, rows, chunk):
    out = torch.empty(rows.shape[0], device=rows.device)
    for i in range(0, rows.shape[0], chunk):
        out[i:i + chunk] = value(rows[i:i + chunk])
    return out


def bench_size(n, h, hidden, warmup, reps, chunk):
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    policy, value = MLPPolicy(hidden).to(dev), MLPValue(hidden).to(dev)
    gamma, lam = 0.995, 0.95
    rows = (h + 1) * n
    print(f"\n== {n} battles x horizon {h}, H = {hidden}: {rows} value rows ==", flush=True)
    res = {}
    env0 = FootsiesEnv(num_envs=n, device=dev, seed=0)
    col0 = RolloutCollector(env0, policy, horizon=h)
    res["collect"] = cuda_time(col0.collect, reps, warmup)
    del col0, env0
    env1 = FootsiesEnv(num_envs=n, device=dev, seed=0)
    col1 = RolloutCollector(env1, policy, horizon=h, value=value, gamma=gamma, gae_lambda=lam)
    assert col1.mode == "horizon"
    res["collect_value_gae"] = cuda_time(col1.collect, reps, warmup)
    out = col1.collect()
    torch.cuda.synchronize()
    obs_rows = col1.obs.view(-1, 8)
    vals = torch.empty(rows, device=dev)
    with torch.no_grad():
        res["fg_value_mlp"] = cuda_time(lambda: value.fused_values(obs_rows, vals), reps, warmup)
        chunked = rows > chunk
        res["torch_value"] = cuda_time(lambda: torch_values(value, obs_rows, chunk), max(1, reps // 2), 1)
        ref = torch_values(value, obs_rows, chunk)
        value.fused_values(obs_rows, vals)
        err = float(((vals - ref).abs() / (1.0 + ref.abs())).max())
        del ref
        rew, dones, v = out["rewards"], out["dones"], out["values"]
        adv, ret = torch.empty_like(rew), torch.empty_like(rew)
        res["fg_gae"] = cuda_time(lambda: compute_gae(rew, dones, v, gamma, lam, adv, ret), reps, warmup)
        donef = dones.float()
        res["torch_gae_loop"] = cuda_time(lambda: example_gae_loop(rew, donef, v, gamma, lam), max(1, reps // 2), 1)
        ref_adv, ref_ret = example_gae_loop(rew, donef, v, gamma, lam)
        compute_gae(rew, dones, v, gamma, lam, adv, ret)
        same = bool(torch.equal(adv, ref_adv) and torch.equal(ret, ref_ret))
    print(f"collect() horizon mode, no value network   {res['collect']:9.3f} ms  ({res['collect'] * 1e3 / h:7.2f} us per step)")
    print(f"collect() with MLPValue (rollout+value+GAE) {res['collect_value_gae']:9.3f} ms  "
          f"(+{res['collect_value_gae'] - res['collect']:.3f} ms)")
    t = res["fg_value_mlp"] * 1e-3
    print(f"fg_value_mlp over {rows} rows                {res['fg_value_mlp']:9.3f} ms  {rows / t / 1e9:6.2f} G rows/s  "
          f"{2 * MACS_PER_ROW * rows / t / 1e12:6.1f} TFLOP/s of split-MMA work  {MUFU_PER_ROW * rows / t / 1e12:5.2f} T MUFU/s  "
          f"{36 * rows / t / 1e9:7.1f} GB/s (obs in, value out)")
    print(f"torch MLPValue.forward, same rows{' (chunks of %d rows)' % chunk if chunked else ''}  "
          f"{res['torch_value']:9.3f} ms  ({res['torch_value'] / res['fg_value_mlp']:.1f} x fg_value_mlp)")
    print(f"  max |v - v_torch| / (1 + |v_torch|) = {err:.3e}")
    gb = (GAE_BYTES_PER_ELEM * h * n + 4 * n) / 1e9
    print(f"fg_gae                                      {res['fg_gae']:9.3f} ms  {gb / (res['fg_gae'] * 1e-3):7.1f} GB/s "
          f"({gb * 1e3:.1f} MB moved{', fits in L2' if gb < 0.1 else ''})")
    print(f"example's torch GAE loop ({9 * h} launches)   {res['torch_gae_loop']:9.3f} ms  "
          f"({res['torch_gae_loop'] / res['fg_gae']:.1f} x fg_gae)   bit-identical: {same}")
    del col1, env1
    torch.cuda.empty_cache()
    return res


def bench_example_iteration(n, h, iters, warmup):
    """One PPO iteration of examples/ppo_footsies.py (defaults: 2 epochs x 8 minibatches), before (torch value pass + GAE
    loop after collect()) and after (collect() with the value network); the two alternate."""
    dev = torch.device("cuda:0")
    gamma, lam, clip, ent_c = 0.995, 0.95, 0.2, 0.01
    variants = {}
    for name in ("before", "after"):
        torch.manual_seed(0)
        policy, value = MLPPolicy(64).to(dev), MLPValue(64).to(dev)
        params = list(policy.parameters()) + list(value.parameters())
        env = FootsiesEnv(num_envs=n, device=dev, seed=0)
        col = RolloutCollector(env, policy, horizon=h, value=value if name == "after" else None, gamma=gamma, gae_lambda=lam)
        variants[name] = (policy, value, params, torch.optim.Adam(params, lr=1e-3), col)

    def iteration(name):
        policy, value, params, opt, col = variants[name]
        out = col.collect()
        obs, act, logp_old = out["obs"], out["actions"].long(), out["logp"]
        with torch.no_grad():
            if name == "before":
                v = value(torch.cat([obs, out["last_obs"][None]], 0))
                adv, ret = example_gae_loop(out["rewards"], out["dones"].float(), v, gamma, lam)
            else:
                adv, ret = out["advantages"], out["returns"]
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        flat = lambda x: x.reshape(h * n, *x.shape[2:])     # noqa: E731
        fo, fa, fl, fadv, fret = flat(obs), flat(act), flat(logp_old), flat(adv), flat(ret)
        for _ in range(2):
            perm = torch.randperm(h * n, device=dev)
            for mb in perm.chunk(8):
                lp_all = torch.log_softmax(policy(fo[mb]), -1)
                lp = lp_all.gather(1, fa[mb, None]).squeeze(1)
                ratio = (lp - fl[mb]).exp()
                pg = -torch.min(ratio * fadv[mb], ratio.clamp(1 - clip, 1 + clip) * fadv[mb]).mean()
                vl = 0.5 * (value(fo[mb]) - fret[mb]).pow(2).mean()
                ent = -(lp_all.exp() * lp_all).sum(-1).mean()
                loss = pg + 0.5 * vl - ent_c * ent
                opt.zero_grad(set_to_none=True)
                loss.backward()
                torch.nn.utils.clip_grad_norm_(params, 0.5)
                opt.step()

    for _ in range(warmup):
        for name in variants:
            iteration(name)
    times = {k: [] for k in variants}
    for _ in range(iters):
        for name in variants:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            iteration(name)
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
    print(f"\n== PPO example iteration, {n} battles x horizon {h}, 2 epochs x 8 minibatches ({iters} each, alternating) ==")
    for name, ts in times.items():
        ts = sorted(ts)
        print(f"{name:6s}: median {ts[len(ts) // 2] * 1e3:8.2f} ms  min {ts[0] * 1e3:8.2f}  max {ts[-1] * 1e3:8.2f}")


def accuracy(rows=129 * 16384):
    """The bar of tests/test_value_gae.py: parameters x3, observations drawn over the observation space."""
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(rows)
    ri = lambda hi: torch.randint(0, hi, (rows,), generator=g, device=dev).float()   # noqa: E731
    pos = lambda: torch.rand(rows, generator=g, device=dev) * 9.2 - 4.6              # noqa: E731
    obs = torch.stack([ri(4), ri(4), ri(15), ri(15), ri(56), ri(56), pos(), pos()], dim=1).contiguous()
    print(f"\n== fg_value_mlp vs torch fp32 MLPValue.forward, parameters x3, {rows} rows ==")
    for hidden in (32, 64):
        torch.manual_seed(hidden)
        v = MLPValue(hidden).to(dev)
        with torch.no_grad():
            for prm in v.net.parameters():
                prm.mul_(3.0)
            ref = v(obs)
        out = torch.empty(rows, device=dev)
        v.fused_values(obs, out)
        d = (out - ref).abs()
        print(f"H = {hidden}: max |v - v_torch| = {float(d.max()):.3e}, max |v - v_torch| / (1 + |v_torch|) = "
              f"{float((d / (1 + ref.abs())).max()):.3e}  (bar 2e-5; |v_torch| up to {float(ref.abs().max()):.2f})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[16384, 1 << 20])
    ap.add_argument("--horizon", type=int, default=128)
    ap.add_argument("--hidden", type=int, default=64)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=1 << 24, help="rows per torch value call (torch runs in chunks above it)")
    ap.add_argument("--example-iters", type=int, default=6)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, q = gpu_info()
    print(f"GPU: {name}; nvidia-smi name, power limit, max SM clock: {q}")
    print(f"torch {torch.__version__}; work per value row (H = 64): {MACS_PER_ROW} MMA multiply-adds, {MUFU_PER_ROW} MUFU")
    accuracy()
    for n in a.envs:
        bench_size(n, a.horizon, a.hidden, a.warmup, a.reps if n <= 65536 else max(3, a.reps // 2), a.chunk)
    bench_example_iteration(a.envs[0], a.horizon, a.example_iters, 2)


if __name__ == "__main__":
    main()
