"""Whole-horizon rollouts with delayed observations (FootsiesEnv frame_delay, fg_rollout_mlp_delayed).

CPU: the ctypes mirror of fg_delay_ring matches the header as gcc compiles it, and a null handle or ring is refused.
GPU: the one-launch horizon equals, bit for bit, the eager per-step path (policy sample(s) on the delayed observation,
fg_step, fg_delay_ring_step) -- buffers, state planes, the queue itself, statistics and pool counters -- against the bot, a
second policy, a pool and a pool with the bot; the delayed observations, rewards and dones equal the CPU oracle's;
env.step() / env.reset() between collects; values and GAE; the ABI's rejections; one mebi-battle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("obs", "actions", "logp", "rewards", "dones", "last_obs")


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_delay_ring_struct_matches_the_header_as_gcc_sees_it(tmp_path):
    from footsies_gym_b200 import _capi
    cls = _capi.FgDelayRing
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "footsies_b200.h"', "int main(void) {",
             'printf("fg_delay_ring %zu\\n", sizeof(fg_delay_ring));']
    for fname, _ in cls._fields_:
        lines.append(f'printf("{fname} %zu\\n", offsetof(fg_delay_ring, {fname}));')
    lines += ["return 0; }"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["fg_delay_ring"]) == C.sizeof(cls)
    for fname, _ in cls._fields_:
        assert int(got[fname]) == getattr(cls, fname).offset, fname


def test_null_handle_and_null_ring_are_refused():
    from footsies_gym_b200 import _capi
    lib = _capi.load()
    f = lib.fg_rollout_mlp_delayed
    assert f.argtypes == [C.c_void_p, C.POINTER(_capi.FgRolloutBuffers), C.POINTER(_capi.FgOpponentPool), C.c_int32,
                          C.POINTER(_capi.FgDelayRing), C.c_void_p]
    r = _capi.FgRolloutBuffers(struct_size=C.sizeof(_capi.FgRolloutBuffers), hidden=64, horizon=8)
    ring = _capi.FgDelayRing(struct_size=C.sizeof(_capi.FgDelayRing), depth=4, pos=0)
    assert f(None, C.byref(r), None, -1, None, None) == -1
    assert b"fg_delay_ring is null" in lib.fg_last_error()
    bad = _capi.FgDelayRing(struct_size=8, depth=4, pos=0)
    assert f(None, C.byref(r), None, -1, C.byref(bad), None) == -1
    assert b"struct_size" in lib.fg_last_error()
    assert f(None, C.byref(r), None, -1, C.byref(ring), None) == -1
    assert b"null handle" in lib.fg_last_error()


# ---------------------------------------------------------------------------------------------------------------- GPU
def _dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    return torch.device("cuda:0")


def _mlp(hidden, dev, gain=2.0):
    from footsies_gym_b200.rollout import MLPPolicy
    p = MLPPolicy(hidden).to(dev)
    with torch.no_grad():
        for prm in p.net.parameters():
            prm.mul_(gain)
    return p


def _is_bot(m):
    return isinstance(m, str) and m == "bot"


def _queue(env, sl=slice(None)):
    """The env's frame_delay queue of battles `sl`, oldest slot first (independent of the ring position), and what it
    shows."""
    pos = env._ring_pos
    roll = lambda t: torch.roll(t[:, sl], -pos, 0)            # noqa: E731
    return dict(ring_obs=roll(env._ring_obs), ring_frame=roll(env._ring_frame), ring_misc=roll(env._ring_misc),
                delayed_obs=env._delayed_obs[sl], delayed_frame=env._delayed_frame[sl], delayed_misc=env._delayed_misc[sl])


def _env_equal(env, tenv, sl, where):
    assert torch.equal(env.state[:, sl], tenv.state), where
    assert torch.equal(env.info_frame[sl], tenv.info_frame), where
    assert torch.equal(env.info_misc[sl], tenv.info_misc), where
    q, tq = _queue(env, sl), _queue(tenv)
    for k in q:
        assert torch.equal(q[k], tq[k]), (where, k)


def _twin(env, col, s, e, member=None):
    """An eager per-step (fused="step") collector on an env holding battles [s, e) of `env` exactly as they are now:
    state planes, the queue and what it shows, info outputs, the policy counter.  member: the P2 of those battles (an
    MLPPolicy, "bot"), or None for the env's own opponent."""
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    if member is None:
        bot = env._opponent_mode == "bot"
        member = "bot" if bot else col.opponent_policy
    bot = _is_bot(member)
    tenv = FootsiesEnv(num_envs=e - s, device=env.device, first_env_index=s, opponent="bot" if bot else "self_play",
                       frame_delay=env.frame_delay, dense_reward=env.dense_reward, frame_skip=env.frame_skip,
                       skip_unactionable=env.skip_unactionable)
    kw = {} if bot else dict(opponent_policy=member, mirror_opponent=col.mirror_opponent)
    tcol = RolloutCollector(tenv, col.policy, horizon=col.horizon, fused="step", seed=col._seed, **kw)
    assert tcol.mode == "step"
    tenv.state.copy_(env.state[:, s:e])
    tenv.info_frame.copy_(env.info_frame[s:e])
    tenv.info_misc.copy_(env.info_misc[s:e])
    tenv._ring_obs.copy_(env._ring_obs[:, s:e])
    tenv._ring_frame.copy_(env._ring_frame[:, s:e])
    tenv._ring_misc.copy_(env._ring_misc[:, s:e])
    tenv._ring_pos = env._ring_pos
    tenv._delayed_obs.copy_(env._delayed_obs[s:e])
    tenv._delayed_frame.copy_(env._delayed_frame[s:e])
    tenv._delayed_misc.copy_(env._delayed_misc[s:e])
    tcol._drawn.copy_(col._drawn)
    return tenv, tcol


def _collect_against_twins(env, col, rounds):
    """`rounds` collects of `col`, each against eager twins of every non-empty range built from the state before it."""
    ranges = col.opponent_ranges or [(0, env.num_envs)]
    members = col.opponent_pool or [None]
    for r in range(rounds):
        twins = {m: _twin(env, col, s, e, members[m]) for m, (s, e) in enumerate(ranges) if s < e}
        tstats0 = {m: t[0].stats.clone() for m, t in twins.items()}
        pool0 = col.opponent_pool_stats() if col.opponent_pool else None
        handle0 = env.stats.clone()
        torch.cuda.synchronize()
        out = col.collect()
        touts = {m: t[1].collect() for m, t in twins.items()}
        torch.cuda.synchronize()
        for m, (s, e) in enumerate(ranges):
            if s == e:
                continue
            tenv, tcol = twins[m]
            tout = touts[m]
            where = (r, m)
            for k in KEYS:
                assert torch.equal(out[k][s:e] if k == "last_obs" else out[k][:, s:e], tout[k]), (where, k)
            if col.actions_p2 is not None and not _is_bot(members[m]):
                for k in ("actions_p2", "logp_p2"):
                    assert torch.equal(out[k][:, s:e], tout[k]), (where, k)
            _env_equal(env, tenv, slice(s, e), where)
            dstats = tenv.stats - tstats0[m]
            if col.opponent_pool:
                assert torch.equal((col.opponent_pool_stats() - pool0)[m], dstats[:4]), where
            else:
                assert torch.equal((env.stats - handle0)[:12], dstats[:12]), where
        if col.opponent_pool:
            tot = sum(twins[m][0].stats - tstats0[m] for m in twins)
            assert torch.equal((env.stats - handle0)[:12], tot[:12]), r
    return out


def _collector(n, delay, hidden, opp, dense=True, frame_skip=1, skip=False, horizon=50, seed=3):
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    torch.manual_seed(hidden * 31 + delay)
    env = FootsiesEnv(num_envs=n, device=dev, seed=seed, frame_delay=delay, opponent="bot" if opp == "bot" else "self_play",
                      dense_reward=dense, frame_skip=frame_skip, skip_unactionable=skip)
    kw = {}
    if opp in ("mirror", "selfplay"):
        kw = dict(opponent_policy=_mlp(hidden, dev), mirror_opponent=opp == "mirror")
    elif opp in ("pool", "pool_bot"):
        kw = dict(opponent_pool=[_mlp(hidden, dev), "bot" if opp == "pool_bot" else _mlp(hidden, dev), _mlp(hidden, dev)],
                  mirror_opponent=True)
    col = RolloutCollector(env, _mlp(hidden, dev), horizon=horizon, seed=17, **kw)
    assert col.mode == "horizon"
    return env, col


_N16, _N32 = 16384 + 300, 131072 + 300       # 16-battle warps / 32-battle warps picked by the launch


@pytest.mark.gpu
@pytest.mark.parametrize("delay,hidden,dense,opp,frame_skip,skip,n", [
    (1, 64, True, "bot", 1, False, _N16),
    (3, 32, False, "mirror", 3, False, _N16),
    (8, 128, True, "mirror", 1, True, _N16),
    (1, 32, True, "selfplay", 1, False, _N16),
    (3, 64, True, "pool", 1, True, _N16),
    (3, 64, False, "pool_bot", 3, False, _N16),
    (8, 32, True, "pool_bot", 1, True, _N16),
    (3, 128, False, "pool_bot", 1, False, _N16),
    (1, 128, True, "pool", 3, True, _N16),
    (3, 128, False, "bot", 3, True, _N16),
    (3, 64, True, "mirror", 1, False, _N32),
    (1, 32, False, "pool_bot", 1, True, _N32),
    (8, 64, True, "bot", 3, True, _N32),
    (3, 64, False, "pool", 1, False, _N32),
])
def test_horizon_kernel_equals_the_eager_step_path(delay, hidden, dense, opp, frame_skip, skip, n):
    """Three consecutive collects of 50 steps: with depth 2 / 4 / 9 the ring position moves by 0 / 2 / 5 per collect."""
    env, col = _collector(n, delay, hidden, opp, dense=dense, frame_skip=frame_skip, skip=skip)
    if col.opponent_pool:
        col.assign_opponents([2, 1, 1])
    out = _collect_against_twins(env, col, 3)
    assert out["dones"].any()
    # the delay is real: the buffer's observations are not the battles' current ones
    assert not torch.equal(env._delayed_frame, env.info_frame)


@pytest.mark.gpu
@pytest.mark.parametrize("delay", [1, 3, 7])
def test_delayed_rollout_equals_the_oracle(oracle, delay):
    """Every battle's collected actions replayed into the CPU reference with the same frame_delay: its delayed
    observations, rewards and terminations equal the rollout buffers."""
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    torch.manual_seed(delay)
    n, horizon = 384, 90
    env = FootsiesEnv(num_envs=n, device=dev, seed=2, frame_delay=delay)
    col = RolloutCollector(env, _mlp(64, dev), horizon=horizon, seed=5)
    assert col.mode == "horizon"
    orc = oracle.OracleBatch(n, p2_bot=True, frame_delay=delay, seed=2)
    orc.reset()
    assert np.array_equal(col.obs[horizon].cpu().numpy(), orc.trace["obs"])
    dones = 0
    for r in range(2):
        out = col.collect()
        obs, acts = out["obs"].cpu().numpy(), out["actions"].cpu().numpy()
        rew, done = out["rewards"].cpu().numpy(), out["dones"].cpu().numpy()
        last = out["last_obs"].cpu().numpy()
        for t in range(horizon):
            assert np.array_equal(obs[t], orc.trace["obs"]), (r, t)
            orc.step(acts[t])
            assert np.array_equal(rew[t], orc.trace["reward"]), (r, t)
            assert np.array_equal(done[t].astype(np.int32), orc.trace["terminated"]), (r, t)
        assert np.array_equal(last, orc.trace["obs"]), r
        assert np.array_equal(env._delayed_frame.cpu().numpy(), orc.trace["info_frame"]), r
        dones += int(done.sum())
    assert dones > 0


@pytest.mark.gpu
def test_env_steps_and_resets_between_collects():
    """collect(), env.step() x 3, env.reset(mask), collect() on the horizon kernel equals the same on the eager path."""
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    torch.manual_seed(7)
    n, horizon, delay = 1000, 50, 3
    pol = _mlp(64, dev)
    envs = [FootsiesEnv(num_envs=n, device=dev, seed=4, frame_delay=delay) for _ in range(2)]
    cols = [RolloutCollector(envs[0], pol, horizon=horizon, seed=9),
            RolloutCollector(envs[1], pol, horizon=horizon, seed=9, fused="step")]
    assert [c.mode for c in cols] == ["horizon", "step"]
    rng = np.random.default_rng(1)
    for r in range(2):
        outs = [c.collect() for c in cols]
        torch.cuda.synchronize()
        for k in KEYS:
            assert torch.equal(outs[0][k], outs[1][k]), (r, k)
        _env_equal(envs[0], envs[1], slice(None), r)
        for _ in range(3):
            a = torch.from_numpy(rng.integers(0, 8, size=n, dtype=np.uint8))
            stepped = [env.step(a) for env in envs]
            for k in ("guard", "move", "move_frame", "position"):
                assert torch.equal(stepped[0][0][k], stepped[1][0][k]), k
        mask = torch.from_numpy(rng.random(n) < 0.3)
        for env in envs:
            env.reset(options={"mask": mask})
        _env_equal(envs[0], envs[1], slice(None), ("reset", r))
    shown = envs[0]._delayed_obs.clone()
    outs = [c.collect() for c in cols]
    torch.cuda.synchronize()
    assert torch.equal(outs[0]["obs"][0], shown)                    # obs[0]: what the env showed when collect() began
    for k in KEYS:
        assert torch.equal(outs[0][k], outs[1][k]), k
    _env_equal(envs[0], envs[1], slice(None), "end")


@pytest.mark.gpu
def test_values_and_gae_on_the_delayed_buffer():
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import MLPValue, RolloutCollector, compute_gae
    dev = _dev()
    torch.manual_seed(11)
    env = FootsiesEnv(num_envs=2000, device=dev, seed=1, frame_delay=4)
    value = MLPValue(64).to(dev)
    col = RolloutCollector(env, _mlp(64, dev), horizon=60, seed=2, value=value, gamma=0.97, gae_lambda=0.9)
    assert col.mode == "horizon"
    for _ in range(2):
        out = col.collect()
        v = torch.empty_like(out["values"])
        value.fused_values(col.obs, v)
        assert torch.equal(out["values"], v)
        adv, ret = compute_gae(out["rewards"], out["dones"], v, 0.97, 0.9)
        assert torch.equal(out["advantages"], adv) and torch.equal(out["returns"], ret)
        with torch.no_grad():
            ref = value(col.obs.view(-1, 8)).view_as(v)
        assert torch.allclose(out["values"], ref, rtol=1e-4, atol=1e-5)


def _raw_call(col, edit=None, pool=None, bot_member=-1):
    from footsies_gym_b200 import _capi
    env, pol = col.env, col.policy
    l1, l2, l3 = pol.net[0], pol.net[2], pol.net[4]
    r = _capi.FgRolloutBuffers(struct_size=C.sizeof(_capi.FgRolloutBuffers), hidden=pol.hidden, horizon=col.horizon, seed=17)
    for k, t in dict(scale=pol.scale, w1=l1.weight, b1=l1.bias, w2=l2.weight, b2=l2.bias, w3=l3.weight, b3=l3.bias,
                     counter_base=col._drawn, obs=col.obs, actions=col.actions, logp=col.logp, rewards=col.rewards,
                     dones=col.dones).items():
        setattr(r, k, t.data_ptr())
    ring = _capi.FgDelayRing(struct_size=C.sizeof(_capi.FgDelayRing), depth=env.frame_delay + 1, pos=env._ring_pos)
    for k, t in dict(ring_obs=env._ring_obs, ring_frame=env._ring_frame, ring_misc=env._ring_misc, out_obs=env._delayed_obs,
                     out_frame=env._delayed_frame, out_misc=env._delayed_misc).items():
        setattr(ring, k, t.data_ptr())
    if edit:
        edit(ring)
    rc = env._lib.fg_rollout_mlp_delayed(env._handle, C.byref(r), pool, bot_member, C.byref(ring), env._stream())
    return rc, env._lib.fg_last_error().decode()


@pytest.mark.gpu
def test_abi_rejections():
    from footsies_gym_b200 import FootsiesEnv, _capi
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    env = FootsiesEnv(num_envs=640, device=dev, seed=3, frame_delay=3)
    col = RolloutCollector(env, _mlp(64, dev), horizon=8, seed=17)
    launches = env.launch_count()
    s = lambda name, value: (lambda o: setattr(o, name, value))    # noqa: E731
    cases = [
        (s("depth", 1), "depth"), (s("depth", 0), "depth"), (s("pos", 4), "pos"), (s("pos", -1), "pos"),
        (s("ring_obs", None), "null buffer"), (s("ring_frame", None), "null buffer"), (s("ring_misc", None), "null buffer"),
        (s("out_obs", None), "null buffer"), (s("out_frame", None), "null buffer"), (s("out_misc", None), "null buffer"),
        (s("ring_obs", env._ring_obs.data_ptr() + 4), "16-byte"), (s("out_obs", env._delayed_obs.data_ptr() + 8), "16-byte"),
        (s("ring_misc", env._ring_misc.data_ptr() + 1), "4-byte"), (s("out_misc", env._delayed_misc.data_ptr() + 2), "4-byte"),
        (s("struct_size", 16), "struct_size"),
    ]
    for edit, msg in cases:
        rc, err = _raw_call(col, edit)
        assert rc == -1 and msg in err, (msg, rc, err)
    rc, err = _raw_call(col, bot_member=0)                           # a bot member without a pool
    assert rc == -1 and "bot_member" in err, err
    bad_pool = _capi.FgOpponentPool(struct_size=8, count=1)          # the pool's own checks apply
    rc, err = _raw_call(col, pool=C.byref(bad_pool))
    assert rc == -1 and "fg_opponent_pool" in err, err
    rc = env._lib.fg_rollout_mlp_delayed(env._handle, None, None, -1, None, env._stream())
    assert rc == -1 and "fg_delay_ring is null" in env._lib.fg_last_error().decode()
    assert env.launch_count() == launches                           # nothing was launched
    rc, err = _raw_call(col)
    assert rc == 0, err
    torch.cuda.synchronize()
    assert env.launch_count() == launches + 1


@pytest.mark.gpu
def test_one_mebibattle_delay_4():
    env, col = _collector(1 << 20, 4, 64, "bot", horizon=128)
    out = _collect_against_twins(env, col, 1)
    assert out["dones"].any()
