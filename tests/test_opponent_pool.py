"""Self-play against an opponent pool (fg_rollout_mlp_pool, RolloutCollector(opponent_pool=...)).

CPU: the ctypes mirrors match the header as gcc compiles it, null handles / pools are refused, and the share-to-range
arithmetic covers every battle once with block-aligned boundaries.  GPU: every member's range of a pool rollout equals,
bit for bit, a rollout of just those battles against that member alone through the existing single-opponent kernel, and
the per-member counters equal that twin's episode statistics."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("obs", "actions", "logp", "actions_p2", "logp_p2", "rewards", "dones", "last_obs")
STAT4 = ("episodes", "p1_wins", "p2_wins", "double_ko")


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_pool_structs_match_the_header_as_gcc_sees_it(tmp_path):
    from footsies_gym_b200 import _capi
    pairs = {"fg_mlp_weights": _capi.FgMlpWeights, "fg_opponent_pool": _capi.FgOpponentPool}
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "footsies_b200.h"', "int main(void) {",
             'printf("FG_POOL_MAX %d\\n", FG_POOL_MAX);', 'printf("FG_POOL_BLOCK %d\\n", FG_POOL_BLOCK);']
    for cname, cls in pairs.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["return 0; }"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["FG_POOL_MAX"]) == _capi.FG_POOL_MAX and int(got["FG_POOL_BLOCK"]) == _capi.FG_POOL_BLOCK
    for cname, cls in pairs.items():
        assert int(got[cname]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, (cname, fname)


def test_null_handle_and_null_pool_are_refused():
    from footsies_gym_b200 import _capi
    lib = _capi.load()
    r = _capi.FgRolloutBuffers(struct_size=C.sizeof(_capi.FgRolloutBuffers), hidden=64, horizon=8)
    pool = _capi.FgOpponentPool(struct_size=C.sizeof(_capi.FgOpponentPool), count=1)
    assert lib.fg_rollout_mlp_pool(None, C.byref(r), None, None) == -1
    assert b"fg_opponent_pool is null" in lib.fg_last_error()
    bad = _capi.FgOpponentPool(struct_size=8, count=1)
    assert lib.fg_rollout_mlp_pool(None, C.byref(r), C.byref(bad), None) == -1
    assert b"struct_size" in lib.fg_last_error()
    assert lib.fg_rollout_mlp_pool(None, C.byref(r), C.byref(pool), None) == -1     # null handle


@pytest.mark.parametrize("n", [1, 127, 128, 1000, 16384, 131072 + 37, 1 << 20])
@pytest.mark.parametrize("shares", [[1], [1, 1], [3, 0, 1, 2], [0, 0, 5], [1, 0], [0.1, 0.7, 0.2],
                                    [1] * 16, [2, 1, 0, 0, 1, 3, 0, 1, 1, 0, 0, 2, 1, 1, 0, 7]])
def test_share_ranges_are_aligned_and_cover_every_battle_once(n, shares):
    from footsies_gym_b200.rollout import opponent_ranges
    block = 128
    ranges = opponent_ranges(n, shares)
    assert len(ranges) == len(shares)
    assert ranges[0][0] == 0 and ranges[-1][1] == n
    for (s0, e0), (s1, _) in zip(ranges, ranges[1:]):
        assert e0 == s1
    for k, (s, e) in enumerate(ranges):
        assert s <= e
        if e != n:
            assert e % block == 0, (k, ranges)
        if shares[k] == 0:
            assert s == e, (k, ranges)
    # largest remainder over the whole blocks: each member is within one block of its exact quota
    blocks = n // block
    last = max(i for i, s in enumerate(shares) if s > 0)
    for k, (s, e) in enumerate(ranges):
        got = (e - s) // block if k != last else (e - s - n % block) // block
        assert abs(got - shares[k] / sum(shares) * blocks) < 1.0 + 1e-9, (k, ranges)
    # the leftover battles of the last partial block belong to the last member with a non-zero share
    assert ranges[last][1] == n and (n % block == 0 or ranges[last][1] - ranges[last][0] >= n % block)


def test_share_ranges_largest_remainder_and_rejections():
    from footsies_gym_b200.rollout import opponent_ranges
    # 7 whole blocks at 3 : 0 : 1 : 2 -> quotas 3.5, 0, 1.17, 2.33 -> 3 + 1 (largest remainder), 0, 1, 2; 104 left over
    assert opponent_ranges(1000, [3, 0, 1, 2]) == [(0, 512), (512, 512), (512, 640), (640, 1000)]
    assert opponent_ranges(256, [1, 1, 1]) == [(0, 128), (128, 256), (256, 256)]     # tie: the lower index wins
    assert opponent_ranges(100, [1, 1]) == [(0, 0), (0, 100)]
    assert opponent_ranges(300, [1, 0]) == [(0, 300), (300, 300)]
    for bad in ([], [0, 0], [-1, 2], [float("nan")], [1] * 17, [float("inf"), 1]):
        with pytest.raises(ValueError):
            opponent_ranges(1000, bad)


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


def _stat4(env):
    s = env.episode_stats()
    return np.array([s[k] for k in STAT4], dtype=np.int64)


def _pool_equals_twins(hidden, n, shares, dense=True, frame_skip=1, skip=False, mirror=False, horizon=130, rounds=2,
                       live_member=False):
    """Pool rollout against, per non-empty range, a twin env of just those battles (num_envs = end - start,
    first_env_index = start) played by the single-opponent kernel with that member as P2."""
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    torch.manual_seed(hidden * 7 + n)
    p1 = _mlp(hidden, dev)
    members = [_mlp(hidden, dev) for _ in shares]
    if live_member:
        members[0] = p1                                     # the learner itself is a member
    kw = dict(seed=3, opponent="self_play", dense_reward=dense, frame_skip=frame_skip, skip_unactionable=skip)
    env = FootsiesEnv(num_envs=n, device=dev, **kw)
    col = RolloutCollector(env, p1, horizon=horizon, use_cuda_graph=False, seed=17, opponent_pool=members,
                           mirror_opponent=mirror)
    assert col.mode == "horizon"
    ranges = col.assign_opponents(shares)
    assert ranges == col.opponent_ranges
    twins = {}
    for m, (s, e) in enumerate(ranges):
        if s < e:
            tenv = FootsiesEnv(num_envs=e - s, device=dev, first_env_index=s, **kw)
            twins[m] = (tenv, RolloutCollector(tenv, p1, horizon=horizon, use_cuda_graph=False, seed=17,
                                               opponent_policy=members[m], mirror_opponent=mirror))
    start = _stat4(env)
    for r in range(rounds):
        out = col.collect()
        touts = {m: (t[1].collect(), _stat4(t[0])) for m, t in twins.items()}
        torch.cuda.synchronize()
        pool_stats = col.opponent_pool_stats().cpu().numpy()
        state = env.get_state()
        for m, (s, e) in enumerate(ranges):
            if s == e:
                assert not pool_stats[m].any(), (r, m)
                continue
            tout, tstats = touts[m]
            for k in KEYS:
                assert torch.equal(out[k][s:e] if k == "last_obs" else out[k][:, s:e], tout[k]), (r, m, k)
            assert state[s:e].tobytes() == twins[m][0].get_state().tobytes(), (r, m)
            assert np.array_equal(pool_stats[m], tstats), (r, m, pool_stats[m], tstats)
            assert torch.equal(env.info_frame[s:e], twins[m][0].info_frame), (r, m)
        # the per-member counters add up to what the handle counted over the same collects
        assert np.array_equal(pool_stats.sum(0), _stat4(env) - start), r
        assert (pool_stats[:, 0] == pool_stats[:, 1:].sum(1)).all()
    assert pool_stats[:, 0].sum() > 0 and out["dones"].any()


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,n,shares,dense,frame_skip,skip,mirror", [
    (64, 1000, [3, 0, 1, 2], True, 1, False, True),          # ragged tail, an empty range in the middle
    (64, 777, [0, 1, 1, 1], False, 2, False, False),         # empty first range, sparse reward, frame skip
    (32, 1000, [1, 2, 0, 1], True, 1, True, False),          # fused frame skipping
    (32, 555, [2, 1, 1], False, 1, False, True),
    (128, 1000, [1, 2, 0, 1], True, 1, False, False),        # H = 128: the FFMA kernel
    (128, 700, [1, 1, 1], False, 3, True, True),
])
def test_pool_ranges_equal_single_opponent_twins(hidden, n, shares, dense, frame_skip, skip, mirror):
    _pool_equals_twins(hidden, n, shares, dense=dense, frame_skip=frame_skip, skip=skip, mirror=mirror, horizon=150)


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,n,shares,skip", [(64, 1000, [3, 0, 1, 2], False), (32, 700, [1, 1, 0, 2], True)])
def test_pool_ranges_equal_twins_with_32_battle_warps(monkeypatch, hidden, n, shares, skip):
    """The 32-battle-warp shape (128-battle CTAs, selected from 131 072 battles up) forced onto small batches."""
    monkeypatch.setenv("FOOTSIES_B200_ROLLOUT_MT", "2")
    _pool_equals_twins(hidden, n, shares, skip=skip, mirror=True)


@pytest.mark.gpu
def test_pool_at_the_size_that_selects_32_battle_warps():
    """131 072 + 300 battles: the pool launch picks 128-battle CTAs by itself while the smaller twins run 64-battle CTAs."""
    _pool_equals_twins(64, 131072 + 300, [1, 1, 1, 1], horizon=64, rounds=2, mirror=True)


@pytest.mark.gpu
def test_pool_with_the_live_policy_as_a_member():
    _pool_equals_twins(64, 640, [1, 1, 1], mirror=True, live_member=True)


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,mirror", [(64, True), (128, False)])
def test_one_member_pool_equals_opponent_policy(hidden, mirror):
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    torch.manual_seed(5)
    n, horizon = 1000, 130
    p1, p2 = _mlp(hidden, dev), _mlp(hidden, dev)
    envs = [FootsiesEnv(num_envs=n, device=dev, seed=3, opponent="self_play") for _ in range(2)]
    a = RolloutCollector(envs[0], p1, horizon=horizon, seed=17, opponent_policy=p2, mirror_opponent=mirror)
    b = RolloutCollector(envs[1], p1, horizon=horizon, seed=17, opponent_pool=[p2], mirror_opponent=mirror)
    assert a.mode == b.mode == "horizon" and b.opponent_ranges == [(0, n)]
    for r in range(2):
        oa, ob = a.collect(), b.collect()
        torch.cuda.synchronize()
        for k in KEYS:
            assert torch.equal(oa[k], ob[k]), (r, k)
        assert envs[0].get_state().tobytes() == envs[1].get_state().tobytes()
        assert envs[0].episode_stats() == envs[1].episode_stats()
        assert np.array_equal(b.opponent_pool_stats().cpu().numpy()[0], _stat4(envs[1]))
    assert int(b.opponent_pool_stats()[0, 0]) > 0


@pytest.mark.gpu
def test_load_state_dict_into_a_member_changes_only_its_range():
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    torch.manual_seed(9)
    n, horizon = 768, 100
    p1 = _mlp(64, dev)
    base = [_mlp(64, dev) for _ in range(3)]
    snapshot = _mlp(64, dev).state_dict()
    envs, cols, pools = [], [], []
    for _ in range(2):
        pool = [_mlp(64, dev) for _ in range(3)]
        for m, src in zip(pool, base):
            m.load_state_dict(src.state_dict())
        env = FootsiesEnv(num_envs=n, device=dev, seed=3, opponent="self_play")
        envs.append(env); pools.append(pool)
        cols.append(RolloutCollector(env, p1, horizon=horizon, seed=17, opponent_pool=pool))
    ranges = cols[0].opponent_ranges
    assert ranges == [(0, 256), (256, 512), (512, 768)]
    outs = [c.collect() for c in cols]
    for k in KEYS:
        assert torch.equal(outs[0][k], outs[1][k]), k
    pools[0][1].load_state_dict(snapshot)                   # in place: the next collect() plays the snapshot
    outs = [c.collect() for c in cols]
    torch.cuda.synchronize()
    s, e = ranges[1]
    for k in ("actions_p2", "logp_p2"):
        assert torch.equal(outs[0][k][:, :s], outs[1][k][:, :s]) and torch.equal(outs[0][k][:, e:], outs[1][k][:, e:]), k
        assert not torch.equal(outs[0][k][:, s:e], outs[1][k][:, s:e]), k
    for k in ("obs", "actions", "rewards", "dones"):
        assert torch.equal(outs[0][k][:, :s], outs[1][k][:, :s]) and torch.equal(outs[0][k][:, e:], outs[1][k][:, e:]), k
    st = [env.get_state() for env in envs]
    assert st[0][:s].tobytes() == st[1][:s].tobytes() and st[0][e:].tobytes() == st[1][e:].tobytes()
    assert st[0][s:e].tobytes() != st[1][s:e].tobytes()


def _raw_pool_call(col, r_edit=None, pool_edit=None):
    from footsies_gym_b200 import _capi
    env, pol = col.env, col.policy
    l1, l2, l3 = pol.net[0], pol.net[2], pol.net[4]
    r = _capi.FgRolloutBuffers(struct_size=C.sizeof(_capi.FgRolloutBuffers), hidden=pol.hidden, horizon=col.horizon,
                               seed=17)
    for k, t in dict(scale=pol.scale, w1=l1.weight, b1=l1.bias, w2=l2.weight, b2=l2.bias, w3=l3.weight, b3=l3.bias,
                     counter_base=col._drawn, obs=col.obs, actions=col.actions, logp=col.logp, rewards=col.rewards,
                     dones=col.dones, actions_p2=col.actions_p2, logp_p2=col.logp_p2).items():
        setattr(r, k, t.data_ptr())
    pool = col._pool_struct()
    if r_edit:
        r_edit(r)
    if pool_edit:
        pool_edit(pool)
    lib = env._lib
    rc = lib.fg_rollout_mlp_pool(env._handle, C.byref(r), C.byref(pool), env._stream())
    return rc, lib.fg_last_error().decode()


@pytest.mark.gpu
def test_abi_rejections():
    from footsies_gym_b200 import FootsiesEnv, _capi
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    n = 640
    p1 = _mlp(64, dev)
    members = [_mlp(64, dev) for _ in range(3)]
    env = FootsiesEnv(num_envs=n, device=dev, seed=3, opponent="self_play")
    col = RolloutCollector(env, p1, horizon=8, seed=17, opponent_pool=members)
    lib = env._lib
    launches = env.launch_count()

    def end(*vals):
        def f(p):
            for k, v in enumerate(vals):
                p.end[k] = v
        return f

    def setattr_(name, value):
        return lambda o: setattr(o, name, value)

    cases = [
        (None, setattr_("struct_size", C.sizeof(_capi.FgOpponentPool) - 8), "struct_size"),
        (None, setattr_("count", 0), "count"),
        (None, setattr_("count", 17), "count"),
        (None, end(100, 256, 640), "multiple of FG_POOL_BLOCK"),         # misaligned
        (None, end(256, 128, 640), "non-decreasing"),                    # decreasing
        (None, end(128, 256, 512), "end[count - 1] must be num_envs"),   # short
        (None, end(128, 256, 768), "at most num_envs"),                  # beyond the batch
        (None, lambda p: setattr(p.member[2], "w3", None), "null member"),
        (None, lambda p: setattr(p.member[1], "w2", p.member[1].w2 + 4), "16-byte aligned"),
        (None, lambda p: setattr(p, "stats", p.stats + 4), "8-byte aligned"),
        (setattr_("hidden", 48), None, "hidden size"),
        (setattr_("actions_p2", None), None, "null pointer"),
        (setattr_("struct_size", 8), None, "fg_rollout_buffers"),
    ]
    for r_edit, pool_edit, msg in cases:
        rc, err = _raw_pool_call(col, r_edit, pool_edit)
        assert rc == -1 and msg in err, (msg, rc, err)
    rc = lib.fg_rollout_mlp_pool(env._handle, None, None, env._stream())
    assert rc == -1 and "fg_opponent_pool is null" in lib.fg_last_error().decode()
    assert env.launch_count() == launches                            # nothing was launched
    # a handle whose P2 is the in-game bot cannot take a pool
    bot_env = FootsiesEnv(num_envs=n, device=dev, seed=3)
    bot_col = RolloutCollector(bot_env, p1, horizon=8, seed=17)
    bot_col.actions_p2 = col.actions_p2; bot_col.logp_p2 = col.logp_p2
    bot_col.opponent_pool, bot_col.opponent_ranges, bot_col._pool_stats = members, col.opponent_ranges, col._pool_stats
    rc, err = _raw_pool_call(bot_col)
    assert rc == -1 and "p2_bot = 0" in err, err
    # and the valid call goes through
    rc, err = _raw_pool_call(col)
    assert rc == 0, err
    torch.cuda.synchronize()
    assert env.launch_count() == launches + 1


@pytest.mark.gpu
def test_collector_rejects_what_the_pool_cannot_run():
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    p1, m = _mlp(64, dev), _mlp(64, dev)
    sp = FootsiesEnv(num_envs=256, device=dev, seed=3, opponent="self_play")
    with pytest.raises(ValueError):
        RolloutCollector(sp, p1, horizon=8, opponent_policy=m, opponent_pool=[m])
    with pytest.raises(ValueError):
        RolloutCollector(FootsiesEnv(num_envs=256, device=dev, seed=3), p1, horizon=8, opponent_pool=[m])   # bot P2
    with pytest.raises(ValueError):
        RolloutCollector(sp, p1, horizon=8, opponent_pool=[_mlp(32, dev)])                                # hidden
    with pytest.raises(ValueError):
        RolloutCollector(sp, p1, horizon=8, opponent_pool=[m] * 17)
    with pytest.raises(ValueError):
        RolloutCollector(sp, p1, horizon=8, opponent_pool=[torch.nn.Linear(8, 8).to(dev)])
    with pytest.raises(ValueError):
        RolloutCollector(sp, p1, horizon=8, opponent_pool=[m], fused="step")
    with pytest.raises(ValueError):
        RolloutCollector(FootsiesEnv(num_envs=256, device=dev, seed=3, opponent="self_play", autoreset=False), p1,
                         horizon=8, opponent_pool=[m])
    col = RolloutCollector(sp, p1, horizon=8, opponent_pool=[m, m])
    with pytest.raises(ValueError):
        col.assign_opponents([1, 2, 3])
    with pytest.raises(ValueError):
        col.assign_opponents([0, 0])
    assert col.assign_opponents([0, 1]) == [(0, 0), (0, 256)]


@pytest.mark.gpu
def test_one_mebibattle_with_sixteen_members():
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    torch.manual_seed(16)
    n = 1 << 20
    p1 = _mlp(64, dev)
    members = [_mlp(64, dev) for _ in range(16)]
    env = FootsiesEnv(num_envs=n, device=dev, seed=3, opponent="self_play")
    col = RolloutCollector(env, p1, horizon=64, seed=17, opponent_pool=members, mirror_opponent=True)
    shares = list(range(1, 17))
    ranges = col.assign_opponents(shares)
    start = _stat4(env)
    done_count = np.zeros(16, dtype=np.int64)
    for _ in range(2):
        out = col.collect()
        per_battle = out["dones"].sum(0).cpu().numpy()
        done_count += [per_battle[s:e].sum() for s, e in ranges]
    st = col.opponent_pool_stats().cpu().numpy()
    assert np.array_equal(st.sum(0), _stat4(env) - start)
    assert (st[:, 0] == st[:, 1:].sum(1)).all() and (st[:, 0] > 0).all()
    assert np.array_equal(st[:, 0], done_count)            # one finished episode per done flag of the member's range
    assert st[15, 0] > st[0, 0]                             # 16 times the battles, more finished episodes
