"""The in-game bot as an opponent-pool member (fg_rollout_mlp_pool_bot, RolloutCollector(opponent_pool=[..., "bot"])).

CPU: the entry point is exported with the header's signature, and null handles / pools are refused.  GPU: every range of
a pool rollout equals, bit for bit, a twin env of just those battles that holds the same state (planes copied, the same
carried-over observation row, policy-step counter and first_env_index) run by the single-opponent kernel: a bot twin
(opponent="bot") for the bot's range, a self-play twin with that member as P2 for the others.  The twins are rebuilt
from the state copied just before every collect, so ranges may move between collects, in mid-episode."""
import ctypes as C

import numpy as np
import pytest
import torch

KEYS = ("obs", "actions", "logp", "rewards", "dones", "last_obs")


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_pool_bot_entry_point_is_exported_and_bound():
    from footsies_gym_b200 import _capi
    assert "fg_rollout_mlp_pool_bot" in _capi.EXPORTS
    lib = _capi.load()
    f = lib.fg_rollout_mlp_pool_bot
    assert f.restype is C.c_int32
    assert f.argtypes == [C.c_void_p, C.POINTER(_capi.FgRolloutBuffers), C.POINTER(_capi.FgOpponentPool), C.c_int32,
                          C.c_void_p]


def test_pool_bot_refuses_null_handle_and_null_pool():
    from footsies_gym_b200 import _capi
    lib = _capi.load()
    r = _capi.FgRolloutBuffers(struct_size=C.sizeof(_capi.FgRolloutBuffers), hidden=64, horizon=8)
    pool = _capi.FgOpponentPool(struct_size=C.sizeof(_capi.FgOpponentPool), count=1)
    assert lib.fg_rollout_mlp_pool_bot(None, C.byref(r), None, 0, None) == -1
    assert b"fg_opponent_pool is null" in lib.fg_last_error()
    bad = _capi.FgOpponentPool(struct_size=8, count=1)
    assert lib.fg_rollout_mlp_pool_bot(None, C.byref(r), C.byref(bad), 0, None) == -1
    assert b"struct_size" in lib.fg_last_error()
    assert lib.fg_rollout_mlp_pool_bot(None, C.byref(r), C.byref(pool), 0, None) == -1     # null handle
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


def _pool_env(n, dense=True, frame_skip=1, skip=False, seed=3):
    from footsies_gym_b200 import FootsiesEnv
    return FootsiesEnv(num_envs=n, device=_dev(), seed=seed, opponent="self_play", dense_reward=dense,
                       frame_skip=frame_skip, skip_unactionable=skip)


def _twin(env, col, m, s, e, horizon=None):
    """A single-opponent env + collector holding battles [s, e) of `env` / `col` as they are now."""
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    member = col.opponent_pool[m]
    bot = _is_bot(member)
    tenv = FootsiesEnv(num_envs=e - s, device=env.device, first_env_index=s, opponent="bot" if bot else "self_play",
                       dense_reward=env.dense_reward, frame_skip=env.frame_skip, skip_unactionable=env.skip_unactionable)
    kw = {} if bot else dict(opponent_policy=member, mirror_opponent=col.mirror_opponent)
    h = horizon or col.horizon
    tcol = RolloutCollector(tenv, col.policy, horizon=h, use_cuda_graph=False, seed=col._seed, **kw)
    assert tcol.mode == "horizon"
    tenv.state.copy_(env.state[:, s:e])
    tcol.obs[h].copy_(col.obs[col.horizon][s:e])
    tcol._drawn.copy_(col._drawn)
    return tenv, tcol


def _collect_against_twins(env, col, shares_per_round):
    """One pool collect per entry of shares_per_round (ranges re-assigned before it), every non-empty range compared
    with its twin built from the state just before the collect.  Returns the pool-stats delta of each round."""
    deltas = []
    for r, shares in enumerate(shares_per_round):
        ranges = col.assign_opponents(shares)
        twins = {}
        for m, (s, e) in enumerate(ranges):
            if s < e:
                tenv, tcol = _twin(env, col, m, s, e)
                twins[m] = (tenv, tcol, tenv.stats.clone())
        torch.cuda.synchronize()
        held_p2 = env.get_state()["actor_input"][:, 1].copy()
        pool0, handle0 = col.opponent_pool_stats(), env.stats.clone()
        out = col.collect()
        touts = {m: t[1].collect() for m, t in twins.items()}
        torch.cuda.synchronize()
        dpool = (col.opponent_pool_stats() - pool0).cpu().numpy()
        dhandle = (env.stats - handle0).cpu().numpy()
        state = env.get_state()
        for m, (s, e) in enumerate(ranges):
            if s == e:
                assert not dpool[m].any(), (r, m)
                continue
            tenv, tcol, tstats0 = twins[m]
            tout = touts[m]
            for k in KEYS:
                assert torch.equal(out[k][s:e] if k == "last_obs" else out[k][:, s:e], tout[k]), (r, m, k)
            if _is_bot(col.opponent_pool[m]):
                assert torch.equal(out["logp_p2"][:, s:e], torch.zeros_like(out["logp_p2"][:, s:e])), (r, m)
                assert np.array_equal(out["actions_p2"][0, s:e].cpu().numpy(), held_p2[s:e]), (r, m)
            else:
                assert torch.equal(out["actions_p2"][:, s:e], tout["actions_p2"]), (r, m)
                assert torch.equal(out["logp_p2"][:, s:e], tout["logp_p2"]), (r, m)
            assert state[s:e].tobytes() == tenv.get_state().tobytes(), (r, m)
            assert torch.equal(env.info_frame[s:e], tenv.info_frame), (r, m)
            assert np.array_equal(dpool[m], (tenv.stats - tstats0)[:4].cpu().numpy()), (r, m, dpool[m])
        # the members' counters add up to what the handle counted
        assert np.array_equal(dpool.sum(0), dhandle[:4]), (r, dpool.sum(0), dhandle[:4])
        assert (dpool[:, 0] == dpool[:, 1:].sum(1)).all()
        deltas.append(dpool)
    return deltas


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [32, 64, 128])
def test_bot_alone_equals_a_bot_env(hidden):
    """opponent_pool=["bot"] on a self-play env against a p2_bot = 1 twin of the whole batch, over 2 horizons: every
    output, the state planes, info_frame, the handle's statistics and the bot's pool row."""
    from footsies_gym_b200.rollout import RolloutCollector
    torch.manual_seed(hidden)
    n, horizon = 1000, 130
    env = _pool_env(n)
    col = RolloutCollector(env, _mlp(hidden, env.device), horizon=horizon, use_cuda_graph=False, seed=17,
                           opponent_pool=["bot"])
    assert col.mode == "horizon" and col.opponent_ranges == [(0, n)]
    tenv, tcol = _twin(env, col, 0, 0, n)
    s0, t0 = env.stats.clone(), tenv.stats.clone()
    for r in range(2):
        out, tout = col.collect(), tcol.collect()
        torch.cuda.synchronize()
        for k in KEYS:
            assert torch.equal(out[k], tout[k]), (r, k)
        assert torch.equal(out["logp_p2"], torch.zeros_like(out["logp_p2"]))
        assert torch.equal(env.state, tenv.state), r
        assert torch.equal(env.info_frame, tenv.info_frame), r
        assert torch.equal(env.stats - s0, tenv.stats - t0), r
        assert torch.equal(col.opponent_pool_stats()[0], (tenv.stats - t0)[:4]), r
    assert out["dones"].any() and int(col.opponent_pool_stats()[0, 0]) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,n,pool,shares,dense,frame_skip,skip,mirror", [
    (64, 1000, [0, "bot", 2, 3], [1, 2, 0, 1], True, 1, False, True),      # bot in the middle, an empty range after it
    (64, 777, [0, 1, 2, "bot"], [0, 1, 1, 1], False, 3, False, False),     # bot as the ragged tail, sparse, frame skip
    (64, 1000, [0, "bot", 2, 3], [1, 0, 1, 1], True, 1, False, True),      # the bot's range empty
    (32, 1000, ["bot", 1, 2, 3], [1, 2, 0, 1], True, 1, True, False),      # fused frame skipping
    (32, 555, [0, "bot", 2], [2, 1, 1], False, 1, False, True),
    (128, 1000, [0, 1, "bot", 3], [1, 2, 1, 1], True, 1, False, False),    # H = 128: the FFMA kernel
    (128, 700, [0, 1, "bot"], [1, 1, 1], False, 3, True, True),
])
def test_mixed_pool_ranges_equal_their_twins(hidden, n, pool, shares, dense, frame_skip, skip, mirror):
    from footsies_gym_b200.rollout import RolloutCollector
    torch.manual_seed(hidden * 7 + n)
    env = _pool_env(n, dense=dense, frame_skip=frame_skip, skip=skip)
    members = [m if _is_bot(m) else _mlp(hidden, env.device) for m in pool]
    col = RolloutCollector(env, _mlp(hidden, env.device), horizon=150, use_cuda_graph=False, seed=17,
                           opponent_pool=members, mirror_opponent=mirror)
    deltas = _collect_against_twins(env, col, [shares, shares])
    assert sum(d[:, 0].sum() for d in deltas) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,n,pool,shares,skip", [
    (64, 1000, [0, "bot", 2, 3], [3, 2, 0, 1], False),
    (32, 700, [0, 1, 2, "bot"], [1, 1, 0, 2], True),
])
def test_mixed_pool_with_32_battle_warps(monkeypatch, hidden, n, pool, shares, skip):
    """The 32-battle-warp shape (128-battle CTAs, selected from 131 072 battles up) forced onto small batches."""
    from footsies_gym_b200.rollout import RolloutCollector
    monkeypatch.setenv("FOOTSIES_B200_ROLLOUT_MT", "2")
    torch.manual_seed(n)
    env = _pool_env(n, skip=skip)
    members = [m if _is_bot(m) else _mlp(hidden, env.device) for m in pool]
    col = RolloutCollector(env, _mlp(hidden, env.device), horizon=130, use_cuda_graph=False, seed=17,
                           opponent_pool=members, mirror_opponent=True)
    _collect_against_twins(env, col, [shares, shares])


@pytest.mark.gpu
def test_mixed_pool_at_the_size_that_selects_32_battle_warps():
    """131 072 + 300 battles: the pool launch picks 128-battle CTAs by itself, the smaller twins 64-battle CTAs."""
    from footsies_gym_b200.rollout import RolloutCollector
    torch.manual_seed(131)
    env = _pool_env(131072 + 300)
    members = [_mlp(64, env.device), "bot", _mlp(64, env.device), _mlp(64, env.device)]
    col = RolloutCollector(env, _mlp(64, env.device), horizon=64, use_cuda_graph=False, seed=17,
                           opponent_pool=members, mirror_opponent=True)
    _collect_against_twins(env, col, [[1, 1, 1, 1], [1, 1, 1, 1]])


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [64, 128])
def test_reassignment_moves_battles_into_and_out_of_the_bot_range_mid_episode(hidden):
    from footsies_gym_b200.rollout import RolloutCollector
    torch.manual_seed(33)
    n = 1024
    env = _pool_env(n)
    members = [_mlp(hidden, env.device), "bot", _mlp(hidden, env.device)]
    col = RolloutCollector(env, _mlp(hidden, env.device), horizon=90, use_cuda_graph=False, seed=17,
                           opponent_pool=members, mirror_opponent=True)
    # [0, 384) [384, 640) [640, 1024) -> [0, 128) [128, 512) [512, 1024) -> [0, 640) [640, 768) [768, 1024)
    deltas = _collect_against_twins(env, col, [[3, 2, 3], [1, 3, 4], [5, 1, 2]])
    assert deltas[1][1, 0] > 0


@pytest.mark.gpu
def test_bot_actions_p2_are_its_held_input_before_each_step():
    """In the bot's battles actions_p2[t] is the input a bot twin holds before step t, read by a horizon-1 twin between
    its collects; logp_p2 is exactly 0."""
    from footsies_gym_b200.rollout import RolloutCollector
    torch.manual_seed(4)
    n, horizon = 640, 40
    env = _pool_env(n, frame_skip=1)
    members = [_mlp(64, env.device), "bot"]
    col = RolloutCollector(env, _mlp(64, env.device), horizon=horizon, use_cuda_graph=False, seed=17,
                           opponent_pool=members)
    col.collect()                                       # start from mid-episode battles
    s, e = col.opponent_ranges[1]
    tenv, tcol = _twin(env, col, 1, s, e, horizon=1)
    out = col.collect()
    held, acts = [], []
    for t in range(horizon):
        torch.cuda.synchronize()
        held.append(tenv.get_state()["actor_input"][:, 1].copy())
        acts.append(tcol.collect()["actions"][0].clone())
    torch.cuda.synchronize()
    assert torch.equal(out["actions"][:, s:e], torch.stack(acts))
    assert np.array_equal(out["actions_p2"][:, s:e].cpu().numpy(), np.stack(held).astype(np.uint8))
    assert (out["logp_p2"][:, s:e] == 0).all()
    assert len(np.unique(np.stack(held))) > 1


@pytest.mark.gpu
def test_adding_the_bot_leaves_every_other_range_unchanged():
    from footsies_gym_b200.rollout import RolloutCollector
    torch.manual_seed(8)
    n, horizon = 1000, 120
    p1 = _mlp(64, _dev())
    nets = [_mlp(64, _dev()) for _ in range(4)]
    shares = [1, 2, 1, 1]
    outs, states, cols = [], [], []
    for with_bot in (False, True):
        env = _pool_env(n)
        pool = list(nets)
        if with_bot:
            pool[1] = "bot"
        col = RolloutCollector(env, p1, horizon=horizon, use_cuda_graph=False, seed=17, opponent_pool=pool,
                               mirror_opponent=True)
        col.assign_opponents(shares)
        o = [{k: v.clone() for k, v in col.collect().items()} for _ in range(2)]
        torch.cuda.synchronize()
        outs.append(o); states.append(env.get_state()); cols.append(col)
    s, e = cols[0].opponent_ranges[1]
    assert cols[1].opponent_ranges == cols[0].opponent_ranges and s < e
    for r in range(2):
        for k in KEYS + ("actions_p2", "logp_p2"):
            a, b = outs[0][r][k], outs[1][r][k]
            if k == "last_obs":
                assert torch.equal(a[:s], b[:s]) and torch.equal(a[e:], b[e:]), (r, k)
            else:
                assert torch.equal(a[:, :s], b[:, :s]) and torch.equal(a[:, e:], b[:, e:]), (r, k)
                assert not torch.equal(a[:, s:e], b[:, s:e]) or k == "dones", (r, k)
    assert states[0][:s].tobytes() == states[1][:s].tobytes() and states[0][e:].tobytes() == states[1][e:].tobytes()
    p0, p1s = cols[0].opponent_pool_stats().cpu().numpy(), cols[1].opponent_pool_stats().cpu().numpy()
    assert np.array_equal(np.delete(p0, 1, 0), np.delete(p1s, 1, 0))


def _raw_bot_call(col, bot_member, pool_edit=None):
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
    if pool_edit:
        pool_edit(pool)
    lib = env._lib
    rc = lib.fg_rollout_mlp_pool_bot(env._handle, C.byref(r), C.byref(pool), bot_member, env._stream())
    return rc, lib.fg_last_error().decode()


@pytest.mark.gpu
def test_abi_and_collector_rejections():
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    n = 640
    p1 = _mlp(64, dev)
    members = [_mlp(64, dev), "bot", _mlp(64, dev)]
    env = _pool_env(n)
    col = RolloutCollector(env, p1, horizon=8, seed=17, opponent_pool=members)
    launches = env.launch_count()
    for bad in (-1, 3):
        rc, err = _raw_bot_call(col, bad)
        assert rc == -1 and "bot_member" in err, (bad, err)
    rc, err = _raw_bot_call(col, 1, lambda p: setattr(p.member[2], "w3", None))     # a network member without weights
    assert rc == -1 and "null member" in err, err
    rc, err = _raw_bot_call(col, 0)                                                 # member 1 is now a null network
    assert rc == -1 and "null member" in err, err
    assert env.launch_count() == launches                                           # nothing was launched
    # a handle whose P2 is already the in-game bot
    bot_env = FootsiesEnv(num_envs=n, device=dev, seed=3)
    bot_col = RolloutCollector(bot_env, p1, horizon=8, seed=17)
    bot_col.actions_p2 = col.actions_p2; bot_col.logp_p2 = col.logp_p2
    bot_col.opponent_pool, bot_col.opponent_ranges, bot_col._pool_stats = members, col.opponent_ranges, col._pool_stats
    bot_col._pool_bot = 1
    bot_launches = bot_env.launch_count()
    rc, err = _raw_bot_call(bot_col, 1)
    assert rc == -1 and "p2_bot = 0" in err, err
    assert bot_env.launch_count() == bot_launches
    # the valid call goes through, with the bot's weight pointers null
    rc, err = _raw_bot_call(col, 1)
    assert rc == 0, err
    torch.cuda.synchronize()
    assert env.launch_count() == launches + 1
    sp = _pool_env(256)
    with pytest.raises(ValueError):
        RolloutCollector(sp, p1, horizon=8, opponent_pool=[p1, "bot", "bot"])
    with pytest.raises(ValueError):
        RolloutCollector(sp, p1, horizon=8, opponent_policy=p1, opponent_pool=["bot"])
    with pytest.raises(ValueError):
        RolloutCollector(sp, p1, horizon=8, opponent_pool=["Bot"])


@pytest.mark.gpu
def test_one_mebibattle_with_sixteen_members_one_of_them_the_bot():
    from footsies_gym_b200.rollout import RolloutCollector
    torch.manual_seed(16)
    n = 1 << 20
    env = _pool_env(n)
    members = [_mlp(64, env.device) for _ in range(16)]
    members[5] = "bot"
    col = RolloutCollector(env, _mlp(64, env.device), horizon=64, seed=17, opponent_pool=members, mirror_opponent=True)
    ranges = col.assign_opponents(list(range(1, 17)))
    start = env.stats[:4].clone()
    done_count = np.zeros(16, dtype=np.int64)
    for _ in range(2):
        out = col.collect()
        per_battle = out["dones"].sum(0).cpu().numpy()
        done_count += [per_battle[s:e].sum() for s, e in ranges]
    st = col.opponent_pool_stats().cpu().numpy()
    assert np.array_equal(st.sum(0), (env.stats[:4] - start).cpu().numpy())
    assert (st[:, 0] == st[:, 1:].sum(1)).all() and (st[:, 0] > 0).all()
    assert np.array_equal(st[:, 0], done_count)
    s, e = ranges[5]
    assert (out["logp_p2"][:, s:e] == 0).all()
    win_rate = st[5, 1] / st[5, 0]
    assert st[5, 0] > 0 and np.isfinite(win_rate)
