"""Value estimates (fg_value_mlp, MLPValue) and GAE advantages / returns (fg_gae, compute_gae) computed on the GPU, alone
and inside RolloutCollector.  The GAE reference is the torch loop the PPO example ran before the library computed it."""
import ctypes as C
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

gpu = pytest.mark.gpu


def _dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    return torch.device("cuda:0")


def _reference_gae(rew, dones, v, gamma, lam):
    """The value-free part of examples/ppo_footsies.py's update before fg_gae, verbatim: v [h + 1, n] are the values."""
    a = types.SimpleNamespace(gamma=gamma, lam=lam)
    h, n = rew.shape
    dev = rew.device
    done = dones.float()
    with torch.no_grad():
        # an env that terminated at step t restarts by itself: the step after is the reset (reward 0); cut the
        # bootstrap at the terminal step
        adv = torch.zeros_like(rew)
        last = torch.zeros(n, device=dev)
        for t in range(h - 1, -1, -1):
            nonterm = 1.0 - done[t]
            delta = rew[t] + a.gamma * v[t + 1] * nonterm - v[t]
            last = delta + a.gamma * a.lam * nonterm * last
            adv[t] = last
        ret = adv + v[:h]
    return adv, ret


def _numpy_gae(rew, dones, v, gamma, lam):
    rew, done, v = rew.double().cpu().numpy(), dones.double().cpu().numpy(), v.double().cpu().numpy()
    h = rew.shape[0]
    adv = np.zeros_like(rew)
    last = np.zeros(rew.shape[1])
    for t in range(h - 1, -1, -1):
        nt = 1.0 - done[t]
        last = rew[t] + gamma * v[t + 1] * nt - v[t] + gamma * lam * nt * last
        adv[t] = last
    return adv, adv + v[:h]


def _random_rollout(h, n, dev, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    choice = torch.tensor([0.0, 0.3, -0.3, 1.0, -1.0], device=dev)
    rew = choice[torch.randint(0, 5, (h, n), generator=g, device=dev)]
    arbitrary = torch.rand((h, n), generator=g, device=dev) < 0.2
    rew = torch.where(arbitrary, torch.randn((h, n), generator=g, device=dev) * 2.0, rew).contiguous()
    dones = torch.rand((h, n), generator=g, device=dev) < 0.02
    dones[h - 1, :: 3] = True                          # a terminal last step too: no bootstrap from values[h] there
    values = torch.randn((h + 1, n), generator=g, device=dev) * 3.0
    return rew, dones.contiguous(), values


def _random_obs(rows, dev, seed):
    """Observations over the observation space: guard 0..3, move 0..14, move frame 0..55, position -4.6 .. 4.6."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    ri = lambda hi: torch.randint(0, hi, (rows,), generator=g, device=dev).float()   # noqa: E731
    pos = lambda: torch.rand(rows, generator=g, device=dev) * 9.2 - 4.6              # noqa: E731
    return torch.stack([ri(4), ri(4), ri(15), ri(15), ri(56), ri(56), pos(), pos()], dim=1).contiguous()


def _value_net(hidden, dev, seed, mul=3.0):
    from footsies_gym_b200.rollout import MLPValue
    torch.manual_seed(seed)
    v = MLPValue(hidden).to(dev)
    with torch.no_grad():
        for prm in v.net.parameters():
            prm.mul_(mul)                              # larger weights than the default init: saturating tanh, |V| of a few
    return v


# ---- 1. fg_gae against the example's own loop ----

@gpu
@pytest.mark.parametrize("h", [1, 7, 128, 300])
@pytest.mark.parametrize("n", [1, 1000, 16384 + 5])
def test_gae_equals_the_example_loop(h, n):
    from footsies_gym_b200.rollout import compute_gae
    dev = _dev()
    gamma, lam = 0.995, 0.95                           # the example's defaults
    rew, dones, values = _random_rollout(h, n, dev, seed=h * 100003 + n)
    adv, ret = compute_gae(rew, dones, values, gamma, lam)
    ref_adv, ref_ret = _reference_gae(rew, dones, values, gamma, lam)
    torch.cuda.synchronize()
    assert torch.equal(adv, ref_adv) and torch.equal(ret, ref_ret)
    # the same through uint8 dones, into caller-supplied outputs
    adv2, ret2 = torch.empty_like(rew), torch.empty_like(rew)
    out = compute_gae(rew, dones.to(torch.uint8), values, gamma, lam, advantages=adv2, returns=ret2)
    assert out[0] is adv2 and out[1] is ret2
    assert torch.equal(adv2, ref_adv) and torch.equal(ret2, ref_ret)
    # semantics against float64
    a64, r64 = _numpy_gae(rew, dones, values, gamma, lam)
    np.testing.assert_allclose(adv.cpu().numpy(), a64, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ret.cpu().numpy(), r64, rtol=1e-5, atol=1e-5)


@gpu
def test_gae_other_discounts_and_a_terminal_cut():
    """gamma * lambda is rounded from its double product; a done at t makes adv[t] = r[t] - v[t] exactly."""
    from footsies_gym_b200.rollout import compute_gae
    dev = _dev()
    rew, dones, values = _random_rollout(64, 4099, dev, seed=5)
    for gamma, lam in ((0.99, 0.95), (0.9, 1.0), (1.0, 0.0), (0.97, 0.9)):
        adv, ret = compute_gae(rew, dones, values, gamma, lam)
        ref_adv, ref_ret = _reference_gae(rew, dones, values, gamma, lam)
        assert torch.equal(adv, ref_adv) and torch.equal(ret, ref_ret), (gamma, lam)
    t = dones.nonzero()
    assert torch.equal(adv[t[:, 0], t[:, 1]], rew[t[:, 0], t[:, 1]] - values[t[:, 0], t[:, 1]])


# ---- 2. fg_value_mlp against MLPValue.forward ----

@gpu
@pytest.mark.parametrize("hidden", [32, 64])
@pytest.mark.parametrize("rows", [1, 15, 17, 10007, 129 * 16384])
def test_fused_values_match_torch(hidden, rows):
    dev = _dev()
    v = _value_net(hidden, dev, seed=hidden)
    obs = _random_obs(rows, dev, seed=rows)
    out = torch.full((rows,), float("nan"), device=dev)
    with torch.no_grad():
        ref = v(obs)
    v.fused_values(obs, out)
    torch.cuda.synchronize()
    err = float(((out - ref).abs() / (1.0 + ref.abs())).max())
    assert err <= 2e-5, err
    assert rows < 1000 or float(ref.abs().max()) > 0.5  # a value head that is not trivially flat


@gpu
def test_fused_values_of_a_rollout_shaped_block():
    """[horizon + 1, N, 8] in, [horizon + 1, N] out: the rows are the flattened leading dimensions."""
    dev = _dev()
    v = _value_net(64, dev, seed=2)
    obs = _random_obs(9 * 333, dev, seed=3).view(9, 333, 8)
    out = torch.empty((9, 333), device=dev)
    v.fused_values(obs, out)
    flat = torch.empty(9 * 333, device=dev)
    v.fused_values(obs.view(-1, 8), flat)
    assert torch.equal(out.view(-1), flat)


@gpu
@pytest.mark.parametrize("hidden", [32, 64])
def test_zero_output_weights_give_the_bias_exactly(hidden):
    dev = _dev()
    v = _value_net(hidden, dev, seed=7)
    with torch.no_grad():
        v.net[4].weight.zero_()
        v.net[4].bias.fill_(-1.2345678)
    obs = _random_obs(1000, dev, seed=1)
    out = torch.empty(1000, device=dev)
    v.fused_values(obs, out)
    assert torch.equal(out, v.net[4].bias.expand(1000))


@gpu
def test_fused_values_rejects_hidden_128():
    from footsies_gym_b200.rollout import MLPValue
    dev = _dev()
    v = MLPValue(128).to(dev)
    obs = _random_obs(100, dev, seed=1)
    with pytest.raises(ValueError):
        v.fused_values(obs, torch.empty(100, device=dev))


# ---- 3. RolloutCollector with a value network ----

def _collector_pair(n, horizon, value_factory, opponent=False, mirror=False):
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
    dev = _dev()
    torch.manual_seed(11)
    pol = MLPPolicy(64).to(dev)
    with torch.no_grad():
        for prm in pol.net.parameters():
            prm.mul_(2.0)
    val = value_factory(dev)
    cols = []
    for mode in ("step", "horizon"):
        env = FootsiesEnv(num_envs=n, device=dev, seed=3, opponent="self_play" if opponent else None)
        cols.append(RolloutCollector(env, pol, horizon=horizon, use_cuda_graph=False, fused=mode, seed=17, value=val,
                                     gamma=0.995, gae_lambda=0.95, opponent_policy=pol if opponent else None,
                                     mirror_opponent=mirror))
    assert [c.mode for c in cols] == ["step", "horizon"]
    return cols, val


@gpu
@pytest.mark.parametrize("opponent,mirror", [(False, False), (True, True)])
def test_collector_values_and_gae_step_vs_horizon(opponent, mirror):
    n, horizon = 1000, 130
    cols, val = _collector_pair(n, horizon, lambda dev: _value_net(64, dev, seed=4), opponent, mirror)
    for r in range(2):
        outs = [c.collect() for c in cols]
        torch.cuda.synchronize()
        for k in ("obs", "actions", "rewards", "dones", "last_obs", "values", "advantages", "returns"):
            assert torch.equal(outs[0][k], outs[1][k]), (r, k)
        out = outs[1]
        assert out["dones"].any()
        assert out["values"].shape == (horizon + 1, n) and out["advantages"].shape == (horizon, n)
        rows = torch.cat([out["obs"], out["last_obs"][None]], 0)
        fresh = torch.empty((horizon + 1, n), device=rows.device)
        val.fused_values(rows.contiguous(), fresh)
        assert torch.equal(out["values"], fresh), r
        ref_adv, ref_ret = _reference_gae(out["rewards"], out["dones"], out["values"], 0.995, 0.95)
        assert torch.equal(out["advantages"], ref_adv) and torch.equal(out["returns"], ref_ret), r


@gpu
def test_collector_with_a_torch_value_module():
    """Any callable value network: a plain nn.Sequential with output [N, 1] in the torch policy mode."""
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
    dev = _dev()
    torch.manual_seed(2)
    pol = MLPPolicy(64).to(dev)
    val = torch.nn.Sequential(torch.nn.Linear(8, 32), torch.nn.Tanh(), torch.nn.Linear(32, 1)).to(dev)
    n, horizon = 500, 40
    env = FootsiesEnv(num_envs=n, device=dev, seed=3)
    col = RolloutCollector(env, pol, horizon=horizon, use_cuda_graph=False, fused=False, value=val, gamma=0.99, gae_lambda=0.9)
    assert col.mode == "torch"
    out = col.collect()
    rows = torch.cat([out["obs"], out["last_obs"][None]], 0)
    with torch.no_grad():
        ref = val(rows.reshape(-1, 8)).squeeze(1).view(horizon + 1, n)
    torch.testing.assert_close(out["values"], ref, rtol=1e-6, atol=1e-6)
    ref_adv, ref_ret = _reference_gae(out["rewards"], out["dones"], out["values"], 0.99, 0.9)
    assert torch.equal(out["advantages"], ref_adv) and torch.equal(out["returns"], ref_ret)


@gpu
def test_collector_without_a_value_network_is_unchanged():
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
    dev = _dev()
    env = FootsiesEnv(num_envs=64, device=dev, seed=3)
    col = RolloutCollector(env, MLPPolicy(64).to(dev), horizon=8)
    out = col.collect()
    assert col.values is None and col.advantages is None and col.returns is None
    assert not {"values", "advantages", "returns"} & set(out)


# ---- 4. CUDA graph: in-place weight updates reach the next replay ----

@gpu
@pytest.mark.parametrize("hidden", [32, 64])
def test_cuda_graph_sees_in_place_value_updates(hidden):
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
    dev = _dev()
    torch.manual_seed(5)
    pol = MLPPolicy(64).to(dev)
    val = _value_net(hidden, dev, seed=6)
    n, horizon = 777, 50
    env = FootsiesEnv(num_envs=n, device=dev, seed=3, autoreset=True)
    col = RolloutCollector(env, pol, horizon=horizon, use_cuda_graph=True, fused="step", value=val, gamma=0.995, gae_lambda=0.95)
    first = {k: t.clone() for k, t in col.collect().items()}
    assert col._graph is not None
    with torch.no_grad():
        for prm in val.net.parameters():
            prm.mul_(-0.5).add_(0.01)
    out = col.collect()
    torch.cuda.synchronize()
    fresh = torch.empty((horizon + 1, n), device=dev)
    val.fused_values(col.obs, fresh)
    assert torch.equal(out["values"], fresh)
    stale = torch.empty_like(fresh)
    _value_net(hidden, dev, seed=6).fused_values(col.obs, stale)          # the weights before the update
    assert not torch.equal(out["values"], stale) and not torch.equal(out["obs"], first["obs"])
    ref_adv, ref_ret = _reference_gae(out["rewards"], out["dones"], out["values"], 0.995, 0.95)
    assert torch.equal(out["advantages"], ref_adv) and torch.equal(out["returns"], ref_ret)


# ---- 5. full size ----

@gpu
def test_full_size_rollout_with_values_and_gae():
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
    dev = _dev()
    torch.manual_seed(0)
    n, horizon = 1 << 20, 128
    env = FootsiesEnv(num_envs=n, device=dev, seed=0)
    col = RolloutCollector(env, MLPPolicy(64).to(dev), horizon=horizon, value=_value_net(64, dev, seed=1),
                           gamma=0.995, gae_lambda=0.95)
    assert col.mode == "horizon"
    out = col.collect()
    torch.cuda.synchronize()
    assert bool(torch.isfinite(out["values"]).all())
    ref_adv, ref_ret = _reference_gae(out["rewards"], out["dones"], out["values"], 0.995, 0.95)
    assert torch.equal(out["advantages"], ref_adv) and torch.equal(out["returns"], ref_ret)


# ---- 6. argument checks ----

@gpu
def test_compute_gae_and_fused_values_reject_bad_tensors():
    from footsies_gym_b200._capi import FootsiesLibraryError
    from footsies_gym_b200.rollout import compute_gae
    dev = _dev()
    h, n = 6, 40
    rew, dones, values = _random_rollout(h, n, dev, seed=1)
    bad = [
        (rew.double(), dones, values),                  # dtype
        (rew, dones.float(), values),
        (rew, dones, values.half()),
        (rew, dones, values[:h]),                       # shape
        (rew, dones[:, :-1], values),
        (rew[:, None], dones, values),
        (rew.cpu(), dones, values),                     # device
        (rew, dones, values.cpu()),
        (rew.t().contiguous().t(), dones, values),      # not contiguous
        (rew[:, :0], dones[:, :0], values[:, :0]),      # empty
        (rew[:0], dones[:0], values[:1]),
    ]
    for args in bad:
        with pytest.raises(ValueError):
            compute_gae(*args, 0.99, 0.95)
    with pytest.raises(ValueError):
        compute_gae(rew, dones, values, 0.99, 0.95, advantages=torch.empty((h, n + 1), device=dev))
    with pytest.raises(ValueError):
        compute_gae(rew, dones, values, 0.99, 0.95, returns=torch.empty((h, n), device=dev, dtype=torch.float64))
    v = _value_net(64, dev, seed=1)
    obs = _random_obs(n, dev, seed=1)
    for o, out in ((obs, torch.empty(n - 1, device=dev)), (obs.double(), torch.empty(n, device=dev)),
                   (obs, torch.empty(n, device=dev, dtype=torch.float64)), (obs[:, :7].contiguous(), torch.empty(n, device=dev)),
                   (obs.cpu(), torch.empty(n)), (obs[:, :4], torch.empty(n, device=dev)), (obs[:0], torch.empty(0, device=dev))):
        with pytest.raises((ValueError, FootsiesLibraryError)):
            v.fused_values(o, out)


def test_c_entry_points_reject_null_and_empty_arguments():
    """fg_value_mlp / fg_gae validate their arguments before touching the device (runs without a GPU)."""
    from footsies_gym_b200 import _capi
    lib = _capi.load()
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    w = [p] * 8
    for i in range(8):
        args = list(w)
        args[i] = None
        assert lib.fg_value_mlp(*args, 64, 10, p, None) == -1
    assert lib.fg_value_mlp(*w, 64, 10, None, None) == -1
    assert lib.fg_value_mlp(*w, 64, 0, p, None) == -1
    assert lib.fg_value_mlp(*w, 128, 10, p, None) == -1
    assert b"hidden size" in lib.fg_policy_last_error()
    assert lib.fg_value_mlp(*w, 16, 10, p, None) == -1
    assert lib.fg_gae(p, p, p, 4, 0, 0.99, 0.95, p, p, None) == -1
    assert lib.fg_gae(p, p, p, 0, 4, 0.99, 0.95, p, p, None) == -1
    for i in (0, 1, 2, 7, 8):
        args = [p, p, p, 4, 4, 0.99, 0.95, p, p, None]
        args[i] = None
        assert lib.fg_gae(*args) == -1
    assert b"fg_gae" in lib.fg_policy_last_error()


def test_python_wrappers_reject_bad_arguments_without_a_gpu():
    from footsies_gym_b200.rollout import MLPValue, compute_gae
    rew = torch.zeros((4, 10))
    with pytest.raises(ValueError):
        compute_gae(rew, torch.zeros((4, 10), dtype=torch.bool), torch.zeros((5, 10)), 0.99, 0.95)    # not on a GPU
    with pytest.raises(ValueError):
        compute_gae(torch.zeros(10), torch.zeros(10, dtype=torch.bool), torch.zeros(11), 0.99, 0.95)  # not [h, n]
    with pytest.raises(ValueError):
        compute_gae(torch.zeros((0, 10)), torch.zeros((0, 10), dtype=torch.bool), torch.zeros((1, 10)), 0.99, 0.95)
    with pytest.raises(ValueError):
        MLPValue(128).fused_values(torch.zeros((4, 8)), torch.zeros(4))
    with pytest.raises(ValueError):
        MLPValue(64).fused_values(torch.zeros((4, 8)), torch.zeros(4))                                  # not on a GPU
    assert MLPValue(32)(torch.zeros((3, 8))).shape == (3,)
