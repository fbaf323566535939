"""On-device rollout collection (BASELINE.json configs[4]: an MLP policy consuming the observation tensor in place).

The reference's training loops step one socket-connected game per process and move every observation through JSON
(footsies.py:518-570, 633-661).  Here a whole horizon of policy-forward -> sample -> FootsiesEnv.step for N battles is
a sequence of device kernels with no host round trip, captured once into a CUDA graph and replayed.

Three policy paths:
  * any torch callable `policy(obs[N, 8]) -> logits[N, 8]` (a dozen small torch kernels per step);
  * `MLPPolicy`, fused="step": one hand-written kernel per step (csrc/policy_kernel.cu, fg_policy_mlp_sample) does
    scale -> 8-H-H-8 tanh MLP -> log-softmax -> sample, and the rollout needs no copies at all: the step kernel is
    re-bound, per captured launch, to write observation t + 1, reward t and done t straight into the rollout buffers,
    and the policy kernel reads observation t from there.  Per step: 2 launches (policy, simulator step).
  * `MLPPolicy`, fused="horizon" (the default whenever the env qualifies: P1 = policy, P2 = in-game bot or a second
    MLPPolicy given as `opponent_policy` (self-play), autoreset, no step mask): ONE launch per horizon (csrc/rollout_kernel.cu, fg_rollout_mlp) -- a CTA keeps its 64 battles in
    registers from the first step to the last and alternates policy inference and the frame update; bit-identical
    to the per-step path.  Self-play against an opponent pool (`opponent_pool=[...]`: up to 16 P2 networks, each on its
    own range of battles, with results per member) runs on this path only (fg_rollout_mlp_pool); one member may be the
    in-game bot, "bot" (fg_rollout_mlp_pool_bot).

An env with frame_delay > 0 runs on every path: the policies act on the delayed observation, as the reference's agent and
its `opponent(obs, info)` callable do (footsies.py:129-131, 533-535), and obs[t + 1] of the rollout buffer receives the
delayed observation; rewards and dones are not delayed.  The whole-horizon kernel advances the env's queue inside its one
launch (fg_rollout_mlp_delayed); the per-step paths run env.step_bound() (which advances the queue with
fg_delay_ring_step) and copy the delayed observation into the buffer, without a CUDA graph: the ring position is a host
integer that a captured launch would replay frozen.

With a value network (`value=`), collect() also returns what a PPO update consumes besides the rollout itself: the values
of all horizon + 1 observation rows (one fg_value_mlp launch for an `MLPValue` with hidden 32 / 64, else one call of the
torch callable) and GAE advantages / returns (one fg_gae launch), after the rollout on the same stream.

PyTorch is plumbing here (parameters, buffers, CUDA graph); the simulator step inside the loop is fg_step.
"""
import ctypes as C
import math
from typing import Callable, List, Optional, Sequence, Tuple

import torch

from . import _capi
from .env import FootsiesEnv

# FootsiesNormalized scales (wrappers/normalization.py:28-55): guard / 3, move index / 14, move_frame / 55, position / 4.6
_OBS_SCALE = (1 / 3.0, 1 / 3.0, 1 / 14.0, 1 / 14.0, 1 / 55.0, 1 / 55.0, 1 / 4.6, 1 / 4.6)


class MLPPolicy(torch.nn.Module):
    """8 -> hidden -> hidden -> 8 logits over the 2^3 input combinations (wrappers/action_comb_disc.py:13-18).
    hidden in {32, 64, 128} can be run by the fused inference kernel."""

    def __init__(self, hidden: int = 64):
        super().__init__()
        self.hidden = int(hidden)
        self.register_buffer("scale", torch.tensor(_OBS_SCALE, dtype=torch.float32))
        self.net = torch.nn.Sequential(torch.nn.Linear(8, hidden), torch.nn.Tanh(), torch.nn.Linear(hidden, hidden),
                                       torch.nn.Tanh(), torch.nn.Linear(hidden, 8))

    def forward(self, obs: torch.Tensor) -> torch.Tensor:
        return self.net(obs * self.scale)

    def fused_sample(self, obs: torch.Tensor, actions: torch.Tensor, logp: Optional[torch.Tensor], seed: int, counter: int,
                     counter_base: Optional[torch.Tensor] = None, obs_copy: Optional[torch.Tensor] = None,
                     first_env_index: int = 0):
        """One launch of fg_policy_mlp_sample on the current stream: actions (uint8 [N]) and logp (float32 [N]) are
        written in place; sampling is a pure function of (seed, counter + counter_base[0], first_env_index + env index)
        -- the global battle index, so that shards of one job draw what the whole batch would; counter_base is an optional
        int64 device tensor (bumped between CUDA-graph replays)."""
        lib = _capi.load()
        l1, l2, l3 = self.net[0], self.net[2], self.net[4]
        ts = [obs, self.scale, l1.weight, l1.bias, l2.weight, l2.bias, l3.weight, l3.bias]
        for t in ts:
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != obs.device:
                raise ValueError("fused policy inference needs contiguous float32 tensors on one device")
        if actions.dtype != torch.uint8 or not actions.is_contiguous():
            raise ValueError("actions must be a contiguous uint8 tensor")
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())   # noqa: E731
        rc = lib.fg_policy_mlp_sample(*[ptr(t) for t in ts], self.hidden, obs.shape[0], int(seed) & (2**64 - 1),
                                      int(counter), ptr(counter_base), ptr(actions), ptr(logp), ptr(obs_copy),
                                      int(first_env_index), C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream))
        if rc != 0:
            raise _capi.FootsiesLibraryError(lib.fg_policy_last_error().decode())

    def fused_sample_p2(self, obs: torch.Tensor, actions: torch.Tensor, logp: Optional[torch.Tensor], seed: int, counter: int,
                        counter_base: Optional[torch.Tensor] = None, mirror: bool = False, first_env_index: int = 0):
        """fused_sample for a policy that drives P2 (fg_policy_mlp_sample_p2): with mirror=True it is fed the mirrored
        observation (per-player fields swapped, positions negated) and its Left / Right bits are mirrored back, so that
        the network that plays P1 can play P2 as well."""
        lib = _capi.load()
        l1, l2, l3 = self.net[0], self.net[2], self.net[4]
        ts = [obs, self.scale, l1.weight, l1.bias, l2.weight, l2.bias, l3.weight, l3.bias]
        for t in ts:
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != obs.device:
                raise ValueError("fused policy inference needs contiguous float32 tensors on one device")
        if actions.dtype != torch.uint8 or not actions.is_contiguous():
            raise ValueError("actions must be a contiguous uint8 tensor")
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())   # noqa: E731
        rc = lib.fg_policy_mlp_sample_p2(*[ptr(t) for t in ts], self.hidden, obs.shape[0], int(seed) & (2**64 - 1),
                                         int(counter), ptr(counter_base), ptr(actions), ptr(logp), int(bool(mirror)),
                                         int(first_env_index), C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream))
        if rc != 0:
            raise _capi.FootsiesLibraryError(lib.fg_policy_last_error().decode())


class MLPValue(torch.nn.Module):
    """Value network 8 -> hidden -> hidden -> 1 (tanh) on the observation times the same `scale` as MLPPolicy.
    hidden in {32, 64} can be run by the fused kernel (fused_values); any hidden size runs as a torch module."""

    def __init__(self, hidden: int = 64):
        super().__init__()
        self.hidden = int(hidden)
        self.register_buffer("scale", torch.tensor(_OBS_SCALE, dtype=torch.float32))
        self.net = torch.nn.Sequential(torch.nn.Linear(8, hidden), torch.nn.Tanh(), torch.nn.Linear(hidden, hidden),
                                       torch.nn.Tanh(), torch.nn.Linear(hidden, 1))

    def forward(self, obs: torch.Tensor) -> torch.Tensor:
        """obs [N, 8] -> values [N]"""
        return self.net(obs * self.scale).squeeze(-1)

    def fused_values(self, obs_rows: torch.Tensor, out: torch.Tensor):
        """One launch of fg_value_mlp on the current stream: out (float32, one value per observation row) receives the
        values of obs_rows (float32 [..., 8], e.g. a whole [horizon + 1, N, 8] rollout buffer).  Agrees with forward() to
        ~1e-5 relative (tensor-core path with split operands, not torch's fp32 GEMM)."""
        if self.hidden not in (32, 64):
            raise ValueError(f"fused_values needs hidden 32 or 64 (got {self.hidden}): use the module itself")
        lib = _capi.load()
        l1, l2, l3 = self.net[0], self.net[2], self.net[4]
        ts = [obs_rows, self.scale, l1.weight, l1.bias, l2.weight, l2.bias, l3.weight, l3.bias]
        for t in ts:
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != obs_rows.device:
                raise ValueError("fused value inference needs contiguous float32 tensors on one device")
        if obs_rows.device.type != "cuda":
            raise ValueError("fused value inference needs CUDA tensors")
        if obs_rows.dim() < 1 or obs_rows.shape[-1] != 8:
            raise ValueError("obs_rows must have 8 features in its last dimension")
        rows = obs_rows.numel() // 8
        if out.dtype != torch.float32 or not out.is_contiguous() or out.device != obs_rows.device or out.numel() != rows:
            raise ValueError(f"out must be a contiguous float32 tensor of {rows} values on the observations' device")
        rc = lib.fg_value_mlp(*[C.c_void_p(t.data_ptr()) for t in ts], self.hidden, rows, C.c_void_p(out.data_ptr()),
                              C.c_void_p(torch.cuda.current_stream(obs_rows.device).cuda_stream))
        if rc != 0:
            raise _capi.FootsiesLibraryError(lib.fg_policy_last_error().decode())


def compute_gae(rewards: torch.Tensor, dones: torch.Tensor, values: torch.Tensor, gamma: float, gae_lambda: float,
                advantages: Optional[torch.Tensor] = None, returns: Optional[torch.Tensor] = None):
    """GAE advantages and returns of a [horizon, N] rollout in one launch of fg_gae on the current stream.

    rewards float32 [h, N]; dones bool / uint8 [h, N] (a done at step t cuts the bootstrap from t + 1); values float32
    [h + 1, N] (values[h]: the observation after the last step); all contiguous on one CUDA device.  advantages / returns:
    optional float32 [h, N] outputs (allocated when None).  Returns (advantages, returns).  Bit-identical to the torch loop
        last = 0
        for t in reversed(range(h)):
            nonterm = 1.0 - dones[t].float()
            delta = rewards[t] + gamma * values[t + 1] * nonterm - values[t]
            last = delta + gamma * gae_lambda * nonterm * last
            advantages[t] = last
        returns = advantages + values[:h]"""
    if rewards.dim() != 2:
        raise ValueError("rewards must be [horizon, N]")
    h, n = rewards.shape
    if h == 0 or n == 0:
        raise ValueError("empty rollout")
    if rewards.device.type != "cuda":
        raise ValueError("compute_gae needs CUDA tensors")
    dev = rewards.device
    if advantages is None:
        advantages = torch.empty((h, n), dtype=torch.float32, device=dev)
    if returns is None:
        returns = torch.empty((h, n), dtype=torch.float32, device=dev)
    for name, t, dtypes, shape in (("rewards", rewards, (torch.float32,), (h, n)),
                                   ("dones", dones, (torch.bool, torch.uint8), (h, n)),
                                   ("values", values, (torch.float32,), (h + 1, n)),
                                   ("advantages", advantages, (torch.float32,), (h, n)),
                                   ("returns", returns, (torch.float32,), (h, n))):
        if t.dtype not in dtypes or tuple(t.shape) != shape or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"{name} must be a contiguous {' / '.join(str(d) for d in dtypes)} tensor of shape {shape} "
                             f"on {dev} (got {t.dtype} {tuple(t.shape)} on {t.device})")
    lib = _capi.load()
    ptr = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731
    # gamma * gae_lambda in double, then rounded once to fp32: what torch does with the Python scalar of the loop above
    rc = lib.fg_gae(ptr(rewards), ptr(dones), ptr(values), h, n, float(gamma), float(gamma) * float(gae_lambda),
                    ptr(advantages), ptr(returns), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    if rc != 0:
        raise _capi.FootsiesLibraryError(lib.fg_policy_last_error().decode())
    return advantages, returns


def mirror_obs(obs: torch.Tensor) -> torch.Tensor:
    """The observation [N, 8] as P2 sees it: per-player fields swapped, positions negated."""
    m = obs[:, [1, 0, 3, 2, 5, 4, 7, 6]].clone()
    m[:, 6:8] = -m[:, 6:8]
    return m


_MIRROR_ACTION = (0, 2, 1, 3, 4, 6, 5, 7)      # Left (1) <-> Right (2)
_P2_SEED_SALT = 0x5DEECE66D2F1A3B7


def opponent_ranges(num_envs: int, shares: Sequence[float]) -> List[Tuple[int, int]]:
    """Contiguous battle ranges [(start, end), ...], one per opponent-pool member, in proportion to non-negative `shares`.

    The num_envs // 128 whole blocks of FG_POOL_BLOCK = 128 battles are divided by largest remainder (ties go to the lower
    index); the battles left over after the last whole block go to the last member with a non-zero share, so that every
    boundary but the final num_envs is a multiple of 128 -- what fg_rollout_mlp_pool asks of fg_opponent_pool.end.  A member
    with share 0 gets an empty range.  The ranges cover 0 .. num_envs exactly once, in member order."""
    shares = [float(s) for s in shares]
    if not 1 <= len(shares) <= _capi.FG_POOL_MAX:
        raise ValueError(f"an opponent pool has 1 .. {_capi.FG_POOL_MAX} members (got {len(shares)})")
    if any(not math.isfinite(s) or s < 0 for s in shares) or sum(shares) <= 0:
        raise ValueError("opponent shares must be finite, non-negative and not all zero")
    if num_envs < 1:
        raise ValueError("num_envs must be positive")
    block = _capi.FG_POOL_BLOCK
    blocks = num_envs // block
    total = sum(shares)
    quota = [s / total * blocks for s in shares]
    count = [int(math.floor(q)) for q in quota]
    order = sorted((i for i in range(len(shares)) if shares[i] > 0), key=lambda i: (-(quota[i] - count[i]), i))
    for k in range(blocks - sum(count)):
        count[order[k % len(order)]] += 1
    last = max(i for i, s in enumerate(shares) if s > 0)
    ranges, start = [], 0
    for i, c in enumerate(count):
        end = num_envs if i >= last else start + c * block
        ranges.append((start, end))
        start = end
    return ranges


class RolloutCollector:
    """Collects `horizon` steps of (obs, action, log-prob, reward, done) for every env of one GPU, entirely on device.

    Buffers (overwritten by every collect()): obs [horizon + 1, N, 8] (obs[t] is what the policy saw at step t, obs[-1]
    the observation after the last step), actions uint8 [horizon, N], logp / rewards float32 [horizon, N], dones bool;
    with a value network also values float32 [horizon + 1, N] (of every obs row) and advantages / returns float32
    [horizon, N] (GAE with gamma, gae_lambda; see compute_gae).

    Opponent pool (`opponent_pool=[p2_0, p2_1, ...]`, self-play): P2 is played by up to 16 MLPPolicy networks at once, each
    on its own contiguous range of battles (`opponent_ranges`, set by assign_opponents), in the one launch per horizon of
    fg_rollout_mlp_pool.  A battle of member m's range draws exactly what it would draw against member m alone.  Results per
    member accumulate in opponent_pool_stats().  Members are ordinary modules, read at every collect(): a snapshot loaded
    with load_state_dict is played from the next collect() on, and the live `policy` may itself be a member.  Ranges only
    change between horizons, but a battle does not restart when they do: a battle re-assigned in mid-episode finishes that
    episode against its new member, and the result counts for the new member.

    One member may be the string "bot": the in-game BattleAI plays its range, bit for bit as a rollout on an
    opponent="bot" env holding the same battle state would (fg_rollout_mlp_pool_bot), so that e.g. past snapshots and the
    scripted opponent share one rollout and the win rate against the bot is a row of opponent_pool_stats().  In its
    battles actions_p2 holds the bot's input at the start of each step and logp_p2 is 0 (not a log-probability).  A battle
    moved into the bot's range continues its episode with empty bot queues and P2's last held input; the first round
    after env.reset() of a battle in the bot's range starts like such an entry (a self-play env's reset does not ask the
    bot for its Fight-transition input), every later round exactly as on a bot env.

    frame_delay > 0: every policy acts on the delayed observation the env shows (see the module docstring), and obs[0] of
    each collect() is what the env shows when it starts, so env.step() / env.reset() calls between collects are picked
    up.  The per-step paths ("step", "torch") run without a CUDA graph then, whatever use_cuda_graph says."""

    def __init__(self, env: FootsiesEnv, policy: Callable[[torch.Tensor], torch.Tensor], horizon: int = 128,
                 use_cuda_graph: bool = True, fused=None, seed: int = 0,
                 opponent_policy: Optional[Callable[[torch.Tensor], torch.Tensor]] = None, mirror_opponent: bool = False,
                 value: Optional[Callable[[torch.Tensor], torch.Tensor]] = None, gamma: float = 0.99, gae_lambda: float = 0.95,
                 opponent_pool: Optional[Sequence] = None):
        """fused: None / True = the most fused path available ("horizon", else "step", else torch ops for a policy that
        is not an MLPPolicy); False = torch ops; "step" / "horizon" = that path or an error.
        opponent_policy: a second policy for P2 (self-play rollouts; the env must take P2's actions from step(), i.e.
        opponent="self_play" / "remote").  It sees the same observation as the reference's `opponent(obs, info)`
        callable (footsies.py:522-527), or its mirror image with mirror_opponent=True (then `policy` itself can be passed
        again: one network plays both sides).  Its actions / log-probabilities are collected in actions_p2 / logp_p2.
        value: a value network, `value(obs[M, 8]) -> [M]` or `[M, 1]`; an MLPValue with hidden 32 / 64 runs on the fused
        kernel (fg_value_mlp).  The policy path is chosen as without it.  Values and advantages are P1's.
        opponent_pool: instead of opponent_policy, a list of 1 .. 16 MLPPolicy networks with `policy`'s hidden size that
        play P2 on separate ranges of battles (see the class docstring; equal shares until assign_opponents is called),
        each on the mirrored observation with mirror_opponent=True.  At most one entry may be the string "bot" (the in-game
        bot, as in FootsiesEnv(opponent="bot")); it counts as a member for shares and statistics, and mirror_opponent does
        not apply to it.  Needs an MLPPolicy `policy`, a self-play env with autoreset and no step mask: the whole-horizon
        kernel (fused=None / True / "horizon"); anything else is a ValueError."""
        if env.by_example:
            raise ValueError("the policy drives P1: create the env with by_example=False")
        self.env, self.policy, self.horizon = env, policy, int(horizon)
        self.opponent_policy, self.mirror_opponent = opponent_policy, bool(mirror_opponent)
        if opponent_policy is not None and (env._opponent_mode == "bot" or env.opponent is not None):
            raise ValueError("opponent_policy needs an env whose P2 actions come from step(): opponent='self_play'")
        self.opponent_pool = None if opponent_pool is None else list(opponent_pool)
        self._pool_bot = None                                       # index of the "bot" member, if any
        if self.opponent_pool is not None:
            self._check_pool(fused)
        can_step = isinstance(policy, MLPPolicy) and policy.hidden in (32, 64, 128)
        if opponent_policy is not None:
            can_step = can_step and isinstance(opponent_policy, MLPPolicy) and opponent_policy.hidden == policy.hidden
        can_horizon = (can_step and env.autoreset and env._step_mask is None
                       and (env._opponent_mode == "bot" or opponent_policy is not None or self.opponent_pool is not None))
        if fused is None or fused is True:
            if fused and not can_step:
                raise ValueError("fused=True needs an MLPPolicy with hidden in {32, 64, 128}")
            self.mode = "horizon" if can_horizon else "step" if can_step else "torch"
        elif fused is False:
            self.mode = "torch"
        elif fused in ("step", "horizon"):
            if not (can_horizon if fused == "horizon" else can_step):
                raise ValueError(f"fused={fused!r} is not available for this policy / env configuration")
            self.mode = fused
        else:
            raise ValueError("fused must be None, a bool, 'step' or 'horizon'")
        self.fused = self.mode != "torch"
        n, dev, h = env.num_envs, env.device, self.horizon
        self.obs = torch.zeros((h + 1, n, 8), dtype=torch.float32, device=dev)
        self.actions = torch.zeros((h, n), dtype=torch.uint8, device=dev)
        self.logp = torch.zeros((h, n), dtype=torch.float32, device=dev)
        self.rewards = torch.zeros((h, n), dtype=torch.float32, device=dev)
        self.dones = torch.zeros((h, n), dtype=torch.bool, device=dev)
        self.actions_p2 = self.logp_p2 = None
        if opponent_policy is not None or self.opponent_pool is not None:
            self.actions_p2 = torch.zeros((h, n), dtype=torch.uint8, device=dev)
            self.logp_p2 = torch.zeros((h, n), dtype=torch.float32, device=dev)
            self._mirror_action = torch.tensor(_MIRROR_ACTION, dtype=torch.uint8, device=dev)
        self.opponent_ranges = None
        if self.opponent_pool is not None:
            self._pool_stats = torch.zeros((len(self.opponent_pool), 4), dtype=torch.int64, device=dev)
            self.assign_opponents()
        self.value, self.gamma, self.gae_lambda = value, float(gamma), float(gae_lambda)
        self.values = self.advantages = self.returns = None
        if value is not None:
            self._fused_value = isinstance(value, MLPValue) and value.hidden in (32, 64)
            self.values = torch.zeros((h + 1, n), dtype=torch.float32, device=dev)
            self.advantages = torch.zeros((h, n), dtype=torch.float32, device=dev)
            self.returns = torch.zeros((h, n), dtype=torch.float32, device=dev)
        self._seed = int(seed)
        self._drawn = torch.zeros(1, dtype=torch.int64, device=dev)   # policy steps taken so far (device side: graph replays bump it)
        self._graph = None
        self.use_cuda_graph = bool(use_cuda_graph)
        if not env.has_reset:
            env.reset()
        self.obs[h].copy_(env._delayed_obs if env.frame_delay else env.obs)   # what the first step will act on

    def _check_pool(self, fused):
        env, pool = self.env, self.opponent_pool
        if self.opponent_policy is not None:
            raise ValueError("opponent_policy and opponent_pool are mutually exclusive")
        if env._opponent_mode == "bot" or env.opponent is not None:
            raise ValueError("opponent_pool needs an env whose P2 actions come from step(): opponent='self_play'")
        if not 1 <= len(pool) <= _capi.FG_POOL_MAX:
            raise ValueError(f"opponent_pool has 1 .. {_capi.FG_POOL_MAX} members (got {len(pool)})")
        if not (isinstance(self.policy, MLPPolicy) and self.policy.hidden in (32, 64, 128)):
            raise ValueError("opponent_pool needs an MLPPolicy with hidden in {32, 64, 128} as the policy")
        bots = [k for k, m in enumerate(pool) if isinstance(m, str) and m == "bot"]
        if len(bots) > 1:
            raise ValueError(f'opponent_pool may hold the in-game bot ("bot") once (found at {bots})')
        self._pool_bot = bots[0] if bots else None
        for k, m in enumerate(pool):
            if k != self._pool_bot and (not isinstance(m, MLPPolicy) or m.hidden != self.policy.hidden):
                raise ValueError(f'opponent_pool[{k}] must be "bot" or an MLPPolicy with the policy\'s hidden size '
                                 f'{self.policy.hidden}')
        if not env.autoreset or env._step_mask is not None:
            raise ValueError("opponent_pool runs on the whole-horizon kernel only: the env needs autoreset and no step mask")
        if fused not in (None, True, "horizon"):
            raise ValueError("opponent_pool runs on the whole-horizon kernel only: fused must be None, True or 'horizon'")

    def assign_opponents(self, shares: Optional[Sequence[float]] = None):
        """Splits this device's battles between the pool members in proportion to non-negative `shares` (default: equal),
        as contiguous block-aligned ranges (see opponent_ranges), from the next collect() on.  Returns the ranges, which
        are also kept in self.opponent_ranges."""
        if self.opponent_pool is None:
            raise ValueError("assign_opponents needs a collector with an opponent_pool")
        if shares is None:
            shares = [1.0] * len(self.opponent_pool)
        if len(shares) != len(self.opponent_pool):
            raise ValueError(f"one share per pool member: {len(self.opponent_pool)} expected, got {len(shares)}")
        self.opponent_ranges = opponent_ranges(self.env.num_envs, shares)
        return self.opponent_ranges

    def opponent_pool_stats(self) -> torch.Tensor:
        """int64 [K, 4] on the device: episodes, P1 wins, P2 wins, double KOs of the battles each pool member has played,
        accumulated over every collect() so far (a copy)."""
        if self.opponent_pool is None:
            raise ValueError("opponent_pool_stats needs a collector with an opponent_pool")
        return self._pool_stats.clone()

    def _pool_struct(self):
        pool = _capi.FgOpponentPool(struct_size=C.sizeof(_capi.FgOpponentPool), count=len(self.opponent_pool),
                                    stats=self._pool_stats.data_ptr())
        for k, m in enumerate(self.opponent_pool):
            pool.end[k] = self.opponent_ranges[k][1]
            if k == self._pool_bot:                                 # the bot's weight pointers stay null
                continue
            l1, l2, l3 = m.net[0], m.net[2], m.net[4]
            for name, t in dict(scale=m.scale, w1=l1.weight, b1=l1.bias, w2=l2.weight, b2=l2.bias, w3=l3.weight,
                                b3=l3.bias).items():
                if t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.env.device:
                    raise ValueError(f"opponent_pool[{k}].{name} must be a contiguous float32 tensor on the env's device")
                setattr(pool.member[k], name, t.data_ptr())
        return pool

    def _horizon_launch(self):
        """fg_rollout_mlp (fg_rollout_mlp_pool with an opponent pool, fg_rollout_mlp_pool_bot when the bot is one of its
        members, fg_rollout_mlp_delayed for any of them with frame_delay > 0): the whole horizon in one launch on the
        current stream."""
        env, pol = self.env, self.policy
        l1, l2, l3 = pol.net[0], pol.net[2], pol.net[4]
        r = _capi.FgRolloutBuffers(struct_size=C.sizeof(_capi.FgRolloutBuffers), hidden=pol.hidden, horizon=self.horizon,
                                   reserved0=0, seed=self._seed & (2**64 - 1))
        ts = dict(scale=pol.scale, w1=l1.weight, b1=l1.bias, w2=l2.weight, b2=l2.bias, w3=l3.weight, b3=l3.bias,
                  counter_base=self._drawn, obs=self.obs, actions=self.actions, logp=self.logp, rewards=self.rewards,
                  dones=self.dones)
        if self.opponent_policy is not None:
            o = self.opponent_policy
            m1, m2, m3 = o.net[0], o.net[2], o.net[4]
            ts.update(p2_scale=o.scale, p2_w1=m1.weight, p2_b1=m1.bias, p2_w2=m2.weight, p2_b2=m2.bias, p2_w3=m3.weight,
                      p2_b3=m3.bias, actions_p2=self.actions_p2, logp_p2=self.logp_p2)
            r.p2_seed = (self._seed ^ _P2_SEED_SALT) & (2**64 - 1)
            r.p2_mirror = int(self.mirror_opponent)
        elif self.opponent_pool is not None:
            ts.update(actions_p2=self.actions_p2, logp_p2=self.logp_p2)
            r.p2_seed = (self._seed ^ _P2_SEED_SALT) & (2**64 - 1)
            r.p2_mirror = int(self.mirror_opponent)
        for k, t in ts.items():
            if not t.is_contiguous() or t.device != env.device:
                raise ValueError(f"fused rollout needs contiguous tensors on the env's device ({k})")
            setattr(r, k, t.data_ptr())
        if env.frame_delay:
            depth = env.frame_delay + 1
            ring = _capi.FgDelayRing(struct_size=C.sizeof(_capi.FgDelayRing), depth=depth, pos=env._ring_pos, reserved0=0)
            for k, t in dict(ring_obs=env._ring_obs, ring_frame=env._ring_frame, ring_misc=env._ring_misc,
                             out_obs=env._delayed_obs, out_frame=env._delayed_frame, out_misc=env._delayed_misc).items():
                setattr(ring, k, t.data_ptr())
            pool = None if self.opponent_pool is None else C.byref(self._pool_struct())
            bot = -1 if self._pool_bot is None else self._pool_bot
            _capi.check(env._lib.fg_rollout_mlp_delayed(env._handle, C.byref(r), pool, bot, C.byref(ring), env._stream()))
            env._ring_pos = (env._ring_pos + self.horizon) % depth
        elif self.opponent_pool is not None:
            pool = self._pool_struct()
            if self._pool_bot is None:
                _capi.check(env._lib.fg_rollout_mlp_pool(env._handle, C.byref(r), C.byref(pool), env._stream()))
            else:
                _capi.check(env._lib.fg_rollout_mlp_pool_bot(env._handle, C.byref(r), C.byref(pool), self._pool_bot,
                                                             env._stream()))
        else:
            _capi.check(env._lib.fg_rollout_mlp(env._handle, C.byref(r), env._stream()))
        self._drawn.add_(self.horizon)

    def _values_and_gae(self):
        """Values of all (horizon + 1) x N observation rows, then GAE: two launches on the current stream."""
        if self._fused_value:
            self.value.fused_values(self.obs, self.values)
        else:
            v = self.value(self.obs.view(-1, 8))
            if v.dim() == 2 and v.shape[1] == 1:
                v = v.squeeze(1)
            self.values.view(-1).copy_(v)
        compute_gae(self.rewards, self.dones, self.values, self.gamma, self.gae_lambda, self.advantages, self.returns)

    @torch.no_grad()
    def _one_horizon(self):
        self._rollout()
        if self.value is not None:
            self._values_and_gae()

    def _rollout(self):
        env, h = self.env, self.horizon
        if env.frame_delay:
            self.obs[h].copy_(env._delayed_obs)                     # what the env shows now (env.step() / reset() since)
        if self.mode == "horizon":
            return self._horizon_launch()
        self.obs[0].copy_(self.obs[h])                              # carry the last observation over
        for t in range(h):
            if self.mode == "step":
                self.policy.fused_sample(self.obs[t], self.actions[t], self.logp[t], self._seed, t, self._drawn,
                                         first_env_index=env.first_env_index)
            else:
                logits = self.policy(self.obs[t])
                logp_all = torch.log_softmax(logits, dim=-1)
                a = torch.multinomial(logp_all.exp(), 1).squeeze(1)
                self.logp[t].copy_(logp_all.gather(1, a.unsqueeze(1)).squeeze(1))
                self.actions[t].copy_(a)                            # int64 -> uint8 bitmask (Left 1 | Right 2 | Attack 4)
            if self.opponent_policy is None:
                env.bind_actions(self.actions[t])
            else:
                if self.mode == "step":
                    self.opponent_policy.fused_sample_p2(self.obs[t], self.actions_p2[t], self.logp_p2[t],
                                                         self._seed ^ _P2_SEED_SALT, t, self._drawn, self.mirror_opponent,
                                                         first_env_index=env.first_env_index)
                else:
                    o = mirror_obs(self.obs[t]) if self.mirror_opponent else self.obs[t]
                    logp_all = torch.log_softmax(self.opponent_policy(o), dim=-1)
                    a = torch.multinomial(logp_all.exp(), 1).squeeze(1)
                    self.logp_p2[t].copy_(logp_all.gather(1, a.unsqueeze(1)).squeeze(1))
                    self.actions_p2[t].copy_(self._mirror_action[a] if self.mirror_opponent else a)
                env.bind_actions(self.actions[t], self.actions_p2[t])
            env.bind_outputs(obs=self.obs[t + 1], reward=self.rewards[t], terminated=self.dones[t])
            env.step_bound()
            if env.frame_delay:
                self.obs[t + 1].copy_(env._delayed_obs)             # the queue has taken the true observation already
        self._drawn.add_(h)

    def collect(self):
        """Runs one horizon (and with a value network its values and GAE); returns the rollout buffers (views,
        overwritten by the next call)."""
        dev = self.env.device
        # horizon: one launch, nothing for a graph to save; frame_delay: the ring position is a host integer
        if not self.use_cuda_graph or self.mode == "horizon" or self.env.frame_delay:
            self._one_horizon()
        else:
            if self._graph is None:
                stream = torch.cuda.Stream(device=dev)
                stream.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(stream):
                    self._one_horizon()                             # warm-up outside the capture (lazy inits)
                torch.cuda.current_stream(dev).wait_stream(stream)
                torch.cuda.synchronize(dev)
                self._graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._graph):
                    self._one_horizon()
            self._graph.replay()
        out = {"obs": self.obs[:self.horizon], "actions": self.actions, "logp": self.logp, "rewards": self.rewards,
               "dones": self.dones, "last_obs": self.obs[self.horizon]}
        if self.actions_p2 is not None:
            out.update(actions_p2=self.actions_p2, logp_p2=self.logp_p2)
        if self.value is not None:
            out.update(values=self.values, advantages=self.advantages, returns=self.returns)
        return out
