"""The learned-policy side against float64: the fused policy kernels (fg_policy_mlp_sample / _p2, tensor-core path for
H = 32 / 64, FFMA2 path for H = 128), the whole-horizon rollout kernels through RolloutCollector, the value head
(fg_value_mlp) and the sampler (policy_sample + hash3).

Tolerance: a fixed bar cannot follow training -- as weights grow, torch's own fp32 forward pass drifts from float64 by
more than any fixed bar a correct kernel passes, while a priori worst-case bounds are so loose that a kernel which lost
half its operand precision passes them.  So the yardstick is fp32's own error on the same network: e32 = |torch fp32 on
the CPU - float64| over a fixed set of 65 536 observations, and a kernel is correct when its error against float64 is
within K = 32 times e32, max and RMS (see `check_rule`).  The CPU part proves in CI that this rule rejects a kernel that
dropped the lo halves of its split operands and accepts one with MUFU-grade tanh errors; the GPU part applies it to every
call site.

The sampler is checked draw for draw: with W3 = 0 every path computes logits equal to b3 exactly, so the action of every
row follows from b3's float64 CDF and the 24-bit uniform of a numpy hash3; the hash itself is checked for uniformity and
independence on the CPU."""
import copy
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")

gpu = pytest.mark.gpu

# ---- the tolerance rule ----

# Kernel error against float64 may be at most K times fp32's own error on the same network (max over rows, and RMS over
# rows).  An fp32 emulation of the kernels (MUFU ex2 / rcp tanh, __expf / __logf) sits at 1-6 x e32 in the regimes below,
# while the float64 forward pass with the lo halves of the split weights dropped (2^-11 relative) sits at 280 - 3 600 x:
# K = 32 leaves a correct kernel 5 x of headroom and still sees a lost half.  Measured on a B200 (1 000 W): 0.2 - 5.7 x
# at every site, except the value head with |b3| ~ 50 (14 x at H = 32, 25 x at H = 64, max and RMS alike): the bias is
# the MMA accumulator's starting value, so each of the 6 / 12 MMAs rounds a sum of size |V|, where fp32's forward pass
# rounds it once -- a systematic offset of ~1e-6 |V| that grows with the number of k-steps.
K_E32 = 32.0
# The floor covers what no forward pass can beat: the last bits of __logf / the fp32 log-softmax at |log p|, and a row
# where e32 happens to be 0 (W3 = 0 makes fp32 exact).
FLOOR_REL = 2.0 ** -20

N_YARDSTICK = 65536


class Verdict:
    """Errors of `got` against the float64 `ref`, in units of the yardstick, and whether they are within the rule."""

    def __init__(self, got, ref, e32):
        got, ref = np.asarray(got, np.float64).ravel(), np.asarray(ref, np.float64).ravel()
        d = np.abs(got - ref)
        floor = FLOOR_REL * (1.0 + np.abs(ref))
        self.rows = d.size
        self.err_max, self.err_rms = float(d.max()), float(np.sqrt(np.mean(d * d)))
        self.e32_max, self.e32_rms = e32
        self.ratio_max = self.err_max / self.e32_max if self.e32_max > 0 else (0.0 if self.err_max == 0 else np.inf)
        self.ratio_rms = self.err_rms / self.e32_rms if self.e32_rms > 0 else (0.0 if self.err_rms == 0 else np.inf)
        # how far outside the rule (<= 1: inside); the max bound is per row, with that row's floor
        excess_max = float(np.max(d / (K_E32 * self.e32_max + floor)))
        excess_rms = self.err_rms / (K_E32 * self.e32_rms + float(np.sqrt(np.mean(floor * floor))))
        self.excess = max(excess_max, excess_rms)
        self.ok = bool(np.all(np.isfinite(got))) and self.excess <= 1.0

    def __str__(self):
        return (f"max|d| {self.err_max:.3g} ({self.ratio_max:.2f} x e32 {self.e32_max:.3g}), rms {self.err_rms:.3g} "
                f"({self.ratio_rms:.2f} x e32 {self.e32_rms:.3g}), {self.excess:.3g} of the bound, {self.rows} rows")


def check_rule(got, ref, e32, what):
    """max|got - ref| <= K e32_max + floor and rms|got - ref| <= K e32_rms + rms(floor), floor = 2^-20 (1 + |ref|)."""
    v = Verdict(got, ref, e32)
    print(f"{what}: {v}")
    assert v.ok, f"{what}: {v}"
    return v


# ---- networks, observations and references ----

POLICY_REGIMES = ("default", "x3", "x10", "x30", "student_t", "w3_row_small", "w2_block_small", "max_pow2",
                  "max_below_pow2", "w2_zero", "tiny", "w3_zero_big_b3")
VALUE_REGIMES = POLICY_REGIMES + ("b3_50",)
# regimes whose output does not depend on the lo halves of the weights, so no precision loss of the split can show:
# W3 = 0 gives the logits b3 exactly; weights around 1e-30 contribute below fp32's resolution of the biases
_SPLIT_BLIND = ("tiny", "w3_zero_big_b3")
# How far outside the rule the hi-only weights must land.  20 wherever the weights carry the output; in three regimes the
# lo halves carry less of it against fp32's own error and the floor -- small default-init weights (H = 32: 280 x e32),
# W2 = 0 (only W1 and W3 are split) and a value of |b3| ~ 50 (the floor grows with |V|) -- and the measured margin is
# 7 - 15, so these regimes ask for 5.
_MIN_REJECTION = {"default": 5.0, "w2_zero": 5.0, "b3_50": 5.0}


def _random_obs(rows, seed, device="cpu"):
    """Observations over the observation space: guard 0..3, move 0..14, move frame 0..55, position -4.6 .. 4.6 (drawn on
    the CPU, so the same seed gives the same rows everywhere)."""
    g = torch.Generator()
    g.manual_seed(seed)
    ri = lambda hi: torch.randint(0, hi, (rows,), generator=g).float()   # noqa: E731
    pos = lambda: torch.rand(rows, generator=g) * 9.2 - 4.6              # noqa: E731
    return torch.stack([ri(4), ri(4), ri(15), ri(15), ri(56), ri(56), pos(), pos()], dim=1).contiguous().to(device)


def _f32(x):
    return torch.from_numpy(np.asarray(x, np.float32))


def _apply_regime(net, regime, seed):
    """Rewrites the parameters of a freshly initialised MLPPolicy / MLPValue for one weight regime (seeded)."""
    rng = np.random.default_rng(seed)
    l1, l2, l3 = net.net[0], net.net[2], net.net[4]
    lin = (l1, l2, l3)
    h = l2.weight.shape[0]
    with torch.no_grad():
        if regime == "default":
            return
        if regime in ("x10", "x30"):
            for p in net.net.parameters():
                p.mul_(float(regime[1:]))
            return
        if regime == "student_t":
            for m in lin:                            # heavy tails at the default init's scale
                s = 1.0 / np.sqrt(m.weight.shape[1])
                m.weight.copy_(_f32(rng.standard_t(3, m.weight.shape) * s))
                m.bias.copy_(_f32(rng.standard_t(3, m.bias.shape) * s))
            return
        for p in net.net.parameters():               # every other regime starts from x3: a peaky policy
            p.mul_(3.0)
        w2, w3 = l2.weight, l3.weight
        if regime == "x3":
            pass
        elif regime == "w3_row_small":               # the FP16 path picks one scale per matrix
            if w3.shape[0] == 8:
                w3[5].mul_(1e-4)
            else:
                w3[0, : h // 2].mul_(1e-4)
        elif regime == "w2_block_small":
            w2[: h // 2, : h // 2].mul_(1e-4)
        elif regime in ("max_pow2", "max_below_pow2"):   # the exponent boundary of the scale in [2^12, 2^13)
            for w in (w2, w3):
                flat = w.view(-1)
                i = int(flat.abs().argmax())
                p2 = 2.0 ** np.ceil(np.log2(float(flat[i].abs())))
                v = p2 if regime == "max_pow2" else float(np.nextafter(np.float32(p2), np.float32(0)))
                flat[i] = v if float(flat[i]) > 0 else -v
        elif regime == "w2_zero":                    # the exponent clamp (E = 0 -> 40)
            w2.zero_()
        elif regime == "tiny":                       # every weight around 1e-30: the clamp again, with live weights
            for m in lin:
                m.weight.copy_(_f32(rng.standard_normal(m.weight.shape) * 1e-30))
        elif regime == "w3_zero_big_b3":             # logits = b3 exactly, |b3| up to 1e4
            w3.zero_()
            l3.bias.copy_(_f32(rng.uniform(-1e4, 1e4, l3.bias.shape)))
        elif regime == "b3_50":
            l3.bias.copy_(_f32(rng.choice([-50.0, 50.0], l3.bias.shape) * (1 + 0.01 * rng.standard_normal(l3.bias.shape))))
        else:
            raise ValueError(regime)


@functools.lru_cache(maxsize=None)
def _net_cpu(kind, hidden, regime, seed=0):
    from footsies_gym_b200.rollout import MLPPolicy, MLPValue
    torch.manual_seed(1000 * seed + hidden)
    net = (MLPPolicy if kind == "policy" else MLPValue)(hidden)
    _apply_regime(net, regime, seed=hidden * 7 + seed)
    return net.eval()


def _net(kind, hidden, regime, device, seed=0):
    return copy.deepcopy(_net_cpu(kind, hidden, regime, seed)).to(device)


def _params64(net, device):
    l1, l2, l3 = net.net[0], net.net[2], net.net[4]
    return [t.detach().to(device=device, dtype=torch.float64)
            for t in (net.scale, l1.weight, l1.bias, l2.weight, l2.bias, l3.weight, l3.bias)]


def _forward64(params, obs, mirror=False):
    """The module's forward pass in float64 on `obs` (any device): logits [N, 8] or values [N, 1]."""
    from footsies_gym_b200.rollout import mirror_obs
    scale, w1, b1, w2, b2, w3, b3 = params
    x = obs.to(dtype=torch.float64, device=scale.device)
    if mirror:
        x = mirror_obs(x)
    h1 = torch.tanh(x * scale @ w1.T + b1)
    h2 = torch.tanh(h1 @ w2.T + b2)
    return h2 @ w3.T + b3


def _policy_logp64(net, obs, mirror=False, device=None):
    """float64 log-probabilities [N, 8] of an MLPPolicy on obs (as P2 with mirror: on the mirrored observation, indexed by
    the network's own action, i.e. before _MIRROR_ACTION maps it back)."""
    dev = obs.device if device is None else device
    return torch.log_softmax(_forward64(_params64(net, dev), obs, mirror), dim=-1)


def _value64(net, obs):
    return _forward64(_params64(net, obs.device), obs).squeeze(-1)


@functools.lru_cache(maxsize=None)
def _yardstick(kind, hidden, regime, seed=0):
    """(max, rms) of |torch fp32 on the CPU - float64| of one network over N_YARDSTICK fixed observations: every
    log-probability of a policy, the value of a value network."""
    net = _net_cpu(kind, hidden, regime, seed)
    obs = _random_obs(N_YARDSTICK, seed=20251)
    with torch.no_grad():
        if kind == "policy":
            e = (torch.log_softmax(net(obs), dim=-1).double() - _policy_logp64(net, obs)).abs()
        else:
            e = (net(obs).double() - _value64(net, obs)).abs()
    e = e.numpy()
    return float(e.max()), float(np.sqrt(np.mean(e * e)))


# ---- CPU emulations for the negative control ----

def _tf32_rna(w):
    """cvt.rna.tf32.f32: round to 10 explicit mantissa bits, ties away from zero (finite inputs)."""
    u = np.asarray(w, np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xffffe000)).view(np.float32)


def _f16_hi(w):
    """The hi half of policy_mma_stage's FP16 split: w times the power of two that puts max|w| into [2^12, 2^13)
    (biased exponent clamped to [40, 254]), rounded to FP16, scaled back."""
    w = np.asarray(w, np.float32)
    e = int(np.abs(w).max().view(np.uint32) >> 23) if w.size else 0
    e = min(max(e, 40), 254)
    s = np.float32(2.0 ** (139 - e))
    return (w * s).astype(np.float16).astype(np.float64) / np.float64(s)


def _hi_only_params64(net):
    """float64 parameters with the weights cut to the hi half of their split: TF32 for W1, FP16 after the power-of-two
    scale for W2 / W3 -- what a kernel that dropped every lo product would compute with."""
    scale, w1, b1, w2, b2, w3, b3 = _params64(net, "cpu")
    f = lambda t: t.float().numpy()              # noqa: E731   (the fp32 parameters themselves)
    w1 = torch.from_numpy(_tf32_rna(f(w1)).astype(np.float64))
    w2 = torch.from_numpy(_f16_hi(f(w2)))
    w3 = torch.from_numpy(_f16_hi(f(w3)))
    return [scale, w1, b1, w2, b2, w3, b3]


def _emulated_kernel(net, obs, seed):
    """fp32 forward pass with the kernels' approximations as seeded relative errors: tanh = 1 - 2 rcp(ex2(2 x log2 e) + 1)
    with ex2 / rcp each off by up to 2^-22, __expf off by 2^-21 and __logf by 2^-21 absolute in the log-softmax."""
    rng = np.random.default_rng(seed)
    jit = lambda shape, eps: (1.0 + rng.uniform(-eps, eps, shape)).astype(np.float32)   # noqa: E731
    l1, l2, l3 = net.net[0], net.net[2], net.net[4]
    np32 = lambda t: t.detach().float().numpy()  # noqa: E731

    def tanh(x):
        with np.errstate(over="ignore"):
            e = np.exp2(x * np.float32(2.8853900432586669921875)) * jit(x.shape, 2.0 ** -22)
            r = (np.float32(1.0) / (e + np.float32(1.0))) * jit(x.shape, 2.0 ** -22)
        return np.float32(1.0) - np.float32(2.0) * r

    x = obs.float().numpy() * np32(net.scale)
    h1 = tanh(x @ np32(l1.weight).T + np32(l1.bias))
    h2 = tanh(h1 @ np32(l2.weight).T + np32(l2.bias))
    out = h2 @ np32(l3.weight).T + np32(l3.bias)
    if out.shape[1] == 1:
        return out[:, 0]
    m = out.max(axis=1, keepdims=True)
    e = np.exp(out - m) * jit(out.shape, 2.0 ** -21)
    return (out - m) - (np.log(e.sum(axis=1, keepdims=True)) + rng.uniform(-1, 1, (out.shape[0], 1)) * 2.0 ** -21)


def _reference(kind, net, obs, params=None):
    p = _params64(net, "cpu") if params is None else params
    out = _forward64(p, obs)
    return torch.log_softmax(out, dim=-1).numpy() if kind == "policy" else out.squeeze(-1).numpy()


@pytest.mark.parametrize("kind,regime", [("policy", r) for r in POLICY_REGIMES] + [("value", r) for r in VALUE_REGIMES])
def test_rule_rejects_dropped_lo_halves_and_accepts_mufu_errors(kind, regime):
    """The rule on CPU emulations: a forward pass with MUFU-grade tanh / exp / log errors passes; one whose weights lost
    their lo halves fails by a factor >= 20 (_MIN_REJECTION; none in the regimes whose output cannot see the lo halves)."""
    hiddens = (32, 64, 128) if kind == "policy" else (32, 64)
    obs = _random_obs(8192, seed=77)
    for hidden in hiddens:
        net = _net_cpu(kind, hidden, regime)
        e32 = _yardstick(kind, hidden, regime)
        ref = _reference(kind, net, obs)
        emu = _emulated_kernel(net, obs, seed=hidden)
        check_rule(emu, ref, e32, f"{kind} H={hidden} {regime}: MUFU emulation")
        hi = _reference(kind, net, obs, _hi_only_params64(net))
        v = Verdict(hi, ref, e32)
        print(f"{kind} H={hidden} {regime}: hi-only weights {v}; rejection margin {v.excess:.1f}")
        if regime not in _SPLIT_BLIND:
            need = _MIN_REJECTION.get(regime, 20.0)
            assert v.excess >= need, f"{kind} H={hidden} {regime}: hi-only weights only {v.excess:.2f} x outside: {v}"


def test_yardstick_is_fp32_error_of_the_same_network():
    """e32 grows with the weights (what a fixed bar cannot follow) and is 0 only where fp32 is exact."""
    small, big = _yardstick("policy", 64, "default"), _yardstick("policy", 64, "x30")
    assert 0 < small[1] <= small[0] and 0 < big[1] <= big[0]
    assert big[0] > 4 * small[0]
    assert _yardstick("value", 64, "w3_zero_big_b3") == (0.0, 0.0)


# ---- numpy reference of the sampler's randomness (policy_mlp.cuh: hash3, policy_sample) ----

_U64 = np.uint64


def hash3(seed, counter, idx):
    """hash3(seed, counter, idx) in uint64 arithmetic (wrapping like the device code); broadcasts."""
    counter = np.asarray(counter, dtype=np.uint64)
    idx = np.asarray(idx, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = _U64(int(seed) & (2**64 - 1)) + _U64(0x9E3779B97F4A7C15) * (counter * _U64(0x100000001B3) + idx + _U64(1))
        z = (z ^ (z >> _U64(30))) * _U64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> _U64(27))) * _U64(0x94D049BB133111EB)
        return ((z ^ (z >> _U64(31))) >> _U64(32)).astype(np.uint32)


def uniform24(h):
    """policy_sample's u in [0, 1): the top 24 bits of the hash (exact in float64 and fp32)."""
    return (np.asarray(h, np.uint32) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


def _hash3_int(seed, counter, idx):
    m = 2**64 - 1
    z = (seed + 0x9E3779B97F4A7C15 * (counter * 0x100000001B3 + idx + 1)) & m
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
    return (z ^ (z >> 31)) >> 32


def test_numpy_hash3_equals_python_integers():
    rng = np.random.default_rng(5)
    for seed in (0, 1, 17, 2**63, 2**64 - 1, 0x5DEECE66D2F1A3B7):
        c = rng.integers(0, 2**62, 64, dtype=np.uint64)
        i = rng.integers(0, 2**40, 64, dtype=np.uint64)
        got = hash3(seed, c, i)
        assert [int(x) for x in got] == [_hash3_int(seed, int(a), int(b)) for a, b in zip(c, i)]


AMBIGUOUS = 1e-5


def predict_draws(b3, u):
    """Actions the sampler must draw for logits b3 (exact) and uniforms u: the first o with u < CDF_f64(o), and a mask of
    the rows where u lies within AMBIGUOUS of a CDF boundary (fp32's sum may fall either side there)."""
    lp = torch.log_softmax(torch.as_tensor(np.asarray(b3, np.float32), dtype=torch.float64), dim=0).numpy()
    cdf = np.cumsum(np.exp(lp))[:7]
    a = np.searchsorted(cdf, u, side="right")
    amb = np.min(np.abs(u[:, None] - cdf[None, :]), axis=1) < AMBIGUOUS
    return a.astype(np.int64), amb, lp


_P_TINY = 1e-9


def _b3_vectors():
    """Logit vectors b3 for the draw-for-draw checks (float32): uniform, peaky, tied, spread over [-80, 0], and one with
    an action at p = 1e-9 behind enough mass that fp32's running CDF cannot move by it: it must never be drawn."""
    rest = np.array([1.0, 0.5, 0.8, 0.0, 0.2, -0.3, 0.0, 0.6])
    z = np.exp(np.delete(rest, 3)).sum()
    rest[3] = np.log(_P_TINY * z / (1 - _P_TINY))
    return {
        "uniform": np.zeros(8),
        "peaky": np.array([-1.0, 0.0, 9.0, -2.0, 0.5, -0.5, 1.0, 0.0]),
        "tied": np.array([2.0, 2.0, 0.0, 0.0, 2.0, 2.0, -1.0, -1.0]),
        "spread": np.array([-80.0, -2.0, -40.0, 0.0, -11.4, -1.0, -60.0, -5.5]),
        "tiny": rest,
    }


# ---- hash statistics (CPU) ----

_SALT = 0x5DEECE66D2F1A3B7


def test_hash_uniforms_are_uniform_and_independent():
    """u over the (counter, global index) grid of a 128-step horizon x 32 768 battles, three seeds including 2^64 - 1:
    KS and chi-square uniformity, and no correlation between t and t + 1, i and i + 1, P1 and P2 (seed ^ salt).  The
    thresholds are 6 sigma, so a seeded run never flakes."""
    from scipy import stats
    from footsies_gym_b200.rollout import _P2_SEED_SALT
    assert _P2_SEED_SALT == _SALT
    p6 = 2.0 * stats.norm.sf(6.0)                    # two-sided 6 sigma
    t = np.arange(128, dtype=np.uint64)[:, None] + np.uint64(3 * 128)
    i = np.arange(32768, dtype=np.uint64)[None, :] + np.uint64(1 << 20)
    for seed in (0, 0x0123456789ABCDEF, 2**64 - 1):
        u = uniform24(hash3(seed, t, i))
        n = u.size
        ks = stats.kstest(u.ravel(), "uniform")
        counts = np.bincount((u.ravel() * 4096).astype(np.int64), minlength=4096)
        chi = stats.chisquare(counts)
        assert ks.pvalue > p6 and chi.pvalue > p6, (seed, ks, chi)

        def z(a, b):
            r = np.corrcoef(a.ravel(), b.ravel())[0, 1]
            return abs(r) * np.sqrt(a.size)
        zt, zi = z(u[:-1], u[1:]), z(u[:, :-1], u[:, 1:])
        zp = z(u, uniform24(hash3(seed ^ _SALT, t, i)))
        print(f"seed {seed:#x}: {n} draws, KS p {ks.pvalue:.3g}, chi2 p {chi.pvalue:.3g}, |corr| sqrt(n): "
              f"t/t+1 {zt:.2f}, i/i+1 {zi:.2f}, P1/P2 {zp:.2f}")
        assert max(zt, zi, zp) < 6.0, (seed, zt, zi, zp)


# ---- GPU: the call sites against the rule ----

ROW_COUNTS = (1, 15, 17, 31, 33, 10007, 50001)


def _dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    return torch.device("cuda:0")


_OBS_CACHE = {}


def _obs_gpu(rows, dev):
    key = (rows, str(dev))
    if key not in _OBS_CACHE:
        _OBS_CACHE[key] = _random_obs(rows, seed=rows + 3, device=dev)
    return _OBS_CACHE[key]


def _chosen_logp64(lp64, actions, mirror):
    """float64 log-probability of the network's own pick: the reported P2 action is mapped back with _MIRROR_ACTION."""
    from footsies_gym_b200.rollout import _MIRROR_ACTION
    a = actions.long()
    if mirror:
        a = torch.tensor(_MIRROR_ACTION, device=a.device)[a]
    return lp64.gather(-1, a.unsqueeze(-1)).squeeze(-1)


SENTINEL_A, PAD = 0xAB, 64


@gpu
@pytest.mark.parametrize("regime", POLICY_REGIMES)
@pytest.mark.parametrize("hidden", [32, 64, 128])
def test_policy_sample_kernel_against_float64(hidden, regime):
    """fg_policy_mlp_sample and fg_policy_mlp_sample_p2 (mirror on and off) at ragged row counts: the log-probability of
    the drawn action against float64, by the rule; nothing written past the last row."""
    dev = _dev()
    pol = _net("policy", hidden, regime, dev)
    e32 = _yardstick("policy", hidden, regime)
    obs_all = _obs_gpu(max(ROW_COUNTS), dev)
    for site in ("p1", "p2", "p2_mirror"):
        mirror = site == "p2_mirror"
        got, ref = [], []
        for n in ROW_COUNTS:
            obs = obs_all[:n].contiguous()
            actions = torch.full((n + PAD,), SENTINEL_A, dtype=torch.uint8, device=dev)
            logp = torch.full((n + PAD,), float("nan"), dtype=torch.float32, device=dev)
            if site == "p1":
                pol.fused_sample(obs, actions[:n], logp[:n], seed=11 + n, counter=n)
            else:
                pol.fused_sample_p2(obs, actions[:n], logp[:n], seed=11 + n, counter=n, mirror=mirror)
            torch.cuda.synchronize()
            assert bool((actions[n:] == SENTINEL_A).all()) and bool(logp[n:].isnan().all()), (site, n)
            assert int(actions[:n].max()) <= 7
            lp64 = _policy_logp64(pol, obs, mirror=mirror)
            got.append(logp[:n].double())
            ref.append(_chosen_logp64(lp64, actions[:n], mirror))
            check_rule(got[-1].cpu().numpy(), ref[-1].cpu().numpy(), e32, f"policy {site} H={hidden} {regime} rows={n}")
        check_rule(torch.cat(got).cpu().numpy(), torch.cat(ref).cpu().numpy(), e32,
                   f"policy {site} H={hidden} {regime} all rows")


@gpu
@pytest.mark.parametrize("regime", VALUE_REGIMES)
@pytest.mark.parametrize("hidden", [32, 64])
def test_value_kernel_against_float64(hidden, regime):
    """fg_value_mlp at ragged row counts against float64, by the rule; nothing written past the last row.  W3 = 0 gives
    the bias exactly."""
    dev = _dev()
    val = _net("value", hidden, regime, dev)
    e32 = _yardstick("value", hidden, regime)
    obs_all = _obs_gpu(max(ROW_COUNTS), dev)
    got, ref = [], []
    for n in ROW_COUNTS:
        obs = obs_all[:n].contiguous()
        out = torch.full((n + PAD,), float("nan"), dtype=torch.float32, device=dev)
        val.fused_values(obs, out[:n])
        torch.cuda.synchronize()
        assert bool(out[n:].isnan().all()), n
        got.append(out[:n].double())
        ref.append(_value64(val, obs))
        check_rule(got[-1].cpu().numpy(), ref[-1].cpu().numpy(), e32, f"value H={hidden} {regime} rows={n}")
        if regime == "w3_zero_big_b3":
            assert torch.equal(out[:n], val.net[4].bias.expand(n)), n
    check_rule(torch.cat(got).cpu().numpy(), torch.cat(ref).cpu().numpy(), e32, f"value H={hidden} {regime} all rows")


@gpu
@pytest.mark.parametrize("hidden", [32, 64])
def test_value_kernel_past_2_31_floats(hidden):
    """One launch over 2^28 + 3 rows (2^31 + 24 floats of observations: the int64 `rows` contract): a seeded sample of
    rows and the last 4 096 against float64, by the rule."""
    dev = _dev()
    rows = 2**28 + 3
    need = rows * 9 * 4 + (4 << 30)                  # observations + values + working room
    free, _ = torch.cuda.mem_get_info(dev)
    if free < max(need, 24 << 30):
        pytest.skip(f"needs 24 GB of free device memory ({free / 2**30:.1f} GiB free)")
    val = _net("value", hidden, "x3", dev)
    e32 = _yardstick("value", hidden, "x3")
    obs = torch.empty((rows, 8), dtype=torch.float32, device=dev)
    chunk = 1 << 24
    for k, start in enumerate(range(0, rows, chunk)):
        m = min(chunk, rows - start)
        obs[start:start + m] = _random_obs(m, seed=900 + k, device=dev)
    out = torch.full((rows + PAD,), float("nan"), dtype=torch.float32, device=dev)
    val.fused_values(obs, out[:rows])
    torch.cuda.synchronize()
    assert bool(out[rows:].isnan().all())
    g = torch.Generator(device=dev)
    g.manual_seed(hidden)
    idx = torch.cat([torch.randint(0, rows, (65536,), generator=g, device=dev),
                     torch.arange(rows - 4096, rows, device=dev)])
    check_rule(out[idx].double().cpu().numpy(), _value64(val, obs[idx]).cpu().numpy(), e32,
               f"value H={hidden} x3 rows=2^28+3 (sampled + last 4096)")
    del obs, out
    torch.cuda.empty_cache()


# ---- GPU: the whole-horizon kernels through RolloutCollector ----

ROLLOUT_SITES = ("bot_h32", "bot_h64", "bot_h128", "self_play_mirror", "pool3_bot", "frame_delay3", "mt2_bot",
                 "mt2_self_play_mirror")


def _rollout_setup(site, regime, dev, n, horizon, seed=21):
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    hidden = int(site[5:]) if site.startswith("bot_h") else 64
    pol = _net("policy", hidden, regime, dev, seed=1)
    p2 = pool = None
    mirror = False
    delay = 3 if site == "frame_delay3" else 0
    if site in ("bot_h32", "bot_h64", "bot_h128", "frame_delay3", "mt2_bot"):
        env = FootsiesEnv(num_envs=n, device=dev, seed=5, frame_delay=delay)
    else:
        env = FootsiesEnv(num_envs=n, device=dev, seed=5, opponent="self_play")
        mirror = True
        if site == "pool3_bot":
            pool = [_net("policy", hidden, regime, dev, seed=s) for s in (2, 3, 4)] + ["bot"]
        else:
            p2 = _net("policy", hidden, regime, dev, seed=2)
    col = RolloutCollector(env, pol, horizon=horizon, seed=seed, opponent_policy=p2, mirror_opponent=mirror,
                           opponent_pool=pool)
    assert col.mode == "horizon"
    return col, pol, p2, pool, hidden, mirror


@gpu
@pytest.mark.parametrize("regime", ["x3", "x30"])
@pytest.mark.parametrize("site", ROLLOUT_SITES)
def test_rollout_kernels_against_float64(monkeypatch, site, regime):
    """Every (t, battle) of two collects of the whole-horizon kernel: logp (and logp_p2) against float64 of the network
    on obs[t] (its mirror for P2), by the rule.  Each kernel variant stages its observation rows differently."""
    if site.startswith("mt2_"):
        monkeypatch.setenv("FOOTSIES_B200_ROLLOUT_MT", "2")
    dev = _dev()
    n, horizon = 1100, 48
    col, pol, p2, pool, hidden, mirror = _rollout_setup(site, regime, dev, n, horizon)
    e32 = _yardstick("policy", hidden, regime, 1)
    for c in range(2):
        out = col.collect()
        torch.cuda.synchronize()
        obs = out["obs"]
        lp64 = _policy_logp64(pol, obs.reshape(-1, 8)).view(horizon, n, 8)
        check_rule(out["logp"].double().cpu().numpy(), _chosen_logp64(lp64, out["actions"], False).cpu().numpy(), e32,
                   f"rollout {site} {regime} collect {c} P1")
        if p2 is not None:
            lp2 = _policy_logp64(p2, obs.reshape(-1, 8), mirror=mirror).view(horizon, n, 8)
            check_rule(out["logp_p2"].double().cpu().numpy(),
                       _chosen_logp64(lp2, out["actions_p2"], mirror).cpu().numpy(),
                       _yardstick("policy", hidden, regime, 2), f"rollout {site} {regime} collect {c} P2")
        if pool is not None:
            for k, (a, b) in enumerate(col.opponent_ranges):
                if pool[k] == "bot" or a == b:
                    continue
                lpk = _policy_logp64(pool[k], obs[:, a:b].reshape(-1, 8), mirror=mirror).view(horizon, b - a, 8)
                check_rule(out["logp_p2"][:, a:b].double().cpu().numpy(),
                           _chosen_logp64(lpk, out["actions_p2"][:, a:b], mirror).cpu().numpy(),
                           _yardstick("policy", hidden, regime, k + 2), f"rollout {site} {regime} collect {c} member {k}")


# ---- GPU: draw for draw on exact logits ----

def _exact_logit_policy(hidden, b3, dev, seed=0):
    """An x3 policy with W3 = 0 and the given b3: every path computes logits equal to b3 exactly (FP16 path: the clamped
    scale 2^99 and its inverse 2^-107 are powers of two; FFMA2 path: the partial sums are zeros)."""
    pol = _net("policy", hidden, "x3", dev, seed=seed)
    with torch.no_grad():
        pol.net[4].weight.zero_()
        pol.net[4].bias.copy_(torch.as_tensor(np.asarray(b3, np.float32), device=dev))
    return pol


class DrawCheck:
    """Accumulates draw-for-draw comparisons of one site: predicted vs drawn actions off the ambiguous rows, logp against
    float64 log_softmax(b3) within the floor."""

    def __init__(self, what):
        self.what, self.rows, self.ambiguous = what, 0, 0

    def add(self, b3, u, actions, logp, mirror=False, tiny_action=None):
        from footsies_gym_b200.rollout import _MIRROR_ACTION
        pred, amb, lp = predict_draws(b3, u)
        a = np.asarray(actions, np.int64)
        own = np.asarray(_MIRROR_ACTION)[a] if mirror else a       # the network's own pick
        self.rows += a.size
        self.ambiguous += int(amb.sum())
        bad = (own != pred) & ~amb
        assert not bad.any(), (f"{self.what}: {int(bad.sum())} draws differ from the prediction, e.g. row "
                               f"{int(np.argmax(bad))}: u {u[bad][0]!r} drew {own[bad][0]} predicted {pred[bad][0]}")
        ref = lp[own]
        d = np.abs(np.asarray(logp, np.float64) - ref)
        assert np.all(d <= FLOOR_REL * (1 + np.abs(ref))), (self.what, float(d.max()))
        if tiny_action is not None:
            assert not (own == tiny_action).any(), f"{self.what}: the p = 1e-9 action was drawn"

    def finish(self):
        print(f"{self.what}: {self.rows} draws, {self.ambiguous} ambiguous ({self.ambiguous / max(self.rows, 1):.2e})")
        assert self.rows > 0 and self.ambiguous < 1e-3 * self.rows, (self.what, self.rows, self.ambiguous)


@gpu
@pytest.mark.parametrize("hidden", [32, 64, 128])
def test_per_step_kernels_draw_for_draw(hidden):
    """fg_policy_mlp_sample with counter, counter_base and first_env_index != 0, and fg_policy_mlp_sample_p2 with mirror
    (the mapped-back action): every unambiguous draw equals the prediction from b3's float64 CDF and hash3."""
    dev = _dev()
    n = 200_003
    obs = _obs_gpu(n, dev)
    seed, counter, base, first = 0xFEEDFACE12345678, 1234, 987654321, 3_000_000_017
    cb = torch.tensor([base], dtype=torch.int64, device=dev)
    u1 = uniform24(hash3(seed, counter + base, first + np.arange(n, dtype=np.uint64)))
    u2 = uniform24(hash3(seed ^ _SALT, counter, np.arange(n, dtype=np.uint64)))
    chk1, chk2 = DrawCheck(f"per-step P1 H={hidden}"), DrawCheck(f"per-step P2 mirror H={hidden}")
    for name, b3 in _b3_vectors().items():
        pol = _exact_logit_policy(hidden, b3, dev)
        tiny = 3 if name == "tiny" else None
        a = torch.zeros(n, dtype=torch.uint8, device=dev)
        lp = torch.zeros(n, dtype=torch.float32, device=dev)
        pol.fused_sample(obs, a, lp, seed=seed, counter=counter, counter_base=cb, first_env_index=first)
        torch.cuda.synchronize()
        chk1.add(b3, u1, a.cpu().numpy(), lp.cpu().numpy(), tiny_action=tiny)
        pol.fused_sample_p2(obs, a, lp, seed=seed ^ _SALT, counter=counter, mirror=True)
        torch.cuda.synchronize()
        chk2.add(b3, u2, a.cpu().numpy(), lp.cpu().numpy(), mirror=True, tiny_action=tiny)
    chk1.finish()
    chk2.finish()


DRAW_SITES = ("bot_h32", "bot_h64", "bot_h128", "mt2_bot", "frame_delay3", "self_play_mirror", "mt2_self_play_mirror",
              "pool3_bot")


@gpu
@pytest.mark.parametrize("site", DRAW_SITES)
def test_rollout_kernels_draw_for_draw(monkeypatch, site):
    """Three consecutive collects of the whole-horizon kernel (the counter advances by the horizon) on exact logits:
    P1 draws with (seed, drawn + t, first_env_index + i), P2 with seed ^ salt and the mirrored-back action, each pool
    member from its own b3 on its own range."""
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    if site.startswith("mt2_"):
        monkeypatch.setenv("FOOTSIES_B200_ROLLOUT_MT", "2")
    dev = _dev()
    hidden = int(site[5:]) if site.startswith("bot_h") else 64
    n, horizon, seed, first = 1100, 100, 0x0DDBA11C0FFEE, 40_000
    vecs = _b3_vectors()
    p1_vecs = ("peaky", "tiny", "spread")            # P1's b3 in collect 0, 1, 2
    pol = _exact_logit_policy(hidden, vecs["peaky"], dev)
    p2 = pool = None
    if site in ("self_play_mirror", "mt2_self_play_mirror", "pool3_bot"):
        env = FootsiesEnv(num_envs=n, device=dev, seed=5, opponent="self_play", first_env_index=first)
        if site == "pool3_bot":
            pool = [_exact_logit_policy(hidden, vecs[k], dev, seed=s) for s, k in ((2, "tied"), (3, "spread"), (4, "tiny"))]
            pool.append("bot")
        else:
            p2 = _exact_logit_policy(hidden, vecs["uniform"], dev, seed=2)
    else:
        env = FootsiesEnv(num_envs=n, device=dev, seed=5, first_env_index=first,
                          frame_delay=3 if site == "frame_delay3" else 0)
    col = RolloutCollector(env, pol, horizon=horizon, seed=seed, opponent_policy=p2, mirror_opponent=p2 is not None or
                           pool is not None, opponent_pool=pool)
    assert col.mode == "horizon"
    chk1, chk2 = DrawCheck(f"rollout {site} P1"), DrawCheck(f"rollout {site} P2")
    idx = first + np.arange(n, dtype=np.uint64)
    for c in range(3):
        # P1's b3 changes between collects (the kernel reads the weights at every launch)
        b3 = vecs[p1_vecs[c]]
        with torch.no_grad():
            pol.net[4].bias.copy_(torch.as_tensor(np.asarray(b3, np.float32), device=dev))
        out = col.collect()
        torch.cuda.synchronize()
        t = np.arange(c * horizon, (c + 1) * horizon, dtype=np.uint64)[:, None]
        u1 = uniform24(hash3(seed, t, idx[None, :]))
        chk1.add(b3, u1.ravel(), out["actions"].cpu().numpy().ravel(), out["logp"].cpu().numpy().ravel(),
                 tiny_action=3 if p1_vecs[c] == "tiny" else None)
        u2 = uniform24(hash3(seed ^ _SALT, t, idx[None, :]))
        a2, l2 = (out["actions_p2"].cpu().numpy(), out["logp_p2"].cpu().numpy()) if "actions_p2" in out else (None, None)
        if p2 is not None:
            chk2.add(vecs["uniform"], u2.ravel(), a2.ravel(), l2.ravel(), mirror=True)
        if pool is not None:
            for k, (lo, hi) in enumerate(col.opponent_ranges):
                if pool[k] == "bot" or lo == hi:
                    continue
                kb3 = pool[k].net[4].bias.detach().cpu().numpy()
                chk2.add(kb3, u2[:, lo:hi].ravel(), a2[:, lo:hi].ravel(), l2[:, lo:hi].ravel(), mirror=True,
                         tiny_action=3 if k == 2 else None)
    chk1.finish()
    if p2 is not None or pool is not None:
        chk2.finish()


@gpu
@pytest.mark.parametrize("hidden", [64, 128])
def test_rollout_action_counts_follow_float64_probabilities(hidden):
    """General weights (x3): over 2^20 rollout draws the count of every action is within 6 sigma of the sum of its
    float64 probabilities on the observations the policy saw."""
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import RolloutCollector
    dev = _dev()
    n, horizon = 8192, 128
    pol = _net("policy", hidden, "x3", dev, seed=1)
    col = RolloutCollector(FootsiesEnv(num_envs=n, device=dev, seed=9), pol, horizon=horizon, seed=99)
    out = col.collect()
    torch.cuda.synchronize()
    p = _policy_logp64(pol, out["obs"].reshape(-1, 8)).exp()
    expect, var = p.sum(0), (p * (1 - p)).sum(0)
    counts = torch.bincount(out["actions"].reshape(-1).long(), minlength=8).double()
    z = ((counts - expect) / var.clamp_min(1e-12).sqrt()).cpu().numpy()
    print(f"H={hidden}: {n * horizon} draws, counts {counts.tolist()}, z {np.round(z, 2).tolist()}")
    assert np.all(np.abs(z) < 6.0), z
