"""The CPU oracle (oracle/footsies_oracle.c, the hand-written restatement every GPU parity test is judged by) against
the REFERENCE'S OWN battle code: /root/reference/Assets/Script/*.cs transliterated mechanically by tools/cs2cpp.py and
compiled into oracle/_ref/libfootsies_ref.so (oracle/Makefile.ref; harness oracle/ref_shim/ref_harness.cpp).

The transliteration is generated from the reference's source and never committed.  Where it is not built, each test
compares the oracle's traces with stored ones instead: one 64-bit digest per step, in tests/golden/ref_trace_digests.npz.
Those digests were recorded from the oracle as of commit a4b2496.  Its source had not changed since the last run beside
the reference engine (profiles/r03_oracle_vs_ref_fuzz.log: 479 random configurations, every trace byte-identical).
Where the engine is built, every comparison runs against it directly, and FOOTSIES_RECORD_TRACE_DIGESTS=1 rewrites the
stored digests from that run.

Every tape of tests/parity_cases.py -- the same seeded action sequences the CUDA path replays on the B200 -- goes through
both engines; after reset and after every step EVERY field of the trace must be byte-identical: fighter state incl. the
Left / Right history and the Attack run length read from the real 180-entry arrays, frame counter, recorded inputs,
hit / block / guard-break events, battle_over, the xorshift128 state and draw count, the bots' held inputs, observation,
info, reward (float64 and float32), termination.  Bar: bit-exact, floats compared as bytes (0 ulp).

This is the pin SURVEY.md section 8(c) asks for: a shared misreading of the C# between the oracle and the known-answer
tests can no longer pass, because the second engine is the C# text itself.  What stays unpinned is only what is NOT in
/root/reference (closed-source UnityEngine.Random / Rect / Time and Mono's fp32 evaluation), restated in
oracle/ref_shim/unity_shim.h and stated as such in DESIGN.md."""
import functools
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_binding as ob
import parity_cases as pc
import ref_binding as rb

needs_ref_engine = pytest.mark.skipif(not rb.available(), reason="the transliterated reference engine (oracle/_ref) is not built")

EVENT_MASK = 0x3F      # bits 6-7 (proximity notification) are instrumentation inside the hand-written oracle only
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_trace_digests.npz")
RECORD = os.environ.get("FOOTSIES_RECORD_TRACE_DIGESTS") == "1"
_recorded = {}


def assert_traces_equal(o, r, where):
    for name in ob.TRACE_DTYPE.names:
        a, b = o[name], r[name]
        if name == "events":
            a, b = a & EVENT_MASK, b & EVENT_MASK
        if a.tobytes() == b.tobytes():
            continue
        if a.dtype.names:
            for f in a.dtype.names:
                if a[f].tobytes() != b[f].tobytes():
                    i = tuple(np.argwhere(a[f] != b[f])[0])
                    raise AssertionError(f"[{where}] f.{f} differs at (env, player) {i}: oracle={a[f][i]!r} reference={b[f][i]!r}")
        i = tuple(np.argwhere(a != b)[0])
        raise AssertionError(f"[{where}] {name} differs at {i}: oracle={a[i]!r} reference={b[i]!r}")


def trace_digest(trace, fields=None):
    """64-bit digest of the trace fields of every battle (events without the oracle-only bits), in TRACE_DTYPE order."""
    h = hashlib.blake2b(digest_size=8)
    for name in fields or ob.TRACE_DTYPE.names:
        a = trace[name]
        h.update(np.ascontiguousarray(a & EVENT_MASK if name == "events" else a).tobytes())
    return int.from_bytes(h.digest(), "little")


class ReferenceSide:
    """The reference side of one comparison: the transliterated engine when it is built (stepped alongside the oracle,
    traces compared field by field), else the per-step trace digests stored under `key` in GOLDEN."""

    def __init__(self, key, n, fields=None, **kw):
        self.key, self.fields, self.digests = key, fields, []
        self.engine = rb.RefBatch(n, **kw) if rb.available() else None
        self.expected = None
        if self.engine is None and not RECORD:
            with np.load(GOLDEN) as g:
                assert key in g.files, f"no recorded reference traces for {key}"
                self.expected = g[key]

    # the engine, if any, gets the same calls as the oracle
    def reset(self, mask=None):
        if self.engine is not None:
            self.engine.reset(mask)

    def step(self, a1, a2=None, repeat=1):
        if self.engine is not None:
            self.engine.step(a1, a2, repeat=repeat)

    def seed(self, seed_base, mask=None):
        if self.engine is not None:
            self.engine.seed(seed_base, mask)

    def set_rng_tape(self, env, raw):
        if self.engine is not None:
            self.engine.set_rng_tape(env, raw)

    def _check(self, digest, where):
        i = len(self.digests)
        self.digests.append(digest)
        if self.expected is not None:
            assert i < len(self.expected) and int(self.expected[i]) == digest, \
                f"[{where}] the oracle's trace differs from the recorded one"

    def check(self, o_trace, where):
        if self.engine is not None:
            if self.fields:
                for name in self.fields:
                    assert o_trace[name].tobytes() == self.engine.trace[name].tobytes(), (where, name)
            else:
                assert_traces_equal(o_trace, self.engine.trace, where)
        self._check(trace_digest(o_trace, self.fields), where)

    def check_totals(self, o):
        st = o.stats()
        if self.engine is not None:
            sr = self.engine.stats()
            assert st == sr, (st, sr)
            assert o.frames_simulated() == self.engine.frames_simulated()
        blob = json.dumps([st, o.frames_simulated()], sort_keys=True).encode()
        self._check(int.from_bytes(hashlib.blake2b(blob, digest_size=8).digest(), "little"), "stats")
        return st

    def finish(self):
        if RECORD:
            _recorded[self.key] = np.array(self.digests, dtype=np.uint64)


@pytest.fixture(scope="module", autouse=True)
def _write_recorded_digests():
    yield
    if RECORD and _recorded:
        stored = dict(np.load(GOLDEN)) if os.path.exists(GOLDEN) else {}
        stored.update(_recorded)
        np.savez_compressed(GOLDEN, **stored)


@pytest.fixture
def reference(request):
    """reference(n, fields=None, **batch kwargs) -> a ReferenceSide keyed by the test's name and call order."""
    made = []

    def make(n, fields=None, **kw):
        made.append(ReferenceSide(f"{request.node.name}#{len(made)}", n, fields, **kw))
        return made[-1]
    yield make
    for side in made:
        side.finish()


def run_pair(reference, make_env, oracle, n, steps, *, p1_bot=False, p2_bot=True, dense=True, frame_skip=1, autoreset=True, stale=True,
             seed=0, tape1=None, tape2=None, first_env_index=0, check_every=1, frame_delay=0):
    """Drop-in for parity_cases.run_case: same tapes, but the two implementations under comparison are the two CPU engines."""
    kw = dict(p1_bot=p1_bot, p2_bot=p2_bot, dense_reward=dense, autoreset=autoreset, stale_intro_input=stale,
              first_env_index=first_env_index, seed=seed, threads=8, frame_delay=frame_delay)
    o, r = ob.OracleBatch(n, **kw), reference(n, **kw)
    o.reset()
    r.reset()
    r.check(o.trace, "reset")
    zero = np.zeros(n, np.uint8)
    for t in range(steps):
        a1 = zero if p1_bot else tape1[t]
        a2 = None if p2_bot else tape2[t]
        o.step(a1, a2, repeat=frame_skip)
        r.step(a1, a2, repeat=frame_skip)
        r.check(o.trace, f"step {t}")
    st = dict(r.check_totals(o))
    st["episode_frames"] = st.pop("frames")
    return st


CASES = [name for name in dir(pc) if name.startswith("case_") and name != "case_fused_frame_skip"]


@pytest.mark.parametrize("name", CASES, ids=[c[5:] for c in CASES])
def test_every_parity_tape_oracle_equals_transliterated_reference(monkeypatch, reference, name):
    monkeypatch.setattr(pc, "run_case", functools.partial(run_pair, reference))
    # config B (the trace bit-exactness gate) at 512 battles x 2048 frames; the others at 1/16 of their GPU size
    getattr(pc, name)(None, None, scale=0.125 if name.startswith("case_config_b") else 0.0625)


@pytest.mark.parametrize("k,p2_bot", pc.FUSED_PARAMS)
def test_frame_skip_tapes_oracle_equals_transliterated_reference(monkeypatch, reference, k, p2_bot):
    monkeypatch.setattr(pc, "run_case", functools.partial(run_pair, reference))
    pc.case_fused_frame_skip(None, None, k, p2_bot, scale=0.03125)


@pytest.mark.parametrize("frame_delay,dense", [(3, True), (1, False)])
def test_frame_delay_queue(reference, frame_delay, dense):
    rng = np.random.default_rng(17)
    n, steps = 96, 900
    run_pair(reference, None, None, n, steps, dense=dense, frame_delay=frame_delay, tape1=pc.tape_sticky(rng, steps, n), seed=5)


@pytest.mark.parametrize("by_example", [False, True])
def test_masked_hard_reset_and_reseed_mid_episode(reference, by_example):
    """RESET command in the middle of an episode (BattleCore.cs:143-146) and SEED (:170-173) on a subset of the battles;
    by_example: P1's spectator-wrapped bot is not Reset() by the new round."""
    rng = np.random.default_rng(8)
    n = 128
    kw = dict(p1_bot=by_example, p2_bot=True, seed=1, threads=8)
    o, r = ob.OracleBatch(n, **kw), reference(n, **kw)
    o.reset()
    r.reset()
    for t in range(700):
        a = rng.integers(0, 8, size=n, dtype=np.uint8)
        o.step(a)
        r.step(a)
        if t % 50 == 25:
            mask = rng.random(n) < 0.3
            for b in (o, r):
                b.seed(1000 + t, mask)
                b.reset(mask)
        r.check(o.trace, f"step {t}")


def test_bot_decisions_on_injected_draw_tapes(reference):
    """The bot's decision tree on a chosen draw sequence (tests of BattleAI.SelectMovement / SelectAttack branches that a
    seeded stream visits rarely): both engines consume the same raw 32-bit draws."""
    rng = np.random.default_rng(99)
    n, steps = 64, 1200
    kw = dict(p1_bot=False, p2_bot=True, seed=0, threads=1)
    o, r = ob.OracleBatch(n, **kw), reference(n, fields=("f", "frame", "bot_input", "rng_draws", "obs", "reward", "terminated"), **kw)
    for e in range(n):
        raw = rng.integers(0, 2 ** 32, size=4000, dtype=np.uint64).astype(np.uint32)
        o.set_rng_tape(e, raw)
        r.set_rng_tape(e, raw)
    o.reset()
    r.reset()
    tape = pc.tape_sticky(rng, steps, n)
    for t in range(steps):
        o.step(tape[t])
        r.step(tape[t])
        r.check(o.trace, f"step {t}")


@needs_ref_engine
def test_save_load_battle_state_through_the_games_own_commands():
    """STATE_SAVE / STATE_LOAD (BattleCore.SaveState / LoadState, Fighter.SaveState / LoadState, FighterState ctor --
    all transliterated): saved states are identical, and a state saved by one engine continues identically in the other."""
    rng = np.random.default_rng(23)
    n, steps = 48, 400
    kw = dict(p2_bot=False, seed=0, threads=1)
    o, r = ob.OracleBatch(n, **kw), rb.RefBatch(n, **kw)
    o.reset()
    r.reset()
    t1, t2 = pc.tape_sticky(rng, steps, n), pc.tape_sticky(rng, steps, n)
    saved = {}
    for t in range(steps):
        o.step(t1[t], t2[t])
        r.step(t1[t], t2[t])
        if t % 37 == 5:
            for e in range(0, n, 5):
                so, sr = o.save_battle_state(e), r.save_battle_state(e)
                so.pop("roundStartTime"), sr.pop("roundStartTime")      # wall-clock bookkeeping, not battle state
                assert so == sr, (t, e)
                if not (o.trace["terminated"][e] or e in saved):
                    saved[e] = (t, r.save_battle_state(e))
    # cross-load: what the reference engine saved goes into the oracle (and back into the reference), then both continue
    assert len(saved) >= 5
    for e, (t, state) in saved.items():
        if o.trace["terminated"][e]:
            continue
        o.load_battle_state(e, state)
        r.load_battle_state(e, state)
    for t in range(200):
        a1, a2 = t1[t], t2[t]
        o.step(a1, a2)
        r.step(a1, a2)
        # reward included: after a load both engines reward the next step against the guard bars the agent saw last
        # (footsies.py:530, 556-558), and the episode's cumulative reward runs on across the load
        for name in ("f", "frame", "obs", "terminated", "battle_over", "reward", "reward_f64"):
            assert o.trace[name].tobytes() == r.trace[name].tobytes(), (t, name)


@pytest.mark.parametrize("engine", ["oracle", pytest.param("reference_transliteration", marks=needs_ref_engine)])
@pytest.mark.parametrize("dense,p2_bot", [(True, True), (False, True), (True, False)])
def test_reference_held_invariants_on_the_cpu_engines(engine, dense, p2_bot):
    """tests/invariants.py (observation_space bounds, episode reward sum == +-1, three blocks then guard break) over both
    CPU engines; the B200 tests run the same checker over a million battles."""
    import torch
    from invariants import ReferenceInvariants
    rng = np.random.default_rng(31)
    n, steps = 192, 1500
    cls = ob.OracleBatch if engine == "oracle" else rb.RefBatch
    b = cls(n, p2_bot=p2_bot, dense_reward=dense, seed=2, threads=8)
    inv = ReferenceInvariants(n, "cpu", dense=dense)

    def tensors(tr):
        misc = np.concatenate([tr["info_action"], tr["info_hitstun"]], axis=1).astype(np.uint8)
        return (torch.from_numpy(tr["obs"].copy()), torch.from_numpy(tr["reward"].copy()),
                torch.from_numpy(tr["terminated"].astype(bool)), torch.from_numpy(tr["info_frame"].copy()), torch.from_numpy(misc))
    obs, _, _, frame, misc = tensors(b.reset())
    inv.reset(obs, frame, misc)
    t1 = pc.tape_sticky(rng, steps, n, weights=[1, 1, 3, 0.3, 2, 0.5, 2, 0.3])
    t2 = pc.tape_sticky(rng, steps, n, weights=[1, 0.5, 5, 0.2, 1, 0.2, 1, 0.1])
    for t in range(steps):
        inv.update(*tensors(b.step(t1[t], None if p2_bot else t2[t])), where=f"step {t}")
    assert inv.episodes > 50 and inv.blocks > 20 and (p2_bot or inv.breaks > 0)
