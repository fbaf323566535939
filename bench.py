#!/usr/bin/env python3
"""Throughput benchmark of the batched FOOTSIES frame update (BASELINE.json metric: env-frames/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--envs-per-gpu E] [--dump-outputs DIR]

One "step" = one FootsiesEnv.step over every env of the rank (frame-skip 1: one BattleCore fight frame per
env).  Workload (config D of SURVEY.md §8, weak-scaled so that each GPU's working set exceeds the 126 MB L2):
random-action P1 (iid uniform over the 8 input bitmasks) vs the in-game BattleAI, auto-reset on KO.
Env-frames are counted by the kernel's own simulated-frame counter, not as N x K.

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (CUDA events, max over ranks);
`e2e` = the same metric through the host-buffer C-ABI call (pinned host actions in, results out);
`roofline` = algorithmic HBM bytes per launch / measured launch time vs MEASURED_PEAKS.json;
`cpu_baseline` = the reference's own battle code on this box's host cores (rank 0, N = 1 only): oracle/_ref, the C# compiled
natively through the mechanical transliteration of tools/cs2cpp.py (kind "reference"; the prebuilt library travels with the
snapshot), with the hand-written C restatement (kind "port") beside it in `cpu_baseline_c_port`.
`--impl reference` times that CPU path alone on the same workload definition.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "env_frames_per_sec"
UNIT = "env-frames/s"
DEFAULT_ENVS_PER_GPU = 4 * 1024 * 1024
STRONG_WORKLOAD = ("D: random-action P1 vs in-game BattleAI, frame-skip 1, auto-reset, {t} envs sharded over {w} GPU(s) "
                   "(BASELINE configs[3]; per-GPU shards below ~2 Mi envs fit the 126 MB L2)")
WORKLOAD = ("D-weak: random-action P1 vs in-game BattleAI, frame-skip 1, auto-reset, "
            "{n} envs per GPU (BASELINE configs[3] weak-scaled so the per-GPU working set exceeds L2)")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=DEFAULT_ENVS_PER_GPU)
    ap.add_argument("--total-envs", type=int, default=0,
                    help="strong scaling: shard this many envs over the ranks (BASELINE configs[3]: 1048576); "
                         "default 0 = weak scaling with --envs-per-gpu envs on every GPU")
    ap.add_argument("--burnin", type=int, default=600,
                    help="untimed steps before the warm-up so that episodes are desynchronised (steady state)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 20)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work budget of the cpu_baseline leg")
    ap.add_argument("--workload", default="step", choices=["step", "rollout"],
                    help="step (default): the single-frame step kernel, BASELINE's headline metric; rollout: BASELINE "
                         "configs[4], 16384 envs per GPU x 128-step horizon with the fused MLP policy kernel in the loop "
                         "(one horizon = one bench step), weak scaling, one stats all-reduce at the end")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (rank 0, a fixed seeded sample "
                         "of the envs) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def dump_outputs(out_dir, n, sample, arrays):
    """Writes each device tensor of `arrays` ({name: (tensor, env axis)}) at a fixed, seeded sample of `sample` of the
    N envs as float32 (float64 for integers wider than 16 bits, which float32 may not hold exactly), plus the sampled
    env indices.  The caller picks `sample` so that the whole dump stays under 64 MB."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, sample), replace=False))
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    for name, (t, axis) in arrays.items():
        a = t.index_select(axis, torch.from_numpy(idx).to(t.device)).cpu().numpy()
        wide = a.dtype.kind in "iu" and a.dtype.itemsize > 2
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64 if wide else np.float32))


def measured_traffic(bytes_per_env_alg, n):
    """DRAM bytes per launch of the step kernel from the committed `ncu --set full` capture (profiles/traffic.json,
    written by tools/ncu_summary.py from dram__bytes_read.sum + dram__bytes_write.sum), scaled to this launch's envs."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(path))
        return float(t["dram_bytes_per_env_step"]) * n, t.get("source")
    except Exception:  # noqa: BLE001
        return None, None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:  # noqa: BLE001
                self.proc.kill()

    def summary(self, t0, t1):
        rows = []
        for ts, ln in self.lines:
            if t0 <= ts <= t1 + 0.06:
                parts = [x.strip() for x in ln.split(",")]
                if len(parts) >= 9:
                    rows.append(parts)
        if not rows:
            return None
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows)}


def cpu_engine(kind):
    """("reference" | "port", batch class, library): oracle/_ref -- the reference's own C# battle code compiled through the
    mechanical transliteration of tools/cs2cpp.py (prebuilt, travels with the snapshot) -- or the C restatement oracle/."""
    import oracle_binding as ob
    if kind == "reference":
        import ref_binding as rb
        if rb.available():
            try:
                return "reference", rb.RefBatch, rb.lib()
            except Exception as e:  # noqa: BLE001
                print(f"oracle/_ref unavailable ({e}); falling back to the C port", file=sys.stderr)
    return "port", ob.OracleBatch, ob.lib()


def cpu_throughput(kind, n_envs, threads, seconds=None, steps=None, warmup=3, seed=1234, inner=1):
    """The CPU path on the same workload definition (random P1 vs BattleAI, frame-skip 1, auto-reset) on `threads` host
    threads; timed for `seconds` or for exactly `steps` steps, a step being `inner` consecutive env-steps of the sample batch
    (so that `--steps 20` is seconds of CPU work, not milliseconds).  Returns (kind, frames/s, frames, elapsed, steps)."""
    import numpy as np
    kind, cls, L = cpu_engine(kind)
    orc = cls(n_envs, p2_bot=True, seed=0, threads=threads)
    L.fo_reset(orc.h, None, None)
    rng = np.random.default_rng(seed)
    tapes = [rng.integers(0, 8, size=n_envs, dtype=np.uint8) for _ in range(16)]
    for i in range(warmup * inner):
        L.fo_step(orc.h, tapes[i % 16].ctypes.data, None, 1, None, threads)
    f0 = orc.frames_simulated()
    t0 = time.perf_counter()
    done = 0
    while True:
        for j in range(inner):
            L.fo_step(orc.h, tapes[(done * inner + j) % 16].ctypes.data, None, 1, None, threads)
        done += 1
        if (steps is not None and done >= steps) or (seconds is not None and time.perf_counter() - t0 >= seconds):
            break
    dt = time.perf_counter() - t0
    frames = orc.frames_simulated() - f0
    return kind, frames / dt, frames, dt, done


REF_STEP_ENV_STEPS = 256
REF_SAMPLE_ENVS = {"reference": 4096, "port": 32768}     # a transliterated game object graph is ~0.6 MB per battle


def cpu_baseline_entry(kind, threads, seconds=None, steps=None, warmup=3, inner=1):
    kind, v, frames, dt, done = cpu_throughput(kind, REF_SAMPLE_ENVS[kind], threads, seconds=seconds, steps=steps, warmup=warmup,
                                               inner=inner)
    what = ("oracle/_ref: the reference's own Assets/Script battle code (BattleCore, Fighter, BattleAI, ...) transliterated "
            "mechanically into C++ (tools/cs2cpp.py) and compiled natively" if kind == "reference"
            else "oracle/: scalar C restatement of the reference's battle code")
    sample = (f"{REF_SAMPLE_ENVS[kind]} envs x {done * inner} steps ({frames} env-frames, {dt:.1f} s) of the same random-vs-bot workload "
              f"on {threads} host threads; {what} (the Unity game binary itself cannot run offline)")
    return {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample}, dt, done


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores: oracle/_ref (the
    reference's C# compiled through the transliteration) when it is there, else the C port; rank 0 only."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    # one `step` of this arm = REF_STEP_ENV_STEPS consecutive env-steps of the 4096-battle sample (~1 M env-frames: a few
    # tenths of a second on a many-core host), so that `--steps 20` times seconds of CPU work
    base, dt, done = cpu_baseline_entry("reference", threads, steps=args.steps, warmup=min(args.warmup, 3),
                                        inner=REF_STEP_ENV_STEPS)
    port, _, _ = cpu_baseline_entry("port", threads, seconds=3.0)
    value = base["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": done, "warmup": min(args.warmup, 3), "ms_per_step": dt / max(done, 1) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32+fp32", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(n=args.envs_per_gpu), "reference_sample": base["sample"],
                   "note": "reference game binary + FootsiesEnv not runnable offline (no Unity/mono, no binary); this is its "
                           "battle code compiled natively (kind 'reference') -- far faster than the game process, whose "
                           "configured ceiling is 300 env-frames/s; the hand-written C restatement is timed beside it",
                   "c_port_beside_it": port},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def emit(line):
    """The one JSON line goes to the process's ORIGINAL stdout; everything else any library prints to fd 1 while the
    benchmark runs (e.g. NCCL's version banner) is diverted to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)


def run_rollout(args, rank, world, dev, dist):
    """--workload rollout: BASELINE configs[4] on N GPUs.  One bench step = one 128-step horizon for 16384 envs per
    GPU, one launch of the whole-horizon rollout kernel (fg_rollout_mlp: MLP policy inference + sampling + simulator step,
    battle state in registers for the whole horizon, rollout buffers written in place)."""
    import torch
    from footsies_gym_b200 import FootsiesEnv
    from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
    n, horizon = 16384, 128
    steps = args.steps
    env = FootsiesEnv(num_envs=n, device=dev, opponent=None, seed=0, first_env_index=rank * n)
    torch.manual_seed(0)
    col = RolloutCollector(env, MLPPolicy(64).to(dev), horizon=horizon, use_cuda_graph=True, seed=rank)
    assert col.mode == "horizon", col.mode
    for _ in range(max(args.warmup, 3)):
        col.collect()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    f0 = env.episode_stats()["env_frames"]
    l0 = env.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = col.collect()
    e1.record()
    torch.cuda.synchronize(dev)
    if args.dump_outputs and rank == 0:
        # obs [horizon, N, 8], actions / logp / rewards / dones [horizon, N], last_obs [N, 8]: ~6 KB per env
        dump_outputs(args.dump_outputs, n, 4096, {k: (v, 0 if k == "last_obs" else 1) for k, v in out.items()})
    if world > 1:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    f = torch.tensor([env.episode_stats()["env_frames"] - f0], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(f, op=dist.ReduceOp.SUM)
    stats = env.all_reduce_stats()
    if rank == 0:
        ms = float(t.item())
        emit({"metric": METRIC, "value": int(f.item()) / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
              "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
              "vs_baseline": None, "dtype": "int32+fp32", "data": "synthetic",
              "config": {"workload": "E: PPO rollout, MLP 8-64-64-8 policy fused with the simulator step into one launch per "
                                     "horizon (fg_rollout_mlp), 16384 envs per GPU x 128-step horizon per bench step, "
                                     "vs in-game BattleAI, frame-skip 1 (BASELINE configs[4])",
                         "envs_per_gpu": n, "horizon": horizon, "l2": "working set fits L2 (latency-bound regime); not the "
                         "roofline workload"},
              "gpu_launches": env.launch_count() - l0, "episode_stats_all_ranks": stats})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    sys.stdout.flush()
    os.dup2(2, 1)
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from footsies_gym_b200 import FootsiesEnv, _capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the one JSON line: whatever NCCL_DEBUG level the caller chose goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    if args.workload == "rollout":
        run_rollout(args, rank, world, dev, dist)
        return
    if args.total_envs > 0:
        from footsies_gym_b200.distributed import shard_range
        first_index, n = shard_range(args.total_envs, rank, world)
    else:
        n, first_index = args.envs_per_gpu, rank * args.envs_per_gpu
    env = FootsiesEnv(num_envs=n, device=dev, opponent=None, seed=0, first_env_index=first_index)
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    n_tapes = 8
    tapes = [torch.randint(0, 8, (n,), generator=gen, device=dev, dtype=torch.uint8) for _ in range(n_tapes)]

    def device_step(i):
        env.bind_actions(tapes[i % n_tapes])     # zero-copy: the kernel reads the resident tape directly
        env.step_bound()

    # burn-in: all envs start synchronised on frame -1 (low divergence, optimistic); run until episodes have
    # desynchronised so that the timed region measures the steady state of a long rollout
    for i in range(args.burnin):
        device_step(i)
    for i in range(max(args.warmup, 3)):
        device_step(i)
    torch.cuda.synchronize(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)

    # ---------------- timed region: exactly `steps` device-resident steps, back to back ----------------
    # an event after every block of `block` steps gives the spread; the value is the whole window
    block = max(1, args.steps // 25)
    barrier()
    # a few untimed lead-in steps keep the GPU busy while the window opens, so that a short window does not time the
    # idle GPU's start-up; the frame counter is snapshotted in stream order where the window begins
    for i in range(4):
        device_step(i)
    env_frames = _capi.STAT_NAMES.index("env_frames")
    frames_before = env.stats[env_frames].clone()
    launches_before = env.launch_count()
    events, marks = [torch.cuda.Event(enable_timing=True)], [0]
    wall0 = time.time()
    events[0].record()
    for i in range(args.steps):
        device_step(i)
        if (i + 1) % block == 0 or i + 1 == args.steps:
            events.append(torch.cuda.Event(enable_timing=True))
            events[-1].record()
            marks.append(i + 1)
    barrier()
    wall1 = time.time()
    if args.dump_outputs and rank == 0:
        # what step_bound() returned for the last timed step: obs [N, 8], reward, terminated, truncated, info frame /
        # actions / hitstun (info's observation keys are views of obs); ~76 bytes per env
        dump_outputs(args.dump_outputs, n, 1 << 18,
                     {"obs": (env.obs, 0), "reward": (env.reward, 0), "terminated": (env.terminated, 0),
                      "truncated": (env.truncated, 0), "info_frame": (env.info_frame, 0), "info_misc": (env.info_misc, 0)})
    ms_local = events[0].elapsed_time(events[-1])
    per_step_ms = sorted(events[j].elapsed_time(events[j + 1]) / (marks[j + 1] - marks[j]) for j in range(len(events) - 1))
    frames_local = int((env.stats[env_frames] - frames_before).item())
    launches = env.launch_count() - launches_before

    clocks = None
    if rank == 0:
        clocks = sampler.summary(wall0, wall1) or {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        clocks["sampled"] = "nvidia-smi -lms 50 during the %d timed steps (%.2f s)" % (args.steps, wall1 - wall0)
        sampler.stop()

    t = torch.tensor([ms_local, -per_step_ms[0], per_step_ms[-1]], dtype=torch.float64, device=dev)
    f = torch.tensor([frames_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(f, op=dist.ReduceOp.SUM)
    ms_total, ms_step_min, ms_step_max = float(t[0].item()), -float(t[1].item()), float(t[2].item())
    frames_total = float(f.item())
    value = frames_total / (ms_total * 1e-3)

    # ---------------- e2e: the host-buffer C-ABI call (pinned host actions in, results out), median of blocks -------------
    e2e_steps = args.e2e_steps or min(args.steps, 20)
    host_tapes = [tp.cpu().pin_memory() for tp in tapes[:4]]
    env.bind_actions(torch.zeros(n, dtype=torch.uint8, device=dev))   # staging buffer for the host actions

    def e2e_measure(call, e2e_blocks=9):
        for i in range(2):
            call(host_tapes[i % 4])
        fb = env.episode_stats()["env_frames"]
        barrier()
        dts = []
        for b in range(e2e_blocks):
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                call(host_tapes[i % 4])          # returns when the results are in host memory
            dts.append(time.perf_counter() - t0)
        torch.cuda.synchronize(dev)
        fr = (env.episode_stats()["env_frames"] - fb) / e2e_blocks
        dts.sort()
        te = torch.tensor([dts[len(dts) // 2], -dts[0], dts[-1]], dtype=torch.float64, device=dev)
        fe = torch.tensor([fr], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
            dist.all_reduce(fe, op=dist.ReduceOp.SUM)
        return float(fe.item()) / float(te[0].item()), float(fe.item()) / float(te[2].item()), float(fe.item()) / -float(te[1].item())

    e2e_value, e2e_lo, e2e_hi = e2e_measure(env.step_host_packed)
    h2d, d2h = env.host_io_bytes_per_step(packed=True)
    e2e_compact_value, _, _ = e2e_measure(env.step_host)
    h2d_c, d2h_c = env.host_io_bytes_per_step()

    # ---------------- end-of-rollout statistics all-reduce (the only collective on the path) ----------------
    stats = env.all_reduce_stats()

    # ---------------- extras every rank takes part in: BASELINE configs[3] as written and configs[4] ----------------
    extra = {}

    def agg(ms, frames):
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        ff = torch.tensor([frames], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(ff, op=dist.ReduceOp.SUM)
        return float(tt.item()), float(ff.item())

    if not args.no_extra:
        from footsies_gym_b200.distributed import shard_range
        total = 1 << 20
        first_s, n_s = shard_range(total, rank, world)
        es = FootsiesEnv(num_envs=n_s, device=dev, opponent=None, seed=0, first_env_index=first_s)
        es.reset()
        ts = [torch.randint(0, 8, (n_s,), generator=gen, device=dev, dtype=torch.uint8) for _ in range(4)]

        def one_s(i):
            es.bind_actions(ts[i % 4])
            es.step_bound()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for i in range(300):
                one_s(i)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        gs = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gs):
            for i in range(200):
                one_s(i)
        gs.replay()
        barrier()
        f0 = es.episode_stats()["env_frames"]
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(5):
            gs.replay()
        s1.record()
        barrier()
        ms_s, fr_s = agg(s0.elapsed_time(s1), es.episode_stats()["env_frames"] - f0)
        hs = [tp.cpu().pin_memory() for tp in ts]
        for i in range(2):
            es.step_host_packed(hs[i % 4])
        f0 = es.episode_stats()["env_frames"]
        barrier()
        t0 = time.perf_counter()
        for i in range(40):
            es.step_host_packed(hs[i % 4])
        dt_s = time.perf_counter() - t0
        ms_e, fr_e = agg(dt_s * 1e3, es.episode_stats()["env_frames"] - f0)
        es.close()
        extra["D_1048576_envs_sharded_strong"] = {
            "env_frames_per_sec": fr_s / (ms_s * 1e-3), "ms_per_step": ms_s / 1000.0, "e2e_env_frames_per_sec": fr_e / (ms_e * 1e-3),
            "total_envs": total, "envs_per_gpu": n_s, "n_gpus": world, "scaling": "strong",
            "note": "BASELINE configs[3] as written: 1 048 576 envs sharded over the ranks by global env index, random P1 vs "
                    "BattleAI, frame-skip 1; CUDA-graph replay of 5 x 200 launches, max over ranks; shards fit the 126 MB L2 "
                    "(latency-bound regime, not the roofline workload); e2e = fg_step_host_packed, 40 calls"}

        from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
        er = FootsiesEnv(num_envs=16384, device=dev, opponent=None, seed=0, first_env_index=rank * 16384)
        torch.manual_seed(0)
        col = RolloutCollector(er, MLPPolicy(64).to(dev), horizon=128, use_cuda_graph=True, seed=0)
        for _ in range(3):
            col.collect()
        barrier()
        f0 = er.episode_stats()["env_frames"]
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(50):
            col.collect()
        s1.record()
        barrier()
        ms_r, fr_r = agg(s0.elapsed_time(s1), er.episode_stats()["env_frames"] - f0)
        er.close()
        extra["E_ppo_rollout_16384_per_gpu"] = {
            "env_frames_per_sec": fr_r / (ms_r * 1e-3), "ms_per_horizon": ms_r / 50.0, "n_gpus": world, "mode": col.mode,
            "note": "BASELINE configs[4] on every rank: 16384 envs per GPU x 128-step horizon, MLP 8-64-64-8 policy + sampling + "
                    "simulator step in ONE launch per horizon (fg_rollout_mlp); 50 horizons, max over ranks, frames summed"}

    # ---------------- extra single-GPU workloads (parity-gate configs, informational) ----------------
    if rank == 0 and world == 1 and not args.no_extra:
        def quick(n_envs, frame_skip, self_play, steps=200):
            """Device-resident throughput of another configuration; the `steps` launches are captured into one CUDA
            graph and replayed, so that small batches are not timed on the Python launch overhead (~15 us/step)."""
            e = FootsiesEnv(num_envs=n_envs, device=dev, opponent="self_play" if self_play else None,
                            frame_skip=frame_skip, seed=0)
            e.reset()
            a1 = [torch.randint(0, 8, (n_envs,), generator=gen, device=dev, dtype=torch.uint8) for _ in range(4)]
            a2 = [torch.randint(0, 8, (n_envs,), generator=gen, device=dev, dtype=torch.uint8) for _ in range(4)]

            def one(i):
                e.bind_actions(a1[i % 4], a2[i % 4] if self_play else None)
                e.step_bound()
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for i in range(300):                 # burn-in: desynchronise the episodes
                    one(i)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for i in range(steps):
                    one(i)
            graph.replay()
            torch.cuda.synchronize(dev)
            f0 = e.episode_stats()["env_frames"]
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(3):
                graph.replay()
            s1.record()
            torch.cuda.synchronize(dev)
            ms = s0.elapsed_time(s1)
            fr = e.episode_stats()["env_frames"] - f0
            e.close()
            return {"env_frames_per_sec": fr / (ms * 1e-3), "ms_per_step": ms / (3 * steps), "envs": n_envs,
                    "frame_skip": frame_skip, "opponent": "self_play" if self_play else "bot",
                    "note": "CUDA-graph replay of %d launches; working set fits L2 (launch/latency-bound regime)" % steps}
        extra["B_4096_bot_k1"] = quick(4096, 1, False)
        extra["C_65536_selfplay_k4"] = quick(65536, 4, True)
        extra["1Mi_bot_k1"] = quick(1 << 20, 1, False)
        extra["1Mi_bot_k4"] = quick(1 << 20, 4, False, steps=100)

        def ppo_rollout(n_envs=16384, horizon=128, reps=5):
            """configs[4]: torch MLP policy (8-64-64-8) consuming env.obs in place, sampling Discrete(8) actions into
            the tensor the step kernel is bound to; the whole horizon is one CUDA graph.  Policy time included."""
            from footsies_gym_b200.rollout import MLPPolicy, RolloutCollector
            e = FootsiesEnv(num_envs=n_envs, device=dev, opponent=None, seed=0)
            pol = MLPPolicy().to(dev)
            out = {}
            for name, graph, fused in (("horizon_kernel", False, "horizon"), ("fused_policy_kernel_cuda_graph", True, "step"),
                                       ("torch_policy_cuda_graph", True, False), ("torch_policy_eager", False, False)):
                col = RolloutCollector(e, pol, horizon=horizon, use_cuda_graph=graph, fused=fused)
                col.collect()
                torch.cuda.synchronize(dev)
                f0 = e.episode_stats()["env_frames"]
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                for _ in range(reps):
                    col.collect()
                s1.record()
                torch.cuda.synchronize(dev)
                ms = s0.elapsed_time(s1)
                fr = e.episode_stats()["env_frames"] - f0
                out[name] = {"env_frames_per_sec": fr / (ms * 1e-3), "ms_per_horizon": ms / reps}
            e.close()
            out.update(envs=n_envs, horizon=horizon, policy="MLP 8-64-64-8 tanh fp32, categorical sampling",
                       note="per GPU; policy forward + sampling + rollout-buffer writes inside the timed region; horizon_kernel "
                            "is one launch per horizon (fg_rollout_mlp, battle state in registers throughout); "
                            "fused_policy_kernel is 2 launches per step (fg_policy_mlp_sample + fg_step) with zero-copy "
                            "rollout buffers")
            return out
        extra["E_ppo_rollout_16384x128"] = ppo_rollout()

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    cpu_baseline = cpu_port = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        cpu_baseline, _, _ = cpu_baseline_entry("reference", threads, seconds=args.cpu_seconds)
        cpu_port, _, _ = cpu_baseline_entry("port", threads, seconds=args.cpu_seconds / 2)

    if rank == 0:
        peak, peak_src = measured_peaks()
        bytes_per_env = env.algorithmic_bytes_per_env_step
        ms_per_launch = ms_total / args.steps
        achieved = bytes_per_env * n / (ms_per_launch * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic(bytes_per_env, n)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_launch,
            "ms_per_step_min": ms_step_min, "ms_per_step_max": ms_step_max,
            "timing": "`steps` launches back to back after the burn-in and warm-up; value and ms_per_step are the whole "
                      "window (CUDA events on the launching stream, max over ranks); min / max are the fastest / slowest "
                      "of up to 25 equal blocks of the window, per step",
            "higher_is_better": True,
            "scaling": "strong" if args.total_envs > 0 else "weak", "vs_baseline": None, "dtype": "int32+fp32",
            "data": "synthetic",
            "config": {"workload": (STRONG_WORKLOAD.format(t=args.total_envs, w=world) if args.total_envs > 0
                                    else WORKLOAD.format(n=n)),
                       "envs_per_gpu": n, "frame_skip": 1, "opponent": "bot",
                       "actions": "iid uniform over 8 bitmasks, torch.Generator(device).manual_seed(1234 + rank)",
                       "l2": (f"inputs larger than L2: {2 * 64 * n / 1e6:.0f} MB of state traffic + "
                              f"{46 * n / 1e6:.0f} MB of outputs per step vs 126 MB L2; no flush"
                              if (2 * 64 + 46) * n > 2 * 126e6 else
                              f"NOT larger than L2: {(2 * 64 + 46) * n / 1e6:.0f} MB touched per step vs 126 MB L2 and no "
                              f"flush -> informational only, use the default weak-scaling workload for the roofline"),
                       "frames_counted": "kernel simulated-frame counter (FG_STAT_ENV_FRAMES)",
                       "burnin_steps": args.burnin},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": bytes_per_env * n,
                         "algorithmic_bytes_per_env_frame": bytes_per_env, "peak_source": peak_src,
                         "kernel": "step_kernel<K=1, P2 bot, dense>"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "blocks": 9, "value_slowest_block": e2e_lo, "value_fastest_block": e2e_hi,
                    "api": "FootsiesEnv.step_host_packed -> fg_step_host_packed: pinned host actions in, one lossless 16-byte "
                           "record per battle out (NUMA-local pinned block from fg_host_alloc; 1 Mi-env slices pipelined "
                           "over two streams, one contiguous copy per slice); median of 9 blocks of `steps` calls, "
                           "wall clock around calls that return with the results in host memory, max over ranks",
                    "natural_width_layout": {"value": e2e_compact_value, "h2d_bytes_per_step": h2d_c,
                                             "d2h_bytes_per_step": d2h_c,
                                             "api": "FootsiesEnv.step_host -> fg_step_host_compact (27 bytes per battle: every "
                                                    "field in its natural width, six copies per slice)"},
                    "scaling_efficiency_note": "driver computes efficiency from the per-N lines"},
            "gpu_launches": launches,
            "clocks": clocks,
            "episode_stats_all_ranks": stats,
        }
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
            line["cpu_baseline_c_port"] = cpu_port
        if extra:
            line["extra"] = extra
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
