// rollout_kernel.cu -- BASELINE.json configs[4] as ONE launch per horizon: policy inference -> sample -> FootsiesEnv.step,
// `horizon` times, for every battle of the device, with the battle state held in registers for the whole horizon.
//
// Battles never interact and the policy only couples them through its (read-only) weights, so a horizon needs no
// grid-wide synchronisation: a CTA owns its battles from the first step to the last.  Two CTA shapes share the per-battle
// horizon loop (rollout_horizon: autoreset or K frames, fused frame skipping, outputs, frame_delay queue, statistics):
//   rollout_mma_kernel (H = 32 / 64): 4 warps, every warp owns 16 MT battles -- policy on the tensor cores, no CTA barrier
//                  inside the horizon loop (below);
//   rollout_kernel (H = 128): 4 warps own 64 battles, 2 per lane.  Per step and CTA:
//     policy phase   all warps: warp w computes hidden units w * H/4 .. of every battle of the CTA, lanes = battles
//                    (policy_mlp.cuh: weight fetches are warp-wide shared-memory broadcasts, activations
//                    cross between warps through shared memory), ending with the partial logits in shared memory;
//     simulator phase  one thread per battle: assemble the 8 logits, log-softmax, sample the input bitmask, then the
//                    reference frame update (frame_logic.cuh; autoreset, bot query, reward and termination exactly as
//                    step_kernel does it); action t / log-probability t / observation t + 1 / reward t / done t go to the
//                    rollout buffers and observation t + 1 stays in shared memory for the next policy phase.
// Against the two launches per step of the per-step path (policy kernel + step kernel in a CUDA graph) this removes
// 2 x horizon launches, every state load / store but one, and the observation round trip through L2.  Several CTAs are
// resident per SM.  (Tried twice -- by blockIdx and by per-SM arrival order (%smid + atomic) -- starting every second
// co-resident CTA half a step late so that simulator and policy phases interleave: no measurable effect for any delay;
// one CTA per SM runs a step in 4.7 us, two in 6.5 us, so co-residency already overlaps most of the work.  Removed.)
// Results are bit-identical to the per-step path (tests/test_rollout.py).
// One parameter block (RolloutParams) serves every mode; launch_rollout picks the kernel from it:
//   P2 (P2POL, POOL, BOTM): the in-game bot; a second policy (p2_policy); an opponent pool (pool.count > 0) of up to
//     FG_POOL_MAX networks, member m on the battles [end[m - 1], end[m]) -- the boundaries are multiples of FG_POOL_BLOCK, a
//     multiple of every CTA's battle count, so a CTA stages one member's weights in the single P2 policy's place, runs the
//     same horizon loop and also flushes its statistics into that member's counters (tests/test_opponent_pool.py); a pool
//     with the in-game bot as member bot_member, whose CTAs branch (CTA-uniformly) into the P2 = bot horizon loop: RNG plane
//     loaded and stored, bot queried by reset_env / simulate_frame, no P2 weights and no P2 policy pass, actions_p2 receives
//     the bot's held input at the start of each step and logp_p2 zero (tests/test_opponent_pool_bot.py).
//   DELAY (ring.depth > 0): every step pushes the battle's new state into the caller's frame_delay ring (delay_ring.cuh, the
//     rule fg_delay_ring_step applies) and the emitted, delayed observation is what both policies read next and what
//     obs[t + 1] receives; the bot, rewards, dones and fused frame skipping see the true state
//     (tests/test_rollout_frame_delay.py).
//   SKIP: fg_config.skip_unactionable (fused FootsiesFrameSkipped).
// Compiled with -fmad=false like the step kernel; the policy arithmetic uses explicit fmaf.
#include <stdlib.h>

#include "delay_ring.cuh"
#include "rollout_kernel.h"
#include "policy_mma.cuh"

namespace fgk {

using namespace fgp;

template <int H, bool P2POL>
struct RolloutSmem {
    static constexpr int kE = 2;                                // battles per lane: 4 do not fit the registers at H = 128
    static constexpr int kW = kPolicyWarps;
    static constexpr int kEnvs = 32 * kE;
    using PL = PolicySmemBcast<H, kEnvs, kW>;
    static constexpr size_t kTables = 0;
    static constexpr size_t kPolicy = (sizeof(Tables) + 127) / 128 * 128;                             // P1 weights + activations
    static constexpr size_t kPolicy2 = kPolicy + (PL::kBytes + 15) / 16 * 16;                         // P2 weights (P2POL)
    static constexpr size_t kObs = kPolicy2 + (P2POL ? (sizeof(float) * PL::kWeightFloats + 15) / 16 * 16 : 0);   // float4 [kEnvs][2]
    static constexpr size_t kStats = kObs + sizeof(float4) * 2 * kEnvs;                             // u64 [FG_STAT_COUNT]
    static constexpr size_t kBytes = kStats + sizeof(unsigned long long) * FG_STAT_COUNT;
};

// ---- opponent pool: a CTA's P2 weights are those of the member whose range holds its battles ----
// member of the CTA whose first battle is `first`: the number of boundaries end[0 .. count - 2] at or below it (end is
// non-decreasing and first < n = end[count - 1]).  Unrolled with constant indices so that the parameter arrays are read
// from the constant bank instead of being copied to local memory for a dynamic index.
__device__ __forceinline__ int pool_member(const RolloutPool &pool, long long first) {
    int m = 0;
#pragma unroll
    for (int k = 0; k < FG_POOL_MAX - 1; k++) m += (k < pool.count - 1 && first >= pool.end[k]) ? 1 : 0;
    return m;
}
__device__ __forceinline__ PolicyWeights pool_weights(const RolloutPool &pool, int m) {
    PolicyWeights w = pool.member[0];
#pragma unroll
    for (int k = 1; k < FG_POOL_MAX; k++)
        if (k == m) w = pool.member[k];
    return w;
}
// after the CTA's final statistics flush (and its barrier): the member's episodes, P1 wins, P2 wins, double KOs
__device__ __forceinline__ void pool_flush(const RolloutPool &pool, int m, const unsigned long long *s_stats, int tid) {
    static_assert(FG_STAT_EPISODES == 0 && FG_STAT_P1_WINS == 1 && FG_STAT_P2_WINS == 2 && FG_STAT_DOUBLE_KO == 3, "stats[m][4] order");
    if (pool.stats && tid < 4 && s_stats[tid]) atomicAdd(&pool.stats[(size_t)m * 4 + tid], s_stats[tid]);
}

// ---- frame_delay queue (DELAY = true): one lane's queue state across the horizon ----
// Step t pushes the battle's new state at ring position (pos + t) % depth exactly as fg_delay_ring_step does after an
// fg_step (delay_ring_push); the emitted, delayed observation replaces the true one in obs[t + 1] and in the policy's input
// rows.  The entry to emit and the newest entry's frame are loaded before the frame update (prefetch): the same thread
// wrote them in an earlier step, and their latency hides under the frame update instead of lengthening the chain from
// policy to frame update.  The DELAY = false version is empty and its calls compile to nothing.
template <bool DELAY> struct DelayQueue {
    __device__ __forceinline__ DelayQueue(const RolloutParams &, bool, int) {}
    __device__ __forceinline__ void prefetch(const RolloutParams &, bool, int) {}
    __device__ __forceinline__ void push(const RolloutParams &, int, int32_t, uint32_t, const float4 *, float4 &, float4 &) {}
    __device__ __forceinline__ void finish(const RolloutParams &, int, float4, float4) const {}
    __device__ __forceinline__ void advance(const RolloutParams &) {}
};
template <> struct DelayQueue<true> {
    int slot;                   // (pos + t) % depth
    int32_t shown_frame;        // info frame and misc of the delayed state emitted last (what out_* receive at the end)
    uint32_t shown_misc;
    DelayEntry oldest;          // slot + 1: the entry this step emits
    int32_t newest_frame;       // frame of slot - 1

    static __device__ __forceinline__ DelayRingRef ref(const RolloutParams &rp) {
        return { rp.ring.obs, rp.ring.frame, rp.ring.misc, (size_t)rp.sim.n };
    }
    __device__ __forceinline__ DelayQueue(const RolloutParams &rp, bool valid, int i) : slot(rp.ring.pos) {
        shown_frame = valid ? rp.ring.out_frame[i] : 0;
        shown_misc = valid ? rp.ring.out_misc[i] : 0u;
    }
    __device__ __forceinline__ void prefetch(const RolloutParams &rp, bool valid, int i) {
        if (valid) {
            const int d = rp.ring.depth;
            oldest = ref(rp).load(slot + 1 == d ? 0 : slot + 1, i);
            newest_frame = rp.ring.frame[(size_t)(slot == 0 ? d - 1 : slot - 1) * rp.sim.n + i];
        }
    }
    // a, b: the step's observation in, the delayed one out; shown_obs: the lane's policy input row (the last emitted
    // observation, which a battle that did not advance keeps)
    __device__ __forceinline__ void push(const RolloutParams &rp, int i, int32_t frame, uint32_t misc, const float4 *shown_obs, float4 &a,
                                         float4 &b) {
        const DelayEntry now = { a, b, frame, misc };
        DelayEntry emit;
        if (delay_ring_push(ref(rp), i, rp.ring.depth, slot, false, now, oldest, newest_frame, emit)) {
            a = emit.a; b = emit.b; shown_frame = emit.frame; shown_misc = emit.misc;
        } else {
            a = shown_obs[0]; b = shown_obs[1];
        }
    }
    __device__ __forceinline__ void finish(const RolloutParams &rp, int i, float4 a, float4 b) const {
        rp.ring.out_obs[2 * (size_t)i] = a; rp.ring.out_obs[2 * (size_t)i + 1] = b;
        rp.ring.out_frame[i] = shown_frame; rp.ring.out_misc[i] = shown_misc;
    }
    __device__ __forceinline__ void advance(const RolloutParams &rp) { slot = slot + 1 == rp.ring.depth ? 0 : slot + 1; }
};

// ---- the per-battle pieces both CTA shapes share; obs[2 * row], obs[2 * row + 1] is the lane's policy input row ----
// (n, K = frame_skip and horizon come from the kernel's registers: read from rp inside, after the stores to global memory,
// they would be loaded again)
// the observation the first step acts on: the last one of the previous horizon, carried over into slot 0
__device__ __forceinline__ void carry_first_obs(const RolloutParams &rp, int n, int horizon, bool valid, int i, float4 *obs, int row) {
    float4 a = make_float4(0, 0, 0, 0), b = a;
    if (valid) {
        const size_t src = ((size_t)horizon * n + i) * 2;
        a = rp.obs[src]; b = rp.obs[src + 1];
        rp.obs[(size_t)i * 2] = a; rp.obs[(size_t)i * 2 + 1] = b;
    }
    obs[2 * row] = a; obs[2 * row + 1] = b;
}

// a bot member's P2 record of step t: its input held when the step begins; no log-probability
__device__ __forceinline__ void record_bot_p2(const RolloutParams &rp, const Env &e, int n, int t, int i) {
    rp.actions_p2[(size_t)t * n + i] = (uint8_t)((e.misc >> FGM_ACTOR2_SHIFT) & 7u);
    rp.logp_p2[(size_t)t * n + i] = 0.0f;
}

// The lane's battle through the whole horizon once the CTA has staged its weights, shared by both CTA shapes.  Per step:
// policy(t, drawn, in1, in2) -- the shape's policy phase, which samples P1's input and, with a second policy or pool
// member, P2's -- then FootsiesEnv.step in the same order of events as step_kernel: autoreset or K frames, fused frame
// skipping, the step's outputs (the input row obs[2 * row], obs[2 * row + 1] receives observation t + 1, delayed with
// DELAY) and the statistics flush.  The battle state, its statistics and its queue are locals of this function, not
// references handed to a callee: so the kernels compile to the code they had with the step written out in each body.
// Threads that simulate no battle (sim_thread false: whole warps) take part in the policy phase and the barriers only.
// n, frame_skip and horizon are read once: read from rp after the stores to global memory, they would be loaded again.
template <bool DENSE, bool P2BOT, bool BOT, bool SKIP, bool POOL, bool DELAY, bool CTA_SYNC, class Policy>
__device__ __forceinline__ void rollout_horizon(const RolloutParams &rp, const Tables &T, unsigned long long *s_stats, float4 *obs,
                                                int row, int n, int horizon, int i, int tid, int lane, int member, bool sim_thread,
                                                bool valid, const Policy &policy) {
    const Params &p = rp.sim;
    Env e;
    if (valid) load_env<P2BOT>(p, i, e);
    if (sim_thread) carry_first_obs(rp, n, horizon, valid, i, obs, row);
    __syncthreads();                                            // tables, weights, statistics: staged
    const unsigned long long drawn = rp.counter_base ? *rp.counter_base : 0ull;
    StatAcc acc = { 0u, 0u, 0u, 0u };
    uint32_t frames_since_flush = 0u;
    const int K = p.frame_skip;
    DelayQueue<DELAY> dq(rp, valid, i);

    for (int t = 0; t < horizon; t++) {
        uint32_t in1 = 0u, in2 = 0u;
        policy(t, drawn, in1, in2);
        if (BOT && valid) record_bot_p2(rp, e, n, t, i);
        if (sim_thread) {                                       // FootsiesEnv.step (whole warps: __any_sync inside)
            double reward = 0.0;
            bool terminal = false, ran = false;
            if constexpr (DELAY) dq.prefetch(rp, valid, i);
            if (valid) {
                if ((e.misc >> FGM_DONE_SHIFT) & 1u) {                  // next-step autoreset: this step only resets
                    reset_env<false, P2BOT>(T, e, p.stale_intro != 0);
                    acc.s += 0x10000u;
                } else {
                    ran = true;
                    if (P2BOT) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
                    for (int kk = 0; kk < K; kk++) {
                        if (!terminal) {
                            simulate_frame<false, P2BOT, DENSE, false>(T, e, in1, in2, reward, terminal, acc);
                            acc.s += 1u << 24;
                            if (P2BOT) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
                        }
                    }
                }
            }
            if (SKIP) {
                // fused FootsiesFrameSkipped (fg_config.skip_unactionable), exactly as in step_kernel: warp-synchronous so that the
                // statistics fold stays a warp-uniform decision
                bool more = ran && !terminal && obs_is_skippable(e);
                while (__any_sync(kFull, more)) {
                    for (int kk = 0; kk < K; kk++) {
                        if (more && !terminal) {
                            simulate_frame<false, P2BOT, DENSE, false>(T, e, 0u, in2, reward, terminal, acc);
                            acc.s += 1u << 24;
                            if (P2BOT) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
                        }
                    }
                    more = more && !terminal && obs_is_skippable(e);
                    frames_since_flush += (uint32_t)K;
                    if (frames_since_flush >= kStatFlushFrames) { flush_stats(acc, s_stats, lane); frames_since_flush = 0u; }
                }
            }
            if (valid) {
                StepOutputs o;
                make_outputs(e, o);
                float4 a = make_float4(o.obs[0], o.obs[1], o.obs[2], o.obs[3]), b = make_float4(o.obs[4], o.obs[5], o.obs[6], o.obs[7]);
                if constexpr (DELAY) dq.push(rp, i, e.frame, o.info_misc, obs + 2 * row, a, b);        // a, b become the delayed observation
                const size_t dst = ((size_t)(t + 1) * n + i) * 2;
                rp.obs[dst] = a; rp.obs[dst + 1] = b;
                rp.rewards[(size_t)t * n + i] = (float)reward;
                rp.dones[(size_t)t * n + i] = terminal ? 1 : 0;
                obs[2 * row] = a; obs[2 * row + 1] = b;
                if (t == horizon - 1) { p.info_frame[i] = e.frame; p.info_misc[i] = o.info_misc; if constexpr (DELAY) dq.finish(rp, i, a, b); }
            }
            if constexpr (DELAY) dq.advance(rp);
            frames_since_flush += (uint32_t)K;                          // uniform across the warp
            if (frames_since_flush >= kStatFlushFrames) { flush_stats(acc, s_stats, lane); frames_since_flush = 0u; }
        }
        if (CTA_SYNC) __syncthreads();
        else __syncwarp();                                      // observation rows are in place for the next policy pass
    }
    if (sim_thread) {
        if (valid) store_env<P2BOT>(p, i, e);
        flush_stats(acc, s_stats, lane);
    }
    __syncthreads();
    if (tid < FG_STAT_COUNT && s_stats[tid]) atomicAdd(&p.stats[tid], s_stats[tid]);
    if constexpr (POOL) pool_flush(rp.pool, member, s_stats, tid);
}

// One CTA's whole horizon.  BOT (opponent pool with the in-game bot as a member, the CTA in the bot's range): P2 is the
// bot exactly as in the P2POL = false kernel, in the P2POL shared-memory layout, with no P2 weights staged or policy pass.
// (tid is read in the kernel itself, where the compiler bounds it by __launch_bounds__.)
template <int H, bool DENSE, bool P2POL, bool SKIP, bool POOL, bool BOT, bool DELAY>
__device__ __forceinline__ void rollout_cta(const RolloutParams &rp, const int tid) {
    using SM = RolloutSmem<H, P2POL>;
    using PL = typename SM::PL;
    constexpr bool kP2Pol = P2POL && !BOT;
    constexpr bool kP2Bot = !kP2Pol;                            // P2 = in-game bot (needs the RNG plane) or the second policy
    constexpr int E = SM::kE, W = SM::kW;
    constexpr int kEnvs = SM::kEnvs, kRollThreads = 32 * W;
    static_assert(kEnvs <= kRollThreads, "one simulator thread per battle");
    static_assert(!POOL || (P2POL && FG_POOL_BLOCK % kEnvs == 0), "a pool CTA plays against one member");
    static_assert(!BOT || POOL, "the bot is a pool member");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Tables &Tw = *reinterpret_cast<Tables *>(smem_raw + SM::kTables);
    const Tables &T = Tw;
    float *pw = reinterpret_cast<float *>(smem_raw + SM::kPolicy);
    float *pact = pw + PL::kWeightFloats;                       // activations, shared by both policies
    float *pw2 = reinterpret_cast<float *>(smem_raw + SM::kPolicy2);
    float4 *obs_s = reinterpret_cast<float4 *>(smem_raw + SM::kObs);
    unsigned long long *s_stats = reinterpret_cast<unsigned long long *>(smem_raw + SM::kStats);
    const Params &p = rp.sim;
    const int lane = tid & 31, warp = tid >> 5;
    const int n = p.n, horizon = rp.horizon;
    const int base = blockIdx.x * kEnvs;
    const int stid = tid;                                       // simulator thread index = battle within the CTA
    const bool sim_thread = stid < kEnvs;                       // whole warps: kEnvs is a multiple of 32
    const int i = base + stid;                                  // simulator mapping: one battle per thread
    const bool valid = sim_thread && i < n;

    load_tables(&Tw, p.tables);
    policy_stage_bcast<H, kEnvs, W>(pw, rp.w, tid, kRollThreads);
    int member = 0;
    if constexpr (POOL) {
        member = pool_member(rp.pool, base);
        if (!BOT) policy_stage_bcast<H, kEnvs, W>(pw2, pool_weights(rp.pool, member), tid, kRollThreads);
    } else if (P2POL) policy_stage_bcast<H, kEnvs, W>(pw2, rp.w_p2, tid, kRollThreads);
    if (tid < FG_STAT_COUNT) s_stats[tid] = 0ull;
    rollout_horizon<DENSE, kP2Bot, BOT, SKIP, POOL, DELAY, true>(
        rp, T, s_stats, obs_s, stid, n, horizon, i, tid, lane, member, sim_thread, valid,
        [&](int t, unsigned long long drawn, uint32_t &in1, uint32_t &in2) {
            // ---- policy phase (two CTA barriers inside) ----
            {
                float x[E][8];
#pragma unroll
                for (int q = 0; q < E; q++) {
                    const float4 a = obs_s[2 * (lane + 32 * q)], b = obs_s[2 * (lane + 32 * q) + 1];
                    x[q][0] = a.x; x[q][1] = a.y; x[q][2] = a.z; x[q][3] = a.w;
                    x[q][4] = b.x; x[q][5] = b.y; x[q][6] = b.z; x[q][7] = b.w;
                }
                policy_partials_bcast<H, E, W>(pw, pact, warp, lane, x);
            }
            if (valid) {
                float lg[8], lp;
                policy_logits_of<H, kEnvs, W>(pw, pact, stid, lg);
                in1 = (uint32_t)policy_sample(lg, hash3(rp.seed, drawn + (unsigned long long)t, (uint64_t)(p.first_env_index + i)), lp);
                rp.actions[(size_t)t * n + i] = (uint8_t)in1;
                rp.logp[(size_t)t * n + i] = lp;
            }
            if (kP2Pol) {
                // the second policy on the same observation rows (mirrored if asked): the sampling threads above have read
                // P1's partial sums before they arrive at the barriers in here, so the activation buffers can be reused
                float x[E][8];
#pragma unroll
                for (int q = 0; q < E; q++) {
                    const float4 a = obs_s[2 * (lane + 32 * q)], b = obs_s[2 * (lane + 32 * q) + 1];
                    x[q][0] = a.x; x[q][1] = a.y; x[q][2] = a.z; x[q][3] = a.w;
                    x[q][4] = b.x; x[q][5] = b.y; x[q][6] = b.z; x[q][7] = b.w;
                    if (rp.p2_mirror) policy_mirror_obs(x[q]);
                }
                policy_partials_bcast<H, E, W>(pw2, pact, warp, lane, x);
                if (valid) {
                    float lg[8], lp;
                    policy_logits_of<H, kEnvs, W>(pw2, pact, stid, lg);
                    int a2 = policy_sample(lg, hash3(rp.seed_p2, drawn + (unsigned long long)t, (uint64_t)(p.first_env_index + i)), lp);
                    if (rp.p2_mirror) a2 = policy_mirror_action(a2);
                    in2 = (uint32_t)a2;
                    rp.actions_p2[(size_t)t * n + i] = (uint8_t)a2;
                    rp.logp_p2[(size_t)t * n + i] = lp;
                }
            }
        });
}

template <int H, bool DENSE, bool P2POL, bool SKIP, bool POOL, bool BOTM, bool DELAY>
__global__ void __launch_bounds__(32 * kPolicyWarps) rollout_kernel(const RolloutParams rp) {
    const int tid = threadIdx.x;
    if constexpr (BOTM) {                                       // CTA-uniform: a CTA's battles belong to one member
        if (pool_member(rp.pool, (long long)blockIdx.x * RolloutSmem<H, P2POL>::kEnvs) == rp.bot_member) {
            rollout_cta<H, DENSE, P2POL, SKIP, POOL, true, DELAY>(rp, tid);
            return;
        }
    }
    rollout_cta<H, DENSE, P2POL, SKIP, POOL, false, DELAY>(rp, tid);
}

// ---- tensor-core version (H <= 64): every WARP owns 16 MT battles for the whole horizon -- policy (policy_mma.cuh: mma.sync
// m16n8k8 with the 3 x TF32 split, activations never leave the registers between layers) and simulator alike -- so the
// horizon loop contains no CTA barrier at all: warps drift apart and one warp's simulator phase overlaps its neighbours'
// tensor-core phases.  MT = 2: 32 battles per warp, every lane simulates one; MT = 1: 16 battles per warp (lanes 16-31 only
// feed the MMA), twice the warps per SM -- what a batch of 16 384 battles (111 per SM) needs to keep two warps per scheduler.
template <int H, bool P2POL>
struct RolloutMmaSmem {
    static constexpr int kW = 4;
    using PL = PolicyMmaSmem<H>;
    static constexpr size_t kTables = 0;
    static constexpr size_t kPolicy = (sizeof(Tables) + 127) / 128 * 128;
    static constexpr size_t kPolicy2 = kPolicy + (PL::kBytes + 15) / 16 * 16;
    static constexpr size_t kObs = kPolicy2 + (P2POL ? (PL::kBytes + 15) / 16 * 16 : 0);      // float [kW][32][8]
    static constexpr size_t kLogits = kObs + sizeof(float) * kW * 256;                       // float [kW][32][8]
    static constexpr size_t kStats = kLogits + sizeof(float) * kW * 256;
    static constexpr size_t kBytes = kStats + sizeof(unsigned long long) * FG_STAT_COUNT;
};

// One CTA's whole horizon; BOT as in rollout_cta.
template <int H, int MT, bool DENSE, bool P2POL, bool SKIP, bool POOL, bool BOT, bool DELAY>
__device__ __forceinline__ void rollout_mma_cta(const RolloutParams &rp, const int tid) {
    using SM = RolloutMmaSmem<H, P2POL>;
    constexpr bool kP2Pol = P2POL && !BOT;
    constexpr bool kP2Bot = !kP2Pol;
    constexpr int W = SM::kW;
    constexpr int kWarpEnvs = 16 * MT, kEnvs = kWarpEnvs * W;
    static_assert(!POOL || (P2POL && FG_POOL_BLOCK % kEnvs == 0), "a pool CTA plays against one member");
    static_assert(!BOT || POOL, "the bot is a pool member");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Tables &Tw = *reinterpret_cast<Tables *>(smem_raw + SM::kTables);
    const Tables &T = Tw;
    float *pw = reinterpret_cast<float *>(smem_raw + SM::kPolicy);
    float *pw2 = reinterpret_cast<float *>(smem_raw + SM::kPolicy2);
    unsigned long long *s_stats = reinterpret_cast<unsigned long long *>(smem_raw + SM::kStats);
    const Params &p = rp.sim;
    const int lane = tid & 31, warp = tid >> 5;
    float *obs_w = reinterpret_cast<float *>(smem_raw + SM::kObs) + warp * 256;      // this warp's observation rows
    float *lg_w = reinterpret_cast<float *>(smem_raw + SM::kLogits) + warp * 256;    // ... and logits
    const int n = p.n, horizon = rp.horizon;
    const int i = blockIdx.x * kEnvs + warp * kWarpEnvs + lane;                      // one battle per simulating lane
    const bool valid = lane < kWarpEnvs && i < n;

    load_tables(&Tw, p.tables);
    policy_mma_stage<H>(pw, rp.w, tid, 32 * W);
    int member = 0;
    if constexpr (POOL) {
        member = pool_member(rp.pool, (long long)blockIdx.x * kEnvs);
        if (!BOT) policy_mma_stage<H>(pw2, pool_weights(rp.pool, member), tid, 32 * W);
    } else if (P2POL) policy_mma_stage<H>(pw2, rp.w_p2, tid, 32 * W);
    if (tid < FG_STAT_COUNT) s_stats[tid] = 0ull;
    rollout_horizon<DENSE, kP2Bot, BOT, SKIP, POOL, DELAY, false>(
        rp, T, s_stats, reinterpret_cast<float4 *>(obs_w), lane, n, horizon, i, tid, lane, member, true, valid,
        [&](int t, unsigned long long drawn, uint32_t &in1, uint32_t &in2) {
            // ---- policy: the warp's battles through the MLP on the tensor cores, then one lane per battle samples ----
            // (the random words do not depend on the logits: their 64-bit multiply chains are issued before the MMAs, under
            // whose latency they complete)
            const uint32_t rnd1 = hash3(rp.seed, drawn + (unsigned long long)t, (uint64_t)(p.first_env_index + i));
            const uint32_t rnd2 = kP2Pol ? hash3(rp.seed_p2, drawn + (unsigned long long)t, (uint64_t)(p.first_env_index + i)) : 0u;
            policy_mma_logits<H, MT, false>(pw, obs_w, lg_w, lane);
            if (valid) {
                const float4 l0 = reinterpret_cast<const float4 *>(lg_w)[2 * lane], l1 = reinterpret_cast<const float4 *>(lg_w)[2 * lane + 1];
                const float lg[8] = { l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w };
                float lp;
                in1 = (uint32_t)policy_sample(lg, rnd1, lp);
                rp.actions[(size_t)t * n + i] = (uint8_t)in1;
                rp.logp[(size_t)t * n + i] = lp;
            }
            if (kP2Pol) {
                if (rp.p2_mirror) policy_mma_logits<H, MT, true>(pw2, obs_w, lg_w, lane);
                else policy_mma_logits<H, MT, false>(pw2, obs_w, lg_w, lane);
                if (valid) {
                    const float4 l0 = reinterpret_cast<const float4 *>(lg_w)[2 * lane], l1 = reinterpret_cast<const float4 *>(lg_w)[2 * lane + 1];
                    const float lg[8] = { l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w };
                    float lp;
                    int a2 = policy_sample(lg, rnd2, lp);
                    if (rp.p2_mirror) a2 = policy_mirror_action(a2);
                    in2 = (uint32_t)a2;
                    rp.actions_p2[(size_t)t * n + i] = (uint8_t)a2;
                    rp.logp_p2[(size_t)t * n + i] = lp;
                }
            }
        });
}

template <int H, int MT, bool DENSE, bool P2POL, bool SKIP, bool POOL, bool BOTM, bool DELAY>
__global__ void __launch_bounds__(32 * RolloutMmaSmem<H, P2POL>::kW, 1) rollout_mma_kernel(const RolloutParams rp) {
    const int tid = threadIdx.x;
    if constexpr (BOTM) {                                       // CTA-uniform: a CTA's battles belong to one member
        if (pool_member(rp.pool, (long long)blockIdx.x * (16 * MT * RolloutMmaSmem<H, P2POL>::kW)) == rp.bot_member) {
            rollout_mma_cta<H, MT, DENSE, P2POL, SKIP, POOL, true, DELAY>(rp, tid);
            return;
        }
    }
    rollout_mma_cta<H, MT, DENSE, P2POL, SKIP, POOL, false, DELAY>(rp, tid);
}

inline int rollout_mt(int n) {
    // Measured (profiles/r02f_rollout_mma.log, H = 64, us per step, 16-battle / 32-battle warps / round-1 FFMA2 kernel):
    // 16 384 battles 4.49 / 5.90 / 6.37; 131 072: 28.0 / 31.3 / -; 1 Mi: 216 / 227 / 262 -- more, lighter warps hide the
    // simulator's latency under the neighbours' tensor-core phases at every size, so 16-battle warps are the default
    // (developer knob: FOOTSIES_B200_ROLLOUT_MT = 1 | 2).
    int mt = n >= 131072 ? 2 : 1;
    if (const char *v = getenv("FOOTSIES_B200_ROLLOUT_MT")) mt = atoi(v) == 2 ? 2 : 1;
    // (7-warp CTAs, which would spread 16 384 battles evenly as 147 x 112, measured 4.55 us per step against 4.46 for 4 warps.)
    // (8-battle warps -- half-empty M tiles, twice the warps, 124 registers -- are the same bits and SLOWER from 8192 battles up:
    // 16 384 battles 4.98 vs 3.35 us per step; only 4096 battles gain, 2.30 vs 2.46.  A one-off start stagger between the two
    // CTAs of an SM changes nothing: 3.33 vs 3.32.  tools/probes/half_tile_and_stagger_experiment.patch,
    // profiles/r03h_rollout_half_tiles.log, r03i_rollout_stagger.log.  Step time against batch size -- 4096: 2.46, 8192: 2.48,
    // 16 384: 3.35, 32 768: 6.33 -- says the kernel leaves the latency-bound regime right at one CTA per SM.)
    // (Compiling the 32-battle-warp bot kernel for 3 CTAs per SM -- 168 registers instead of 190, 24 bytes of spill, 12
    // instead of 8 warps per SM -- LOSES: 1 Mi battles 143.1 vs 137.5 us per step, 131 072: 19.3 vs 18.7,
    // profiles/r03f_rollout_mt2_blocks.log.)
    // Two policies (self-play): 32-battle warps from 131 072 battles up (1 Mi: 479 us per step against 567).
    return mt;
}

// once per device and kernel: the dynamic shared memory opt-in; then one CTA of kThreads threads per kEnvs battles
template <auto kKernel, size_t kBytes, int kEnvs, int kThreads>
static cudaError_t launch_cta(cudaStream_t s, const RolloutParams &rp) {
    static fg::DeviceOnceFlags configured;
    if (cudaError_t e = fg::configure_once_per_device(configured, [] {
            return cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBytes); }))
        return e;
    kKernel<<<(rp.sim.n + kEnvs - 1) / kEnvs, kThreads, kBytes, s>>>(rp);
    return cudaSuccess;
}

// the shape: the tensor-core kernel for H <= 64 (16- or 32-battle warps by batch size), the FFMA kernel for H = 128
template <int H, bool DENSE, bool P2POL, bool SKIP, bool POOL, bool BOTM, bool DELAY>
static cudaError_t launch_rollout_k(cudaStream_t s, const RolloutParams &rp) {
    if constexpr (H <= kMmaMaxHidden) {
        using SM = RolloutMmaSmem<H, P2POL>;
        if (rollout_mt(rp.sim.n) == 1)
            return launch_cta<rollout_mma_kernel<H, 1, DENSE, P2POL, SKIP, POOL, BOTM, DELAY>, SM::kBytes, 16 * SM::kW, 32 * SM::kW>(s, rp);
        return launch_cta<rollout_mma_kernel<H, 2, DENSE, P2POL, SKIP, POOL, BOTM, DELAY>, SM::kBytes, 32 * SM::kW, 32 * SM::kW>(s, rp);
    } else {
        using SM = RolloutSmem<H, P2POL>;
        return launch_cta<rollout_kernel<H, DENSE, P2POL, SKIP, POOL, BOTM, DELAY>, SM::kBytes, SM::kEnvs, 32 * SM::kW>(s, rp);
    }
}
// the P2 mode: a pool (with the bot as a member or without), a second policy, or the bot
template <int H, bool DENSE, bool DELAY, bool SKIP>
static cudaError_t launch_rollout_p(cudaStream_t s, const RolloutParams &rp) {
    if (rp.pool.count > 0)
        return rp.bot_member >= 0 ? launch_rollout_k<H, DENSE, true, SKIP, true, true, DELAY>(s, rp)
                                  : launch_rollout_k<H, DENSE, true, SKIP, true, false, DELAY>(s, rp);
    return rp.p2_policy ? launch_rollout_k<H, DENSE, true, SKIP, false, false, DELAY>(s, rp)
                        : launch_rollout_k<H, DENSE, false, SKIP, false, false, DELAY>(s, rp);
}

// One translation unit per hidden size, reward mode and DELAY (build.py compiles this file with -DFG_ROLLOUT_H=..
// -DFG_ROLLOUT_DENSE=.. -DFG_ROLLOUT_DELAY=.. so that the kernels compile in parallel) plus one without the defines that
// holds the dispatcher.
#define FG_ROLLOUT_DECL(H, D, DL) cudaError_t launch_rollout_##H##_##D##_##DL(cudaStream_t s, const RolloutParams &rp)
#define FG_ROLLOUT_DECLS(H) FG_ROLLOUT_DECL(H, 0, 0); FG_ROLLOUT_DECL(H, 0, 1); FG_ROLLOUT_DECL(H, 1, 0); FG_ROLLOUT_DECL(H, 1, 1)
FG_ROLLOUT_DECLS(32); FG_ROLLOUT_DECLS(64); FG_ROLLOUT_DECLS(128);
#if defined(FG_ROLLOUT_H)
#define FG_ROLLOUT_DEF2(H, D, DL) FG_ROLLOUT_DECL(H, D, DL) { \
    return rp.sim.skip_unactionable ? launch_rollout_p<H, (D != 0), (DL != 0), true>(s, rp) : launch_rollout_p<H, (D != 0), (DL != 0), false>(s, rp); }
#define FG_ROLLOUT_DEF(H, D, DL) FG_ROLLOUT_DEF2(H, D, DL)
FG_ROLLOUT_DEF(FG_ROLLOUT_H, FG_ROLLOUT_DENSE, FG_ROLLOUT_DELAY)
#else
#define FG_ROLLOUT_CASE(H) case H: return dense ? (delay ? launch_rollout_##H##_1_1(s, rp) : launch_rollout_##H##_1_0(s, rp)) \
                                                : (delay ? launch_rollout_##H##_0_1(s, rp) : launch_rollout_##H##_0_0(s, rp))
cudaError_t launch_rollout(bool dense, cudaStream_t s, const RolloutParams &rp) {
    const bool delay = rp.ring.depth > 0;
    switch (rp.hidden) {
    FG_ROLLOUT_CASE(32);
    FG_ROLLOUT_CASE(64);
    FG_ROLLOUT_CASE(128);
    default: return cudaErrorInvalidValue;
    }
}
#endif

}  // namespace fgk
