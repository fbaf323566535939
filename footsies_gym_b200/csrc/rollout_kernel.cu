// rollout_kernel.cu -- BASELINE.json configs[4] as ONE launch per horizon: policy inference -> sample -> FootsiesEnv.step,
// `horizon` times, for every battle of the device, with the battle state held in registers for the whole horizon.
//
// Battles never interact and the policy only couples them through its (read-only) weights, so a horizon needs no
// grid-wide synchronisation: a CTA of W = 4 warps owns 32 x E battles from the first step to the last.  Per step and CTA:
//   policy phase   all W warps: warp w computes hidden units w * H/W .. of every battle of the CTA, lanes = battles
//                  (policy_mlp.cuh: weight fetches are warp-wide shared-memory broadcasts, activations
//                  cross between warps through shared memory), ending with the partial logits in shared memory;
//   simulator phase  one thread per battle: assemble the 8 logits, log-softmax, sample the input bitmask, then the
//                  reference frame update (frame_logic.cuh; autoreset, bot query, reward and termination exactly as
//                  step_kernel does it); action t / log-probability t / observation t + 1 / reward t / done t go to the
//                  rollout buffers and observation t + 1 stays in shared memory for the next policy phase.
// Against the two launches per step of the per-step path (policy kernel + step kernel in a CUDA graph) this removes
// 2 x horizon launches, every state load / store but one, and the observation round trip through L2.  Several CTAs are
// resident per SM.  (Tried twice -- by blockIdx and by per-SM arrival order (%smid + atomic) -- starting every second
// co-resident CTA half a step late so that simulator and policy phases interleave: no measurable effect for any delay;
// one CTA per SM runs a step in 4.7 us, two in 6.5 us, so co-residency already overlaps most of the work.  Removed.)
// Results are bit-identical to the per-step path (tests/test_rollout.py).
// Opponent pool (fg_rollout_mlp_pool, POOL = true): P2 is played by up to FG_POOL_MAX networks, member m on the battles
// [end[m - 1], end[m]).  The boundaries are multiples of FG_POOL_BLOCK, a multiple of every CTA's battle count, so a CTA
// stages one member's weights in the single P2 policy's place and runs the same horizon loop; its final statistics flush
// also lands in that member's counters.  Every range equals a single-opponent rollout of just those battles
// (tests/test_opponent_pool.py); the POOL = false instantiations are the kernels as they were.
// Compiled with -fmad=false like the step kernel; the policy arithmetic uses explicit fmaf.
#include <stdlib.h>
#include <type_traits>

#include "rollout_kernel.h"
#include "policy_mma.cuh"

namespace fgk {

using namespace fgp;

template <int H, int E, int W, bool P2POL>
struct RolloutSmem {
    static constexpr int kEnvs = 32 * E;
    using PL = PolicySmemBcast<H, kEnvs, W>;
    static constexpr size_t kTables = 0;
    static constexpr size_t kPolicy = (sizeof(Tables) + 127) / 128 * 128;                             // P1 weights + activations
    static constexpr size_t kPolicy2 = kPolicy + (PL::kBytes + 15) / 16 * 16;                         // P2 weights (P2POL)
    static constexpr size_t kObs = kPolicy2 + (P2POL ? (sizeof(float) * PL::kWeightFloats + 15) / 16 * 16 : 0);   // float4 [kEnvs][2]
    static constexpr size_t kStats = kObs + sizeof(float4) * 2 * kEnvs;                             // u64 [FG_STAT_COUNT]
    static constexpr size_t kBytes = kStats + sizeof(unsigned long long) * FG_STAT_COUNT;
};

// ---- opponent pool (fg_rollout_mlp_pool): a CTA's P2 weights are those of the member whose range holds its battles ----
template <bool POOL> struct RolloutArgs { using type = RolloutParams; };
template <> struct RolloutArgs<true> { using type = RolloutPoolParams; };

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

template <int H, int E, int W, bool DENSE, bool P2POL, bool SKIP, bool POOL = false>
__global__ void __launch_bounds__(32 * W) rollout_kernel(const typename RolloutArgs<POOL>::type rp) {
    using SM = RolloutSmem<H, E, W, P2POL>;
    using PL = typename SM::PL;
    constexpr bool kP2Bot = !P2POL;                             // P2 = in-game bot (needs the RNG plane) or the second policy
    constexpr int kEnvs = SM::kEnvs, kRollThreads = 32 * W;
    static_assert(kEnvs <= kRollThreads, "one simulator thread per battle");
    static_assert(!POOL || (P2POL && FG_POOL_BLOCK % kEnvs == 0), "a pool CTA plays against one member");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Tables &Tw = *reinterpret_cast<Tables *>(smem_raw + SM::kTables);
    const Tables &T = Tw;
    float *pw = reinterpret_cast<float *>(smem_raw + SM::kPolicy);
    float *pact = pw + PL::kWeightFloats;                       // activations, shared by both policies
    float *pw2 = reinterpret_cast<float *>(smem_raw + SM::kPolicy2);
    float4 *obs_s = reinterpret_cast<float4 *>(smem_raw + SM::kObs);
    unsigned long long *s_stats = reinterpret_cast<unsigned long long *>(smem_raw + SM::kStats);
    const Params &p = rp.sim;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
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
        policy_stage_bcast<H, kEnvs, W>(pw2, pool_weights(rp.pool, member), tid, kRollThreads);
    } else if (P2POL) policy_stage_bcast<H, kEnvs, W>(pw2, rp.w_p2, tid, kRollThreads);
    if (tid < FG_STAT_COUNT) s_stats[tid] = 0ull;
    Env e;
    if (valid) load_env<kP2Bot>(p, i, e);
    if (sim_thread) {
        // the observation the first step acts on: the last one of the previous horizon, carried over into slot 0
        float4 a = make_float4(0, 0, 0, 0), b = a;
        if (valid) {
            const size_t src = ((size_t)horizon * n + i) * 2;
            a = rp.obs[src]; b = rp.obs[src + 1];
            rp.obs[(size_t)i * 2] = a; rp.obs[(size_t)i * 2 + 1] = b;
        }
        obs_s[2 * stid] = a; obs_s[2 * stid + 1] = b;
    }
    __syncthreads();
    const unsigned long long drawn = rp.counter_base ? *rp.counter_base : 0ull;
    StatAcc acc = { 0u, 0u, 0u, 0u };
    uint32_t frames_since_flush = 0u;
    const int K = p.frame_skip;

    for (int t = 0; t < horizon; t++) {
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
        uint32_t in1 = 0u, in2 = 0u;
        if (valid) {
            float lg[8], lp;
            policy_logits_of<H, kEnvs, W>(pw, pact, stid, lg);
            in1 = (uint32_t)policy_sample(lg, hash3(rp.seed, drawn + (unsigned long long)t, (uint64_t)(p.first_env_index + i)), lp);
            rp.actions[(size_t)t * n + i] = (uint8_t)in1;
            rp.logp[(size_t)t * n + i] = lp;
        }
        if (P2POL) {
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
        // ---- sample + FootsiesEnv.step for the CTA's battles (same order of events as step_kernel) ----
        if (sim_thread) {
            double reward = 0.0;
            bool terminal = false, ran = false;
            if (valid) {
                if ((e.misc >> FGM_DONE_SHIFT) & 1u) {                  // next-step autoreset: this step only resets
                    reset_env<false, kP2Bot>(T, e, p.stale_intro != 0);
                    acc.s += 0x10000u;
                } else {
                    ran = true;
                    if (kP2Bot) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
                    for (int kk = 0; kk < K; kk++) {
                        if (!terminal) {
                            simulate_frame<false, kP2Bot, DENSE, false>(T, e, in1, in2, reward, terminal, acc);
                            acc.s += 1u << 24;
                            if (kP2Bot) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
                        }
                    }
                }
            }
            if (SKIP) {
                // fused FootsiesFrameSkipped (fg_config.skip_unactionable), exactly as in step_kernel: warp-synchronous so that the statistics fold
                // stays a warp-uniform decision
                bool more = ran && !terminal && obs_is_skippable(e);
                while (__any_sync(kFull, more)) {
                    for (int kk = 0; kk < K; kk++) {
                        if (more && !terminal) {
                            simulate_frame<false, kP2Bot, DENSE, false>(T, e, 0u, in2, reward, terminal, acc);
                            acc.s += 1u << 24;
                            if (kP2Bot) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
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
                const float4 a = make_float4(o.obs[0], o.obs[1], o.obs[2], o.obs[3]), b = make_float4(o.obs[4], o.obs[5], o.obs[6], o.obs[7]);
                const size_t dst = ((size_t)(t + 1) * n + i) * 2;
                rp.obs[dst] = a; rp.obs[dst + 1] = b;
                rp.rewards[(size_t)t * n + i] = (float)reward;
                rp.dones[(size_t)t * n + i] = terminal ? 1 : 0;
                obs_s[2 * stid] = a; obs_s[2 * stid + 1] = b;
                if (t == horizon - 1) { p.info_frame[i] = e.frame; p.info_misc[i] = o.info_misc; }
            }
            frames_since_flush += (uint32_t)K;                          // uniform across the warp
            if (frames_since_flush >= kStatFlushFrames) { flush_stats(acc, s_stats, lane); frames_since_flush = 0u; }
        }
        __syncthreads();
    }
    if (sim_thread) {
        if (valid) store_env<kP2Bot>(p, i, e);
        flush_stats(acc, s_stats, lane);
    }
    __syncthreads();
    if (tid < FG_STAT_COUNT && s_stats[tid]) atomicAdd(&p.stats[tid], s_stats[tid]);
    if constexpr (POOL) pool_flush(rp.pool, member, s_stats, tid);
}

// ---- tensor-core version (H <= 64): every WARP owns 16 MT battles for the whole horizon -- policy (policy_mma.cuh: mma.sync
// m16n8k8 with the 3 x TF32 split, activations never leave the registers between layers) and simulator alike -- so the
// horizon loop contains no CTA barrier at all: warps drift apart and one warp's simulator phase overlaps its neighbours'
// tensor-core phases.  MT = 2: 32 battles per warp, every lane simulates one; MT = 1: 16 battles per warp (lanes 16-31 only
// feed the MMA), twice the warps per SM -- what a batch of 16 384 battles (111 per SM) needs to keep two warps per scheduler.
template <int H, int W, bool P2POL>
struct RolloutMmaSmem {
    using PL = PolicyMmaSmem<H>;
    static constexpr size_t kTables = 0;
    static constexpr size_t kPolicy = (sizeof(Tables) + 127) / 128 * 128;
    static constexpr size_t kPolicy2 = kPolicy + (PL::kBytes + 15) / 16 * 16;
    static constexpr size_t kObs = kPolicy2 + (P2POL ? (PL::kBytes + 15) / 16 * 16 : 0);      // float [W][32][8]
    static constexpr size_t kLogits = kObs + sizeof(float) * W * 256;                        // float [W][32][8]
    static constexpr size_t kStats = kLogits + sizeof(float) * W * 256;
    static constexpr size_t kBytes = kStats + sizeof(unsigned long long) * FG_STAT_COUNT;
};

// developer knob: CTAs per SM the 32-battle-warp shape is compiled for.  Measured (profiles/r03f_rollout_mt2_blocks.log): forcing 3
// (168 registers instead of 190, 24 bytes of spill, 12 instead of 8 warps per SM) LOSES -- 1 Mi battles 143.1 vs 137.5 us per
// step, 131 072: 19.3 vs 18.7.
#ifndef FG_ROLLOUT_MT2_MIN_BLOCKS
#define FG_ROLLOUT_MT2_MIN_BLOCKS 1
#endif
template <int H, int W, int MT, bool DENSE, bool P2POL, bool SKIP, bool POOL = false>
__global__ void __launch_bounds__(32 * W, (MT == 2 && !P2POL) ? FG_ROLLOUT_MT2_MIN_BLOCKS : 1)
rollout_mma_kernel(const typename RolloutArgs<POOL>::type rp) {
    using SM = RolloutMmaSmem<H, W, P2POL>;
    constexpr bool kP2Bot = !P2POL;
    constexpr int kWarpEnvs = 16 * MT, kEnvs = kWarpEnvs * W;
    static_assert(!POOL || (P2POL && FG_POOL_BLOCK % kEnvs == 0), "a pool CTA plays against one member");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Tables &Tw = *reinterpret_cast<Tables *>(smem_raw + SM::kTables);
    const Tables &T = Tw;
    float *pw = reinterpret_cast<float *>(smem_raw + SM::kPolicy);
    float *pw2 = reinterpret_cast<float *>(smem_raw + SM::kPolicy2);
    unsigned long long *s_stats = reinterpret_cast<unsigned long long *>(smem_raw + SM::kStats);
    const Params &p = rp.sim;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
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
        policy_mma_stage<H>(pw2, pool_weights(rp.pool, member), tid, 32 * W);
    } else if (P2POL) policy_mma_stage<H>(pw2, rp.w_p2, tid, 32 * W);
    if (tid < FG_STAT_COUNT) s_stats[tid] = 0ull;
    Env e;
    if (valid) load_env<kP2Bot>(p, i, e);
    {
        // the observation the first step acts on: the last one of the previous horizon, carried over into slot 0
        float4 a = make_float4(0, 0, 0, 0), b = a;
        if (valid) {
            const size_t src = ((size_t)horizon * n + i) * 2;
            a = rp.obs[src]; b = rp.obs[src + 1];
            rp.obs[(size_t)i * 2] = a; rp.obs[(size_t)i * 2 + 1] = b;
        }
        reinterpret_cast<float4 *>(obs_w)[2 * lane] = a; reinterpret_cast<float4 *>(obs_w)[2 * lane + 1] = b;
    }
    __syncthreads();                                            // tables, weight fragments, statistics: the only CTA barrier before the end
    const unsigned long long drawn = rp.counter_base ? *rp.counter_base : 0ull;
    StatAcc acc = { 0u, 0u, 0u, 0u };
    uint32_t frames_since_flush = 0u;
    const int K = p.frame_skip;

    for (int t = 0; t < horizon; t++) {
        // ---- policy: the warp's battles through the MLP on the tensor cores, then one lane per battle samples ----
        // (the random words do not depend on the logits: their 64-bit multiply chains are issued before the MMAs, under
        // whose latency they complete)
        const uint32_t rnd1 = hash3(rp.seed, drawn + (unsigned long long)t, (uint64_t)(p.first_env_index + i));
        const uint32_t rnd2 = P2POL ? hash3(rp.seed_p2, drawn + (unsigned long long)t, (uint64_t)(p.first_env_index + i)) : 0u;
        policy_mma_logits<H, MT, false>(pw, obs_w, lg_w, lane);
        uint32_t in1 = 0u, in2 = 0u;
        if (valid) {
            const float4 l0 = reinterpret_cast<const float4 *>(lg_w)[2 * lane], l1 = reinterpret_cast<const float4 *>(lg_w)[2 * lane + 1];
            const float lg[8] = { l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w };
            float lp;
            in1 = (uint32_t)policy_sample(lg, rnd1, lp);
            rp.actions[(size_t)t * n + i] = (uint8_t)in1;
            rp.logp[(size_t)t * n + i] = lp;
        }
        if (P2POL) {
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
        // ---- FootsiesEnv.step for the warp's battles (same order of events as step_kernel) ----
        double reward = 0.0;
        bool terminal = false, ran = false;
        if (valid) {
            if ((e.misc >> FGM_DONE_SHIFT) & 1u) {                      // next-step autoreset: this step only resets
                reset_env<false, kP2Bot>(T, e, p.stale_intro != 0);
                acc.s += 0x10000u;
            } else {
                ran = true;
                if (kP2Bot) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
                for (int kk = 0; kk < K; kk++) {
                    if (!terminal) {
                        simulate_frame<false, kP2Bot, DENSE, false>(T, e, in1, in2, reward, terminal, acc);
                        acc.s += 1u << 24;
                        if (kP2Bot) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
                    }
                }
            }
        }
        if (SKIP) {                                                     // fused FootsiesFrameSkipped, exactly as in step_kernel
            bool more = ran && !terminal && obs_is_skippable(e);
            while (__any_sync(kFull, more)) {
                for (int kk = 0; kk < K; kk++) {
                    if (more && !terminal) {
                        simulate_frame<false, kP2Bot, DENSE, false>(T, e, 0u, in2, reward, terminal, acc);
                        acc.s += 1u << 24;
                        if (kP2Bot) in2 = (e.misc >> FGM_ACTOR2_SHIFT) & 7u;
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
            const float4 a = make_float4(o.obs[0], o.obs[1], o.obs[2], o.obs[3]), b = make_float4(o.obs[4], o.obs[5], o.obs[6], o.obs[7]);
            const size_t dst = ((size_t)(t + 1) * n + i) * 2;
            rp.obs[dst] = a; rp.obs[dst + 1] = b;
            rp.rewards[(size_t)t * n + i] = (float)reward;
            rp.dones[(size_t)t * n + i] = terminal ? 1 : 0;
            reinterpret_cast<float4 *>(obs_w)[2 * lane] = a; reinterpret_cast<float4 *>(obs_w)[2 * lane + 1] = b;
            if (t == horizon - 1) { p.info_frame[i] = e.frame; p.info_misc[i] = o.info_misc; }
        }
        frames_since_flush += (uint32_t)K;                              // uniform across the warp
        if (frames_since_flush >= kStatFlushFrames) { flush_stats(acc, s_stats, lane); frames_since_flush = 0u; }
        __syncwarp();                                                   // observation rows are in place for the next policy pass
    }
    if (valid) store_env<kP2Bot>(p, i, e);
    flush_stats(acc, s_stats, lane);
    __syncthreads();
    if (tid < FG_STAT_COUNT && s_stats[tid]) atomicAdd(&p.stats[tid], s_stats[tid]);
    if constexpr (POOL) pool_flush(rp.pool, member, s_stats, tid);
}

// RP = RolloutParams, or RolloutPoolParams for the opponent-pool instantiations (POOL)
template <class RP> constexpr bool kIsPool = std::is_same<RP, RolloutPoolParams>::value;

template <int H, int W, int MT, bool DENSE, bool P2POL, bool SKIP, class RP>
static cudaError_t launch_rollout_mma_s(cudaStream_t s, const RP &rp) {
    constexpr bool POOL = kIsPool<RP>;
    constexpr size_t bytes = RolloutMmaSmem<H, W, P2POL>::kBytes;
    static fg::DeviceOnceFlags configured;
    if (cudaError_t e = fg::configure_once_per_device(configured, [] {
            return cudaFuncSetAttribute(rollout_mma_kernel<H, W, MT, DENSE, P2POL, SKIP, POOL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); }))
        return e;
    constexpr int kEnvs = 16 * MT * W;
    const int grid = (rp.sim.n + kEnvs - 1) / kEnvs;
    rollout_mma_kernel<H, W, MT, DENSE, P2POL, SKIP, POOL><<<grid, 32 * W, bytes, s>>>(rp);
    return cudaSuccess;
}
template <int H, int W, bool DENSE, class RP>
static cudaError_t launch_rollout_mma_w(int mt, cudaStream_t s, const RP &rp) {
    const bool skip = rp.sim.skip_unactionable != 0;
#define FG_MMA_GO(MT, P2, SK) launch_rollout_mma_s<H, W, MT, DENSE, P2, SK>(s, rp)
    if (kIsPool<RP> || rp.p2_policy) {
        if (mt == 1) return skip ? FG_MMA_GO(1, true, true) : FG_MMA_GO(1, true, false);
        return skip ? FG_MMA_GO(2, true, true) : FG_MMA_GO(2, true, false);
    }
    if constexpr (!kIsPool<RP>) {
        if (mt == 1) return skip ? FG_MMA_GO(1, false, true) : FG_MMA_GO(1, false, false);
        return skip ? FG_MMA_GO(2, false, true) : FG_MMA_GO(2, false, false);
    }
#undef FG_MMA_GO
    return cudaErrorInvalidValue;
}
template <int H, bool DENSE, class RP>
static cudaError_t launch_rollout_mma(cudaStream_t s, const RP &rp) {
    // Measured (profiles/r02f_rollout_mma.log, H = 64, us per step, 16-battle / 32-battle warps / round-1 FFMA2 kernel):
    // 16 384 battles 4.49 / 5.90 / 6.37; 131 072: 28.0 / 31.3 / -; 1 Mi: 216 / 227 / 262 -- more, lighter warps hide the
    // simulator's latency under the neighbours' tensor-core phases at every size, so 16-battle warps are the default
    // (developer knob: FOOTSIES_B200_ROLLOUT_MT = 1 | 2).
    int mt = rp.sim.n >= 131072 ? 2 : 1;
    if (const char *v = getenv("FOOTSIES_B200_ROLLOUT_MT")) mt = atoi(v) == 2 ? 2 : 1;
    // (7-warp CTAs, which would spread 16 384 battles evenly as 147 x 112, measured 4.55 us per step against 4.46 for 4 warps.)
    // (8-battle warps -- half-empty M tiles, twice the warps, 124 registers -- are the same bits and SLOWER from 8192 battles up:
    // 16 384 battles 4.98 vs 3.35 us per step; only 4096 battles gain, 2.30 vs 2.46.  A one-off start stagger between the two
    // CTAs of an SM changes nothing: 3.33 vs 3.32.  tools/probes/half_tile_and_stagger_experiment.patch,
    // profiles/r03h_rollout_half_tiles.log, r03i_rollout_stagger.log.  Step time against batch size -- 4096: 2.46, 8192: 2.48,
    // 16 384: 3.35, 32 768: 6.33 -- says the kernel leaves the latency-bound regime right at one CTA per SM.)
    // Two policies (self-play): 32-battle warps from 131 072 battles up (1 Mi: 479 us per step against 567).
    return launch_rollout_mma_w<H, 4, DENSE>(mt, s, rp);
}

template <int H, int E, int W, bool DENSE, bool P2POL, bool SKIP, class RP>
static cudaError_t launch_rollout_s(cudaStream_t s, const RP &rp) {
    constexpr bool POOL = kIsPool<RP>;
    constexpr size_t bytes = RolloutSmem<H, E, W, P2POL>::kBytes;
    static fg::DeviceOnceFlags configured;
    if (cudaError_t e = fg::configure_once_per_device(configured, [] {
            return cudaFuncSetAttribute(rollout_kernel<H, E, W, DENSE, P2POL, SKIP, POOL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); }))
        return e;
    constexpr int kEnvs = RolloutSmem<H, E, W, P2POL>::kEnvs;
    const int grid = (rp.sim.n + kEnvs - 1) / kEnvs;
    rollout_kernel<H, E, W, DENSE, P2POL, SKIP, POOL><<<grid, 32 * W, bytes, s>>>(rp);
    return cudaSuccess;
}
template <int H, int E, int W, bool DENSE, bool P2POL, class RP>
static cudaError_t launch_rollout_v(cudaStream_t s, const RP &rp) {
    return rp.sim.skip_unactionable ? launch_rollout_s<H, E, W, DENSE, P2POL, true>(s, rp) : launch_rollout_s<H, E, W, DENSE, P2POL, false>(s, rp);
}

template <int H, bool DENSE, class RP>
static cudaError_t launch_rollout_h(cudaStream_t s, const RP &rp) {
    if constexpr (H <= kMmaMaxHidden) {
        if (!getenv("FOOTSIES_B200_ROLLOUT_FFMA")) return launch_rollout_mma<H, DENSE>(s, rp);   // knob: the round-1 FFMA2 kernel for A/B runs
    }
    // battles per lane (measured, tools/rollout_sweep.py, H = 64, us per step): 16 384 battles E = 2 / 4: 6.5 / 7.2 (too few
    // CTAs for E = 4); 131 072: 37.5 / 34.6; 1 Mi: 288 / 264
    int e = rp.sim.n >= 65536 ? 4 : 2;
    if (const char *v = getenv("FOOTSIES_B200_ROLLOUT_E")) e = atoi(v);   // developer knob
    constexpr int E4 = H <= 64 ? 4 : 2;                                  // H = 128: 4 battles per lane do not fit the registers
    if (kIsPool<RP> || rp.p2_policy)       // two weight sets in shared memory: always 2 battles per lane
        return launch_rollout_v<H, 2, kPolicyWarps, DENSE, true>(s, rp);
    if constexpr (!kIsPool<RP>) {
        if (e == 1) return launch_rollout_v<H, 1, kPolicyWarps, DENSE, false>(s, rp);
        return e == 4 ? launch_rollout_v<H, E4, kPolicyWarps, DENSE, false>(s, rp) : launch_rollout_v<H, 2, kPolicyWarps, DENSE, false>(s, rp);
    }
    return cudaErrorInvalidValue;
}

// One translation unit per hidden size and reward mode (build.py compiles this file with -DFG_ROLLOUT_H=.. -DFG_ROLLOUT_DENSE=..
// so that the kernels compile in parallel) plus one without the defines that holds the dispatcher.
#define FG_ROLLOUT_DECL(H, D) cudaError_t launch_rollout_##H##_##D(cudaStream_t s, const RolloutParams &rp)
FG_ROLLOUT_DECL(32, 0); FG_ROLLOUT_DECL(32, 1); FG_ROLLOUT_DECL(64, 0); FG_ROLLOUT_DECL(64, 1); FG_ROLLOUT_DECL(128, 0); FG_ROLLOUT_DECL(128, 1);
#define FG_ROLLOUT_POOL_DECL(H, D) cudaError_t launch_rollout_pool_##H##_##D(cudaStream_t s, const RolloutPoolParams &rp)
FG_ROLLOUT_POOL_DECL(32, 0); FG_ROLLOUT_POOL_DECL(32, 1); FG_ROLLOUT_POOL_DECL(64, 0); FG_ROLLOUT_POOL_DECL(64, 1);
FG_ROLLOUT_POOL_DECL(128, 0); FG_ROLLOUT_POOL_DECL(128, 1);
#ifdef FG_ROLLOUT_H
#define FG_ROLLOUT_DEF2(H, D) FG_ROLLOUT_DECL(H, D) { return launch_rollout_h<H, (D != 0)>(s, rp); } \
    FG_ROLLOUT_POOL_DECL(H, D) { return launch_rollout_h<H, (D != 0)>(s, rp); }
#define FG_ROLLOUT_DEF(H, D) FG_ROLLOUT_DEF2(H, D)
FG_ROLLOUT_DEF(FG_ROLLOUT_H, FG_ROLLOUT_DENSE)
#else
cudaError_t launch_rollout(bool dense, cudaStream_t s, const RolloutParams &rp) {
    switch (rp.hidden) {
    case 32: return dense ? launch_rollout_32_1(s, rp) : launch_rollout_32_0(s, rp);
    case 64: return dense ? launch_rollout_64_1(s, rp) : launch_rollout_64_0(s, rp);
    case 128: return dense ? launch_rollout_128_1(s, rp) : launch_rollout_128_0(s, rp);
    default: return cudaErrorInvalidValue;
    }
}
cudaError_t launch_rollout_pool(bool dense, cudaStream_t s, const RolloutPoolParams &rp) {
    switch (rp.hidden) {
    case 32: return dense ? launch_rollout_pool_32_1(s, rp) : launch_rollout_pool_32_0(s, rp);
    case 64: return dense ? launch_rollout_pool_64_1(s, rp) : launch_rollout_pool_64_0(s, rp);
    case 128: return dense ? launch_rollout_pool_128_1(s, rp) : launch_rollout_pool_128_0(s, rp);
    default: return cudaErrorInvalidValue;
    }
}
#endif

}  // namespace fgk
