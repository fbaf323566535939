#ifndef FOOTSIES_B200_ROLLOUT_KERNEL_H
#define FOOTSIES_B200_ROLLOUT_KERNEL_H
// rollout_kernel.h -- host-side interface of the whole-horizon rollout kernel (rollout_kernel.cu), used by the C ABI.
#include "policy_mlp.cuh"
#include "step_kernel.cuh"

namespace fgk {

struct RolloutParams {
    Params sim;                 // state planes, statistics, tables, info outputs, n, frame_skip, stale_intro
    fgp::PolicyWeights w;
    unsigned long long seed;
    const unsigned long long *counter_base;   // optional device word: policy steps drawn before this horizon
    int hidden, horizon;
    float4 *obs;                // [horizon + 1][n][2]
    uint8_t *actions;           // [horizon][n]
    float *logp;                // [horizon][n]
    float *rewards;             // [horizon][n]
    uint8_t *dones;             // [horizon][n]
    // P2 driven by a second policy instead of the in-game bot (self-play rollouts): same observation rows, optionally
    // mirrored; its own weights, seed and output slots
    int p2_policy, p2_mirror;
    fgp::PolicyWeights w_p2;
    unsigned long long seed_p2;
    uint8_t *actions_p2;        // [horizon][n]
    float *logp_p2;             // [horizon][n]
};

// P2 from an opponent pool (fg_rollout_mlp_pool): member m plays the battles [end[m - 1], end[m]).  The boundaries are
// multiples of FG_POOL_BLOCK (or n), so each CTA belongs to one member, stages its weights where the single P2 policy's go
// and adds its episode results to stats[member][0..3] (optional) when it flushes its statistics at the end.  A separate
// parameter struct, so that the kernels of the other modes keep their parameters and their code.
struct RolloutPool {
    fgp::PolicyWeights member[FG_POOL_MAX];
    long long end[FG_POOL_MAX];
    int count;
    unsigned long long *stats;  // [count][4] or null
};
struct RolloutPoolParams : RolloutParams {
    RolloutPool pool;
};
// The same with member bot_member played by the in-game BattleAI (fg_rollout_mlp_pool_bot): its CTAs run the P2 = bot
// horizon loop, and its weight pointers are never read.
struct RolloutPoolBotParams : RolloutPoolParams {
    int bot_member;
};

// Observations delayed by frame_delay = depth - 1 steps (fg_rollout_mlp_delayed): the queue of every battle is the caller's
// ring (delay_ring.cuh), advanced once per step at position (pos + t) % depth; out_* receive the delayed state after the
// last step.  One parameter struct for every P2 mode: pool.count = 0 is no pool, bot_member = -1 no bot member.
struct RolloutRing {
    float4 *obs;                // [depth][n][2]
    int32_t *frame;             // [depth][n]
    uint32_t *misc;             // [depth][n]
    float4 *out_obs;            // [n][2]
    int32_t *out_frame;         // [n]
    uint32_t *out_misc;         // [n]
    int depth, pos;
};
struct RolloutDelayParams : RolloutPoolBotParams {
    RolloutRing ring;
};

// P1 = the MLP policy, P2 = the in-game BattleAI or a second MLP policy (p2_policy), autoreset on.  Returns
// cudaErrorInvalidValue for other hidden sizes.
cudaError_t launch_rollout(bool dense, cudaStream_t s, const RolloutParams &rp);
// Any of the modes below or above with the frame_delay queue (P2 from rp.pool when rp.pool.count > 0).
cudaError_t launch_rollout_delayed(bool dense, cudaStream_t s, const RolloutDelayParams &rp);
// The same with P2 from an opponent pool (rp.p2_policy = 1; w_p2 is not read).
cudaError_t launch_rollout_pool(bool dense, cudaStream_t s, const RolloutPoolParams &rp);
// The same with member rp.bot_member played by the in-game bot (its weights are not read).
cudaError_t launch_rollout_pool_bot(bool dense, cudaStream_t s, const RolloutPoolBotParams &rp);

}  // namespace fgk
#endif
