#ifndef FOOTSIES_B200_ROLLOUT_KERNEL_H
#define FOOTSIES_B200_ROLLOUT_KERNEL_H
// rollout_kernel.h -- host-side interface of the whole-horizon rollout kernel (rollout_kernel.cu), used by the C ABI.
#include "policy_mlp.cuh"
#include "step_kernel.cuh"

namespace fgk {

// P2 from an opponent pool: member m plays the battles [end[m - 1], end[m]).  The boundaries are multiples of FG_POOL_BLOCK
// (or n), so each CTA belongs to one member, stages its weights where the single P2 policy's go and adds its episode
// results to stats[member][0..3] (optional) when it flushes its statistics at the end.
struct RolloutPool {
    fgp::PolicyWeights member[FG_POOL_MAX];
    long long end[FG_POOL_MAX];
    int count;
    unsigned long long *stats;  // [count][4] or null
};

// Observations delayed by frame_delay = depth - 1 steps: the queue of every battle is the caller's ring (delay_ring.cuh),
// advanced once per step at position (pos + t) % depth; out_* receive the delayed state after the last step.
struct RolloutRing {
    float4 *obs;                // [depth][n][2]
    int32_t *frame;             // [depth][n]
    uint32_t *misc;             // [depth][n]
    float4 *out_obs;            // [n][2]
    int32_t *out_frame;         // [n]
    uint32_t *out_misc;         // [n]
    int depth, pos;
};

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
    RolloutPool pool;           // P2 from an opponent pool when pool.count > 0 (then p2_policy = 1 and w_p2 is not read)
    int bot_member;             // the pool member played by the in-game bot (its weights are not read), or -1
    RolloutRing ring;           // ring.depth = 0: no frame_delay
};

// P1 = the MLP policy, P2 = the in-game BattleAI, a second MLP policy (p2_policy) or an opponent pool, autoreset on, with
// the frame_delay queue when ring.depth > 0.  Returns cudaErrorInvalidValue for other hidden sizes.
cudaError_t launch_rollout(bool dense, cudaStream_t s, const RolloutParams &rp);

}  // namespace fgk
#endif
