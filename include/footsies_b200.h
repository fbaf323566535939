/*
 * footsies_b200.h -- C ABI of the B200-native batched FOOTSIES simulator (libfootsies_b200.so).
 *
 * The reference (martinhoT/Footsies-Gym) has no FFI: its de-facto boundary is the Gymnasium API of
 * FootsiesEnv (footsies-gym/footsies_gym/envs/footsies.py:20-588) on top of a TCP protocol to the Unity
 * game (footsies.py:261-334, Assets/Script/SocketHelper.cs:48-82, TrainingRemoteControl.cs:18-107).
 * This library replaces everything below that API -- process, sockets, JSON and the C# battle engine --
 * for N independent battles per call.  Each entry point names the reference interface it stands in for.
 *
 * Conventions: plain pointers and sizes only; every function returns FG_OK (0) or a negative fg_status;
 * fg_last_error() returns a thread-local message for the last failure; nothing throws.  The library never
 * allocates or frees the buffers passed to fg_bind (the host language owns them, e.g. torch tensors).
 * `stream` arguments are a cudaStream_t passed as void* (NULL = default stream); device-buffer entry
 * points only enqueue work and return.  One handle per GPU / host thread; handles share no mutable state.
 */
#ifndef FOOTSIES_B200_H
#define FOOTSIES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2 (round 2): fg_env_state.p1_bot_memory, first_env_index argument of fg_policy_mlp_sample[_p2], packed host layout
 * (fg_packed_result, fg_step_host_packed, fg_reset_host_packed, fg_packed_reward_table), fg_host_alloc / fg_host_free.
 * Added since, backward compatible (new entry points only, so still 2): fg_value_mlp, fg_gae, fg_rollout_mlp_pool. */
#define FG_ABI_VERSION 2

typedef enum {
    FG_OK = 0,
    FG_ERR_INVALID_ARGUMENT = -1,
    FG_ERR_NOT_BOUND = -2,
    FG_ERR_CUDA = -3,
    FG_ERR_NO_DEVICE = -4,
    FG_ERR_INVALID_STATE = -5
} fg_status;

/* Opponent / actor wiring (GameManager.cs:184-205 flags --p1-bot / --p2-bot, footsies.py:230-247). */
typedef struct {
    int32_t struct_size;        /* sizeof(fg_config), for ABI evolution                                   */
    int32_t num_envs;           /* battles stepped per call on this device                                */
    int32_t device;             /* CUDA device ordinal                                                    */
    int32_t p1_bot;             /* 1: P1 is the in-game BattleAI (FootsiesEnv by_example)                 */
    int32_t p2_bot;             /* 1: P2 is the in-game BattleAI (opponent=None); 0: P2 from actions_p2   */
    int32_t dense_reward;       /* FootsiesEnv dense_reward (footsies.py:388-405), else sparse (:382-386) */
    int32_t frame_skip;         /* K >= 1 frames fused per fg_step with the same action; stops at KO      */
    int32_t autoreset;          /* 0: finished battles freeze until fg_reset; 1: the step after a terminal
                                   one performs the reset and returns the frame -1 state                  */
    int32_t stale_intro_input;  /* 1 = reference behaviour: the Intro frame replays the actors' last input */
    int32_t skip_unactionable;  /* 1: FootsiesFrameSkipped (wrappers/frame_skip.py:46-80) fused into fg_step: after the
                                   step, a battle whose observation P1 cannot act on (frame_skip.py:56-66) keeps stepping
                                   with P1's no-op input inside the same launch; rewards are summed                 */
    int64_t first_env_index;    /* global index of env 0 (multi-GPU sharding; seeds use global indices)   */
} fg_config;

/* Compact battle state: 4 planes of 16 bytes per env (64 B/env), structure-of-arrays, 16-byte aligned.
 * Layout of the words is private to the library (see csrc/state_codec.h); use fg_get_state/fg_set_state. */
#define FG_STATE_PLANES 4
#define FG_STATE_PLANE_BYTES_PER_ENV 16

enum { FG_STAT_EPISODES = 0, FG_STAT_P1_WINS, FG_STAT_P2_WINS, FG_STAT_DOUBLE_KO, FG_STAT_EPISODE_FRAMES,
       FG_STAT_P1_SPECIALS, FG_STAT_P1_SPECIALS_NEUTRAL, FG_STAT_GUARD_BREAKS, FG_STAT_HITS, FG_STAT_BLOCKS,
       FG_STAT_ENV_FRAMES,      /* fight frames simulated: the env-frames counter of the throughput metric */
       FG_STAT_RESETS, FG_STAT_COUNT = 16 };

/* All pointers are DEVICE pointers owned by the caller and must stay valid while bound. */
typedef struct {
    int32_t struct_size;
    int32_t reserved0;
    void *state[FG_STATE_PLANES];   /* each: 16 * num_envs bytes, 16-byte aligned                         */
    uint64_t *stats;                /* [FG_STAT_COUNT] episode statistics (wrappers/statistics.py:26-50 and
                                       the win-rate loop footsies.py:657-661), accumulated by warp reductions */
    const uint8_t *actions_p1;      /* [num_envs] bitmask Left=1 Right=2 Attack=4 (InputData.cs:8-14; the
                                       3 bytes FootsiesEnv._send_action sends, footsies.py:323-334, packed) */
    const uint8_t *actions_p2;      /* [num_envs] same for P2; may be NULL when p2_bot                     */
    float *obs;                     /* [num_envs][8]: guard p1,p2 | move index p1,p2 | move_frame p1,p2 |
                                       position p1,p2  (FootsiesEnv._extract_obs, footsies.py:336-368)     */
    float *reward;                  /* [num_envs] (footsies.py:382-405)                                    */
    uint8_t *terminated;            /* [num_envs] p1Vital == 0 or p2Vital == 0 (footsies.py:555)           */
    int32_t *info_frame;            /* [num_envs] info["frame"] (footsies.py:370-380)                      */
    uint8_t *info_misc;             /* [num_envs][4]: p1_action mask, p2_action mask, p1_hitstun, p2_hitstun */
    const uint8_t *step_mask;       /* optional [num_envs]: fg_step only advances envs with a non-zero entry (NULL =
                                       all); the others keep their state and outputs (used by the batched
                                       FootsiesFrameSkipped wrapper, wrappers/frame_skip.py:46-80)          */
} fg_buffers;

/* Expanded, readable per-env state (superset of EnvironmentState.cs:12-26; the fields of
 * FighterState.cs:26-56 that survive compaction).  Same field order as the test oracle's trace. */
typedef struct {
    float pos_x;
    float velocity_x;
    int32_t action_id;          /* CommonActionID value (Fighter.cs:42-61), e.g. 110                      */
    int32_t action_frame;
    int32_t hitstun;
    int32_t guard;
    int32_t vital;
    int32_t hit_count;
    int32_t buffer_id;          /* -1 or 110                                                              */
    int32_t reserve_id;         /* -1 or 310                                                              */
    int32_t is_input_backward;
    int32_t is_reserve_prox;
    int32_t shake;              /* spriteShakePosition                                                    */
    int32_t has_won;            /* always 0: WIN is unreachable in training (SURVEY App. B-12)            */
    int32_t input0;             /* input applied on the most recent frame                                 */
    uint32_t hist_left;         /* bit i: Left held i frames ago, i < 16                                  */
    uint32_t hist_right;
    int32_t attack_run;         /* consecutive most-recent frames with Attack held, saturating at 59      */
} fg_fighter_state;

typedef struct {
    fg_fighter_state f[2];
    int32_t frame;              /* BattleCore.frameCount                                                  */
    int32_t recorded_input[2];  /* p{1,2}MostRecentAction (BattleCore.cs:463-464)                         */
    int32_t done;               /* battle is over and waiting for a reset                                 */
    int32_t cum_reward_index;   /* index into the dense-reward automaton                                  */
    int32_t actor_input[2];     /* input each actor holds for the next frame (bots: already decided)      */
    uint32_t rng_state[4];      /* per-env xorshift128 standing in for UnityEngine.Random                 */
    uint32_t bot_queue[2];      /* per bot: move position[0:9) remaining[9:16) attack position[16:24) remaining[24:31) */
    int32_t p1_bot_memory;      /* by_example only: what P1's BattleAI keeps across rounds -- it is never Reset() because the
                                   game wraps it in a spectator actor (BattleCore.cs:274, GameManager.cs:200-201).  bit 8: it
                                   has been queried at least once (fightStates no longer null, BattleAI.cs:30,47); while `done`:
                                   bits [0:3) distance bucket, [3:8) opponent action index of its last recorded FightState */
} fg_env_state;

typedef struct fg_handle fg_handle;

/* Library / build identification. */
int32_t fg_abi_version(void);
const char *fg_last_error(void);
/* Bytes of algorithmic HBM traffic of ONE single-frame fg_step for one env (state read + write, actions,
 * obs, reward, terminated, info) under the given config -- the numerator of the roofline in bench.py. */
int32_t fg_algorithmic_bytes_per_env_step(const fg_config *cfg);

/* Replaces: FootsiesEnv.__init__ + _instantiate_game + _connect_to_game (footsies.py:34-290). */
int32_t fg_create(const fg_config *cfg, fg_handle **out);
/* Replaces: FootsiesEnv.close (footsies.py:572-578). */
void fg_destroy(fg_handle *h);
int32_t fg_bind(fg_handle *h, const fg_buffers *buffers);

/* Replaces: remote-control SEED (footsies.py:454-456, BattleCore.cs:170-173): per env
 * Random.InitState(seed_base + global env index).  mask: device uint8[num_envs] or NULL = all. */
int32_t fg_seed(fg_handle *h, int64_t seed_base, const uint8_t *mask, void *stream);
/* Replaces: FootsiesEnv.reset / remote-control RESET (footsies.py:482-515, BattleCore.cs:143-146, 262-291):
 * Stop -> Intro -> one Intro frame -> Fight; writes the frame -1 observation.  mask as above. */
int32_t fg_reset(fg_handle *h, const uint8_t *mask, void *stream);
/* Replaces: FootsiesEnv.step (footsies.py:518-570) for all envs: frame_skip fused BattleCore fight frames
 * (BattleCore.cs:201-220, 347-364) + bot query (TrainingManager.cs:59-77) + obs / reward / termination. */
int32_t fg_step(fg_handle *h, void *stream);
/* Same as fg_step but with HOST buffers (the reference-facing call: actions come from and results go to
 * host memory like the reference's socket messages): H2D actions, step, D2H results, synchronises.
 * Any output pointer may be NULL to skip that copy.  actions_p2 may be NULL when p2_bot. */
int32_t fg_step_host(fg_handle *h, const uint8_t *actions_p1, const uint8_t *actions_p2, float *obs,
                     float *reward, uint8_t *terminated, int32_t *info_frame, uint8_t *info_misc, void *stream);
/* Host-buffer variant of fg_reset: mask is a HOST uint8[num_envs] or NULL; copies back obs / info. */
int32_t fg_reset_host(fg_handle *h, const uint8_t *mask, float *obs, int32_t *info_frame, uint8_t *info_misc,
                      void *stream);

/* Compact host layout of one step's results: what FootsiesEnv.step returns (footsies.py:336-380, 555-570) with every
 * field in its natural width -- the reference's guard / move / move_frame are Python ints, here bytes -- 27 bytes per
 * battle instead of the 45 of the device layout, because the host-buffer call is bound by PCIe.  All pointers are HOST
 * pointers (pinned memory for full PCIe speed); any pointer may be NULL to skip that field, except that position and
 * obs_u8 go together. */
typedef struct {
    int32_t struct_size;
    int32_t reserved0;
    float *position;                /* [num_envs][2] obs["position"]                                           */
    uint8_t *obs_u8;                /* [num_envs][6] obs["guard"] p1,p2 | obs["move"] index p1,p2 | obs["move_frame"] p1,p2 */
    float *reward;                  /* [num_envs]                                                              */
    uint8_t *terminated;            /* [num_envs]                                                              */
    int32_t *info_frame;            /* [num_envs]                                                              */
    uint8_t *info_misc;             /* [num_envs][4] as in fg_buffers                                          */
} fg_host_outputs;
/* fg_step_host / fg_reset_host delivering the compact layout.  Batches above 1 Mi battles are cut into slices that are
 * pipelined over two library-owned streams (upload + simulate slice c+1 while slice c's results cross PCIe); the call
 * is ordered after prior work on `stream` and returns when every result is in host memory. */
int32_t fg_step_host_compact(fg_handle *h, const uint8_t *actions_p1, const uint8_t *actions_p2,
                             const fg_host_outputs *out, void *stream);
int32_t fg_reset_host_compact(fg_handle *h, const uint8_t *mask, const fg_host_outputs *out, void *stream);

/* ---- packed host layout: ONE 16-byte record per battle and ONE device->host copy per slice ------------------------------
 * The host-buffer calls are bound by the host link, not by the GPU, so the bytes per battle decide their throughput:
 * 45 (device layout) -> 27 (fg_host_outputs) -> 16 here.  Everything FootsiesEnv.step returns is in the record, losslessly:
 *   position[2]  obs["position"] as float32, bit for bit
 *   w0  [0:2) guard p1  [2:4) guard p2  [4:8) move index p1  [8:12) move index p2  [12:18) move_frame p1  [18:24) move_frame
 *       p2  [24] terminated  [25:28) info p1_action mask  [28:31) info p2_action mask        (footsies.py:336-380, 555)
 *   w1  [0:5) p1_hitstun  [5:10) p2_hitstun  [10:17) index of the reward in the table fg_packed_reward_table returns
 *       (the dense reward only ever takes a few dozen distinct float32 values: +-0.3 steps and the terminal
 *       compensations of footsies.py:388-405)  [17:32) info frame + 1, saturating at 32767 (frame -1 = reset -> 0)
 * Needs frame_skip = 1, no fused frame skipping (their summed rewards are not table values) and no frame_delay. */
typedef struct {
    float position[2];
    uint32_t w0, w1;
} fg_packed_result;
#define FG_PACKED_REWARD_TABLE_SIZE 128
/* table[i] for i < *count are the float32 rewards a record can carry, in ascending order (count <= 128). */
int32_t fg_packed_reward_table(fg_handle *h, float *table, int32_t *count);
/* fg_step_host / fg_reset_host delivering packed records to out[num_envs] (HOST memory, pinned for full link speed).
 * Large batches are pipelined in slices like fg_step_host_compact; each slice is one contiguous copy. */
int32_t fg_step_host_packed(fg_handle *h, const uint8_t *actions_p1, const uint8_t *actions_p2, fg_packed_result *out,
                            void *stream);
int32_t fg_reset_host_packed(fg_handle *h, const uint8_t *mask, fg_packed_result *out, void *stream);
/* Pinned host memory placed on the NUMA node of the GPU (the calling thread is bound to that node's CPUs while the pages
 * are allocated and first touched, then gets its affinity back): device<->host copies then stay on the socket the GPU
 * hangs off.  Returns NULL on failure (fg_last_error).  Free with fg_host_free. */
void *fg_host_alloc(int32_t device, uint64_t bytes);
void fg_host_free(void *p);

/* Replaces: the frame_delay queue of FootsiesEnv (footsies.py:129-131, 502-504, 533-535) for all envs: pushes the state
 * the last fg_step / fg_reset wrote to the bound obs / info buffers into slot `pos` of a ring of depth = frame_delay + 1
 * slots (into every slot for envs that step just reset) and emits the oldest slot, (pos + 1) % depth, to out_*.  The
 * caller owns the ring (DEVICE memory: ring_obs [depth][num_envs][8] floats, ring_frame [depth][num_envs], ring_misc
 * [depth][num_envs][4]) and advances pos by one (mod depth) per step.  Reward and termination are not delayed.  Battles
 * held back by the bound step mask keep their queue (their slots are rotated along with pos) and their last out_* entry. */
int32_t fg_delay_ring_step(fg_handle *h, int32_t depth, int32_t pos, float *ring_obs, int32_t *ring_frame, uint8_t *ring_misc,
                           float *out_obs, int32_t *out_frame, uint8_t *out_misc, void *stream);

/* Replaces: remote-control STATE_SAVE / STATE_LOAD (footsies.py:432-444, BattleCore.cs:667-683) at the level
 * of the compact state.  out / in are HOST arrays of `count` entries starting at env `first`. Synchronous. */
int32_t fg_get_state(fg_handle *h, int32_t first, int32_t count, fg_env_state *out);
int32_t fg_set_state(fg_handle *h, int32_t first, int32_t count, const fg_env_state *in);
/* Copies the statistics vector to the host (synchronises `stream`). */
int32_t fg_read_stats(fg_handle *h, uint64_t *out /* FG_STAT_COUNT */, void *stream);
/* Number of kernels this handle has launched so far (bench.py's gpu_launches claim). */
int64_t fg_launch_count(fg_handle *h);

/* BASELINE.json configs[4] (PPO rollout with an MLP policy reading the observation tensor in place; the reference's
 * agents run their policy in Python between two socket round trips, footsies.py:633-661): fused inference of
 * obs * scale -> Linear(8, H) -> tanh -> Linear(H, H) -> tanh -> Linear(H, 8) -> log-softmax -> categorical sample
 * for every env in one launch.  All pointers are DEVICE pointers; weights are row-major [out][in] like torch.nn.Linear.
 * hidden must be 32, 64 or 128.  actions receives the sampled index 0..7 = the input bitmask of fg_buffers.actions_p1
 * (wrappers/action_comb_disc.py:13-18); logp (optional) its log-probability; obs_copy (optional, [num_envs][8]) a copy
 * of obs, e.g. the rollout-buffer slot of this step.  The sample is a pure function of (seed, counter + *counter_base,
 * first_env_index + env index) -- the GLOBAL battle index, so that samples do not depend on how the battles are sharded
 * (pass fg_config.first_env_index); counter_base is an optional DEVICE word, so that a captured CUDA graph draws fresh
 * numbers on every replay by bumping it. */
int32_t fg_policy_mlp_sample(const float *obs, const float *scale, const float *w1, const float *b1, const float *w2,
                             const float *b2, const float *w3, const float *b3, int32_t hidden, int32_t num_envs,
                             uint64_t seed, uint64_t counter, const uint64_t *counter_base, uint8_t *actions, float *logp,
                             float *obs_copy, int64_t first_env_index, void *stream);
/* The same for a policy that drives P2: writes fg_buffers.actions_p2-style bitmasks; mirror = 1 feeds it the mirrored
 * observation and mirrors its action back (see fg_rollout_buffers.p2_mirror). */
int32_t fg_policy_mlp_sample_p2(const float *obs, const float *scale, const float *w1, const float *b1, const float *w2,
                                const float *b2, const float *w3, const float *b3, int32_t hidden, int32_t num_envs,
                                uint64_t seed, uint64_t counter, const uint64_t *counter_base, uint8_t *actions, float *logp,
                                int32_t mirror, int64_t first_env_index, void *stream);
const char *fg_policy_last_error(void);

/* BASELINE.json configs[4] as ONE launch per horizon: for t = 0 .. horizon - 1 { policy(obs[t]) -> sample -> actions[t],
 * logp[t]; FootsiesEnv.step -> obs[t + 1], rewards[t], dones[t] } for every battle of the handle, with the battle state in
 * registers throughout (csrc/rollout_kernel.cu).  obs[0] is first overwritten with obs[horizon] (the observation the
 * previous horizon, or the reset, ended on).  Bit-identical to `horizon` rounds of fg_policy_mlp_sample(counter = t) +
 * fg_step (+ fg_policy_mlp_sample_p2 for a policy-driven P2).  Needs p1_bot = 0, autoreset = 1, no step mask.  All pointers
 * are DEVICE pointers. */
typedef struct {
    int32_t struct_size;
    int32_t hidden;                 /* 32, 64 or 128                                                           */
    int32_t horizon;
    int32_t reserved0;
    const float *scale, *w1, *b1, *w2, *b2, *w3, *b3;   /* as in fg_policy_mlp_sample                          */
    uint64_t seed;
    const uint64_t *counter_base;   /* optional device word: policy steps drawn before this horizon            */
    float *obs;                     /* [horizon + 1][num_envs][8]                                              */
    uint8_t *actions;               /* [horizon][num_envs]                                                     */
    float *logp;                    /* [horizon][num_envs]                                                     */
    float *rewards;                 /* [horizon][num_envs]                                                     */
    uint8_t *dones;                 /* [horizon][num_envs]                                                     */
    /* P2 driven by a second MLP policy (self-play rollouts; required when p2_bot = 0, ignored otherwise): it reads the
     * same observation rows -- as the reference's `opponent(obs, info)` callable does, footsies.py:522-527 -- or, with
     * p2_mirror = 1, their mirror image (per-player fields swapped, positions negated; the sampled Left / Right bits are
     * mirrored back), so that one network can play both sides.  Same hidden size as P1's policy. */
    const float *p2_scale, *p2_w1, *p2_b1, *p2_w2, *p2_b2, *p2_w3, *p2_b3;
    uint64_t p2_seed;
    uint8_t *actions_p2;            /* [horizon][num_envs]                                                     */
    float *logp_p2;                 /* [horizon][num_envs]                                                     */
    int32_t p2_mirror;
    int32_t reserved1;
} fg_rollout_buffers;
int32_t fg_rollout_mlp(fg_handle *h, const fg_rollout_buffers *r, void *stream);

/* Self-play against an opponent pool: fg_rollout_mlp with P2 played by up to FG_POOL_MAX MLP policies at once, one per
 * contiguous range of battles -- member m plays the local battles [end[m - 1], end[m]) (end[-1] = 0), e.g. the learner
 * and frozen snapshots of it for fictitious self-play.  The reference has no counterpart; its nearest equivalent is the
 * per-process `opponent(obs, info)` callable (footsies.py:522-527).
 *   - end is non-decreasing; every boundary is a multiple of FG_POOL_BLOCK or equal to num_envs, and end[count - 1] =
 *     num_envs.  Empty ranges are allowed.  (A CTA of the kernel owns 64 or 128 battles, so it never spans two members.)
 *   - Every member has the learner's hidden size r->hidden; its weights are DEVICE pointers in torch.nn.Linear layout
 *     (w2 16-byte aligned).  r->p2_scale .. r->p2_b3 are ignored; p2_seed, actions_p2, logp_p2 and p2_mirror keep their
 *     meaning (the mirror applies to every member).  P2's samples depend on (p2_seed, step, GLOBAL battle index) only, so
 *     a battle of member m's range draws exactly what it would draw against member m alone.
 *   - stats (optional, DEVICE, 8-byte aligned, [count][4]): episodes, P1 wins, P2 wins and double KOs of each member's
 *     battles are ADDED to it, next to the handle's own statistics (which count every battle as before).
 * Needs p2_bot = 0 and everything fg_rollout_mlp needs.  Results are bit-identical to fg_rollout_mlp run on a handle of
 * just member m's battles (num_envs = end[m] - end[m - 1], first_env_index shifted by end[m - 1]) with member m as P2. */
#define FG_POOL_MAX 16
#define FG_POOL_BLOCK 128
typedef struct { const float *scale, *w1, *b1, *w2, *b2, *w3, *b3; } fg_mlp_weights;
typedef struct {
    int32_t struct_size, count;              /* 1 .. FG_POOL_MAX                                                       */
    fg_mlp_weights member[FG_POOL_MAX];      /* device pointers, torch.nn.Linear layout                                */
    int64_t end[FG_POOL_MAX];                /* non-decreasing, see above; empty ranges allowed                         */
    uint64_t *stats;                         /* optional device [count][4]: episodes, P1 wins, P2 wins, double KOs (accumulated) */
} fg_opponent_pool;
int32_t fg_rollout_mlp_pool(fg_handle *h, const fg_rollout_buffers *r, const fg_opponent_pool *pool, void *stream);

/* Critic side of an actor-critic (PPO) rollout, for any source of rollout buffers.  Handle-free like fg_policy_mlp_sample;
 * errors are reported through fg_policy_last_error().  All pointers are DEVICE pointers.
 *
 * fg_value_mlp: values[i] = V(obs[i] * scale) for a value network obs * scale -> Linear(8, H) -> tanh -> Linear(H, H) ->
 * tanh -> Linear(H, 1), for rows i = 0 .. rows - 1 of obs [rows][8] (e.g. a whole [horizon + 1][num_envs][8] rollout
 * buffer: rows may exceed INT32_MAX).  Weights row-major [out][in] like torch.nn.Linear: w1 [H][8], b1 [H], w2 [H][H],
 * b2 [H], w3 [1][H], b3 [1]; scale [8].  hidden must be 32 or 64.  It stands in for the separate torch value MLP of the
 * PPO example (examples/ppo_footsies.py before this entry point), on the tensor-core path of the policy kernel: agrees
 * with torch's fp32 forward to ~1e-5 relative. */
int32_t fg_value_mlp(const float *obs, const float *scale, const float *w1, const float *b1, const float *w2,
                     const float *b2, const float *w3, const float *b3, int32_t hidden, int64_t rows,
                     float *values, void *stream);
/* fg_gae: generalised advantage estimation over rewards [horizon][num_envs], dones [horizon][num_envs] (0 / 1 flags, e.g.
 * fg_rollout_buffers.dones) and values [horizon + 1][num_envs] (values[horizon] = the value of the observation after the
 * last step); writes advantages and returns [horizon][num_envs].  A done at step t cuts the bootstrap from t + 1 (the
 * autoreset step after it is an ordinary transition).  Per battle, for t = horizon - 1 .. 0, in fp32 and in this order:
 *   nt = 1 - dones[t];  delta = (rewards[t] + (gamma * values[t + 1]) * nt) - values[t];
 *   last = delta + (gamma_lambda * nt) * last  (last = 0 before t = horizon - 1);  advantages[t] = last;
 *   returns[t] = advantages[t] + values[t]
 * -- the torch loop of the PPO example (examples/ppo_footsies.py before this entry point) operation for operation, so the
 * results are bit-identical to it when gamma_lambda is gamma * lambda rounded to float from the double product. */
int32_t fg_gae(const float *rewards, const uint8_t *dones, const float *values, int32_t horizon, int32_t num_envs,
               float gamma, float gamma_lambda, float *advantages, float *returns, void *stream);

#ifdef __cplusplus
}
#endif
#endif
