// policy_kernel.cu -- fused inference of a small MLP policy over the step kernel's observation tensor:
// scale -> Linear(8, H) -> tanh -> Linear(H, H) -> tanh -> Linear(H, 8) -> log-softmax -> categorical sample, one launch.
//
// BASELINE.json configs[4] (PPO rollout, a torch MLP policy consuming obs in place, 16 384 envs per GPU) is bound by
// the dozen tiny torch kernels a policy step costs (~110 us per step, against ~6 us for the simulator step).  This
// kernel replaces them for the 8-H-H-8 tanh MLP of footsies_gym_b200.rollout.MLPPolicy: weights are staged once per CTA
// in shared memory; a CTA of 4 warps handles 64 battles at a time (warp = a quarter of the hidden units, lane = two
// battles; policy_mlp.cuh); the sampled action is written as the uint8 input bitmask the step kernel is bound to, next
// to its log-probability, and (optionally) the observation row is copied into the rollout buffer on the way.
// The per-step path for configurations the whole-horizon kernel (rollout_kernel.cu) does not cover (self-play, masks).
// Also the critic side of an actor-critic rollout: the value network on the same tensor-core path (fg_value_mlp) and GAE
// advantages / returns (fg_gae).
#include "device_once.h"
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/footsies_b200.h"
#include "policy_mlp.cuh"
#include "policy_mma.cuh"

namespace {

using namespace fgp;

constexpr int kPolThreads = 32 * kPolicyWarps;
constexpr int kPolE = 2;                       // battles per lane
constexpr int kPolEnvs = 32 * kPolE;           // battles per CTA pass

struct PolicyParams {
    const float *obs;          // [n, 8]
    PolicyWeights w;
    uint8_t *actions;          // [n]
    float *logp;               // [n] or null
    float *obs_copy;           // [n, 8] or null: rollout-buffer slot for this step's observations
    unsigned long long seed, counter;
    const unsigned long long *counter_base;   // optional device word added to `counter` (CUDA-graph replays bump it)
    int n, hidden;
    int mirror;                // 1: the policy drives P2 from the mirrored observation, its action is mirrored back
    long long first_env;       // global index of battle 0 (fg_config.first_env_index): samples do not depend on the sharding
};

template <int H>
__global__ void __launch_bounds__(kPolThreads) policy_mlp_sample_kernel(const PolicyParams p) {
    extern __shared__ __align__(16) float sm[];
    policy_stage_bcast<H, kPolEnvs, kPolicyWarps>(sm, p.w, threadIdx.x, kPolThreads);
    __syncthreads();
    const unsigned long long counter = p.counter + (p.counter_base ? *p.counter_base : 0ull);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int base = blockIdx.x * kPolEnvs; base < p.n; base += gridDim.x * kPolEnvs) {
        float x[kPolE][8];
#pragma unroll
        for (int q = 0; q < kPolE; q++) {
            const int env = base + lane + 32 * q;
            const bool valid = env < p.n;
            const float4 a = valid ? reinterpret_cast<const float4 *>(p.obs)[2 * (size_t)env] : make_float4(0, 0, 0, 0);
            const float4 b = valid ? reinterpret_cast<const float4 *>(p.obs)[2 * (size_t)env + 1] : make_float4(0, 0, 0, 0);
            if (valid && p.obs_copy && warp == 0) {
                reinterpret_cast<float4 *>(p.obs_copy)[2 * (size_t)env] = a;
                reinterpret_cast<float4 *>(p.obs_copy)[2 * (size_t)env + 1] = b;
            }
            x[q][0] = a.x; x[q][1] = a.y; x[q][2] = a.z; x[q][3] = a.w;
            x[q][4] = b.x; x[q][5] = b.y; x[q][6] = b.z; x[q][7] = b.w;
            if (p.mirror) policy_mirror_obs(x[q]);
        }
        policy_partials_bcast<H, kPolE, kPolicyWarps>(sm, sm + PolicySmemBcast<H, kPolEnvs, kPolicyWarps>::kWeightFloats, warp, lane, x);     // two CTA barriers inside
        const int env = base + tid;                             // one sampling thread per battle
        if (tid < kPolEnvs && env < p.n) {
            float lg[8], lp;
            policy_logits_of<H, kPolEnvs, kPolicyWarps>(sm, sm + PolicySmemBcast<H, kPolEnvs, kPolicyWarps>::kWeightFloats, tid, lg);
            int a = policy_sample(lg, hash3(p.seed, counter, (uint64_t)(p.first_env + env)), lp);
            if (p.mirror) a = policy_mirror_action(a);
            p.actions[env] = (uint8_t)a;
            if (p.logp) p.logp[env] = lp;
        }
        // no barrier needed here: the next pass writes the activations (nobody reads them any more) and only touches
        // the partial sums after its first barrier, which the sampling threads reach after they are done reading
    }
}

// The same policy step on the tensor-core path (policy_mma.cuh) for H <= 64: a warp owns 32 battles for the whole forward
// pass; the CTA's warps share nothing but the staged weight fragments.  Persistent: every warp walks groups of 32 battles.
constexpr int kMmaWarps = 4;
template <int H>
struct PolicyMmaKernelSmem {
    static constexpr size_t kObs = (PolicyMmaSmem<H>::kBytes + 15) / 16 * 16;             // float [kMmaWarps][32][8]
    static constexpr size_t kLogits = kObs + sizeof(float) * kMmaWarps * 256;
    static constexpr size_t kBytes = kLogits + sizeof(float) * kMmaWarps * 256;
};
template <int H, bool MIRROR>
__global__ void __launch_bounds__(32 * kMmaWarps) policy_mma_sample_kernel(const PolicyParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *sm = reinterpret_cast<float *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float *obs_w = reinterpret_cast<float *>(smem_raw + PolicyMmaKernelSmem<H>::kObs) + warp * 256;
    float *lg_w = reinterpret_cast<float *>(smem_raw + PolicyMmaKernelSmem<H>::kLogits) + warp * 256;
    policy_mma_stage<H>(sm, p.w, tid, 32 * kMmaWarps);
    __syncthreads();
    const unsigned long long counter = p.counter + (p.counter_base ? *p.counter_base : 0ull);
    for (int base = (blockIdx.x * kMmaWarps + warp) * 32; base < p.n; base += gridDim.x * kMmaWarps * 32) {
        const int env = base + lane;
        const bool valid = env < p.n;
        const float4 a = valid ? reinterpret_cast<const float4 *>(p.obs)[2 * (size_t)env] : make_float4(0, 0, 0, 0);
        const float4 b = valid ? reinterpret_cast<const float4 *>(p.obs)[2 * (size_t)env + 1] : make_float4(0, 0, 0, 0);
        if (valid && p.obs_copy) {
            reinterpret_cast<float4 *>(p.obs_copy)[2 * (size_t)env] = a;
            reinterpret_cast<float4 *>(p.obs_copy)[2 * (size_t)env + 1] = b;
        }
        __syncwarp();                                           // the previous group's fragment loads are done
        reinterpret_cast<float4 *>(obs_w)[2 * lane] = a;
        reinterpret_cast<float4 *>(obs_w)[2 * lane + 1] = b;
        __syncwarp();
        policy_mma_logits<H, 2, MIRROR>(sm, obs_w, lg_w, lane);
        if (valid) {
            const float4 l0 = reinterpret_cast<const float4 *>(lg_w)[2 * lane], l1 = reinterpret_cast<const float4 *>(lg_w)[2 * lane + 1];
            const float lg[8] = { l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w };
            float lp;
            int act = policy_sample(lg, hash3(p.seed, counter, (uint64_t)(p.first_env + env)), lp);
            if (MIRROR) act = policy_mirror_action(act);
            p.actions[env] = (uint8_t)act;
            if (p.logp) p.logp[env] = lp;
        }
    }
}

// Value network V(obs * scale) = Linear(H, 1)(tanh(Linear(H, H)(tanh(Linear(8, H)(obs * scale))))) over `rows` observation
// rows -- the critic of an actor-critic rollout, over all (horizon + 1) x N rows of a rollout buffer in one launch.  It is
// the policy's forward pass (policy_mma_logits) with W3 staged as ONE real output row: the value is logit column 0.  Same
// shape as policy_mma_sample_kernel: persistent grid, weights staged once per CTA, a warp evaluates 32 rows at a time.
template <int H>
__global__ void __launch_bounds__(32 * kMmaWarps) value_mma_kernel(const float *__restrict__ obs, const PolicyWeights w,
                                                                   long long rows, float *__restrict__ values) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *sm = reinterpret_cast<float *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float *obs_w = reinterpret_cast<float *>(smem_raw + PolicyMmaKernelSmem<H>::kObs) + warp * 256;
    float *lg_w = reinterpret_cast<float *>(smem_raw + PolicyMmaKernelSmem<H>::kLogits) + warp * 256;
    policy_mma_stage<H, 1>(sm, w, tid, 32 * kMmaWarps);
    __syncthreads();
    for (long long base = ((long long)blockIdx.x * kMmaWarps + warp) * 32; base < rows; base += (long long)gridDim.x * kMmaWarps * 32) {
        const long long row = base + lane;
        const bool valid = row < rows;
        const float4 a = valid ? reinterpret_cast<const float4 *>(obs)[2 * row] : make_float4(0, 0, 0, 0);
        const float4 b = valid ? reinterpret_cast<const float4 *>(obs)[2 * row + 1] : make_float4(0, 0, 0, 0);
        __syncwarp();                                           // the previous group's fragment loads are done
        reinterpret_cast<float4 *>(obs_w)[2 * lane] = a;
        reinterpret_cast<float4 *>(obs_w)[2 * lane + 1] = b;
        __syncwarp();
        policy_mma_logits<H, 2, false>(sm, obs_w, lg_w, lane);
        if (valid) values[row] = lg_w[8 * lane];
    }
}

// GAE(gamma, lambda) over a [horizon][n] rollout: one thread per battle walks t = horizon - 1 .. 0; loads and stores of one
// time step are coalesced across the warp.  The arithmetic is the fp32 sequence of the torch loop it replaces
// (examples/ppo_footsies.py before the value pass moved into the library), operation for operation -- the library is
// compiled with -fmad=false, so none of it is contracted:
//   nt = 1 - done[t];  delta = (r[t] + (g * v[t + 1]) * nt) - v[t];  last = delta + (gl * nt) * last;
//   adv[t] = last;  ret[t] = adv[t] + v[t]
// The recursion is a dependency chain of `horizon` steps per thread, so the loads of the next kGaeAhead time steps are
// issued before their arithmetic (the unrolled block below): the chain waits on one memory latency per block, not per step.
constexpr int kGaeThreads = 256;
constexpr int kGaeAhead = 8;
__device__ __forceinline__ void gae_step(float r, uint8_t d, float v, float g, float gl, float &vnext, float &last,
                                         float *adv, float *ret) {
    const float nt = d ? 0.0f : 1.0f;                           // = 1 - done for a 0 / 1 flag
    const float delta = (r + (g * vnext) * nt) - v;
    last = delta + (gl * nt) * last;
    *adv = last;
    *ret = last + v;
    vnext = v;
}
__global__ void __launch_bounds__(kGaeThreads) gae_kernel(const float *__restrict__ rewards, const uint8_t *__restrict__ dones,
                                                          const float *__restrict__ values, int horizon, int n, float g, float gl,
                                                          float *__restrict__ adv, float *__restrict__ ret) {
    const int i = blockIdx.x * kGaeThreads + threadIdx.x;
    if (i >= n) return;
    const size_t N = (size_t)n;
    float vnext = values[(size_t)horizon * N + i], last = 0.0f;
    int t = horizon - 1;
    for (; t >= kGaeAhead - 1; t -= kGaeAhead) {
        float r[kGaeAhead], v[kGaeAhead];
        uint8_t d[kGaeAhead];
#pragma unroll
        for (int u = 0; u < kGaeAhead; u++) {
            const size_t k = (size_t)(t - u) * N + i;
            r[u] = rewards[k]; d[u] = dones[k]; v[u] = values[k];
        }
#pragma unroll
        for (int u = 0; u < kGaeAhead; u++) {
            const size_t k = (size_t)(t - u) * N + i;
            gae_step(r[u], d[u], v[u], g, gl, vnext, last, adv + k, ret + k);
        }
    }
    for (; t >= 0; t--) {
        const size_t k = (size_t)t * N + i;
        gae_step(rewards[k], dones[k], values[k], g, gl, vnext, last, adv + k, ret + k);
    }
}

thread_local char g_perr[256] = "";

}  // namespace

extern "C" {

const char *fg_policy_last_error(void) { return g_perr; }

static int32_t policy_sample_impl(const float *obs, const float *scale, const float *w1, const float *b1, const float *w2,
                                  const float *b2, const float *w3, const float *b3, int32_t hidden, int32_t num_envs,
                                  uint64_t seed, uint64_t counter, const uint64_t *counter_base, uint8_t *actions, float *logp,
                                  float *obs_copy, int32_t mirror, int64_t first_env_index, void *stream) {
    if (!obs || !scale || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !actions || num_envs <= 0) {
        snprintf(g_perr, sizeof g_perr, "fg_policy_mlp_sample: null argument or empty batch");
        return FG_ERR_INVALID_ARGUMENT;
    }
    if (hidden != 32 && hidden != 64 && hidden != 128) {
        snprintf(g_perr, sizeof g_perr, "fg_policy_mlp_sample: hidden size must be 32, 64 or 128");
        return FG_ERR_INVALID_ARGUMENT;
    }
    PolicyParams p = { obs, { scale, w1, b1, w2, b2, w3, b3 }, actions, logp, obs_copy, seed, counter,
                       (const unsigned long long *)counter_base, num_envs, hidden, mirror, (long long)first_env_index };
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int grid = (num_envs + kPolEnvs - 1) / kPolEnvs;
    if (grid > sms * 4) grid = sms * 4;            // persistent: the weight staging is amortised over several passes
    const size_t bytes = hidden == 32 ? PolicySmemBcast<32, kPolEnvs, kPolicyWarps>::kBytes : hidden == 64 ? PolicySmemBcast<64, kPolEnvs, kPolicyWarps>::kBytes
                                      : PolicySmemBcast<128, kPolEnvs, kPolicyWarps>::kBytes;
    cudaError_t e = cudaSuccess;
    cudaStream_t s = (cudaStream_t)stream;
    if (hidden <= kMmaMaxHidden) {                  // tensor-core path (policy_mma.cuh)
        int mgrid = (num_envs + 32 * kMmaWarps - 1) / (32 * kMmaWarps);
        if (mgrid > sms * 4) mgrid = sms * 4;
#define FG_POLICY_MMA_LAUNCH(HH, MM) do { \
        constexpr size_t mbytes = PolicyMmaKernelSmem<HH>::kBytes; \
        static fg::DeviceOnceFlags configured; \
        e = fg::configure_once_per_device(configured, [] { \
            return cudaFuncSetAttribute(policy_mma_sample_kernel<HH, MM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mbytes); }); \
        if (e == cudaSuccess) policy_mma_sample_kernel<HH, MM><<<mgrid, 32 * kMmaWarps, mbytes, s>>>(p); } while (0)
        if (hidden == 32) { if (mirror) FG_POLICY_MMA_LAUNCH(32, true); else FG_POLICY_MMA_LAUNCH(32, false); }
        else { if (mirror) FG_POLICY_MMA_LAUNCH(64, true); else FG_POLICY_MMA_LAUNCH(64, false); }
#undef FG_POLICY_MMA_LAUNCH
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) {
            snprintf(g_perr, sizeof g_perr, "fg_policy_mlp_sample: %s", cudaGetErrorString(e));
            return FG_ERR_CUDA;
        }
        return FG_OK;
    }
#define FG_POLICY_LAUNCH(HH) do { \
        static fg::DeviceOnceFlags configured; \
        e = fg::configure_once_per_device(configured, [bytes] { \
            return cudaFuncSetAttribute(policy_mlp_sample_kernel<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); }); \
        if (e == cudaSuccess) policy_mlp_sample_kernel<HH><<<grid, kPolThreads, bytes, s>>>(p); } while (0)
    if (hidden == 32) FG_POLICY_LAUNCH(32);
    else if (hidden == 64) FG_POLICY_LAUNCH(64);
    else FG_POLICY_LAUNCH(128);
#undef FG_POLICY_LAUNCH
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_perr, sizeof g_perr, "fg_policy_mlp_sample: %s", cudaGetErrorString(e));
        return FG_ERR_CUDA;
    }
    return FG_OK;
}

int32_t fg_policy_mlp_sample(const float *obs, const float *scale, const float *w1, const float *b1, const float *w2,
                             const float *b2, const float *w3, const float *b3, int32_t hidden, int32_t num_envs,
                             uint64_t seed, uint64_t counter, const uint64_t *counter_base, uint8_t *actions, float *logp,
                             float *obs_copy, int64_t first_env_index, void *stream) {
    return policy_sample_impl(obs, scale, w1, b1, w2, b2, w3, b3, hidden, num_envs, seed, counter, counter_base, actions, logp,
                              obs_copy, 0, first_env_index, stream);
}

int32_t fg_policy_mlp_sample_p2(const float *obs, const float *scale, const float *w1, const float *b1, const float *w2,
                                const float *b2, const float *w3, const float *b3, int32_t hidden, int32_t num_envs,
                                uint64_t seed, uint64_t counter, const uint64_t *counter_base, uint8_t *actions, float *logp,
                                int32_t mirror, int64_t first_env_index, void *stream) {
    return policy_sample_impl(obs, scale, w1, b1, w2, b2, w3, b3, hidden, num_envs, seed, counter, counter_base, actions, logp,
                              nullptr, mirror != 0, first_env_index, stream);
}

int32_t fg_value_mlp(const float *obs, const float *scale, const float *w1, const float *b1, const float *w2,
                     const float *b2, const float *w3, const float *b3, int32_t hidden, int64_t rows,
                     float *values, void *stream) {
    if (!obs || !scale || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !values || rows <= 0) {
        snprintf(g_perr, sizeof g_perr, "fg_value_mlp: null argument or no rows");
        return FG_ERR_INVALID_ARGUMENT;
    }
    if (hidden != 32 && hidden != 64) {
        snprintf(g_perr, sizeof g_perr, "fg_value_mlp: hidden size must be 32 or 64");
        return FG_ERR_INVALID_ARGUMENT;
    }
    const PolicyWeights w = { scale, w1, b1, w2, b2, w3, b3 };
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long grid = (rows + 32 * kMmaWarps - 1) / (32 * kMmaWarps);
    if (grid > sms * 4) grid = sms * 4;             // persistent: the weight staging is amortised over many row groups
    cudaError_t e = cudaSuccess;
    cudaStream_t s = (cudaStream_t)stream;
#define FG_VALUE_LAUNCH(HH) do { \
        constexpr size_t vbytes = PolicyMmaKernelSmem<HH>::kBytes; \
        static fg::DeviceOnceFlags configured; \
        e = fg::configure_once_per_device(configured, [] { \
            return cudaFuncSetAttribute(value_mma_kernel<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)vbytes); }); \
        if (e == cudaSuccess) value_mma_kernel<HH><<<(unsigned)grid, 32 * kMmaWarps, vbytes, s>>>(obs, w, (long long)rows, values); } while (0)
    if (hidden == 32) FG_VALUE_LAUNCH(32);
    else FG_VALUE_LAUNCH(64);
#undef FG_VALUE_LAUNCH
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_perr, sizeof g_perr, "fg_value_mlp: %s", cudaGetErrorString(e));
        return FG_ERR_CUDA;
    }
    return FG_OK;
}

int32_t fg_gae(const float *rewards, const uint8_t *dones, const float *values, int32_t horizon, int32_t num_envs,
               float gamma, float gamma_lambda, float *advantages, float *returns, void *stream) {
    if (!rewards || !dones || !values || !advantages || !returns || horizon <= 0 || num_envs <= 0) {
        snprintf(g_perr, sizeof g_perr, "fg_gae: null argument or empty rollout");
        return FG_ERR_INVALID_ARGUMENT;
    }
    const int grid = (num_envs + kGaeThreads - 1) / kGaeThreads;
    gae_kernel<<<grid, kGaeThreads, 0, (cudaStream_t)stream>>>(rewards, dones, values, horizon, num_envs, gamma, gamma_lambda,
                                                               advantages, returns);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_perr, sizeof g_perr, "fg_gae: %s", cudaGetErrorString(e));
        return FG_ERR_CUDA;
    }
    return FG_OK;
}

}  // extern "C"
