// footsies_kernels.cu -- C ABI of the batched FOOTSIES simulator (include/footsies_b200.h) on top of the kernels in
// step_kernel.cuh.
#include <sched.h>
#include <stdlib.h>
#include <algorithm>

#include "delay_ring.cuh"
#include "rollout_kernel.h"
#include "step_kernel.cuh"

using namespace fg;
using namespace fgk;

namespace {

thread_local char g_err[512] = "";
int fail(int code, const char *fmt, const char *detail = "") {
    snprintf(g_err, sizeof g_err, fmt, detail);
    return code;
}
#define CUDA_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) \
    return fail(FG_ERR_CUDA, #expr ": %s", cudaGetErrorString(_e)); } while (0)

}  // namespace

struct fg_handle {
    fg_config cfg;
    fg_buffers buf;
    bool bound;
    Tables *d_tables;
    int sm_count;
    int64_t launches;
    int64_t step_calls;    // fg_step calls so far: every other one walks the battles backwards (L2 reuse across launches)
    uint8_t *d_mask;       // staging for fg_reset_host
    int large_shape_min_envs;
    int pdl_min_envs;      // batch size from which the step kernel is launched with programmatic dependent launch
    // host-buffer path (fg_step_host*): slices of host_chunk_envs battles are pipelined over two library-owned
    // streams, so that the D2H copies of slice c run while slice c+1 is being simulated and its actions uploaded
    int host_chunk_envs;
    int host_lead_div;      // the first slice of a sliced call is host_chunk_envs / host_lead_div battles (see SlicePlan)
    uint4 *d_packed;       // [num_envs] packed host layout (fg_packed_result)
    float *d_reward_table; // [FG_PACKED_REWARD_TABLE_SIZE] ascending; h_reward_table is the host copy
    uint32_t *d_pack_error;
    float h_reward_table[FG_PACKED_REWARD_TABLE_SIZE];
    int reward_table_count;
    float2 *d_position;    // [num_envs] compact host layout: position p1,p2
    uint8_t *d_obs_u8;     // [num_envs][6] compact host layout: guard p1,p2 | move p1,p2 | move_frame p1,p2
    cudaStream_t s_compute, s_copy;
    cudaEvent_t ev_fork, ev_join;
    std::vector<cudaEvent_t> ev_slice;
};

namespace {

int grid_for(const fg_handle *h, int blocks_per_sm) {
    int want = (h->cfg.num_envs + kThreads - 1) / kThreads;
    int cap = h->sm_count * blocks_per_sm;
    return want < cap ? (want > 0 ? want : 1) : cap;
}

// Kernel parameters for the envs [first, first + count) of the handle (count < 0: all of them).
Params make_params(const fg_handle *h, int first = 0, int count = -1) {
    Params p;
    memset(&p, 0, sizeof p);
    const size_t o = (size_t)first;
    p.pl_f1 = (uint4 *)h->buf.state[FG_PLANE_F1] + o; p.pl_f2 = (uint4 *)h->buf.state[FG_PLANE_F2] + o;
    p.pl_env = (uint4 *)h->buf.state[FG_PLANE_ENV] + o; p.pl_rng = (uint4 *)h->buf.state[FG_PLANE_RNG] + o;
    p.stats = (unsigned long long *)h->buf.stats;
    p.act1 = h->buf.actions_p1 ? h->buf.actions_p1 + o : nullptr;
    p.act2 = h->buf.actions_p2 ? h->buf.actions_p2 + o : nullptr;
    p.obs = (float4 *)h->buf.obs + 2 * o; p.reward = h->buf.reward + o; p.terminated = h->buf.terminated + o;
    p.info_frame = h->buf.info_frame + o; p.info_misc = (uint32_t *)h->buf.info_misc + o;
    p.step_mask = h->buf.step_mask ? h->buf.step_mask + o : nullptr;
    p.tables = h->d_tables;
    p.first_env_index = h->cfg.first_env_index + first;
    p.reverse = (int)(h->step_calls & 1);
    p.pdl = (count < 0 ? h->cfg.num_envs - first : count) >= h->pdl_min_envs;
    p.n = count < 0 ? h->cfg.num_envs - first : count; p.frame_skip = h->cfg.frame_skip; p.autoreset = h->cfg.autoreset;
    p.stale_intro = h->cfg.stale_intro_input;
    p.skip_unactionable = h->cfg.skip_unactionable;
    p.large_shape_min_envs = h->large_shape_min_envs;
    return p;
}

template <bool KF>
cudaError_t launch_step_k(const fg_config &c, int sm_count, cudaStream_t s, const Params &p) {
    const bool d = c.dense_reward != 0, m = p.step_mask != nullptr;
    if (c.p1_bot && c.p2_bot) return launch_step_d<KF, true, true>(d, m, sm_count, s, p);
    if (c.p1_bot) return launch_step_d<KF, true, false>(d, m, sm_count, s, p);
    if (c.p2_bot) return launch_step_d<KF, false, true>(d, m, sm_count, s, p);
    return launch_step_d<KF, false, false>(d, m, sm_count, s, p);
}

template <bool B1, bool B2>
cudaError_t launch_reset(int grid, cudaStream_t s, const Params &p) {
    static DeviceOnceFlags configured;
    if (cudaError_t e = configure_once_per_device(configured, [] {
            return cudaFuncSetAttribute(reset_kernel<B1, B2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Tables)); }))
        return e;
    reset_kernel<B1, B2><<<grid, kThreads, sizeof(Tables), s>>>(p);
    return cudaSuccess;
}

int check_bound(const fg_handle *h) {
    if (!h) return fail(FG_ERR_INVALID_ARGUMENT, "null handle%s");
    if (!h->bound) return fail(FG_ERR_NOT_BOUND, "fg_bind has not been called%s");
    return FG_OK;
}

// ---- host-buffer path -------------------------------------------------------------------------------------------
// Where the results of a host-buffer call go.  obs_f32 is the device layout ([n][8] floats, 32 B); position + obs_u8 is
// the compact host layout (8 + 6 B: the integer-valued observation fields travel as bytes), produced by pack_obs_kernel.
struct HostOut {
    float *obs_f32;
    float *position;
    uint8_t *obs_u8;
    float *reward;
    uint8_t *terminated;
    int32_t *info_frame;
    uint8_t *info_misc;
};

// obs [n][8] f32 -> position [n] float2 + obs_u8 [n][6].  Two envs per thread: 4 x 128-bit loads, one 128-bit and three
// 32-bit stores, all coalesced.  The six integer-valued fields are exact in a byte (guard 0..3, move index 0..14,
// move_frame 0..55: FootsiesEnv.observation_space, footsies.py:157-168).
__global__ void __launch_bounds__(256) pack_obs_kernel(const float4 *__restrict__ obs, float2 *__restrict__ position,
                                                        uint8_t *__restrict__ obs_u8, int n) {
    const int pairs = n >> 1;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < pairs; j += gridDim.x * blockDim.x) {
        const float4 a0 = obs[4 * (size_t)j], a1 = obs[4 * (size_t)j + 1], b0 = obs[4 * (size_t)j + 2], b1 = obs[4 * (size_t)j + 3];
        reinterpret_cast<float4 *>(position)[j] = make_float4(a1.z, a1.w, b1.z, b1.w);
        const uint32_t A[6] = { (uint32_t)a0.x, (uint32_t)a0.y, (uint32_t)a0.z, (uint32_t)a0.w, (uint32_t)a1.x, (uint32_t)a1.y };
        const uint32_t B[6] = { (uint32_t)b0.x, (uint32_t)b0.y, (uint32_t)b0.z, (uint32_t)b0.w, (uint32_t)b1.x, (uint32_t)b1.y };
        uint32_t *o = reinterpret_cast<uint32_t *>(obs_u8) + 3 * (size_t)j;
        o[0] = A[0] | A[1] << 8 | A[2] << 16 | A[3] << 24;
        o[1] = A[4] | A[5] << 8 | B[0] << 16 | B[1] << 24;
        o[2] = B[2] | B[3] << 8 | B[4] << 16 | B[5] << 24;
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const int i = n - 1;
        const float4 a0 = obs[2 * (size_t)i], a1 = obs[2 * (size_t)i + 1];
        position[i] = make_float2(a1.z, a1.w);
        const float v[6] = { a0.x, a0.y, a0.z, a0.w, a1.x, a1.y };
        for (int k = 0; k < 6; k++) obs_u8[6 * (size_t)i + k] = (uint8_t)v[k];
    }
}

// The frame_delay queue of FootsiesEnv (delay_ring.cuh) after an fg_step: one thread per battle pushes the state the step
// kernel just produced at ring position `pos` and emits the delayed state to out_*.  44 B read + 44 B written + 44 B
// emitted per battle and step.
__global__ void __launch_bounds__(256) delay_ring_kernel(const float4 *__restrict__ obs, const int32_t *__restrict__ frame,
                                                         const uint32_t *__restrict__ misc, DelayRingRef ring,
                                                         float4 *__restrict__ out_obs, int32_t *__restrict__ out_frame,
                                                         uint32_t *__restrict__ out_misc, const uint8_t *__restrict__ step_mask,
                                                         int n, int depth, int pos) {
    const int oldest = (pos + 1) % depth, newest = (pos + depth - 1) % depth;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        DelayEntry now, emit;
        now.a = obs[2 * (size_t)i]; now.b = obs[2 * (size_t)i + 1]; now.frame = frame[i]; now.misc = misc[i];
        if (delay_ring_push(ring, i, depth, pos, step_mask && !step_mask[i], now, ring.load(oldest, i),
                            ring.frame[(size_t)newest * n + i], emit)) {
            out_obs[2 * (size_t)i] = emit.a; out_obs[2 * (size_t)i + 1] = emit.b; out_frame[i] = emit.frame; out_misc[i] = emit.misc;
        }
    }
}

int step_range(fg_handle *h, int first, int count, cudaStream_t s) {
    const Params p = make_params(h, first, count);
    // the single-frame kernels carry neither the frame_skip loop nor the fused FootsiesFrameSkipped loop
    const bool single = h->cfg.frame_skip == 1 && !h->cfg.skip_unactionable;
    CUDA_TRY(single ? launch_step_k<false>(h->cfg, h->sm_count, s, p) : launch_step_k<true>(h->cfg, h->sm_count, s, p));
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return FG_OK;
}

// obs / reward / terminated / info of one battle -> one 16-byte fg_packed_result (include/footsies_b200.h).  The reward is
// carried as its index in the ascending table of the float32 values a single-frame step can pay (exact match by binary
// search; a value outside the table raises *error).  One thread per battle, 128-bit coalesced loads and stores.
__global__ void __launch_bounds__(256) pack_records_kernel(const float4 *__restrict__ obs, const float *__restrict__ reward,
                                                            const uint8_t *__restrict__ terminated, const int32_t *__restrict__ frame,
                                                            const uint32_t *__restrict__ misc, const float *__restrict__ table,
                                                            int table_n, uint4 *__restrict__ out, uint32_t *error, int n) {
    __shared__ float tab[FG_PACKED_REWARD_TABLE_SIZE];
    for (int k = threadIdx.x; k < FG_PACKED_REWARD_TABLE_SIZE; k += blockDim.x) tab[k] = k < table_n ? table[k] : 3.0e38f;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 a = obs[2 * (size_t)i], b = obs[2 * (size_t)i + 1];
        const float r = reward[i];
        const uint32_t m = misc[i];
        int lo = 0;
#pragma unroll
        for (int stepw = FG_PACKED_REWARD_TABLE_SIZE / 2; stepw >= 1; stepw >>= 1)      // largest lo with tab[lo] <= r
            if (tab[lo + stepw] <= r) lo += stepw;
        if (tab[lo] != r) atomicOr(error, 1u);
        const int32_t f = frame[i] + 1;
        const uint32_t w0 = (uint32_t)a.x | (uint32_t)a.y << 2 | (uint32_t)a.z << 4 | (uint32_t)a.w << 8 | (uint32_t)b.x << 12
                          | (uint32_t)b.y << 18 | (terminated[i] ? 1u << 24 : 0u) | (m & 7u) << 25 | ((m >> 8) & 7u) << 28;
        const uint32_t w1 = ((m >> 16) & 31u) | ((m >> 24) & 31u) << 5 | (uint32_t)lo << 10
                          | (uint32_t)(f < 0 ? 0 : f > 32767 ? 32767 : f) << 17;
        out[i] = make_uint4(__float_as_uint(b.z), __float_as_uint(b.w), w0, w1);
    }
}

// Library-owned resources of the host-buffer path, created on first use.
// Slices of a host-buffer call: [0, lead), then whole chunks from there on.  The first device->host copy can only start when
// the first slice has been stepped and packed, and nothing overlaps that: a SHORT first slice starts the copy stream earlier
// at the price of one more copy.  Measured on a 4 Mi-battle packed call (profiles/r02z_e2e_lead_slice.log, ms per call,
// interleaved): whole first chunk 1.303 / 1.308 / 1.307, half 1.287 / 1.288 / 1.289, quarter 1.302 / 1.296 / 1.353 -> half.
struct SlicePlan {
    size_t n, chunk, lead;
    int count;
    SlicePlan(const fg_handle *h) {
        n = (size_t)h->cfg.num_envs; chunk = (size_t)h->host_chunk_envs;
        if (n <= chunk) { lead = n; count = 1; return; }
        lead = chunk / (size_t)h->host_lead_div;
        count = 1 + (int)((n - lead + chunk - 1) / chunk);
    }
    size_t first(int c) const { return c == 0 ? 0 : lead + (size_t)(c - 1) * chunk; }
    size_t size(int c) const { const size_t f = first(c), want = c == 0 ? lead : chunk; return n - f < want ? n - f : want; }
};

int host_path_init(fg_handle *h, bool compact, int slices) {
    if (compact && !h->d_position) {
        CUDA_TRY(cudaMalloc(&h->d_position, sizeof(float2) * (size_t)h->cfg.num_envs));
        CUDA_TRY(cudaMalloc(&h->d_obs_u8, 6 * (size_t)h->cfg.num_envs + 8));
    }
    if (slices > 1 && !h->s_compute) {
        CUDA_TRY(cudaStreamCreateWithFlags(&h->s_compute, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    while (slices > 1 && (int)h->ev_slice.size() < slices) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        h->ev_slice.push_back(e);
    }
    return FG_OK;
}

// Results of envs [first, first + m) -> host, on stream s (after the pack kernel when the compact layout is asked for).
int copy_out(fg_handle *h, const HostOut &o, size_t first, size_t m, cudaStream_t s) {
    const fg_buffers &b = h->buf;
    if (o.obs_f32) CUDA_TRY(cudaMemcpyAsync(o.obs_f32 + 8 * first, b.obs + 8 * first, m * 8 * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (o.position) CUDA_TRY(cudaMemcpyAsync(o.position + 2 * first, h->d_position + first, m * sizeof(float2), cudaMemcpyDeviceToHost, s));
    if (o.obs_u8) CUDA_TRY(cudaMemcpyAsync(o.obs_u8 + 6 * first, h->d_obs_u8 + 6 * first, m * 6, cudaMemcpyDeviceToHost, s));
    if (o.reward) CUDA_TRY(cudaMemcpyAsync(o.reward + first, b.reward + first, m * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (o.terminated) CUDA_TRY(cudaMemcpyAsync(o.terminated + first, b.terminated + first, m, cudaMemcpyDeviceToHost, s));
    if (o.info_frame) CUDA_TRY(cudaMemcpyAsync(o.info_frame + first, b.info_frame + first, m * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (o.info_misc) CUDA_TRY(cudaMemcpyAsync(o.info_misc + 4 * first, b.info_misc + 4 * first, m * 4, cudaMemcpyDeviceToHost, s));
    return FG_OK;
}

int pack_range(fg_handle *h, size_t first, size_t m, cudaStream_t s) {
    const int want = (int)((m / 2 + 255) / 256), cap = h->sm_count * 8;
    pack_obs_kernel<<<want < cap ? (want > 0 ? want : 1) : cap, 256, 0, s>>>((const float4 *)h->buf.obs + 2 * first,
                                                                             h->d_position + first, h->d_obs_u8 + 6 * first, (int)m);
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return FG_OK;
}

// FootsiesEnv.step with HOST buffers.  Small batches: H2D, step, (pack), D2H on the caller's stream.  Large batches are
// cut into slices of host_chunk_envs battles (battles are independent, so a slice is just an offset into every buffer):
// uploads + kernels run on one library stream, the D2H copies on another, and slice c's results cross PCIe while
// slice c + 1 is simulated.  Ordered after prior work on `stream`; returns when every result is in host memory.
int host_step(fg_handle *h, const uint8_t *a1, const uint8_t *a2, const HostOut &o, cudaStream_t user) {
    if (int rc = check_bound(h)) return rc;
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    if (!h->cfg.p1_bot && !a1) return fail(FG_ERR_INVALID_ARGUMENT, "actions_p1 is required unless p1_bot%s");
    if (!h->cfg.p2_bot && !a2) return fail(FG_ERR_INVALID_ARGUMENT, "actions_p2 is required unless p2_bot%s");
    const bool compact = o.position || o.obs_u8;
    if (compact && !(o.position && o.obs_u8)) return fail(FG_ERR_INVALID_ARGUMENT, "position and obs_u8 go together%s");
    const SlicePlan plan(h);
    const int slices = plan.count;
    if (int rc = host_path_init(h, compact, slices)) return rc;
    cudaStream_t sc = user, sd = user;
    if (slices > 1) {
        sc = h->s_compute; sd = h->s_copy;
        CUDA_TRY(cudaEventRecord(h->ev_fork, user));
        CUDA_TRY(cudaStreamWaitEvent(sc, h->ev_fork, 0));
    }
    for (int c = 0; c < slices; c++) {
        const size_t first = plan.first(c), m = plan.size(c);
        if (!h->cfg.p1_bot) CUDA_TRY(cudaMemcpyAsync((void *)(h->buf.actions_p1 + first), a1 + first, m, cudaMemcpyHostToDevice, sc));
        if (!h->cfg.p2_bot) CUDA_TRY(cudaMemcpyAsync((void *)(h->buf.actions_p2 + first), a2 + first, m, cudaMemcpyHostToDevice, sc));
        if (int rc = step_range(h, (int)first, (int)m, sc)) return rc;
        if (compact) if (int rc = pack_range(h, first, m, sc)) return rc;
        if (slices > 1) {
            CUDA_TRY(cudaEventRecord(h->ev_slice[c], sc));
            CUDA_TRY(cudaStreamWaitEvent(sd, h->ev_slice[c], 0));
        }
        if (int rc = copy_out(h, o, first, m, sd)) return rc;
    }
    if (slices > 1) {
        CUDA_TRY(cudaEventRecord(h->ev_join, sd));
        CUDA_TRY(cudaStreamWaitEvent(user, h->ev_join, 0));
    }
    CUDA_TRY(cudaStreamSynchronize(sd));
    return FG_OK;
}

// ---- packed host layout -------------------------------------------------------------------------------------------
int packed_init(fg_handle *h) {
    if (h->cfg.frame_skip != 1 || h->cfg.skip_unactionable)
        return fail(FG_ERR_INVALID_STATE, "the packed host layout needs frame_skip = 1 and no fused frame skipping "
                                          "(summed rewards are not table values)%s");
    if (h->d_packed) return FG_OK;
    // every float32 value a single-frame step can pay: 0, the +-0.3 guard steps, +-1 and the dense terminal compensations
    static const double step_r[4] = FT_STEP_REWARD_INIT;
    static const double term_r[FT_NUM_CUM][4][2] = FT_TERM_REWARD_INIT;
    std::vector<float> v = { 0.0f, 1.0f, -1.0f };
    for (int k = 0; k < 4; k++) v.push_back((float)step_r[k]);
    for (int c = 0; c < FT_NUM_CUM; c++) for (int k = 0; k < 4; k++) for (int d = 0; d < 2; d++) v.push_back((float)term_r[c][k][d]);
    std::sort(v.begin(), v.end());
    v.erase(std::unique(v.begin(), v.end()), v.end());
    if ((int)v.size() >= FG_PACKED_REWARD_TABLE_SIZE) return fail(FG_ERR_INVALID_STATE, "reward table overflow%s");
    h->reward_table_count = (int)v.size();
    for (int k = 0; k < FG_PACKED_REWARD_TABLE_SIZE; k++) h->h_reward_table[k] = k < (int)v.size() ? v[k] : 0.0f;
    CUDA_TRY(cudaMalloc(&h->d_reward_table, sizeof h->h_reward_table));
    CUDA_TRY(cudaMemcpy(h->d_reward_table, h->h_reward_table, sizeof h->h_reward_table, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&h->d_pack_error, sizeof(uint32_t)));
    CUDA_TRY(cudaMemset(h->d_pack_error, 0, sizeof(uint32_t)));
    CUDA_TRY(cudaMalloc(&h->d_packed, sizeof(uint4) * (size_t)h->cfg.num_envs));
    return FG_OK;
}

int pack_records_range(fg_handle *h, size_t first, size_t m, cudaStream_t s) {
    const int want = (int)((m + 255) / 256), cap = h->sm_count * 8;
    const fg_buffers &b = h->buf;
    pack_records_kernel<<<want < cap ? (want > 0 ? want : 1) : cap, 256, 0, s>>>(
        (const float4 *)b.obs + 2 * first, b.reward + first, b.terminated + first, b.info_frame + first,
        (const uint32_t *)b.info_misc + first, h->d_reward_table, h->reward_table_count, h->d_packed + first, h->d_pack_error, (int)m);
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return FG_OK;
}

int packed_finish(fg_handle *h, cudaStream_t s) {
    uint32_t err = 0;
    CUDA_TRY(cudaMemcpyAsync(&err, h->d_pack_error, sizeof err, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (err) {
        cudaMemset(h->d_pack_error, 0, sizeof(uint32_t));
        return fail(FG_ERR_INVALID_STATE, "a reward outside the packed reward table was produced%s");
    }
    return FG_OK;
}

// fg_step_host_packed: like host_step, but every slice ends in ONE pack kernel and ONE contiguous device->host copy.
int host_step_packed(fg_handle *h, const uint8_t *a1, const uint8_t *a2, fg_packed_result *out, cudaStream_t user) {
    if (int rc = check_bound(h)) return rc;
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    if (!out) return fail(FG_ERR_INVALID_ARGUMENT, "out is null%s");
    if (!h->cfg.p1_bot && !a1) return fail(FG_ERR_INVALID_ARGUMENT, "actions_p1 is required unless p1_bot%s");
    if (!h->cfg.p2_bot && !a2) return fail(FG_ERR_INVALID_ARGUMENT, "actions_p2 is required unless p2_bot%s");
    if (int rc = packed_init(h)) return rc;
    const SlicePlan plan(h);
    const int slices = plan.count;
    if (int rc = host_path_init(h, false, slices)) return rc;
    cudaStream_t sc = user, sd = user;
    if (slices > 1) {
        sc = h->s_compute; sd = h->s_copy;
        CUDA_TRY(cudaEventRecord(h->ev_fork, user));
        CUDA_TRY(cudaStreamWaitEvent(sc, h->ev_fork, 0));
    }
    h->step_calls++;
    for (int c = 0; c < slices; c++) {
        const size_t first = plan.first(c), m = plan.size(c);
        if (!h->cfg.p1_bot) CUDA_TRY(cudaMemcpyAsync((void *)(h->buf.actions_p1 + first), a1 + first, m, cudaMemcpyHostToDevice, sc));
        if (!h->cfg.p2_bot) CUDA_TRY(cudaMemcpyAsync((void *)(h->buf.actions_p2 + first), a2 + first, m, cudaMemcpyHostToDevice, sc));
        if (int rc = step_range(h, (int)first, (int)m, sc)) return rc;
        if (int rc = pack_records_range(h, first, m, sc)) return rc;
        if (slices > 1) {
            CUDA_TRY(cudaEventRecord(h->ev_slice[c], sc));
            CUDA_TRY(cudaStreamWaitEvent(sd, h->ev_slice[c], 0));
        }
        CUDA_TRY(cudaMemcpyAsync(out + first, h->d_packed + first, m * sizeof(uint4), cudaMemcpyDeviceToHost, sd));
    }
    if (slices > 1) {
        CUDA_TRY(cudaEventRecord(h->ev_join, sd));
        CUDA_TRY(cudaStreamWaitEvent(user, h->ev_join, 0));
    }
    return packed_finish(h, sd);
}

int reset_on(fg_handle *h, const uint8_t *dmask, cudaStream_t s) {
    Params p = make_params(h);
    p.mask = dmask;
    const int grid = grid_for(h, 4);
    cudaError_t le;
    if (h->cfg.p1_bot && h->cfg.p2_bot) le = launch_reset<true, true>(grid, s, p);
    else if (h->cfg.p1_bot) le = launch_reset<true, false>(grid, s, p);
    else if (h->cfg.p2_bot) le = launch_reset<false, true>(grid, s, p);
    else le = launch_reset<false, false>(grid, s, p);
    CUDA_TRY(le);
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return FG_OK;
}

// FootsiesEnv.reset with HOST buffers (mask: host uint8[num_envs] or NULL); not a hot call, one stream.
int host_reset(fg_handle *h, const uint8_t *mask, const HostOut &o, cudaStream_t s) {
    if (int rc = check_bound(h)) return rc;
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    const bool compact = o.position || o.obs_u8;
    if (compact && !(o.position && o.obs_u8)) return fail(FG_ERR_INVALID_ARGUMENT, "position and obs_u8 go together%s");
    const size_t n = (size_t)h->cfg.num_envs;
    if (int rc = host_path_init(h, compact, 1)) return rc;
    const uint8_t *dmask = nullptr;
    if (mask) {
        if (!h->d_mask) CUDA_TRY(cudaMalloc(&h->d_mask, n));
        CUDA_TRY(cudaMemcpyAsync(h->d_mask, mask, n, cudaMemcpyHostToDevice, s));
        dmask = h->d_mask;
    }
    if (int rc = reset_on(h, dmask, s)) return rc;
    if (compact) if (int rc = pack_range(h, 0, n, s)) return rc;
    if (int rc = copy_out(h, o, 0, n, s)) return rc;
    CUDA_TRY(cudaStreamSynchronize(s));
    return FG_OK;
}

int host_reset_packed(fg_handle *h, const uint8_t *mask, fg_packed_result *out, cudaStream_t s) {
    if (int rc = check_bound(h)) return rc;
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    if (!out) return fail(FG_ERR_INVALID_ARGUMENT, "out is null%s");
    if (int rc = packed_init(h)) return rc;
    const size_t n = (size_t)h->cfg.num_envs;
    const uint8_t *dmask = nullptr;
    if (mask) {
        if (!h->d_mask) CUDA_TRY(cudaMalloc(&h->d_mask, n));
        CUDA_TRY(cudaMemcpyAsync(h->d_mask, mask, n, cudaMemcpyHostToDevice, s));
        dmask = h->d_mask;
    }
    if (int rc = reset_on(h, dmask, s)) return rc;
    if (int rc = pack_records_range(h, 0, n, s)) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, h->d_packed, n * sizeof(uint4), cudaMemcpyDeviceToHost, s));
    return packed_finish(h, s);
}

// NUMA node of a CUDA device (/sys/bus/pci/devices/<bdf>/numa_node), -1 if unknown
int gpu_numa_node(int dev) {
    char bdf[64] = "", path[160], buf[32] = "";
    if (cudaDeviceGetPCIBusId(bdf, sizeof bdf, dev) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char *c = bdf; *c; c++) if (*c >= 'A' && *c <= 'Z') *c += 32;
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bdf);
    FILE *f = fopen(path, "r");
    if (!f) return -1;
    if (!fgets(buf, sizeof buf, f)) buf[0] = 0;
    fclose(f);
    return atoi(buf);
}
bool node_cpuset(int node, cpu_set_t *set) {
    char path[96], buf[1024] = "";
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    FILE *f = fopen(path, "r");
    if (!f) return false;
    if (!fgets(buf, sizeof buf, f)) buf[0] = 0;
    fclose(f);
    CPU_ZERO(set);
    int n = 0;
    for (char *tok = strtok(buf, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a, b;
        if (sscanf(tok, "%d-%d", &a, &b) == 2) { for (int c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET(c, set); n++; } }
        else if (sscanf(tok, "%d", &a) == 1 && a < CPU_SETSIZE) { CPU_SET(a, set); n++; }
    }
    return n > 0;
}

}  // namespace

extern "C" {

void *fg_host_alloc(int32_t device, uint64_t bytes) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        fail(FG_ERR_INVALID_ARGUMENT, "fg_host_alloc: no such device%s");
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) { fail(FG_ERR_CUDA, "fg_host_alloc: cudaSetDevice failed%s"); return nullptr; }
    cpu_set_t old_set, node_set;
    const int node = gpu_numa_node(device);
    const bool have_old = sched_getaffinity(0, sizeof old_set, &old_set) == 0;
    const bool bound = node >= 0 && have_old && node_cpuset(node, &node_set) && sched_setaffinity(0, sizeof node_set, &node_set) == 0;
    void *p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e == cudaSuccess) memset(p, 0, bytes);              // first touch from the bound thread places the pages
    if (bound) sched_setaffinity(0, sizeof old_set, &old_set);
    if (e != cudaSuccess) { cudaGetLastError(); fail(FG_ERR_CUDA, "fg_host_alloc: cudaHostAlloc failed%s"); return nullptr; }
    return p;
}
void fg_host_free(void *p) { if (p) cudaFreeHost(p); }

int32_t fg_packed_reward_table(fg_handle *h, float *table, int32_t *count) {
    if (!h || !table || !count) return fail(FG_ERR_INVALID_ARGUMENT, "null argument%s");
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    if (int rc = packed_init(h)) return rc;
    memcpy(table, h->h_reward_table, sizeof h->h_reward_table);
    *count = h->reward_table_count;
    return FG_OK;
}
int32_t fg_step_host_packed(fg_handle *h, const uint8_t *a1, const uint8_t *a2, fg_packed_result *out, void *stream) {
    return host_step_packed(h, a1, a2, out, (cudaStream_t)stream);
}
int32_t fg_reset_host_packed(fg_handle *h, const uint8_t *mask, fg_packed_result *out, void *stream) {
    return host_reset_packed(h, mask, out, (cudaStream_t)stream);
}

int32_t fg_abi_version(void) { return FG_ABI_VERSION; }
const char *fg_last_error(void) { return g_err; }

int32_t fg_algorithmic_bytes_per_env_step(const fg_config *cfg) {
    if (!cfg) return 0;
    const bool rng = cfg->p1_bot || cfg->p2_bot;
    int state = 2 * 16 * (rng ? 4 : 3);                 // planes read + written
    int actions = (cfg->p1_bot ? 0 : 1) + (cfg->p2_bot ? 0 : 1);
    return state + actions + 32 /*obs*/ + 4 /*reward*/ + 1 /*terminated*/ + 4 /*info frame*/ + 4 /*info misc*/;
}

int32_t fg_create(const fg_config *cfg, fg_handle **out) {
    if (!cfg || !out) return fail(FG_ERR_INVALID_ARGUMENT, "null argument%s");
    if (cfg->struct_size != (int32_t)sizeof(fg_config)) return fail(FG_ERR_INVALID_ARGUMENT, "fg_config.struct_size mismatch%s");
    if (cfg->num_envs <= 0) return fail(FG_ERR_INVALID_ARGUMENT, "num_envs must be positive%s");
    if (cfg->frame_skip < 1 || cfg->frame_skip > 64) return fail(FG_ERR_INVALID_ARGUMENT, "frame_skip must be in [1, 64]%s");
    if (cfg->skip_unactionable && cfg->p1_bot) return fail(FG_ERR_INVALID_ARGUMENT, "skip_unactionable needs an agent-controlled P1%s");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(FG_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback%s");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(FG_ERR_INVALID_ARGUMENT, "device ordinal out of range%s");
    CUDA_TRY(cudaSetDevice(cfg->device));
    fg_handle *h = new (std::nothrow) fg_handle();
    if (!h) return fail(FG_ERR_INVALID_STATE, "out of host memory%s");
    h->cfg = *cfg;
    h->bound = false;
    h->launches = 0;
    h->step_calls = 0;
    h->d_mask = nullptr;
    h->d_position = nullptr; h->d_obs_u8 = nullptr;
    h->d_packed = nullptr; h->d_reward_table = nullptr; h->d_pack_error = nullptr; h->reward_table_count = 0;
    h->s_compute = h->s_copy = nullptr;
    h->ev_fork = h->ev_join = nullptr;
    // slice size of the pipelined host-buffer path (measured, tools/e2e_bench.py, 4 Mi battles: no slices 2.28 ms, 2 Mi 2.20, 1 Mi 2.21,
    // 512 Ki 2.27, 256 Ki 2.45, 128 Ki 2.84: below 1 Mi the six copies per slice cost more than the overlap wins)
    h->host_chunk_envs = 1024 * 1024;
    h->host_lead_div = 2;
    if (const char *v = getenv("FOOTSIES_B200_HOST_LEAD_DIV")) { const int d = atoi(v); if (d == 1 || d == 2 || d == 4) h->host_lead_div = d; }
    if (const char *v = getenv("FOOTSIES_B200_HOST_CHUNK_ENVS")) {
        const long long c = atoll(v);
        if (c >= 256) h->host_chunk_envs = (int)((c > (1ll << 30) ? (1ll << 30) : c) / 256 * 256);
    }
    // developer / test knob: force the large CTA shapes onto small batches (or the small shape onto large ones)
    h->large_shape_min_envs = kLargeShapeMinEnvs;
    if (const char *v = getenv("FOOTSIES_B200_LARGE_SHAPE_MIN_ENVS")) h->large_shape_min_envs = atoi(v);
    // programmatic dependent launch (measured, profiles/r02j_pdl_threshold.log, us per launch with / without): K = 1 -- 4096
    // battles 4.2 / 5.2, 65 536: 6.0 / 6.3, 262 144: 10.8 / 11.9, 1 Mi: 33.4 / 35.2, 4 Mi: 115.6 / 122; fused K = 4 -- 1 Mi:
    // 83.8 / 85.4, but 65 536 self-play (config C, under one wave of long-running CTAs): 10.4 / 9.2 -> fused kernels only
    // from 262 144 battles up
    h->pdl_min_envs = (cfg->frame_skip > 1 || cfg->skip_unactionable) ? 262144 : 0;
    if (const char *v = getenv("FOOTSIES_B200_PDL_MIN_ENVS")) h->pdl_min_envs = atoi(v);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    h->sm_count = prop.multiProcessorCount;
    Tables *host = new Tables();
    build_tables(*host);
    cudaError_t e = cudaMalloc(&h->d_tables, sizeof(Tables));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_tables, host, sizeof(Tables), cudaMemcpyHostToDevice);
    delete host;
    if (e != cudaSuccess) { delete h; return fail(FG_ERR_CUDA, "table upload: %s", cudaGetErrorString(e)); }
    *out = h;
    return FG_OK;
}

void fg_destroy(fg_handle *h) {
    if (!h) return;
    cudaSetDevice(h->cfg.device);
    cudaFree(h->d_tables);
    if (h->d_mask) cudaFree(h->d_mask);
    if (h->d_position) cudaFree(h->d_position);
    if (h->d_packed) { cudaFree(h->d_packed); cudaFree(h->d_reward_table); cudaFree(h->d_pack_error); }
    if (h->d_obs_u8) cudaFree(h->d_obs_u8);
    if (h->s_compute) { cudaStreamDestroy(h->s_compute); cudaStreamDestroy(h->s_copy); cudaEventDestroy(h->ev_fork); cudaEventDestroy(h->ev_join); }
    for (cudaEvent_t e : h->ev_slice) cudaEventDestroy(e);
    delete h;
}

int32_t fg_bind(fg_handle *h, const fg_buffers *b) {
    if (!h || !b) return fail(FG_ERR_INVALID_ARGUMENT, "null argument%s");
    if (b->struct_size != (int32_t)sizeof(fg_buffers)) return fail(FG_ERR_INVALID_ARGUMENT, "fg_buffers.struct_size mismatch%s");
    for (int k = 0; k < FG_STATE_PLANES; k++)
        if (!b->state[k] || ((uintptr_t)b->state[k] & 15u)) return fail(FG_ERR_INVALID_ARGUMENT, "state planes must be non-null and 16-byte aligned%s");
    if (!b->stats || !b->obs || !b->reward || !b->terminated || !b->info_frame || !b->info_misc)
        return fail(FG_ERR_INVALID_ARGUMENT, "output buffers must be non-null%s");
    if (((uintptr_t)b->obs & 15u) || ((uintptr_t)b->info_misc & 3u) || ((uintptr_t)b->stats & 7u))
        return fail(FG_ERR_INVALID_ARGUMENT, "obs must be 16-byte, info_misc 4-byte, stats 8-byte aligned%s");
    if (!h->cfg.p1_bot && !b->actions_p1) return fail(FG_ERR_INVALID_ARGUMENT, "actions_p1 is required unless p1_bot%s");
    if (!h->cfg.p2_bot && !b->actions_p2) return fail(FG_ERR_INVALID_ARGUMENT, "actions_p2 is required unless p2_bot%s");
    h->buf = *b;
    h->bound = true;
    return FG_OK;
}

int32_t fg_seed(fg_handle *h, int64_t seed_base, const uint8_t *mask, void *stream) {
    if (int rc = check_bound(h)) return rc;
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    Params p = make_params(h);
    p.mask = mask; p.seed_base = seed_base;
    seed_kernel<<<grid_for(h, 8), kThreads, 0, (cudaStream_t)stream>>>(p);
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return FG_OK;
}

int32_t fg_reset(fg_handle *h, const uint8_t *mask, void *stream) {
    if (int rc = check_bound(h)) return rc;
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    return reset_on(h, mask, (cudaStream_t)stream);
}

int32_t fg_step(fg_handle *h, void *stream) {
    if (int rc = check_bound(h)) return rc;
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    h->step_calls++;
    return step_range(h, 0, -1, (cudaStream_t)stream);
}

int32_t fg_step_host(fg_handle *h, const uint8_t *a1, const uint8_t *a2, float *obs, float *reward,
                     uint8_t *terminated, int32_t *info_frame, uint8_t *info_misc, void *stream) {
    HostOut o = { obs, nullptr, nullptr, reward, terminated, info_frame, info_misc };
    return host_step(h, a1, a2, o, (cudaStream_t)stream);
}

int32_t fg_step_host_compact(fg_handle *h, const uint8_t *a1, const uint8_t *a2, const fg_host_outputs *out, void *stream) {
    if (!out || out->struct_size != (int32_t)sizeof(fg_host_outputs))
        return fail(FG_ERR_INVALID_ARGUMENT, "fg_host_outputs is null or its struct_size does not match%s");
    HostOut o = { nullptr, out->position, out->obs_u8, out->reward, out->terminated, out->info_frame, out->info_misc };
    return host_step(h, a1, a2, o, (cudaStream_t)stream);
}

int32_t fg_reset_host(fg_handle *h, const uint8_t *mask, float *obs, int32_t *info_frame, uint8_t *info_misc, void *stream) {
    HostOut o = { obs, nullptr, nullptr, nullptr, nullptr, info_frame, info_misc };
    return host_reset(h, mask, o, (cudaStream_t)stream);
}

int32_t fg_reset_host_compact(fg_handle *h, const uint8_t *mask, const fg_host_outputs *out, void *stream) {
    if (!out || out->struct_size != (int32_t)sizeof(fg_host_outputs))
        return fail(FG_ERR_INVALID_ARGUMENT, "fg_host_outputs is null or its struct_size does not match%s");
    HostOut o = { nullptr, out->position, out->obs_u8, nullptr, nullptr, out->info_frame, out->info_misc };
    return host_reset(h, mask, o, (cudaStream_t)stream);
}

int32_t fg_get_state(fg_handle *h, int32_t first, int32_t count, fg_env_state *out) {
    if (int rc = check_bound(h)) return rc;
    if (!out || first < 0 || count < 0 || (int64_t)first + count > h->cfg.num_envs)
        return fail(FG_ERR_INVALID_ARGUMENT, "env range out of bounds%s");
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    CUDA_TRY(cudaDeviceSynchronize());
    std::vector<FgVec4> pl[FG_STATE_PLANES];
    for (int k = 0; k < FG_STATE_PLANES; k++) {
        pl[k].resize((size_t)count);
        CUDA_TRY(cudaMemcpy(pl[k].data(), (const FgVec4 *)h->buf.state[k] + first, sizeof(FgVec4) * (size_t)count, cudaMemcpyDeviceToHost));
    }
    for (int i = 0; i < count; i++)
        fg_decode_env(pl[FG_PLANE_F1][i], pl[FG_PLANE_F2][i], pl[FG_PLANE_ENV][i], pl[FG_PLANE_RNG][i], &out[i]);
    return FG_OK;
}

int32_t fg_set_state(fg_handle *h, int32_t first, int32_t count, const fg_env_state *in) {
    if (int rc = check_bound(h)) return rc;
    if (!in || first < 0 || count < 0 || (int64_t)first + count > h->cfg.num_envs)
        return fail(FG_ERR_INVALID_ARGUMENT, "env range out of bounds%s");
    std::vector<FgVec4> pl[FG_STATE_PLANES];
    for (int k = 0; k < FG_STATE_PLANES; k++) pl[k].resize((size_t)count);
    for (int i = 0; i < count; i++)
        if (fg_encode_env(&in[i], &pl[FG_PLANE_F1][i], &pl[FG_PLANE_F2][i], &pl[FG_PLANE_ENV][i], &pl[FG_PLANE_RNG][i]))
            return fail(FG_ERR_INVALID_STATE, "state not representable (unknown action id, WIN/has_won, or field out of range)%s");
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    CUDA_TRY(cudaDeviceSynchronize());
    for (int k = 0; k < FG_STATE_PLANES; k++)
        CUDA_TRY(cudaMemcpy((FgVec4 *)h->buf.state[k] + first, pl[k].data(), sizeof(FgVec4) * (size_t)count, cudaMemcpyHostToDevice));
    return FG_OK;
}

int32_t fg_read_stats(fg_handle *h, uint64_t *out, void *stream) {
    if (int rc = check_bound(h)) return rc;
    if (!out) return fail(FG_ERR_INVALID_ARGUMENT, "null output%s");
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    CUDA_TRY(cudaMemcpyAsync(out, h->buf.stats, sizeof(uint64_t) * FG_STAT_COUNT, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return FG_OK;
}

int32_t fg_delay_ring_step(fg_handle *h, int32_t depth, int32_t pos, float *ring_obs, int32_t *ring_frame, uint8_t *ring_misc,
                           float *out_obs, int32_t *out_frame, uint8_t *out_misc, void *stream) {
    if (int rc = check_bound(h)) return rc;
    if (depth < 2 || pos < 0 || pos >= depth) return fail(FG_ERR_INVALID_ARGUMENT, "depth must be frame_delay + 1 >= 2 and 0 <= pos < depth%s");
    if (!ring_obs || !ring_frame || !ring_misc || !out_obs || !out_frame || !out_misc) return fail(FG_ERR_INVALID_ARGUMENT, "null buffer%s");
    if (((uintptr_t)ring_obs & 15u) || ((uintptr_t)out_obs & 15u) || ((uintptr_t)ring_misc & 3u) || ((uintptr_t)out_misc & 3u))
        return fail(FG_ERR_INVALID_ARGUMENT, "obs buffers must be 16-byte, misc buffers 4-byte aligned%s");
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    const DelayRingRef ring = { (float4 *)ring_obs, ring_frame, (uint32_t *)ring_misc, (size_t)h->cfg.num_envs };
    delay_ring_kernel<<<grid_for(h, 8), 256, 0, (cudaStream_t)stream>>>(
        (const float4 *)h->buf.obs, h->buf.info_frame, (const uint32_t *)h->buf.info_misc, ring, (float4 *)out_obs, out_frame,
        (uint32_t *)out_misc, h->buf.step_mask, h->cfg.num_envs, depth, pos);
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return FG_OK;
}

// The checks and parameter block every fg_rollout_mlp* entry point shares, in this order: the pool struct (with_pool), the
// handle, the buffers struct, the handle's configuration, P2 (the pool and its bot member with a pool, the second policy's
// weights without one), hidden size, horizon, buffer pointers and alignment.  No pool: pool.count = 0, bot_member = -1.
// ring.depth is left 0 (no frame_delay).
static int32_t rollout_params(fg_handle *h, const fg_rollout_buffers *r, bool with_pool, const fg_opponent_pool *pool, bool with_bot,
                              int32_t bot_member, RolloutParams &rp) {
    if (with_pool && (!pool || pool->struct_size != (int32_t)sizeof(fg_opponent_pool)))
        return fail(FG_ERR_INVALID_ARGUMENT, "fg_opponent_pool is null or its struct_size does not match%s");
    if (int rc = check_bound(h)) return rc;
    if (!r || r->struct_size != (int32_t)sizeof(fg_rollout_buffers))
        return fail(FG_ERR_INVALID_ARGUMENT, "fg_rollout_buffers is null or its struct_size does not match%s");
    if (h->cfg.p1_bot || !h->cfg.autoreset || h->buf.step_mask)
        return fail(FG_ERR_INVALID_STATE, with_pool ? "fg_rollout_mlp_pool needs P1 = policy, autoreset on, no step mask%s"
                                                    : "fg_rollout_mlp needs P1 = policy, autoreset on, no step mask "
                                                      "(use fg_policy_mlp_sample + fg_step for other configurations)%s");
    const int64_t n = h->cfg.num_envs;
    const bool p2_policy = !h->cfg.p2_bot;
    if (with_pool) {
        if (!p2_policy)
            return fail(FG_ERR_INVALID_ARGUMENT, "fg_rollout_mlp_pool needs p2_bot = 0: the pool plays P2 (the in-game bot cannot be a member)%s");
        if (pool->count < 1 || pool->count > FG_POOL_MAX) return fail(FG_ERR_INVALID_ARGUMENT, "fg_opponent_pool.count must be in 1..16%s");
        if (with_bot && (bot_member < 0 || bot_member >= pool->count))
            return fail(FG_ERR_INVALID_ARGUMENT, "fg_rollout_mlp_pool_bot: bot_member must be in 0 .. fg_opponent_pool.count - 1%s");
        for (int m = 0; m < pool->count; m++) {
            const int64_t lo = m ? pool->end[m - 1] : 0, e = pool->end[m];
            if (e < lo || e > n) return fail(FG_ERR_INVALID_ARGUMENT, "fg_opponent_pool.end must be non-decreasing and at most num_envs%s");
            if (e % FG_POOL_BLOCK && e != n)
                return fail(FG_ERR_INVALID_ARGUMENT, "fg_opponent_pool.end: every boundary must be a multiple of FG_POOL_BLOCK (128) or num_envs%s");
            if (with_bot && m == bot_member) continue;              // the bot's weight pointers are not read
            const fg_mlp_weights &w = pool->member[m];
            if (!w.scale || !w.w1 || !w.b1 || !w.w2 || !w.b2 || !w.w3 || !w.b3)
                return fail(FG_ERR_INVALID_ARGUMENT, "fg_opponent_pool: null member weight pointer%s");
            if ((uintptr_t)w.w2 & 15u) return fail(FG_ERR_INVALID_ARGUMENT, "fg_opponent_pool: member w2 must be 16-byte aligned%s");
        }
        if (pool->end[pool->count - 1] != n) return fail(FG_ERR_INVALID_ARGUMENT, "fg_opponent_pool.end[count - 1] must be num_envs%s");
        if ((uintptr_t)pool->stats & 7u) return fail(FG_ERR_INVALID_ARGUMENT, "fg_opponent_pool.stats must be 8-byte aligned%s");
    } else if (p2_policy && (!r->p2_scale || !r->p2_w1 || !r->p2_b1 || !r->p2_w2 || !r->p2_b2 || !r->p2_w3 || !r->p2_b3 ||
                             !r->actions_p2 || !r->logp_p2 || ((uintptr_t)r->p2_w2 & 15u))) {
        return fail(FG_ERR_INVALID_ARGUMENT, "p2_bot = 0: fg_rollout_buffers needs the P2 policy (p2_* weights, 16-byte aligned p2_w2, "
                                             "actions_p2, logp_p2)%s");
    }
    if (r->hidden != 32 && r->hidden != 64 && r->hidden != 128)
        return fail(FG_ERR_INVALID_ARGUMENT, with_pool ? "hidden size must be 32, 64 or 128 (the learner's and every member's)%s"
                                                       : "hidden size must be 32, 64 or 128%s");
    if (r->horizon < 1) return fail(FG_ERR_INVALID_ARGUMENT, "horizon must be positive%s");
    if (!r->scale || !r->w1 || !r->b1 || !r->w2 || !r->b2 || !r->w3 || !r->b3 || !r->obs || !r->actions || !r->logp || !r->rewards ||
        !r->dones || (with_pool && (!r->actions_p2 || !r->logp_p2)))
        return fail(FG_ERR_INVALID_ARGUMENT, with_pool ? "fg_rollout_buffers: null pointer (actions_p2 and logp_p2 are required)%s"
                                                       : "fg_rollout_buffers: null pointer%s");
    if (((uintptr_t)r->obs & 15u) || ((uintptr_t)r->w2 & 15u)) return fail(FG_ERR_INVALID_ARGUMENT, "obs and w2 must be 16-byte aligned%s");
    rp = {};
    rp.sim = make_params(h);
    rp.w = { r->scale, r->w1, r->b1, r->w2, r->b2, r->w3, r->b3 };
    rp.seed = r->seed; rp.counter_base = (const unsigned long long *)r->counter_base;
    rp.hidden = r->hidden; rp.horizon = r->horizon;
    rp.obs = (float4 *)r->obs; rp.actions = r->actions; rp.logp = r->logp; rp.rewards = r->rewards; rp.dones = r->dones;
    rp.p2_policy = p2_policy; rp.p2_mirror = p2_policy && r->p2_mirror;
    rp.w_p2 = { r->p2_scale, r->p2_w1, r->p2_b1, r->p2_w2, r->p2_b2, r->p2_w3, r->p2_b3 };   // not read with a pool
    rp.seed_p2 = r->p2_seed; rp.actions_p2 = r->actions_p2; rp.logp_p2 = r->logp_p2;
    if (with_pool) {
        for (int m = 0; m < FG_POOL_MAX; m++) {
            const bool used = m < pool->count;
            const fg_mlp_weights &w = pool->member[used ? m : 0];
            rp.pool.member[m] = { w.scale, w.w1, w.b1, w.w2, w.b2, w.w3, w.b3 };
            rp.pool.end[m] = used ? pool->end[m] : n;
        }
        rp.pool.count = pool->count;
        rp.pool.stats = (unsigned long long *)pool->stats;
    }
    rp.bot_member = with_bot ? bot_member : -1;
    return FG_OK;
}

// the launch every fg_rollout_mlp* entry point ends with, once its checks have passed
static int32_t rollout_launch(fg_handle *h, const RolloutParams &rp, void *stream) {
    CUDA_TRY(cudaSetDevice(h->cfg.device));
    CUDA_TRY(launch_rollout(h->cfg.dense_reward != 0, (cudaStream_t)stream, rp));
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return FG_OK;
}

int32_t fg_rollout_mlp(fg_handle *h, const fg_rollout_buffers *r, void *stream) {
    RolloutParams rp;
    if (int rc = rollout_params(h, r, false, nullptr, false, -1, rp)) return rc;
    return rollout_launch(h, rp, stream);
}

int32_t fg_rollout_mlp_pool(fg_handle *h, const fg_rollout_buffers *r, const fg_opponent_pool *pool, void *stream) {
    RolloutParams rp;
    if (int rc = rollout_params(h, r, true, pool, false, -1, rp)) return rc;
    return rollout_launch(h, rp, stream);
}

int32_t fg_rollout_mlp_pool_bot(fg_handle *h, const fg_rollout_buffers *r, const fg_opponent_pool *pool, int32_t bot_member,
                                void *stream) {
    RolloutParams rp;
    if (int rc = rollout_params(h, r, true, pool, true, bot_member, rp)) return rc;
    return rollout_launch(h, rp, stream);
}

int32_t fg_rollout_mlp_delayed(fg_handle *h, const fg_rollout_buffers *r, const fg_opponent_pool *pool, int32_t bot_member,
                               const fg_delay_ring *ring, void *stream) {
    if (!ring || ring->struct_size != (int32_t)sizeof(fg_delay_ring))
        return fail(FG_ERR_INVALID_ARGUMENT, "fg_delay_ring is null or its struct_size does not match%s");
    RolloutParams rp;
    if (int rc = rollout_params(h, r, pool != nullptr, pool, pool && bot_member != -1, bot_member, rp)) return rc;
    if (!pool && bot_member != -1) return fail(FG_ERR_INVALID_ARGUMENT, "fg_rollout_mlp_delayed: bot_member must be -1 without a pool%s");
    if (ring->depth < 2 || ring->pos < 0 || ring->pos >= ring->depth)
        return fail(FG_ERR_INVALID_ARGUMENT, "fg_delay_ring: depth must be frame_delay + 1 >= 2 and 0 <= pos < depth%s");
    if (!ring->ring_obs || !ring->ring_frame || !ring->ring_misc || !ring->out_obs || !ring->out_frame || !ring->out_misc)
        return fail(FG_ERR_INVALID_ARGUMENT, "fg_delay_ring: null buffer%s");
    if (((uintptr_t)ring->ring_obs & 15u) || ((uintptr_t)ring->out_obs & 15u) || ((uintptr_t)ring->ring_misc & 3u) ||
        ((uintptr_t)ring->out_misc & 3u))
        return fail(FG_ERR_INVALID_ARGUMENT, "fg_delay_ring: obs buffers must be 16-byte, misc buffers 4-byte aligned%s");
    rp.ring = { (float4 *)ring->ring_obs, ring->ring_frame, (uint32_t *)ring->ring_misc, (float4 *)ring->out_obs, ring->out_frame,
                (uint32_t *)ring->out_misc, ring->depth, ring->pos };
    return rollout_launch(h, rp, stream);
}

int64_t fg_launch_count(fg_handle *h) { return h ? h->launches : 0; }

}  // extern "C"
