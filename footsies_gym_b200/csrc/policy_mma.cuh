#ifndef FOOTSIES_B200_POLICY_MMA_CUH
#define FOOTSIES_B200_POLICY_MMA_CUH
// policy_mma.cuh -- the 8-H-H-8 tanh MLP policy on the warp-level tensor-core path (mma.sync m16n8k8, TF32 operands,
// fp32 accumulate) with the 3 x TF32 operand split, for H <= 64 (H = 128 keeps the FFMA2 path of policy_mlp.cuh).
//
// Why (round 2, measured -- profiles/r02_mma_probe.log, profiles/r02d_rollout_battles_per_lane.log): the FFMA2 version
// of the rollout kernel is bound by ISSUE SLOTS and shared-memory weight fetches, not by the FMA pipe (one battle per
// lane instead of two: 10.9 us per step instead of 6.4).  An FFMA2 retires 64 multiply-adds per instruction, an m16n8k8
// MMA 1024; mma.sync sustains 512 TF32 MAC per cycle per SM on B200, i.e. 171 fp32-grade MAC per cycle per SM after the
// three-product split against ~127 for FFMA / FFMA2 -- and needs 16 x fewer instructions and one 128-bit weight fetch per
// 3072 multiply-adds.  Accuracy: a = a_hi + a_lo with a_hi = tf32(a), a_lo = tf32(a - a_hi) (likewise b); the product is
// a_lo*b_hi + a_hi*b_lo + a_hi*b_hi accumulated in fp32 (the dropped a_lo*b_lo term is ~2^-22 relative): the logits agree
// with torch's fp32 result to ~1e-6, the test bar is 2e-5 in log-probability (tests/test_rollout.py).
//
// Mapping: ONE WARP owns 32 battles for the whole forward pass -- two 16-row M tiles -- and nothing is shared between
// warps but the read-only weight fragments, so the rollout kernel needs no CTA barrier inside its horizon loop.  With
// g = lane / 4, t = lane % 4 the m16n8k8 fragments are (PTX ISA, "Matrix fragments for mma.m16n8k8"):
//   A (16 x 8, row): a0 = (g, t)  a1 = (g + 8, t)  a2 = (g, t + 4)  a3 = (g + 8, t + 4)
//   B (8 x 8, col):  b0 = (k = t, n = g)  b1 = (k = t + 4, n = g)
//   C (16 x 8):      c0 = (g, 2t)  c1 = (g, 2t + 1)  c2 = (g + 8, 2t)  c3 = (g + 8, 2t + 1)
// A layer's C tile for units 8j .. 8j + 7 becomes the next layer's A fragment of k-step j WITHOUT leaving the registers:
// the k index of an MMA is a summation index, so its order is free as long as A and B agree -- A column t is taken to be
// unit 8j + 2t and column t + 4 unit 8j + 2t + 1 (a0 = c0, a1 = c2, a2 = c1, a3 = c3), and the weight fragments are staged
// with their rows permuted the same way.
//
// Layers 2 and 3 (FG_POLICY_F16, default): the same split on FP16 operands -- mma.sync m16n8k16, 1024 MAC per cycle per SM,
// twice the TF32 rate, and half as many instructions (layer 2 of H = 64: 96 HMMA.16816 instead of 192 HMMA.1688).  FP16
// carries the same 11 significant bits as TF32, so hi + lo holds 22 bits just the same; what FP16 lacks is exponent
// range, and after a tanh the range is known: the activations are produced as 256 tanh(.) (|x| <= 256, hi and lo normal
// FP16 numbers down to |tanh| = 2^-12) and each weight matrix is scaled by a power of two chosen at staging time so that
// its largest entry lies in [2^12, 2^13).  The biases are staged pre-multiplied by the same factor and the inverse is
// folded into the constant of the next tanh's exp2, so the scaling costs no instruction and no rounding.  Layer 1 sees
// raw observations times a caller-supplied scale (unbounded) and stays on TF32.  With k = 16 the C tiles 2j and 2j + 1 of
// one layer are the A fragment of k-step j of the next in their natural order (a0 = (c0, c1) of tile 2j, a1 = (c2, c3),
// a2 / a3 the same of tile 2j + 1): no row permutation.
#include <cuda_fp16.h>

#include "policy_mlp.cuh"

#ifndef FG_POLICY_F16
#define FG_POLICY_F16 1
#endif
// Layer 2 with the OUTPUT tile as the outer loop (profiles/r03e_rollout_l2_order.log: 1 Mi battles 144.7 -> 138.8 us per step,
// 131 072: 19.3 -> 18.9, 16 384: unchanged; same bits -- a tile's k-steps keep their order): acc[nt] is final after its own
// k-steps, so its tanh (two MUFU per value, the XU pipe) runs under the next tiles' MMAs instead of after all of them.
#ifndef FG_POLICY_L2_NT_OUTER
#define FG_POLICY_L2_NT_OUTER 1
#endif

namespace fgp {

constexpr int kMmaMaxHidden = 64;
constexpr float kActScale = 256.0f;             // FP16 path: hidden activations are carried as kActScale * tanh

// Shared memory of one weight set: per (layer, k-step, n-tile) one float4 per lane = {b0_hi, b1_hi, b0_lo, b1_lo}
// (one conflict-free LDS.128 per fragment), then the biases and the observation scale.
// FP16 path: layers 2 and 3 hold per (k-step of 16, n-tile) one uint4 per lane = {b0_hi, b1_hi, b0_lo, b1_lo} as half2
// pairs; kInv2 / kInv3 = 1 / (kActScale x the layer's weight scale), kMax = scratch of the staging reduction.
template <int H>
struct PolicyMmaSmem {
    static_assert(H % 16 == 0 && H <= kMmaMaxHidden, "hidden size of the MMA path");
    static constexpr int NT = H / 8;                              // n-tiles of a hidden layer = k-steps (of 8) of the next one
    static constexpr int KT = FG_POLICY_F16 ? H / 16 : NT;        // k-steps of layers 2 and 3
    static constexpr int kW1 = 0, kW2 = kW1 + NT * 32, kW3 = kW2 + KT * NT * 32, kFrags = kW3 + KT * 32;   // in float4
    static constexpr int kB1 = kFrags * 4, kB2 = kB1 + H, kB3 = kB2 + H, kScale = kB3 + 8, kInv2 = kScale + 8, kInv3 = kInv2 + 1,
                         kMax = kInv3 + 1, kFloats = kMax + 2;    // in floats
    static constexpr size_t kBytes = sizeof(float) * ((kFloats + 3) / 4 * 4);
};

__device__ __forceinline__ float tf32_hi(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// Activation split on the hot path: hi = x truncated to TF32 (one LOP3), lo = x - hi, exact in fp32 and handed to the MMA
// as it is (the tensor core reads the upper 19 bits of a TF32 operand).  sm_100a has no native cvt.rna.tf32: it is emulated
// in ~5 integer instructions, which made the two conversions per activation a quarter of the policy's instructions
// (16 384 battles: 4.46 -> 4.00 us per step); the weights, split once per launch, keep the rounded conversion.
// |x - hi - tf32(lo)| <= 2^-21 |x|.
// (Tried and dropped, profiles/r02n_rollout_halves.log: computing layer 2 in two halves of its n-tiles to halve the live
// accumulators and fit a third CTA per SM -- 4.43 us per step at 16 384 battles, 200 instead of 184 us at 1 Mi.)
__device__ __forceinline__ void tf32_split(float x, uint32_t &hi, uint32_t &lo) {
    hi = __float_as_uint(x) & 0xffffe000u;
    lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// c += a * b at fp32-grade accuracy: small terms first
__device__ __forceinline__ void mma_3xtf32(float (&c)[4], const uint32_t (&ahi)[4], const uint32_t (&alo)[4], const float4 &b) {
    mma_tf32(c, alo, __float_as_uint(b.x), __float_as_uint(b.y));
    mma_tf32(c, ahi, __float_as_uint(b.z), __float_as_uint(b.w));
    mma_tf32(c, ahi, __float_as_uint(b.x), __float_as_uint(b.y));
}


// ---- FP16 operands (layers 2 and 3) ----
__device__ __forceinline__ uint32_t pack_half2(float x, float y) {      // x -> low half, y -> high half (F2FP.PACK_AB)
    const __half2 h = __floats2half2_rn(x, y);
    return *reinterpret_cast<const uint32_t *>(&h);
}
// Two activations -> the hi and lo halves of one A register.  hi = x truncated to 11 significant bits (exact in FP16 for
// 2^-14 <= |x| < 2^16), lo = x - hi, exact in fp32, rounded to FP16: |x - hi - lo| <= 2^-22 |x|.
__device__ __forceinline__ void f16_split2(float x, float y, uint32_t &hi, uint32_t &lo) {
    const float xh = __uint_as_float(__float_as_uint(x) & 0xffffe000u), yh = __uint_as_float(__float_as_uint(y) & 0xffffe000u);
    hi = pack_half2(xh, yh);
    lo = pack_half2(x - xh, y - yh);
}
__device__ __forceinline__ void mma_f16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_3xf16(float (&c)[4], const uint32_t (&ahi)[4], const uint32_t (&alo)[4], const uint4 &b) {
    mma_f16(c, alo, b.x, b.y);
    mma_f16(c, ahi, b.z, b.w);
    mma_f16(c, ahi, b.x, b.y);
}
// kActScale * tanh(x * inv) with c = inv * 2 log2(e): the scaled activation the FP16 layers consume (same two MUFU
// approximations as fast_tanh; inv is a power of two, so x * c rounds exactly like (x * inv) * 2 log2(e))
__device__ __forceinline__ float scaled_tanh(float x, float c) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * c));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f * kActScale, r, kActScale);
}
constexpr float kTwoLog2e = 2.8853900432586669921875f;

// Stage one weight set (torch.nn.Linear layout: W[out][in]) as pre-split B fragments.  Called by every thread of the CTA
// (nthreads a multiple of 32); the FP16 path contains two CTA barriers (the per-matrix maximum that fixes the scale).
// NOUT = real output rows of layer 3 (W3 [NOUT][H], b3 [NOUT]): 8 for the policy's logits, 1 for a value head.  The
// remaining rows of the 8-wide output tile are staged as zeros and never read from the caller's pointers, and the W3 scale
// comes from the real rows alone; for NOUT = 8 every added condition is constant and the code is the policy's as before.
template <int H, int NOUT = 8>
__device__ __forceinline__ void policy_mma_stage(float *sm, const PolicyWeights &p, int tid, int nthreads) {
    static_assert(NOUT >= 1 && NOUT <= 8, "layer 3 has one n-tile of 8 outputs");
    using L = PolicyMmaSmem<H>;
    constexpr int NT = L::NT;
    float4 *frag = reinterpret_cast<float4 *>(sm);
    auto put = [&](int idx, float b0, float b1) {
        const float h0 = tf32_hi(b0), h1 = tf32_hi(b1);
        frag[idx] = make_float4(h0, h1, tf32_hi(b0 - h0), tf32_hi(b1 - h1));
    };
#if FG_POLICY_F16
    // layer 1: k = observation feature (natural order: t, t + 4), n = unit 8 nt + g
    for (int i = tid; i < NT * 32; i += nthreads) {
        const int nt = i >> 5, lane = i & 31, g = lane >> 2, t = lane & 3;
        put(L::kW1 + i, p.w1[(8 * nt + g) * 8 + t], p.w1[(8 * nt + g) * 8 + t + 4]);
    }
    // largest |w| of W2 and of W3 -> power-of-two scales that put it into [2^12, 2^13)
    uint32_t *smax = reinterpret_cast<uint32_t *>(sm + L::kMax);
    if (tid < 2) smax[tid] = 0u;
    __syncthreads();
    {
        uint32_t m2 = 0u, m3 = 0u;                                  // |w| as bits: ordered like the values
        for (int i = tid; i < H * H; i += nthreads) m2 = max(m2, __float_as_uint(p.w2[i]) & 0x7fffffffu);
        for (int i = tid; i < NOUT * H; i += nthreads) m3 = max(m3, __float_as_uint(p.w3[i]) & 0x7fffffffu);
        m2 = __reduce_max_sync(0xffffffffu, m2); m3 = __reduce_max_sync(0xffffffffu, m3);
        if ((tid & 31) == 0) { atomicMax(&smax[0], m2); atomicMax(&smax[1], m3); }
    }
    __syncthreads();
    // biased exponent E of the maximum (clamped: all-zero / non-finite weights keep the arithmetic finite):
    // weight scale 2^(139 - E), inverse of (kActScale x scale) = 2^(E - 147)
    const int e2 = min(max((int)(smax[0] >> 23), 40), 254), e3 = min(max((int)(smax[1] >> 23), 40), 254);
    const float s2 = __uint_as_float((uint32_t)(266 - e2) << 23), s3 = __uint_as_float((uint32_t)(266 - e3) << 23);
    uint4 *hfrag = reinterpret_cast<uint4 *>(sm);
    auto put16 = [&](int idx, const float *row, float scale) {      // row -> k = 2t, 2t + 1 (b0) and 2t + 8, 2t + 9 (b1)
        const float w0 = row[0] * scale, w1 = row[1] * scale, w2 = row[8] * scale, w3 = row[9] * scale;
        const __half2 h0 = __floats2half2_rn(w0, w1), h1 = __floats2half2_rn(w2, w3);
        const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
        uint4 v;
        v.x = *reinterpret_cast<const uint32_t *>(&h0); v.y = *reinterpret_cast<const uint32_t *>(&h1);
        v.z = pack_half2(w0 - f0.x, w1 - f0.y); v.w = pack_half2(w2 - f1.x, w3 - f1.y);
        hfrag[idx] = v;
    };
    // layer 2: k-step kt (16 inputs), n = output unit 8 nt + g
    for (int i = tid; i < L::KT * NT * 32; i += nthreads) {
        const int lane = i & 31, g = lane >> 2, t = lane & 3, nt = (i >> 5) % NT, kt = (i >> 5) / NT;
        put16(L::kW2 + i, p.w2 + (8 * nt + g) * H + 16 * kt + 2 * t, s2);
    }
    // layer 3: one n-tile (the 8 logits), n = g
    for (int i = tid; i < L::KT * 32; i += nthreads) {
        const int kt = i >> 5, lane = i & 31, g = lane >> 2, t = lane & 3;
        if (NOUT < 8 && g >= NOUT) hfrag[L::kW3 + i] = make_uint4(0u, 0u, 0u, 0u);
        else put16(L::kW3 + i, p.w3 + g * H + 16 * kt + 2 * t, s3);
    }
    // biases of the scaled layers in accumulator units
    for (int i = tid; i < H; i += nthreads) { sm[L::kB1 + i] = p.b1[i]; sm[L::kB2 + i] = p.b2[i] * (kActScale * s2); }
    if (tid < 8) {
        sm[L::kB3 + tid] = (NOUT == 8 || tid < NOUT) ? p.b3[tid] * (kActScale * s3) : 0.0f;
        sm[L::kScale + tid] = p.scale[tid];
    }
    if (tid == 0) {
        sm[L::kInv2] = __uint_as_float((uint32_t)(e2 - 20) << 23);
        sm[L::kInv3] = __uint_as_float((uint32_t)(e3 - 20) << 23);
    }
#else
    // layer 1: k = observation feature (natural order: t, t + 4), n = unit 8 nt + g
    for (int i = tid; i < NT * 32; i += nthreads) {
        const int nt = i >> 5, lane = i & 31, g = lane >> 2, t = lane & 3;
        put(L::kW1 + i, p.w1[(8 * nt + g) * 8 + t], p.w1[(8 * nt + g) * 8 + t + 4]);
    }
    // layer 2: k-step kt, column t <-> input unit 8 kt + 2t, column t + 4 <-> 8 kt + 2t + 1; n = output unit 8 nt + g
    for (int i = tid; i < NT * NT * 32; i += nthreads) {
        const int lane = i & 31, g = lane >> 2, t = lane & 3, nt = (i >> 5) % NT, kt = (i >> 5) / NT;
        put(L::kW2 + i, p.w2[(8 * nt + g) * H + 8 * kt + 2 * t], p.w2[(8 * nt + g) * H + 8 * kt + 2 * t + 1]);
    }
    // layer 3: one n-tile (the 8 logits), n = g
    for (int i = tid; i < NT * 32; i += nthreads) {
        const int kt = i >> 5, lane = i & 31, g = lane >> 2, t = lane & 3;
        if (NOUT < 8 && g >= NOUT) frag[L::kW3 + i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        else put(L::kW3 + i, p.w3[g * H + 8 * kt + 2 * t], p.w3[g * H + 8 * kt + 2 * t + 1]);
    }
    for (int i = tid; i < H; i += nthreads) { sm[L::kB1 + i] = p.b1[i]; sm[L::kB2 + i] = p.b2[i]; }
    if (tid < 8) { sm[L::kB3 + tid] = (NOUT == 8 || tid < NOUT) ? p.b3[tid] : 0.0f; sm[L::kScale + tid] = p.scale[tid]; }
#endif
}

// The 8 logits of the warp's 16 MT battles (for a weight set staged with NOUT < 8: its NOUT outputs in columns 0 .. NOUT - 1,
// zeros after them).  obs_rows: the battles' raw observation rows ([16 MT][8] floats, shared or
// global memory); lg_rows: [16 MT][8] floats of shared memory private to the warp, where row r receives battle r's logits
// (the caller reads its own row after the __syncwarp at the end).  MIRROR shows the network the observation as the other
// player sees it (policy_mirror_obs: per-player fields swap, positions change sign).
// MT = M tiles per warp: 2 (32 battles, every lane simulates one) or 1 (16 battles: twice the warps per SM for small batches).
template <int H, int MT, bool MIRROR>
__device__ __forceinline__ void policy_mma_logits(const float *sm, const float *obs_rows, float *lg_rows, int lane) {
    static_assert(MT == 1 || MT == 2, "one or two M tiles per warp");
    using L = PolicyMmaSmem<H>;
    constexpr int NT = L::NT;
    const float4 *frag = reinterpret_cast<const float4 *>(sm);
    const float *b1 = sm + L::kB1, *b2 = sm + L::kB2, *b3 = sm + L::kB3, *sc = sm + L::kScale;
    const int g = lane >> 2, t = lane & 3;
    // ---- A fragments of layer 1 from the observation rows (features t and t + 4 of rows g, g + 8 of each M tile) ----
    uint32_t xhi[MT][4], xlo[MT][4];
    {
        // mirrored observation: feature f comes from f ^ 1, positions (6, 7) change sign; the scale belongs to the feature
        // as the network sees it
        const int f0 = MIRROR ? (t ^ 1) : t, f1 = MIRROR ? ((t + 4) ^ 1) : t + 4;
        const float s0 = sc[t], s1 = (MIRROR && t >= 2) ? -sc[t + 4] : sc[t + 4];
#pragma unroll
        for (int m = 0; m < MT; m++) {
            const float *r0 = obs_rows + (16 * m + g) * 8, *r1 = r0 + 64;
            tf32_split(r0[f0] * s0, xhi[m][0], xlo[m][0]);
            tf32_split(r1[f0] * s0, xhi[m][1], xlo[m][1]);
            tf32_split(r0[f1] * s1, xhi[m][2], xlo[m][2]);
            tf32_split(r1[f1] * s1, xhi[m][3], xlo[m][3]);
        }
    }
    // ---- layer 1: h[m][nt] = tanh(x W1^T + b1), kept as C tiles ----
    float h[MT][NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
        const float4 b = frag[L::kW1 + nt * 32 + lane];
        const float2 bias = *reinterpret_cast<const float2 *>(b1 + 8 * nt + 2 * t);
#pragma unroll
        for (int m = 0; m < MT; m++) {
            h[m][nt][0] = bias.x; h[m][nt][1] = bias.y; h[m][nt][2] = bias.x; h[m][nt][3] = bias.y;
            mma_3xtf32(h[m][nt], xhi[m], xlo[m], b);
#pragma unroll
            for (int k = 0; k < 4; k++) h[m][nt][k] = FG_POLICY_F16 ? scaled_tanh(h[m][nt][k], kTwoLog2e) : fast_tanh(h[m][nt][k]);
        }
    }
    // ---- layer 2 ----
    float acc[MT][NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
        const float2 bias = *reinterpret_cast<const float2 *>(b2 + 8 * nt + 2 * t);
#pragma unroll
        for (int m = 0; m < MT; m++) { acc[m][nt][0] = bias.x; acc[m][nt][1] = bias.y; acc[m][nt][2] = bias.x; acc[m][nt][3] = bias.y; }
    }
#if FG_POLICY_F16
    constexpr int KT = L::KT;
    const uint4 *hfrag = reinterpret_cast<const uint4 *>(sm);
#if FG_POLICY_L2_NT_OUTER
    // all A fragments first, then one output tile at a time (its k-steps in the same order, hence the same bits): acc[nt]
    // is final after its own KT k-steps, so its tanh can run under the next tiles' MMAs
    uint32_t ahi[KT][MT][4], alo[KT][MT][4];
#pragma unroll
    for (int kt = 0; kt < KT; kt++) {
#pragma unroll
        for (int m = 0; m < MT; m++) {
            f16_split2(h[m][2 * kt][0], h[m][2 * kt][1], ahi[kt][m][0], alo[kt][m][0]);
            f16_split2(h[m][2 * kt][2], h[m][2 * kt][3], ahi[kt][m][1], alo[kt][m][1]);
            f16_split2(h[m][2 * kt + 1][0], h[m][2 * kt + 1][1], ahi[kt][m][2], alo[kt][m][2]);
            f16_split2(h[m][2 * kt + 1][2], h[m][2 * kt + 1][3], ahi[kt][m][3], alo[kt][m][3]);
        }
    }
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
#pragma unroll
        for (int kt = 0; kt < KT; kt++) {
            const uint4 b = hfrag[L::kW2 + (kt * NT + nt) * 32 + lane];
#pragma unroll
            for (int m = 0; m < MT; m++) mma_3xf16(acc[m][nt], ahi[kt][m], alo[kt][m], b);
        }
    }
#else
#pragma unroll
    for (int kt = 0; kt < KT; kt++) {
        uint32_t ahi[MT][4], alo[MT][4];
#pragma unroll
        for (int m = 0; m < MT; m++) {                 // C tiles 2kt, 2kt + 1 -> A fragment of k-step kt
            f16_split2(h[m][2 * kt][0], h[m][2 * kt][1], ahi[m][0], alo[m][0]);
            f16_split2(h[m][2 * kt][2], h[m][2 * kt][3], ahi[m][1], alo[m][1]);
            f16_split2(h[m][2 * kt + 1][0], h[m][2 * kt + 1][1], ahi[m][2], alo[m][2]);
            f16_split2(h[m][2 * kt + 1][2], h[m][2 * kt + 1][3], ahi[m][3], alo[m][3]);
        }
#pragma unroll
        for (int nt = 0; nt < NT; nt++) {
            const uint4 b = hfrag[L::kW2 + (kt * NT + nt) * 32 + lane];
#pragma unroll
            for (int m = 0; m < MT; m++) mma_3xf16(acc[m][nt], ahi[m], alo[m], b);
        }
    }
#endif
    // ---- layer 3 on tanh(layer 2); the accumulators are in units of 1 / inv2, the logits of 1 / inv3 ----
    const float c2 = sm[L::kInv2] * kTwoLog2e, inv3 = sm[L::kInv3];
    float lg[MT][4];
    {
        const float2 bias = *reinterpret_cast<const float2 *>(b3 + 2 * t);
#pragma unroll
        for (int m = 0; m < MT; m++) { lg[m][0] = bias.x; lg[m][1] = bias.y; lg[m][2] = bias.x; lg[m][3] = bias.y; }
    }
#pragma unroll
    for (int kt = 0; kt < KT; kt++) {
        const uint4 b = hfrag[L::kW3 + kt * 32 + lane];
#pragma unroll
        for (int m = 0; m < MT; m++) {
            uint32_t ahi[4], alo[4];
            f16_split2(scaled_tanh(acc[m][2 * kt][0], c2), scaled_tanh(acc[m][2 * kt][1], c2), ahi[0], alo[0]);
            f16_split2(scaled_tanh(acc[m][2 * kt][2], c2), scaled_tanh(acc[m][2 * kt][3], c2), ahi[1], alo[1]);
            f16_split2(scaled_tanh(acc[m][2 * kt + 1][0], c2), scaled_tanh(acc[m][2 * kt + 1][1], c2), ahi[2], alo[2]);
            f16_split2(scaled_tanh(acc[m][2 * kt + 1][2], c2), scaled_tanh(acc[m][2 * kt + 1][3], c2), ahi[3], alo[3]);
            mma_3xf16(lg[m], ahi, alo, b);
        }
    }
#pragma unroll
    for (int m = 0; m < MT; m++) {
#pragma unroll
        for (int k = 0; k < 4; k++) lg[m][k] *= inv3;
    }
#else
#pragma unroll
    for (int kt = 0; kt < NT; kt++) {
        uint32_t ahi[MT][4], alo[MT][4];
#pragma unroll
        for (int m = 0; m < MT; m++) {                 // C tile kt -> A fragment of k-step kt: a0 = c0, a1 = c2, a2 = c1, a3 = c3
            tf32_split(h[m][kt][0], ahi[m][0], alo[m][0]);
            tf32_split(h[m][kt][2], ahi[m][1], alo[m][1]);
            tf32_split(h[m][kt][1], ahi[m][2], alo[m][2]);
            tf32_split(h[m][kt][3], ahi[m][3], alo[m][3]);
        }
#pragma unroll
        for (int nt = 0; nt < NT; nt++) {
            const float4 b = frag[L::kW2 + (kt * NT + nt) * 32 + lane];
#pragma unroll
            for (int m = 0; m < MT; m++) mma_3xtf32(acc[m][nt], ahi[m], alo[m], b);
        }
    }
    // ---- layer 3 on tanh(layer 2) ----
    float lg[MT][4];
    {
        const float2 bias = *reinterpret_cast<const float2 *>(b3 + 2 * t);
#pragma unroll
        for (int m = 0; m < MT; m++) { lg[m][0] = bias.x; lg[m][1] = bias.y; lg[m][2] = bias.x; lg[m][3] = bias.y; }
    }
#pragma unroll
    for (int kt = 0; kt < NT; kt++) {
        const float4 b = frag[L::kW3 + kt * 32 + lane];
#pragma unroll
        for (int m = 0; m < MT; m++) {
            uint32_t ahi[4], alo[4];
            tf32_split(fast_tanh(acc[m][kt][0]), ahi[0], alo[0]);
            tf32_split(fast_tanh(acc[m][kt][2]), ahi[1], alo[1]);
            tf32_split(fast_tanh(acc[m][kt][1]), ahi[2], alo[2]);
            tf32_split(fast_tanh(acc[m][kt][3]), ahi[3], alo[3]);
            mma_3xtf32(lg[m], ahi, alo, b);
        }
    }
#endif
    // ---- logits of row r to lg_rows[r][0 .. 7]: this lane holds columns 2t, 2t + 1 of rows 16 m + g and 16 m + g + 8 ----
    __syncwarp();                                     // the previous step's readers are done with lg_rows
#pragma unroll
    for (int m = 0; m < MT; m++) {
        *reinterpret_cast<float2 *>(lg_rows + (16 * m + g) * 8 + 2 * t) = make_float2(lg[m][0], lg[m][1]);
        *reinterpret_cast<float2 *>(lg_rows + (16 * m + g + 8) * 8 + 2 * t) = make_float2(lg[m][2], lg[m][3]);
    }
    __syncwarp();
}

}  // namespace fgp
#endif
