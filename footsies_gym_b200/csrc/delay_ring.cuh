#ifndef FOOTSIES_B200_DELAY_RING_CUH
#define FOOTSIES_B200_DELAY_RING_CUH
// delay_ring.cuh -- the frame_delay queue of FootsiesEnv for one battle (footsies.py:129-131: deque(maxlen = frame_delay
// + 1); :533-535: append the newest state, emit the oldest; :502-504: a reset refills the queue with the first state), as
// a ring of `depth` slots per battle in device memory.  One rule for both users: delay_ring_kernel (fg_delay_ring_step,
// after an fg_step) and the frame_delay instantiations of the whole-horizon rollout kernel (fg_rollout_mlp_delayed).
#include <stdint.h>

namespace fgk {

// what fg_step writes for a battle besides reward and termination: observation, info frame, info misc
struct DelayEntry {
    float4 a, b;
    int32_t frame;
    uint32_t misc;
};

// the caller's ring: slot s of battle i at [s * n + i] (obs: float4 [depth][n][2])
struct DelayRingRef {
    float4 *obs;
    int32_t *frame;
    uint32_t *misc;
    size_t n;
    __device__ __forceinline__ DelayEntry load(int s, size_t i) const {
        const size_t k = (size_t)s * n + i;
        DelayEntry v;
        v.a = obs[2 * k]; v.b = obs[2 * k + 1]; v.frame = frame[k]; v.misc = misc[k];
        return v;
    }
    __device__ __forceinline__ void store(int s, size_t i, const DelayEntry &v) const {
        const size_t k = (size_t)s * n + i;
        obs[2 * k] = v.a; obs[2 * k + 1] = v.b; frame[k] = v.frame; misc[k] = v.misc;
    }
};

// One step of battle i's queue at ring position pos.  `now` is the state the step produced, `oldest` the entry of slot
// (pos + 1) % depth and `newest_frame` the frame of slot (pos + depth - 1) % depth, both read by the caller BEFORE the
// call -- this function writes neither slot before it is done with them, so a caller can issue the loads early.
//   - a battle that did not advance (held back by a step mask, or over and waiting for its reset: its frame counter still
//     is the newest entry's) keeps its queue; the ring position is shared, so its slots move along with it.  Returns
//     false: it emits nothing new (its last emitted state stands);
//   - a battle the step just reset (frame -1) fills every slot with its first state and emits it;
//   - any other battle writes `now` into slot pos and emits `oldest`.
__device__ __forceinline__ bool delay_ring_push(const DelayRingRef &r, size_t i, int depth, int pos, bool held_back,
                                                const DelayEntry &now, const DelayEntry &oldest, int32_t newest_frame,
                                                DelayEntry &emit) {
    if (held_back || (now.frame != -1 && now.frame == newest_frame)) {
        DelayEntry carry = r.load(depth - 1, i);
        for (int s = 0; s < depth; s++) {
            const DelayEntry t = r.load(s, i);
            r.store(s, i, carry);
            carry = t;
        }
        return false;
    }
    if (now.frame == -1) {
        for (int s = 0; s < depth; s++) r.store(s, i, now);
        emit = now;
    } else {
        r.store(pos, i, now);
        emit = oldest;
    }
    return true;
}

}  // namespace fgk
#endif
