// Episode log of the evaluation path (taco_env_attach_episode_log, include/taco_b200.h): one streaming launch after each step
// reads the step's results and the state planes, accumulates per-env running quantities in two SoA float4 planes of its own and
// appends one TacoEpisode record per finished episode.  The step kernel is not touched; an env without a log never launches this.
//
// Accumulator planes (n_pad float4 each):
//   acc[0] = (ret, sum of |pos - target pos|, sum of |linvel|, max tilt)
//   acc[1] = (max |angvel|, roll_continuous after the episode's first step, live flag, 0)
// live = 1: the log saw the running episode start (taco_env_attach_episode_log: the env had reset_buf != 0; afterwards: every
// episode after one the log saw end), so only whole episodes are recorded.
#pragma once
#include <stdint.h>

#include "../../include/taco_b200.h"
#include "step_params.h"

namespace taco {

static_assert(sizeof(TacoEpisode) == 48 && sizeof(TacoEpisode) % 16 == 0, "TacoEpisode is written as three 16-byte words");

// attach initialisation (also after taco_env_reset_all / _import_state / _checkpoint_load): clear the accumulators; an env
// starts a whole episode with its next step exactly when reset_buf != 0 now (lazy reset, DESIGN.md section 3.4)
__global__ void episode_log_init_kernel(const StepParams p, float4* acc0, float4* acc1) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_pad) return;
    const bool fresh = i < p.n && p.reset_buf[i] != 0;
    acc0[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    acc1[i] = make_float4(0.f, 0.f, fresh ? 1.f : 0.f, 0.f);
}

// |(x, y, z)| rounded op by op (no FMA contraction), so that a float32 replay on the host reproduces it bit for bit
__device__ __forceinline__ float norm3_rn(float x, float y, float z) {
    return sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)));
}

// one thread per env.  step = the RL step index of the step just taken (absolute, or the offset to *step_base in graph mode).
// Appending: one atomicAdd on the counter per warp, each recording lane writes at base + its ballot prefix; slots at or past
// `capacity` are dropped but counted, so the record order is unspecified within a launch and count - capacity are dropped.
__global__ void __launch_bounds__(256) episode_log_update_kernel(const StepParams p, float4* acc0, float4* acc1, TacoEpisode* rec,
                                                                 unsigned long long* count, unsigned long long capacity, uint32_t step,
                                                                 const uint32_t* step_base) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool emit = false;
    int4 w0 = make_int4(0, 0, 0, 0), w1 = w0, w2 = w0;
    if (i < p.n) {
        const float4 s0 = p.S[0][i], s1 = p.S[1][i], s2 = p.S[2][i], s3 = p.S[3][i];
        const float rew = p.rew[i];
        const bool done = p.reset_buf[i] != 0;
        const int progress = p.progress[i];
        const long long gid = p.env_offset + i;
        int task = p.task_mode;
        if (task == TACO_TASK_MIX) task = gid < p.mix_n1 ? TACO_TASK_POS : (gid < p.mix_n2 ? TACO_TASK_ROTATE : TACO_TASK_FLIP);
        float4 a0 = acc0[i], a1 = acc1[i];
        // export_state layout: pos s0.xyz, quat xyzw = (s0.w, s1.x, s1.y, s1.z), linvel (s1.w, s2.x, s2.y), angvel (s2.z, s2.w, s3.x),
        // target pos s3.yzw, roll_continuous s4.w
        const float pe = norm3_rn(__fsub_rn(s0.x, s3.y), __fsub_rn(s0.y, s3.z), __fsub_rn(s0.z, s3.w));
        const float speed = norm3_rn(s1.w, s2.x, s2.y);
        const float angv = norm3_rn(s2.z, s2.w, s3.x);
        const float cz = __fsub_rn(1.0f, __fmul_rn(2.0f, __fadd_rn(__fmul_rn(s0.w, s0.w), __fmul_rn(s1.x, s1.x))));
        const float tilt = acosf(fminf(fmaxf(cz, -1.0f), 1.0f));
        a0.x = __fadd_rn(a0.x, rew);                            // the step kernel's ep_ret += rew
        a0.y = __fadd_rn(a0.y, pe);
        a0.z = __fadd_rn(a0.z, speed);
        a0.w = fmaxf(a0.w, tilt);
        a1.x = fmaxf(a1.x, angv);
        float roll = 0.f;
        if (task == TACO_TASK_FLIP) {
            roll = p.S[4][i].w;
            if (progress == 1) a1.y = roll;                     // after the episode's first step
        }
        if (done) {
            emit = a1.z != 0.f;
            if (emit) {
                const float len = (float)progress;
                const uint32_t end = step + (step_base ? __ldg(step_base) : 0u);
                w0 = make_int4((int)(uint32_t)(unsigned long long)gid, (int)(uint32_t)((unsigned long long)gid >> 32), (int)end, progress);
                w1 = make_int4((int)((uint32_t)task | ((uint32_t)p.time_outs[i] << 16)), __float_as_int(a0.x),
                               __float_as_int(__fdiv_rn(a0.y, len)), __float_as_int(pe));
                w2 = make_int4(__float_as_int(a0.w), __float_as_int(__fdiv_rn(a0.z, len)), __float_as_int(a1.x),
                               __float_as_int(task == TACO_TASK_FLIP ? __fsub_rn(roll, a1.y) : 0.f));
            }
            a0 = make_float4(0.f, 0.f, 0.f, 0.f);               // the next episode starts with the next step: the log sees it whole
            a1 = make_float4(0.f, 0.f, 1.f, 0.f);
        }
        acc0[i] = a0;
        acc1[i] = a1;
    }
    const uint32_t m = __ballot_sync(0xffffffffu, emit);
    if (m == 0u) return;
    const int leader = __ffs(m) - 1;
    unsigned long long base = 0ull;
    if (lane == leader) base = atomicAdd(count, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (emit) {
        const unsigned long long slot = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
        if (slot < capacity) {
            int4* o = reinterpret_cast<int4*>(rec + slot);
            o[0] = w0; o[1] = w1; o[2] = w2;
        }
    }
}

}  // namespace taco
