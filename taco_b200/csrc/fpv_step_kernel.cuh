// Fused FPV environment step: one thread = one env, whole RL step in registers.
//
// Replaces, for the fpv_asymmetry tasks of yinzikang/taco (paths under IsaacGymEnvs/isaacgymenvs/):
//   VecTask.step                      tasks/base/vec_task_asymmetry.py:290-334
//   FpvBase.pre/mid/post_physics_step tasks/fpv_asymmetry.py:317-388
//   refresh_state                     tasks/fpv_asymmetry.py:334-360
//   angvel_control.compute            tasks/control/angvel_control.py:67-88
//   control_allocator / sim_process   tasks/control/fpv_dynamics.py:35-56
//   Battery_Dynamics.sim_process      tasks/control/battery_dynamics.py:47-75
//   RotorDynamics / AeroDynamics      tasks/control/thrust_dynamics.py:52-104,173-199
//   gym.simulate (PhysX, closed)      -> our documented free-body integrator (DESIGN.md, oracle/rigid_body.py)
//   compute_observation_state         tasks/fpv_asymmetry.py:390-421 (+ :711-714,:766-771,:830-838,:929-946)
//   compute_{pos,rotating,flip}_reward tasks/control/task_reward.py:20-143
//   reset_idx and friends             tasks/fpv_asymmetry.py:475-603,:725-759,:783-821,:850-917,:981-1112
//
// This header is compiled twice: fpv_step_fast.cu (FMA contraction on) and
// fpv_step_strict.cu (-fmad=false: every multiply/add rounds separately, like eager torch).
#pragma once
#include <climits>
#include <type_traits>
#include "fpv_math.cuh"
#include "philox.cuh"
#include "step_params.h"
#include "launch_count.h"
#include "../../include/taco_b200.h"

#ifndef TACO_MIN_BLOCKS
#define TACO_MIN_BLOCKS 6     // resident CTAs per SM the register allocation targets: 80 regs, 24 warps/SM (measured best of 4/5/6/7/8)
#endif
#ifndef TACO_MIN_BLOCKS_DR
#define TACO_MIN_BLOCKS_DR 5  // the DR variants keep 14 more per-env model parameters live through the control loop: 96 regs, 20 warps/SM (mix + DR: -2 %, profiles/ab_r02w.txt)
#endif
#ifndef TACO_VARIANT
#error "define TACO_VARIANT (fast / strict) before including fpv_step_kernel.cuh"
#endif

// difficulty-dependent scalars: by-value kernel parameters, or -- in the kernel variants launched in graph mode (DEVDIFF) -- their
// device copy (step_params.h), so that launches captured in a CUDA graph follow taco_env_set_difficulty
#define TACO_DIFF(field, idx) (DEVDIFF ? __ldg(p.diff_dev + (idx)) : p.field)

namespace taco {
namespace TACO_VARIANT {   // distinct symbols per translation unit: the two builds must not be merged by the linker

__device__ constexpr float kTurns[8] = {-3.f, -2.f, -1.f, 0.f, 0.f, 1.f, 2.f, 3.f};   // fpv_asymmetry.py:892-901

__device__ __forceinline__ float4 ldg4(const float4* p) { return __ldg(p); }
// refresh_state's roll unwrap (fpv_asymmetry.py:334-360): the continuous roll follows the roll angle, a step over 1 rad is a wrap
__device__ __forceinline__ void unwrap_roll(const Q4& q, float& roll_old, float& roll_cont) {
    const float roll = roll_of(q);
    float dl = roll - roll_old;
    if (dl > 1.0f) dl = dl - kTwoPi;
    if (dl < -1.0f) dl = dl + kTwoPi;
    roll_cont += dl;
    roll_old = roll;
}

// The history writers.  A CTA writes its 128 rows of an (N, L, 26) history buffer: frames 1..L-1 of the previous buffer shifted
// down by one (coalesced 64-bit copies: a row is 13*L float2, the shift is 13 float2) and the newest frame from shared memory.
// nv = valid rows of this CTA (only the last CTA of a shard whose env count is not a multiple of 128 has nv < 128): rows >= nv
// are never touched, so the buffers may be exactly (num_envs, L, 26) -- e.g. a slot of a caller-owned rollout ring.

// kept part, flat walk over the CTA's keep2 * rows kept float2 (every request 256 contiguous bytes, 13 loads in flight per
// thread): out2 row e, column j <- in2 row e, column 13 + j, for j < keep2 (> 0) and rows of row2 float2
__device__ __forceinline__ void copy_kept_flat(const float2* __restrict__ in2, float2* __restrict__ out2, int row2, int keep2,
                                               int rows, int tid) {
    const int total = rows * keep2;
    constexpr int U = 13;                                       // loads in flight per thread
    for (int k0 = tid; k0 < total; k0 += kBlock * U) {
        float2 v[U];
        int dst[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int k = k0 + u * kBlock;
            const int e = k / keep2, j = k - e * keep2;
            dst[u] = e * row2 + j;
            v[u] = (k < total) ? __ldg(in2 + dst[u] + 13) : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (k0 + u * kBlock < total) out2[dst[u]] = v[u];
    }
}
// newest frame, generic walk: 13 float2 of each of the rows (all 128 if FULL, else nv) at column new2 of rows of row2 float2
template <bool FULL>
__device__ __forceinline__ void write_newest_flat(float2* out2, const float* frames, int row2, int new2, int tid, int nv) {
#pragma unroll
    for (int u = 0; u < 13; ++u) {
        const int k = tid + u * kBlock;
        const int e = k / 13, j = k - e * 13;
        const float* fr = frames + e * kFramePad + 2 * j;
        if (FULL || e < nv) out2[e * row2 + new2 + j] = make_float2(fr[0], fr[1]);
    }
}
// Forms for a full CTA and a compile-time L, with no index arithmetic in the instruction stream: warp w owns the 32 consecutive
// rows [32 w, 32 w + 32) and its lanes run ALONG a row, so every load / store is `base + immediate` (the row and column offsets are
// compile-time constants of the unrolled loops).  Same bytes touched as the flat walk, a third of its instructions (8 per element
// there: division by keep2, address, bounds predicate).
// kept part of rows [row0, row0 + NR) of the CTA by ONE warp (lanes along the row)
template <int LC, int NR>
__device__ __forceinline__ void copy_kept_rows(const float* __restrict__ in, float* __restrict__ out, size_t blk_env0, int row0, int lane) {
    constexpr int row2 = 13 * LC, keep2 = 13 * (LC - 1);
    constexpr int NJ = (keep2 + 31) / 32;                       // column chunks of 32 lanes per row
    constexpr int NJ1 = NJ > 0 ? NJ : 1;
    constexpr int EB = NJ1 <= 2 ? 8 : (NJ1 <= 4 ? 4 : 2);       // rows per batch: <= 16 loads in flight per thread
    static_assert(NR % EB == 0, "rows per warp must be a multiple of the batch");
    if (keep2 > 0) {
        const float2* src = reinterpret_cast<const float2*>(in) + (blk_env0 + row0) * row2 + 13 + lane;
        float2* dst = reinterpret_cast<float2*>(out) + (blk_env0 + row0) * row2 + lane;
#pragma unroll (NR <= 32 ? NR / EB : 4)
        for (int e0 = 0; e0 < NR; e0 += EB) {
            float2 v[EB][NJ1];
#pragma unroll
            for (int e = 0; e < EB; ++e)
#pragma unroll
                for (int c = 0; c < NJ; ++c)
                    if ((c + 1) * 32 <= keep2 || c * 32 + lane < keep2) v[e][c] = __ldg(src + (e0 + e) * row2 + c * 32);
#pragma unroll
            for (int e = 0; e < EB; ++e)
#pragma unroll
                for (int c = 0; c < NJ; ++c)
                    if ((c + 1) * 32 <= keep2 || c * 32 + lane < keep2) dst[(e0 + e) * row2 + c * 32] = v[e][c];
        }
    }
}
// newest frame of the 32 rows [32 w, 32 w + 32) by warp w: two rows per store instruction (13 float2 each, lanes 26..31 idle)
template <int LC>
__device__ __forceinline__ void write_newest_rows(float* __restrict__ out, const float* frames, size_t blk_env0, int tid) {
    constexpr int row2 = 13 * LC, keep2 = 13 * (LC - 1);
    const int w = tid >> 5, lane = tid & 31;
    if (lane < 26) {
        const int sub = lane >= 13 ? 1 : 0, j = lane - 13 * sub;
        const float* fr = frames + (32 * w + sub) * kFramePad + 2 * j;
        float2* d = reinterpret_cast<float2*>(out) + (blk_env0 + 32 * w + sub) * row2 + keep2 + j;
#pragma unroll
        for (int e = 0; e < 32; e += 2) d[e * row2] = make_float2(fr[e * kFramePad], fr[e * kFramePad + 1]);
    }
}
// the flat walks for rows of L frames (FULL: nv == 128)
template <int LC, bool FULL>
__device__ __forceinline__ void write_rows_flat(const float* __restrict__ in, float* __restrict__ out, const float* frames,
                                                int L_rt, size_t blk_env0, int tid, int nv) {
    const int L = LC ? LC : L_rt;
    const int row2 = 13 * L, keep2 = 13 * (L - 1);
    const float2* in2 = reinterpret_cast<const float2*>(in) + blk_env0 * row2;
    float2* out2 = reinterpret_cast<float2*>(out) + blk_env0 * row2;
    if (keep2 > 0) copy_kept_flat(in2, out2, row2, keep2, FULL ? kBlock : nv, tid);
    write_newest_flat<FULL>(out2, frames, row2, keep2, tid, nv);
}
// LC = compile-time L (the README shapes L = 5 / L = 1), 0 = runtime L.  A full CTA with a compile-time L writes the newest frame
// with write_newest_rows and the kept part in one of two forms, chosen per kernel variant by measurement (tools/step_ab.py,
// profiles/ab_r02ab.txt / ab_r02ac.txt):
//   FLAT = false  lanes along the rows (copy_kept_rows): a third of the instructions, but the second column chunk of a 52-element row
//                 fills 20 of 32 lanes -- best for the DR variants (96 registers, 5 CTAs per SM: mix + DR 0.719 against 0.731 ms)
//   FLAT = true   the flat walk (copy_kept_flat): best for the variants at 80 registers / 6 CTAs per SM (flip: 0.560 against
//                 0.584 ms over the first synchronised steps, 0.602 against 0.607 in steady state)
template <int LC, bool FLAT>
__device__ __forceinline__ void write_rows(const float* __restrict__ in, float* __restrict__ out, const float* frames,
                                           int L_rt, size_t blk_env0, int tid, int nv) {
    if (nv == kBlock) {                                                                        // every CTA but (at most) the last
        if constexpr (LC > 0) {
            if constexpr (!FLAT) copy_kept_rows<LC, 32>(in, out, blk_env0, 32 * (tid >> 5), tid & 31);
            else if constexpr (LC > 1)
                copy_kept_flat(reinterpret_cast<const float2*>(in) + blk_env0 * (13 * LC), reinterpret_cast<float2*>(out) + blk_env0 * (13 * LC),
                               13 * LC, 13 * (LC - 1), kBlock, tid);
            write_newest_rows<LC>(out, frames, blk_env0, tid);
        } else write_rows_flat<LC, true>(in, out, frames, L_rt, blk_env0, tid, nv);
    } else write_rows_flat<LC, false>(in, out, frames, L_rt, blk_env0, tid, nv);
}

// The env-owned state history (no rollout ring attached): each env's row of the strip holds strip_frames = L + K - 1 frames, and
// after the step that ran at step index t the env's window is the L frames from offset (t + 1) mod K.  A step writes only the newest
// frame, at the end of the new window: 104 B per env instead of re-reading 4 frames and rewriting 5 (936 B).  The step that wraps the
// offset to 0 first moves the L - 1 kept frames (K .. K + L - 2) to the start of the row (0 .. L - 2) -- the "rebase", once per K
// steps.  K >= L, so the moved frames, their destination and the newest frame (L - 1) are disjoint: no ordering inside the CTA.
// The rebase is the flat walk of copy_kept_flat with another source column, but it reads and writes one buffer: it keeps a loop of
// its own with plain loads rather than copy_kept_flat's __ldg from a second, read-only buffer.
__device__ __forceinline__ void write_strip(const StepParams& p, const float* frames, size_t blk_env0, int tid, int nv) {
    const uint32_t t = p.step_index + (p.step_base ? __ldg(p.step_base) : 0u);
    const int L = p.len_states, q = (int)((t + 1u) % (uint32_t)p.strip_period);
    const int row2 = 13 * p.strip_frames;
    float2* s2 = reinterpret_cast<float2*>(p.states_strip) + blk_env0 * row2;
    if (q == 0 && L > 1) {
        const int keep2 = 13 * (L - 1), src2 = 13 * p.strip_period, total = nv * keep2;
        constexpr int U = 13;                                   // loads in flight per thread
        for (int k0 = tid; k0 < total; k0 += kBlock * U) {
            float2 v[U];
            int dst[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int k = k0 + u * kBlock;
                const int e = k / keep2, j = k - e * keep2;
                dst[u] = e * row2 + j;
                v[u] = (k < total) ? s2[dst[u] + src2] : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (k0 + u * kBlock < total) s2[dst[u]] = v[u];
        }
    }
    write_newest_flat<false>(s2, frames, row2, 13 * (q + L - 1), tid, nv);
}

// TASK: task_mode (mix = per-env task from the global env id).  DR: per-env randomised model parameters live in the
// D planes; when false the rotor polynomial / aero coefficients fold into instruction immediates.
// SUB: physics sub-steps per simulate call (1 / 2 unrolled; 0 = runtime p.substeps).
// DEVDIFF: graph-mode variant (difficulty scalars from device memory; costs two spilled registers, so eager launches do not use it).
// CW: extra warps of the CTA (threads >= 128) that do nothing but the kept-history copy into the slot of an attached rollout ring, from
// the first cycle of the CTA -- the copy depends on nothing the step computes (the env-owned strip, write_strip, has no such copy).  CW = 4 for launches of at most one CTA per SM (the 4096-env scale of
// the reference: one env's instruction stream is latency-bound there, and the copy's four load -> store round trips were a third of
// the kernel's time when they ran after it: 14.4 -> 13.1 us); CW = 0 otherwise (the copy warps' registers cost resident compute
// warps: one copy warp per CTA at 2 Mi envs measured 0.636 against 0.609 ms, profiles/ab_r02y.txt).
// HB: variant for the mapped host-buffer step (taco_env_step_host with pinned buffers): the one-byte results (time-outs, compact
// flags) leave as one 128-byte run per CTA.  A separate instantiation, so that the device-resident step carries none of it
// (as run-time branches it cost that step 1 % over the first synchronised steps, profiles/ab_r02aj.txt).
template <int TASK, bool DR, int SUB, bool DEVDIFF = false, int CW = 0, bool HB = false>
__global__ void __launch_bounds__(kBlock + 32 * CW, CW ? 1 : (DR ? TACO_MIN_BLOCKS_DR : TACO_MIN_BLOCKS)) fpv_step_kernel(const StepParams p) {
    __shared__ __align__(16) float s_clean[kBlock * kFramePad];
    __shared__ __align__(16) float s_noisy[kBlock * kFramePad];
    __shared__ double s_stats[kNumStats];
    __shared__ __align__(16) uint8_t s_hostb[HB ? kBlock : 16];  // byte-wide host results of the CTA (mapped host-buffer step)

    const int tid = threadIdx.x;
    const int blk = blockIdx.x + p.block0;                      // a launch covers CTAs [block0, block0 + gridDim.x): chunked host pipeline
    const int i = blk * kBlock + tid;
    const bool is_copy = CW > 0 && tid >= kBlock;              // copy warps: no env of their own
    const bool valid = !is_copy && i < p.n;
    // split copy: else the compute warps copy after the step, as with CW = 0 (where nothing of this is kept live across the step)
    const bool split_copy = CW > 0 && !p.states_strip && min(kBlock, p.n - blk * kBlock) == kBlock && p.len_states == 5;
    const uint32_t flags = p.flags;
    const bool obs_noise = (flags & TACO_F_OBSERVATION_NOISE) != 0;
    if (tid < kNumStats) s_stats[tid] = 0.0;
    __syncthreads();

    if (CW > 0 && is_copy) {
        if (split_copy) copy_kept_rows<5, kBlock / (CW ? CW : 1)>(p.states_in, p.states_out, (size_t)blk * kBlock, ((tid - kBlock) >> 5) * (kBlock / (CW ? CW : 1)), tid & 31);
        return;                                                 // (the compute warps meet at a named barrier of their own)
    }

    float st_rew = 0.f, st_done = 0.f, st_tout = 0.f, st_epret = 0.f, st_eplen = 0.f, st_nonfin = 0.f, st_ovf = 0.f;
    float* fc = s_clean + tid * kFramePad;
    float* fn = s_noisy + tid * kFramePad;

    const uint32_t vmask = __ballot_sync(0xffffffffu, valid);  // only the last CTA of a ragged shard has partial warps

    if (valid) {
        // ------------------------------------------------------------------ load
        const float4 s0 = p.S[0][i], s1 = p.S[1][i], s2 = p.S[2][i], s3 = p.S[3][i];
        const float4 s4 = p.S[4][i], s5 = p.S[5][i], s6 = p.S[6][i], s7 = p.S[7][i];
        float4 act = ldg4(p.actions + i);
        int progress = p.progress[i];
        uint32_t qm = p.qmeta[i];
        const bool R = p.reset_buf[i] != 0;                    // latched for the whole RL step (fpv_asymmetry.py:318)
        float poly[5], aero[5], lag[4];
        if (DR) {
            const float4 d0 = p.D[0][i], d1 = p.D[1][i], d2 = p.D[2][i], d3 = p.D[3][i];
            poly[0] = d0.x; poly[1] = d0.y; poly[2] = d0.z; poly[3] = d0.w; poly[4] = d1.x;
            aero[0] = d1.y; aero[1] = d1.z; aero[2] = d1.w; aero[3] = d2.x; aero[4] = d2.y;
            lag[0] = d3.x; lag[1] = d3.y; lag[2] = d3.z; lag[3] = d3.w;
        } else {
#pragma unroll
            for (int j = 0; j < 5; ++j) { poly[j] = kPolyNom[j]; aero[j] = kAeroNom[j]; }
#pragma unroll
            for (int j = 0; j < 4; ++j) lag[j] = p.lag_gain_fixed;
        }
        V3 pos = v3(s0.x, s0.y, s0.z);
        Q4 q; q.x = s0.w; q.y = s1.x; q.z = s1.y; q.w = s1.z;
        V3 vel = v3(s1.w, s2.x, s2.y);
        V3 wld = v3(s2.z, s2.w, s3.x);                          // angular velocity, world frame
        V3 tpos = v3(s3.y, s3.z, s3.w);
        Q4 tq; tq.x = 0.f; tq.y = 0.f; tq.z = s4.x; tq.w = s4.y; // target attitude is yaw-only (fpv_asymmetry.py:539-546)
        float roll_old = s4.z, roll_cont = s4.w;
        float om[4] = {s5.x, s5.y, s5.z, s5.w};
        float pe[3] = {s6.x, s6.y, s6.z};
        float cmd = s6.w;                                       // rotate: speed command; flip: flip_radian
        float bu1 = s7.x, bec = s7.y, bt = s7.z, ep_ret = s7.w;

        const float ca = p.clip_actions;                        // vec_task_asymmetry.py:304
        act.x = clampf(act.x, -ca, ca); act.y = clampf(act.y, -ca, ca);
        act.z = clampf(act.z, -ca, ca); act.w = clampf(act.w, -ca, ca);

        const uint32_t g = (uint32_t)(p.env_offset + i);        // global env id = Philox counter word 0
        const uint32_t k0 = p.seed_lo, k1 = p.seed_hi, t_rl = p.step_index + (p.step_base ? __ldg(p.step_base) : 0u);
        int task = TASK;
        const bool is_mix = (TASK == TACO_TASK_MIX);
        if (is_mix) {
            const long long gg = p.env_offset + i;
            task = gg < p.mix_n1 ? TACO_TASK_POS : (gg < p.mix_n2 ? TACO_TASK_ROTATE : TACO_TASK_FLIP);
        }
        const bool at500 = (progress == 500);                   // fpv_asymmetry.py:152,597 (before counters clear)

        // pending-action runs live in a ring indexed by the RL step of the LAUNCH (slot = step_index & 15, the same for
        // every env of the launch -> coalesced planes however desynchronised the episodes are); an env's live runs are
        // the last q_n slots, so the head is implied
        const uint32_t tslot = t_rl & 15u;
        uint32_t q_n = qm_runs(qm);
        int q_len = (int)qm_len(qm);
        uint32_t q_ovf = qm_ovf(qm);

        // ------------------------------------------------------------------ reset draws, generated by the WARP for its resetting envs
        // In steady state ~1 % of the envs reset per step, i.e. ~29 % of the warps hold one or two resetting lanes, and such a warp
        // used to run the whole draw sequence (6 .. 11 Philox blocks, ~90 instructions each) for those lanes alone.  Here the lanes
        // of the warp compute the blocks side by side instead -- lanes 0..15 the blocks of the first resetting env, lanes 16..31 those
        // of the second (block c = lane & 15: reset stream blocks 0..9, block 10 = the command stream's block 0) -- and post them in a
        // mailbox in the warp's own rows of s_clean (not written before the frame at the end of the step; no other warp touches
        // them before the CTA barrier).  The resetting lane reads the blocks where the sequential code computed them: same counters,
        // same keys, same words.  Warps with 3+ resetting lanes (the first step, synchronised time-outs) and partial warps keep the
        // per-lane path.
        bool coop = false;
        const uint4* mbox = reinterpret_cast<const uint4*>(s_clean + (tid & ~31) * kFramePad);
        if (vmask == 0xffffffffu) {
            const uint32_t rmask = __ballot_sync(0xffffffffu, R);
            const int nres = __popc(rmask);
            if (nres == 1 || nres == 2) {
                const int lane = tid & 31, first = __ffs(rmask) - 1, last = 31 - __clz(rmask);
                const uint32_t gs = __shfl_sync(0xffffffffu, g, (lane & 16) ? last : first);
                const uint32_t c = (uint32_t)(lane & 15);
                if (c <= 10u) {
                    const uint4 blk4 = philox4x32_10(gs, t_rl, c < 10u ? c : 0u, c < 10u ? (uint32_t)STREAM_RESET : (uint32_t)STREAM_COMMAND, k0, k1);
                    const_cast<uint4*>(mbox)[lane] = blk4;
                }
                __syncwarp();
                coop = true;
                if (nres == 2 && lane == last) mbox += 16;
            }
        }
        auto reset_block = [&](uint32_t c) -> uint4 { return coop ? mbox[c] : philox4x32_10(g, t_rl, c, STREAM_RESET, k0, k1); };

        // ------------------------------------------------------------------ lazy reset (fpv_asymmetry.py:475-517)
        if (R) {
            const float d = TACO_DIFF(difficulty, 0);          // read where it is used: no register held across the step
            const uint4 b0 = reset_block(0), b1 = reset_block(1), b2 = reset_block(2), b3 = reset_block(3), b4 = reset_block(4);
            const bool flip_env = (task == TACO_TASK_FLIP);
            // copter position (:730-737, :788-793, :855-861, :993-1036)
            if (flags & TACO_F_RANDOM_COPTER_POS) {
                if (flip_env && !is_mix) {
                    pos.x = rr(TACO_DIFF(flip_xy_rng, 1), TACO_DIFF(flip_xy_lo, 2), u01(b0.x));
                    pos.y = rr(TACO_DIFF(flip_xy_rng, 1), TACO_DIFF(flip_xy_lo, 2), u01(b0.y));
                    pos.z = 3.0f + d * rr(4.0f, -2.0f, u01(b0.z));
                } else {
                    pos.x = rr(4.0f, -2.0f, u01(b0.x));
                    pos.y = rr(4.0f, -2.0f, u01(b0.y));
                    pos.z = 2.5f + rr(4.0f, -2.0f, u01(b0.z));
                }
            } else {
                if (is_mix || task == TACO_TASK_POS) { pos.x = 0.f; pos.y = 0.f; pos.z = 2.5f; }
                else {
                    pos.x = rr(1.0f, -0.5f, u01(b0.x));
                    pos.y = rr(1.0f, -0.5f, u01(b0.y));
                    pos.z = flip_env ? 3.0f : 2.5f;
                }
            }
            // attitude: rand_quat feeds its "pitch" draw into the ROLL slot (:698-704); flip is roll-only (:864,:1038)
            if (flags & TACO_F_RANDOM_COPTER_QUAT) {
                const float ea = rr(kTwoPi, -kPi, u01(b1.x));
                if (flip_env) q = quat_from_euler(ea, 0.0f, 0.0f);
                else q = quat_from_euler(ea, rr(kTwoPi, -kPi, u01(b1.y)), rr(kTwoPi, -kPi, u01(b1.z)));
            } else { q.x = 0.f; q.y = 0.f; q.z = 0.f; q.w = 1.f; }
            // velocities (:745-750, :869-878, :1042-1050): flip keeps stale w_y, w_z
            if (flags & TACO_F_RANDOM_COPTER_VEL) {
                if (flip_env) {
                    vel = v3(rr(TACO_DIFF(flip_lin_rng, 3), TACO_DIFF(flip_lin_lo, 4), u01(b2.x)), rr(TACO_DIFF(flip_lin_rng, 3), TACO_DIFF(flip_lin_lo, 4), u01(b2.y)),
                             rr(TACO_DIFF(flip_lin_rng, 3), TACO_DIFF(flip_lin_lo, 4), u01(b2.z)));
                    wld.x = 10.0f * ((b0.w >> 31) ? 1.0f : -1.0f);
                } else {
                    vel = v3(3.0f * rr(2.0f, -1.0f, u01(b2.x)), 3.0f * rr(2.0f, -1.0f, u01(b2.y)), 3.0f * rr(2.0f, -1.0f, u01(b2.z)));
                    wld = v3(3.0f * rr(2.0f, -1.0f, u01(b3.x)), 3.0f * rr(2.0f, -1.0f, u01(b3.y)), 3.0f * rr(2.0f, -1.0f, u01(b3.z)));
                }
            } else {
                vel = v3(0.f, 0.f, 0.f);
                if (!(flip_env && !is_mix)) wld = v3(0.f, 0.f, 0.f);   // FpvFlip leaves angvel untouched (:877-878)
            }
            roll_old = roll_cont = roll_of(q);                   // :752-754
            // controllers (:550-558)
            pe[0] = pe[1] = pe[2] = 0.f;
            bu1 = 0.f; bt = 0.f;
            bec = (flags & TACO_F_RANDOM_VOLTAGE) ? rr(2.2f, 0.0f, u01(b2.w)) : 0.f;
            if (DR) {
                const uint4 b5 = reset_block(5), b6 = reset_block(6), b7 = reset_block(7), b8 = reset_block(8);
                if (flags & TACO_F_RANDOM_ROTORDYNAMIC_COE) {     // thrust_dynamics.py:117-122
                    poly[0] = kPolyNom[0] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b5.x));
                    poly[1] = kPolyNom[1] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b5.y));
                    poly[2] = kPolyNom[2] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b5.z));
                    poly[3] = kPolyNom[3] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b5.w));
                    poly[4] = kPolyNom[4] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b6.x));
                } else {
#pragma unroll
                    for (int j = 0; j < 5; ++j) poly[j] = kPolyNom[j];
                }
                if ((flags & TACO_F_ROTOR_RESPONSE) && (flags & TACO_F_RANDOM_ROTOR_RESPONSE)) {   // thrust_dynamics.py:134-137
                    lag[0] = (1.0f / rr(p.tau_rng, p.tau_lo, u01(b8.x))) * 0.001f;   // python scalar / tensor = tensor.reciprocal() * scalar
                    lag[1] = (1.0f / rr(p.tau_rng, p.tau_lo, u01(b8.y))) * 0.001f;
                    lag[2] = (1.0f / rr(p.tau_rng, p.tau_lo, u01(b8.z))) * 0.001f;
                    lag[3] = (1.0f / rr(p.tau_rng, p.tau_lo, u01(b8.w))) * 0.001f;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) lag[j] = p.lag_gain_fixed;
                }
                if (flags & TACO_F_RANDOM_AERODYNAMIC_COE) {      // thrust_dynamics.py:201-210
                    aero[0] = kAeroNom[0] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b6.y));
                    aero[1] = kAeroNom[1] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b6.z));
                    aero[2] = kAeroNom[2] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b6.w));
                    aero[3] = kAeroNom[3] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b7.x));
                    aero[4] = kAeroNom[4] * rr(TACO_DIFF(dr_rng, 5), TACO_DIFF(dr_lo, 6), u01(b7.y));
                } else {
#pragma unroll
                    for (int j = 0; j < 5; ++j) aero[j] = kAeroNom[j];
                }
                p.D[0][i] = make_float4(poly[0], poly[1], poly[2], poly[3]);
                p.D[1][i] = make_float4(poly[4], aero[0], aero[1], aero[2]);
                p.D[2][i] = make_float4(aero[3], aero[4], 0.f, 0.f);
                p.D[3][i] = make_float4(lag[0], lag[1], lag[2], lag[3]);
            }
            if (flags & TACO_F_RANDOM_ROTOR_SPEED) {              // thrust_dynamics.py:143-146
                const uint4 b9 = reset_block(9);
                om[0] = rr(400.0f, 0.0f, u01(b9.x)); om[1] = rr(400.0f, 0.0f, u01(b9.y));
                om[2] = rr(400.0f, 0.0f, u01(b9.z)); om[3] = rr(400.0f, 0.0f, u01(b9.w));
            } else { om[0] = om[1] = om[2] = om[3] = 0.f; }
            // pending-action queue (:574-578): `delay` slots of zero action
            q_len = p.delay_time;
            if (flags & TACO_F_RAMDOM_DELAY_TIME) q_len = max(p.delay_time - round_normal(b1.w, 3), 0);
            q_n = 0; q_ovf = 0;
            if (q_len > 0) {
                const uint32_t zslot = (tslot + 15u) & 15u;
                p.qact[(size_t)zslot * p.n_pad + i] = make_float4(0.f, 0.f, 0.f, 0.f);
                p.qend[(size_t)zslot * p.n_pad + i] = (uint16_t)q_len;
                q_n = 1;
            }
            // target (:523-548)
            if (flags & TACO_F_RANDOM_TARGET_POS) {
                tpos.x = d * rr(4.0f, -2.0f, u01(b4.x));
                tpos.y = d * rr(4.0f, -2.0f, u01(b4.y));
                tpos.z = 3.0f + d * rr(4.0f, -2.0f, u01(b4.z));
            } else tpos = v3(0.f, 0.f, 3.f);
            const float yaw = (flags & TACO_F_RANDOM_TARGET_YAW) ? rr(kTwoPi, -kPi, u01(b3.w)) : 0.0f;
            sincos_draw(yaw * 0.5f, &tq.z, &tq.w);
        }
        // ------------------------------------------------------------------ command (:587-603, :758, :814-821, :886-917, :1058-1112)
        // (the command stream's block is drawn only where a word of it is consumed: rotate with random_command, flip at progress 500)
        if (R || at500) {
            if (task == TACO_TASK_POS) cmd = 0.f;
            else if (task == TACO_TASK_ROTATE) {
                if (flags & TACO_F_RANDOM_COMMAND) {
                    const uint4 cb = (coop && R) ? mbox[10] : philox4x32_10(g, t_rl, 0, STREAM_COMMAND, k0, k1);
                    cmd = rr(12.0f, -6.0f, u01(cb.y));
                } else cmd = 1.0f;
            } else if (R) cmd = (wld.x > 5.0f) ? kTwoPi : -kTwoPi;   // a reset overrides the redraw at 500 (:886-917)
            else {
                const uint4 cb = philox4x32_10(g, t_rl, 0, STREAM_COMMAND, k0, k1);
                cmd = cmd + kTwoPi * kTurns[cb.x >> 29];
            }
        }
        if (coop) __syncwarp();                                    // mailbox reads done before any lane writes its frame over those rows
        if (R) progress = 0;                                       // :510-511

        // ------------------------------------------------------------------ pre_physics_step (:321-332): enqueue the action
        int T = 10;
        if (flags & TACO_F_RAMDOM_DEPLOY_TIME) {
            const uint4 db = philox4x32_10(g, t_rl, 0, STREAM_DEPLOY, k0, k1);
            T = 10 - round_normal(db.x, 1);
        }
        const int clk = 10 * progress;                              // absolute slot clock of buffer position 0
        if (q_len + T > 100 || q_n >= (uint32_t)kQueueCap) {
            q_ovf = 1;      // reference truncates the write at slot 100 (:329): outside delay_time_max, flagged + counted
            if (q_n >= (uint32_t)kQueueCap) q_n = kQueueCap - 1;   // (flagged envs only) the oldest run is overwritten
        }
        p.qact[(size_t)tslot * p.n_pad + i] = act;
        p.qend[(size_t)tslot * p.n_pad + i] = (uint16_t)min(clk + q_len + T, 65535);
        q_n += 1;
        q_len += T;
        // head run = the oldest of the last q_n slots
        uint32_t q_cur = (tslot + 17u - q_n) & 15u, q_left = q_n;
        float4 dact = make_float4(0.f, 0.f, 0.f, 0.f);
        int run_end = 0;
        if (q_left > 0) {
            dact = p.qact[(size_t)q_cur * p.n_pad + i];
            run_end = p.qend[(size_t)q_cur * p.n_pad + i];
        }

        const float dt = p.dt, h = p.h;
        const float rdt = p.inv_dt;
        auto fdiv_dt = [dt, rdt](float x) { return divc_impl(x, dt, rdt); };   // x / dt, correctly rounded (dt = sim dt)
        const bool battery_on = (flags & TACO_F_BATTERY_CONSUMPTION) != 0;
        const bool track_roll = (task == TACO_TASK_FLIP);
        float volt = 4.35f * 6.0f;                                  // battery_dynamics.py:75
        const Q4 qc0 = conj(q);
        V3 vb = qrot(qc0, vel), wb = qrot(qc0, wld);

        // The control iteration reads the head run at buffer position min(len-1, k) (:366-368), i.e. at slot
        // clk + min(q_len - 1, k), which never decreases in k.  So the head run changes only at the iteration head_k computes, and
        // the values the PID derives from the head run's action (angular_vel_control, :637-650) are formed when it is loaded.
        auto head_k = [&]() { const int r = run_end - clk; return (q_left > 1 && q_len - 1 >= r) ? r : INT_MAX; };
        float u0, hu0, sp[3];
        auto derive = [&]() {
            u0 = (dact.x + 1.0f) / 2.0f * 1000.0f;
            hu0 = u0 / 2.0f;
            sp[0] = dact.y * 20.0f; sp[1] = dact.z * 20.0f; sp[2] = dact.w * 20.0f;
        };
        derive();
        int k_next = head_k();

        // ------------------------------------------------------------------ control_freq_inv x (mid_physics_step + simulate)
        // Two instantiations of the loop, chosen once per launch: GEN tests the debug-delay, battery and rotor-noise switches in every
        // iteration; the other is the configuration of the training defaults (battery on, no rotor noise, no debug output) with
        // none of those tests.
        auto control = [&](auto gen) {
        constexpr bool GEN = decltype(gen)::value;
        for (int k = 0; k < p.cfi; ++k) {
            // refresh_state (:334-360): roll unwrap, body-frame velocities
            if (track_roll) unwrap_roll(q, roll_old, roll_cont);
            if (k > 0) vb = qrot(conj(q), vel);               // wb is carried by the integrator between sub-steps
            // delayed action (:366-368)
            if (k >= k_next) {
                const int slot_abs = clk + min(q_len - 1, k);
                while (slot_abs >= run_end && q_left > 1) {
                    q_cur = (q_cur + 1) & 15u; q_left -= 1;
                    dact = p.qact[(size_t)q_cur * p.n_pad + i];
                    run_end = p.qend[(size_t)q_cur * p.n_pad + i];
                }
                derive();
                k_next = head_k();
            }
            if constexpr (GEN) { if (p.dbg_delay) p.dbg_delay[(size_t)k * p.n_pad + i] = dact; }
            // rate PID (angvel_control.py:67-88)
            float uu[3];
            {
                const float wbv[3] = {wb.x, wb.y, wb.z};
                const float kp[3] = {27.5f, 50.0f, 200.0f};
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    const float e = clampf(sp[a] - wbv[a], -400.0f, 400.0f);
                    const float prev = (pe[a] == 0.0f) ? e : pe[a];
                    const float pt = kp[a] * e;
                    const float dv = clampf(0.5f * fdiv_dt(e - prev), -150.0f, 150.0f);
                    uu[a] = 0.4f * (pt + dv);
                    pe[a] = e;
                }
            }
            // control_allocator (fpv_dynamics.py:35-46)
            float thr[4];
            {
                const float u1 = uu[0], u2 = uu[1];
                const float u3 = fminf(fmaxf(uu[2], -hu0), hu0);      // -u0 / 2 == -(u0 / 2)
                thr[0] = u0 - u1 + u2 - u3;
                thr[1] = u0 - u1 - u2 + u3;
                thr[2] = u0 + u1 - u2 - u3;
                thr[3] = u0 + u1 + u2 + u3;
                const float mx = fmaxf(fmaxf(thr[0], thr[1]), fmaxf(thr[2], thr[3])) - 1000.0f;
                const float sat = fmaxf(mx, 0.0f);
#pragma unroll
                for (int r = 0; r < 4; ++r) thr[r] = clampf(thr[r] - sat, 100.0f, 1000.0f);
            }
            // mechanical power of the previous rotor speeds (fpv_asymmetry.py:614)
            float pm;
            {
                float c[4];
#pragma unroll
                // om * 2 * pi rounds once, as om * (2 pi): the doubling is exact for every float (tests/test_exact_folds.py)
                for (int r = 0; r < 4; ++r) { const float x = TACO_DIVC(om[r] * kTwoPi, 4500.0f); c[r] = 400.0f * (x * x * x); }
                pm = ((c[0] + c[1]) + c[2]) + c[3];
            }
            // battery sag (battery_dynamics.py:47-75)
            if (GEN ? battery_on : true) {
                bt = bt + dt;
                const float pc = TACO_DIVC(TACO_DIVC(pm, 0.75f), 9000.0f);
                bec = bec + pc * dt;
                const float pavg = bec / bt;
                float r0 = (0.0015778f + -7.7608e-5f * pavg) + (float)(0.0069498 * 1500.0);   // b0 + b1*P_avg + b2*C_c (python folds b2*C_c in double)
                r0 = (r0 > 4.5f) ? r0 : 4.5f;
                const float v0 = ((4.35f + -0.1102178f * bec) + 0.0103368f * (bec * bec)) + -4.3778e-4f * (bec * bec * bec);
                bu1 = bu1 + TACO_DIVC(0.00104846f * pc - bu1, 3.3f) * dt;
                const float df = v0 - bu1;
                volt = 0.5f * (df + sqrtf(df * df - 4.0f * r0 * pc)) * 6.0f;
            }
            // rotor lag (thrust_dynamics.py:52-66,80-86) + optional speed noise (:68-78)
            {
                const float y = TACO_DIVC(volt - 23.0f, 3.0f);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const float x = TACO_DIVC(thr[r], 1000.0f);
                    const float p01 = DR ? poly[0] + poly[1] * x : poly[1] * x;    // nominal poly[0] = +0 and poly[1] * x > 0: 0 + a == a bit for bit
                    const float tgt = (((p01 + poly[2] * y) + poly[3] * (x * x)) + poly[4] * x * y) * 100.0f;
                    om[r] = om[r] + lag[r] * (tgt - om[r]);
                }
                if (GEN && (flags & TACO_F_ROTOR_NOISE)) {
                    const uint4 nb = philox4x32_10(g, t_rl, (uint32_t)k, STREAM_ROTOR_NOISE, k0, k1);
                    const float rng = (float)((1.0 + 10.0 / 700.0) - (1.0 - 10.0 / 700.0)), lo = (float)(1.0 - 10.0 / 700.0);
                    om[0] = om[0] * rr(rng, lo, u01(nb.x)); om[1] = om[1] * rr(rng, lo, u01(nb.y));
                    om[2] = om[2] * rr(rng, lo, u01(nb.z)); om[3] = om[3] * rr(rng, lo, u01(nb.w));
                }
            }
            // aerodynamics (thrust_dynamics.py:173-199), real->sim remap (fpv_dynamics.py:48-56), body wrench
            V3 fb, tb;
            {
                float f[4], tqr[4];
#pragma unroll
                for (int r = 0; r < 4; ++r) { f[r] = aero[0] * om[r] * om[r]; tqr[r] = aero[1] * f[r]; }
                const float vxy = norm2(vb.x, vb.y);                                // torch.norm, thrust_dynamics.py:193
                const float f0 = f[2], f1 = f[3], f2 = f[0], f3 = f[1];           // sim rotor (0,1,2,3) <- real (2,3,0,1)
                const float t0 = -tqr[2], t1 = tqr[3], t2 = -tqr[0], t3 = tqr[1];
                fb.x = aero[2] * vb.x;
                fb.y = aero[3] * vb.y;
                fb.z = aero[4] * vxy * vxy + (((f0 + f1) + f2) + f3);
                tb.x = 0.059f * (((f0 + f1) - f2) - f3);
                tb.y = 0.047f * (((f1 + f2) - f0) - f3);
                tb.z = ((t0 + t1) + t2) + t3;
                if (R) { fb = v3(0.f, 0.f, 0.f); tb = v3(0.f, 0.f, 0.f); }        // fpv_asymmetry.py:629-630
            }
            // free rigid body, `substeps` x h (DESIGN.md "integrator"; oracle/rigid_body.c is the specification, operation for
            // operation): force held in the world frame, torque in the body frame, angular velocity carried in body
            // coordinates.  The integrator is ours, so its FMAs are part of the specification (explicit, also in the
            // -fmad=false build); everything that restates the reference's torch expressions rounds every operation.
            {
                // F_w = F_b + w t + u x t,  t = 2 (u x F_b)
                const V3 u = v3(q.x, q.y, q.z);
                V3 t = cross_f(u, fb); t.x = t.x + t.x; t.y = t.y + t.y; t.z = t.z + t.z;
                const V3 ut = cross_f(u, t);
                const V3 fw = v3(__fmaf_rn(q.w, t.x, fb.x) + ut.x, __fmaf_rn(q.w, t.y, fb.y) + ut.y, __fmaf_rn(q.w, t.z, fb.z) + ut.z);
                const V3 acc = v3(fw.x * p.inv_mass, fw.y * p.inv_mass, __fmaf_rn(fw.z, p.inv_mass, -9.81f));
                const int nsub = SUB ? SUB : p.substeps;
#pragma unroll
                for (int s = 0; s < nsub; ++s) {
                    vel.x = __fmaf_rn(h, acc.x, vel.x); vel.y = __fmaf_rn(h, acc.y, vel.y); vel.z = __fmaf_rn(h, acc.z, vel.z);
                    const V3 iw = v3(5e-4f * wb.x, 7e-4f * wb.y, 8e-4f * wb.z);
                    const V3 gy = cross_f(wb, iw);
                    wb.x = __fmaf_rn(h, (tb.x - gy.x) * 2000.0f, wb.x);
                    wb.y = __fmaf_rn(h, (tb.y - gy.y) * (float)(1.0 / 7e-4), wb.y);
                    wb.z = __fmaf_rn(h, (tb.z - gy.z) * 1250.0f, wb.z);
                    pos.x = __fmaf_rn(h, vel.x, pos.x); pos.y = __fmaf_rn(h, vel.y, pos.y); pos.z = __fmaf_rn(h, vel.z, pos.z);
                    const float w2 = __fmaf_rn(wb.z, wb.z, __fmaf_rn(wb.y, wb.y, wb.x * wb.x));
                    const float th2 = w2 * p.half_h2;
                    const float kk = p.half_h * __fmaf_rn(th2, __fmaf_rn(th2, p.c_sin5, p.c_sin3), 1.0f);
                    const float cs = __fmaf_rn(th2, __fmaf_rn(th2, p.c_cos4, -0.5f), 1.0f);
                    const float dx = wb.x * kk, dy = wb.y * kk, dz = wb.z * kk;
                    Q4 r;                                                                   // Hamilton product q * (dx, dy, dz, cs)
                    r.w = __fmaf_rn(-q.z, dz, __fmaf_rn(-q.y, dy, __fmaf_rn(-q.x, dx, q.w * cs)));
                    r.x = __fmaf_rn(-q.z, dy, __fmaf_rn(q.y, dz, __fmaf_rn(q.x, cs, q.w * dx)));
                    r.y = __fmaf_rn(-q.x, dz, __fmaf_rn(q.z, dx, __fmaf_rn(q.y, cs, q.w * dy)));
                    r.z = __fmaf_rn(-q.y, dx, __fmaf_rn(q.x, dy, __fmaf_rn(q.z, cs, q.w * dz)));
                    const float n2 = __fmaf_rn(r.w, r.w, __fmaf_rn(r.z, r.z, __fmaf_rn(r.y, r.y, r.x * r.x)));
                    const float rn = __fmaf_rn(-0.5f, n2, 1.5f);                            // one Newton step of 1/sqrt about 1
                    q.x = r.x * rn; q.y = r.y * rn; q.z = r.z * rn; q.w = r.w * rn;
                }
            }
        }
        };
        if (battery_on && !(flags & TACO_F_ROTOR_NOISE) && !p.dbg_delay) control(std::false_type{});
        else control(std::true_type{});
        wld = qrot(q, wb);                                           // world-frame root state at the end of the RL step

        // ------------------------------------------------------------------ post_physics_step (:374-388)
        progress += 1;
        {   // shift the delay buffer by 10 slots = advance the slot clock; drop exhausted runs
            const int clk2 = clk + 10;
            q_n = q_left;
            while (q_n > 0 && run_end <= clk2) {
                q_cur = (q_cur + 1) & 15u; q_n -= 1;
                if (q_n > 0) run_end = p.qend[(size_t)q_cur * p.n_pad + i];
            }
            q_len = max(q_len - 10, 0);
        }
        // refresh_state
        if (track_roll) unwrap_roll(q, roll_old, roll_cont);
        const Q4 qc = conj(q);
        vb = qrot(qc, vel);
        wb = qrot(qc, wld);
        const V3 rel = v3(tpos.x - pos.x, tpos.y - pos.y, tpos.z - pos.z);
        const V3 relb = qrot(qc, rel);
        const Q4 rq = qmul(qc, tq);
        float m[9];
        rotmat9(rq, m);
        // newest frame (:394-400) + task id / command (:713-714,:768-771,:835-838)
        float c1 = cmd;                                              // command[:,1]
        float o24 = 0.f, o25;
        if (task == TACO_TASK_FLIP) {
            c1 = clampf(cmd - roll_cont, -kTwoPi, kTwoPi);           // :831-832
            o24 = -1.f; o25 = TACO_DIVC(c1 / 2.0f, kPi);
        } else if (task == TACO_TASK_ROTATE) { o24 = 1.f; o25 = TACO_DIVC(c1, 6.0f); }
        else { c1 = 0.f; o25 = 0.f; }
        fc[0] = TACO_DIVC(relb.x, 3.0f); fc[1] = TACO_DIVC(relb.y, 3.0f); fc[2] = TACO_DIVC(relb.z, 3.0f);
#pragma unroll
        for (int j = 0; j < 9; ++j) fc[3 + j] = m[j];
        fc[12] = -vb.x / 2.0f; fc[13] = -vb.y / 2.0f; fc[14] = -vb.z / 2.0f;         // relative velocity = -(own), target is static (:147-148,:357-360)
        fc[15] = TACO_DIVC(-wb.x, kPi); fc[16] = TACO_DIVC(-wb.y, kPi); fc[17] = TACO_DIVC(-wb.z, kPi);
        fc[18] = TACO_DIVC(volt - 23.0f, 3.0f);
        fc[19] = act.x; fc[20] = act.y; fc[21] = act.z; fc[22] = act.w;
        fc[23] = 4.0f * clampf(pos.z, 0.0f, 0.5f) - 1.0f;
        fc[24] = o24; fc[25] = o25;
        bool finite = true;
#pragma unroll
        for (int j = 0; j < 24; ++j) finite = finite && isfinite(fc[j]);
        finite = finite && isfinite(o25);
        if (obs_noise) {                                              // :402-410
            const float d = TACO_DIFF(difficulty, 0);
            float z[12];
#pragma unroll
            for (int s = 0; s < 3; ++s) {
                const uint4 nb = philox4x32_10(g, t_rl, (uint32_t)s, STREAM_OBS_NOISE, k0, k1);
                box_muller(nb.x, nb.y, z[4 * s + 0], z[4 * s + 1]);
                box_muller(nb.z, nb.w, z[4 * s + 2], z[4 * s + 3]);
            }
            const uint4 ub = philox4x32_10(g, t_rl, 3, STREAM_OBS_NOISE, k0, k1);
            const float sp_ = (float)(0.06 / 3 / 3), sv_ = (float)(0.1 / 3 / 2), sw_ = (float)(60.0 / 3 / 180), su_ = (float)(0.06 / 3), sh_ = (float)(0.06 / 3 / 3);
#pragma unroll
            for (int j = 0; j < 26; ++j) fn[j] = fc[j];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                fn[a] = fc[a] + d * (z[a] * sp_);
                fn[12 + a] = fc[12 + a] + d * (z[3 + a] * sv_);
                fn[15 + a] = fc[15 + a] + d * (z[6 + a] * sw_);
            }
            fn[18] = fc[18] + d * (z[9] * su_);
            fn[23] = fc[23] + d * (z[10] * sh_);
            const Q4 nq = quat_from_euler(rr(TACO_DIFF(noise_rng, 7), TACO_DIFF(noise_lo, 8), u01(ub.x)), rr(TACO_DIFF(noise_rng, 7), TACO_DIFF(noise_lo, 8), u01(ub.y)),
                                          rr(TACO_DIFF(noise_rng, 7), TACO_DIFF(noise_lo, 8), u01(ub.z)));
            float mn[9];
            rotmat9(qmul(rq, nq), mn);
#pragma unroll
            for (int j = 0; j < 9; ++j) fn[3 + j] = mn[j];
        }
        // ------------------------------------------------------------------ reward + termination (task_reward.py)
        float rew, dist;
        if (task == TACO_TASK_POS) {                                  // :20-47
            dist = norm3(relb.x, relb.y, relb.z);
            const Q4 mq = qmul(q, conj(tq));                          // quat_diff_rad, torch_jit_utils.py:146-164
            const float nv = norm3(mq.x, mq.y, mq.z);
            const float ang = 2.0f * asinf(fminf(nv, 1.0f));
            rew = TACO_DIVC(two_scale(dist) * two_scale(ang), 100.0f);
        } else if (task == TACO_TASK_ROTATE) {                        // :50-104
            float ex = -rel.x, ey = -rel.y;
            const float en = norm3(ex, ey, 0.0f) + 1e-8f;
            ex = ex / en; ey = ey / en;
            float yx = -ey, yy = ex;                                  // e_z x e_x
            const float yn = norm3(yx, yy, 0.0f) + 1e-8f;
            yx = yx / yn; yy = yy / yn;
            const float hori = norm2(rel.x, rel.y) - 1.2f;
            const float vert = fabsf(rel.z);
            dist = sqrtf(hori * hori + vert * vert);
            const float rvx = -vel.x, rvy = -vel.y, rvz = -vel.z;     // relative_linvel = 0 - v
            const float vn = rvx * ex + rvy * ey;
            const float vt = (rvx * yx + rvy * yy) - c1;
            const float verr = norm3(vn, vt, rvz);
            const float two_s = 2.0f / (((q.x * q.x + q.y * q.y) + q.z * q.z) + q.w * q.w);
            const float hx = 1.0f - two_s * (q.y * q.y + q.z * q.z);
            const float hy = two_s * (q.x * q.y + q.z * q.w);
            const float ddir = 1.0f + (ex * hx + ey * hy) / norm2(hx, hy);
            rew = TACO_DIVC(two_scale(dist) * two_scale(verr) * two_scale(ddir), 100.0f);
        } else {                                                      // :107-143
            dist = norm3(relb.x, relb.y, relb.z);
            const float rp = 1.0f / (1.0f + 1.0f * dist) + 1.0f / (1.0f + 10.0f * dist);
            const float rt = 1.0f / (1.0f + 10.0f * (1.0f - m[0]));
            const float turns = TACO_DIVC(c1 / 2.0f, kPi);
            rew = TACO_DIVC(rp * rt * two_scale(turns), 100.0f);
        }
        const bool die = (pos.z < 0.1f) || (dist > 10.0f);
        const bool tmax = progress >= p.max_len - 1;
        const bool done = tmax || die;
        const bool tout = tmax && done;                               // vec_task_asymmetry.py:323
        // episode statistics (ppo_asymmetry.py:313-339)
        ep_ret += rew;
        st_rew = rew; st_done = done ? 1.f : 0.f; st_tout = tout ? 1.f : 0.f;
        st_epret = done ? ep_ret : 0.f; st_eplen = done ? (float)progress : 0.f;
        st_nonfin = finite ? 0.f : 1.f; st_ovf = q_ovf ? 1.f : 0.f;
        if (done) ep_ret = 0.f;
        // ------------------------------------------------------------------ store
        p.S[0][i] = make_float4(pos.x, pos.y, pos.z, q.x);
        p.S[1][i] = make_float4(q.y, q.z, q.w, vel.x);
        p.S[2][i] = make_float4(vel.y, vel.z, wld.x, wld.y);
        p.S[3][i] = make_float4(wld.z, tpos.x, tpos.y, tpos.z);
        p.S[4][i] = make_float4(tq.z, tq.w, roll_old, roll_cont);
        p.S[5][i] = make_float4(om[0], om[1], om[2], om[3]);
        p.S[6][i] = make_float4(pe[0], pe[1], pe[2], cmd);
        p.S[7][i] = make_float4(bu1, bec, bt, ep_ret);
        p.progress[i] = progress;
        p.qmeta[i] = (q_n << QM_N_SHIFT) | ((uint32_t)min(q_len, 2047) << QM_LEN_SHIFT) | (q_ovf << QM_OVF_SHIFT);
        p.reset_buf[i] = done ? 1ll : 0ll;
        p.time_outs[i] = tout ? 1 : 0;
        p.rew[i] = rew;
        if (p.roll_rew) {       // rows of an attached rollout buffer: rew_buf / done_buf as float32, time-outs as bytes
            p.roll_rew[i] = rew;
            p.roll_done[i] = done ? 1.0f : 0.0f;
            p.roll_tout[i] = tout ? 1 : 0;
        }
        // mapped host-buffer step (taco_env_step_host): results are posted straight into the caller's pinned host memory
        if (p.host_reset) p.host_reset[i] = done ? 1ll : 0ll;
        if (p.host_rew) p.host_rew[i] = rew;
        // the one-byte results go out as ONE 128-byte run per CTA after the barrier below (a warp's 32 single bytes are a 32-byte PCIe
        // write with as much header as payload: the time-out column alone cost 0.07 ms of the 0.82 ms host-buffer step)
        if (HB) {
            if (p.host_tout || p.host_flags) s_hostb[tid] = p.host_flags ? (uint8_t)((done ? 1 : 0) | (tout ? 2 : 0)) : (uint8_t)(tout ? 1 : 0);
        } else {
            if (p.host_tout) p.host_tout[i] = tout ? 1 : 0;
            if (p.host_flags) p.host_flags[i] = (uint8_t)((done ? 1 : 0) | (tout ? 2 : 0));
        }
    } else {
#pragma unroll
        for (int j = 0; j < 26; ++j) { fc[j] = 0.f; fn[j] = 0.f; }
    }

    // ---------------------------------------------------------------------- rollout statistics: warp reduction -> smem -> 1 atomic / block / stat
    // (the 0 / 1 flags as a ballot + popc, the episode lengths as an integer redux: 2 instructions each instead of a 10-instruction
    // shuffle tree; the two float sums keep their butterfly order, so every statistic has the value it had)
    {
        float sv[2] = {st_rew, st_epret};
#pragma unroll
        for (int j = 0; j < 2; ++j) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sv[j] += __shfl_xor_sync(0xffffffffu, sv[j], o);
        }
        const uint32_t b_done = __ballot_sync(0xffffffffu, st_done != 0.f), b_tout = __ballot_sync(0xffffffffu, st_tout != 0.f);
        const uint32_t b_nonfin = __ballot_sync(0xffffffffu, st_nonfin != 0.f), b_ovf = __ballot_sync(0xffffffffu, st_ovf != 0.f);
        const int len_sum = __reduce_add_sync(0xffffffffu, (int)st_eplen);       // episode lengths are integers <= max_len
        if ((tid & 31) == 0) {
            if (sv[0] != 0.f) atomicAdd(&s_stats[0], (double)sv[0]);
            if (b_done) atomicAdd(&s_stats[1], (double)__popc(b_done));
            if (b_tout) atomicAdd(&s_stats[2], (double)__popc(b_tout));
            if (sv[1] != 0.f) atomicAdd(&s_stats[3], (double)sv[1]);
            if (len_sum) atomicAdd(&s_stats[4], (double)len_sum);
            if (b_nonfin) atomicAdd(&s_stats[5], (double)__popc(b_nonfin));
            if (b_ovf) atomicAdd(&s_stats[6], (double)__popc(b_ovf));
        }
    }
    if (CW > 0) asm volatile("bar.sync 1, %0;" ::"n"(kBlock) : "memory");   // the compute warps only: the copy warps may be gone
    else __syncthreads();   // frames + stats visible
    if (HB && (p.host_tout || p.host_flags)) {                  // blk * 128 keeps the 4-byte alignment of a pinned buffer
        uint8_t* hb = (p.host_flags ? p.host_flags : p.host_tout) + (size_t)blk * kBlock;
        const int nvb = min(kBlock, p.n - blk * kBlock);
        if (nvb == kBlock && (reinterpret_cast<uintptr_t>(hb) & 3u) == 0) {
            if (tid < kBlock / 4) reinterpret_cast<uint32_t*>(hb)[tid] = reinterpret_cast<const uint32_t*>(s_hostb)[tid];
        } else if (tid < nvb) hb[tid] = s_hostb[tid];
    }
    if (tid < 7) {
        const double v = s_stats[tid];
        if (v != 0.0) atomicAdd(p.stats + (size_t)(blk % kStatSlots) * kStatStride + tid, v);
    } else if (tid == 7) {
        const int nv = min(kBlock, p.n - blk * kBlock);
        atomicAdd(p.stats + (size_t)(blk % kStatSlots) * kStatStride + 7, (double)nv);
    }

    // ---------------------------------------------------------------------- history shift + newest frame (:392,:413)
    // states: the newest frame into the env-owned strip, or (rollout ring attached) out[e][f][:] = in[e][f+1][:] for f < L-1 and the
    // newest frame last, slot k -> slot k + 1 of the ring.  obs: the same shift between ping-pong buffers.  No in-place hazard.
    const size_t blk_env0 = (size_t)blk * kBlock;
    const int nv = min(kBlock, p.n - blk * kBlock);             // valid rows of this CTA
    if (p.states_strip) write_strip(p, s_clean, blk_env0, tid, nv);
    else if (CW > 0 && split_copy) write_newest_rows<5>(p.states_out, s_clean, blk_env0, tid);   // the copy warps moved the kept part
    else if (p.len_states == 5) write_rows<5, !DR>(p.states_in, p.states_out, s_clean, 5, blk_env0, tid, nv);
    else write_rows<0, false>(p.states_in, p.states_out, s_clean, p.len_states, blk_env0, tid, nv);
    const float* sf = obs_noise ? s_noisy : s_clean;
    if (p.len_obs == 1) write_rows<1, !DR>(p.obs_in, p.obs_out, sf, 1, blk_env0, tid, nv);
    else write_rows<0, false>(p.obs_in, p.obs_out, sf, p.len_obs, blk_env0, tid, nv);
}

#ifndef TACO_COPY_WARPS_SMALL
#define TACO_COPY_WARPS_SMALL 4     // copy warps per CTA for launches of <= kSmallGrid CTAs (0 = off)
#endif
constexpr int kSmallGrid = 148;     // one CTA per SM

template <int TASK, bool DR, bool DEVDIFF>
static void launch_variant(const StepParams& p, int grid, cudaStream_t stream) {
    if (p.substeps == 2) {
        if (TACO_COPY_WARPS_SMALL > 0 && grid <= kSmallGrid && !p.states_strip)   // the ring path's kept-history copy
            fpv_step_kernel<TASK, DR, 2, DEVDIFF, TACO_COPY_WARPS_SMALL><<<grid, kBlock + 32 * TACO_COPY_WARPS_SMALL, 0, stream>>>(p);
        else if (!DEVDIFF && (p.host_tout || p.host_flags)) fpv_step_kernel<TASK, DR, 2, false, 0, true><<<grid, kBlock, 0, stream>>>(p);
        else fpv_step_kernel<TASK, DR, 2, DEVDIFF><<<grid, kBlock, 0, stream>>>(p);
    } else if (p.substeps == 1 && !DEVDIFF) fpv_step_kernel<TASK, DR, 1, DEVDIFF><<<grid, kBlock, 0, stream>>>(p);
    else fpv_step_kernel<TASK, DR, 0, DEVDIFF><<<grid, kBlock, 0, stream>>>(p);
}
template <int TASK>
static void launch_task(const StepParams& p, cudaStream_t stream) {
    const int grid = p.nblocks > 0 ? p.nblocks : p.n_pad / kBlock - p.block0;
    if (p.diff_dev != nullptr) {                       // graph mode (taco_env_graph_begin .. _end)
        if (p.has_dr) launch_variant<TASK, true, true>(p, grid, stream);
        else launch_variant<TASK, false, true>(p, grid, stream);
    } else if (p.has_dr) launch_variant<TASK, true, false>(p, grid, stream);
    else launch_variant<TASK, false, false>(p, grid, stream);
    TACO_LAUNCHED();
}

static inline void launch_any(const StepParams& p, cudaStream_t stream) {
    switch (p.task_mode) {
        case TACO_TASK_POS: launch_task<TACO_TASK_POS>(p, stream); break;
        case TACO_TASK_ROTATE: launch_task<TACO_TASK_ROTATE>(p, stream); break;
        case TACO_TASK_FLIP: launch_task<TACO_TASK_FLIP>(p, stream); break;
        default: launch_task<TACO_TASK_MIX>(p, stream); break;
    }
}

}  // namespace TACO_VARIANT
}  // namespace taco
