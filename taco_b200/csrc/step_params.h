// Kernel parameter block shared by the host library (taco_env.cu) and the two compiled
// variants of the fused step kernel (fpv_step_fast.cu / fpv_step_strict.cu).
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

namespace taco {

constexpr int kBlock = 128;       // envs (threads) per CTA
constexpr int kQueueCap = 16;     // pending-action runs per env (in-domain max is 13, see DESIGN.md)
constexpr int kObs = 26;          // values per frame, fpv_asymmetry.py:107
constexpr int kFramePad = 27;     // smem row stride (odd -> conflict-free column writes)
constexpr int kStatSlots = 64;    // spread of the per-block stats atomics
constexpr int kStatStride = 16;   // doubles per slot (128 B)
constexpr int kNumStats = 8;

// nominal model parameters (thrust_dynamics.py:46-47,156-167): rotor speed polynomial, aero k_f, k_tau, d_x, d_y, k_th
__device__ constexpr float kPolyNom[5] = {0.0f, 12.9466f, 0.1872f, -5.1220f, 0.5906f};
__device__ constexpr float kAeroNom[5] = {1.13e-05f, 0.05f, -0.386f, -0.53f, 0.009f};

// qmeta bit layout: live runs (5 b), actions_remained_length (11 b), overflow flag
constexpr uint32_t QM_N_SHIFT = 4, QM_LEN_SHIFT = 9, QM_OVF_SHIFT = 20;
__host__ __device__ __forceinline__ uint32_t qm_runs(uint32_t qm) { return (qm >> QM_N_SHIFT) & 31u; }
__host__ __device__ __forceinline__ uint32_t qm_len(uint32_t qm) { return (qm >> QM_LEN_SHIFT) & 2047u; }
__host__ __device__ __forceinline__ uint32_t qm_ovf(uint32_t qm) { return (qm >> QM_OVF_SHIFT) & 1u; }
// each field cut to its width (the step kernel packs values already in range: it clamps the length instead)
__host__ __device__ __forceinline__ uint32_t qm_pack(uint32_t runs, uint32_t len, uint32_t ovf) {
    return ((runs & 31u) << QM_N_SHIFT) | ((len & 2047u) << QM_LEN_SHIFT) | ((ovf & 1u) << QM_OVF_SHIFT);
}

struct StepParams {
    int n, n_pad;
    int block0, nblocks;           // CTA range of this launch (nblocks = 0: all remaining CTAs)
    long long env_offset;
    long long mix_n1, mix_n2;      // global task-group boundaries (fpv_asymmetry.py:924-926)
    int task_mode, len_obs, len_states, max_len, cfi, substeps, delay_time;
    uint32_t flags, seed_lo, seed_hi, step_index;   // step_index: absolute RL step, or the offset to *step_base (graph mode)
    const uint32_t* step_base;     // device word added to step_index (null outside graph mode): a captured launch stays valid on replay
    float dt, inv_dt, h, half_h, half_h2, c_sin3, c_sin5, c_cos4, inv_mass, difficulty, clip_actions;
    // host-precomputed (double -> float) bounds of the difficulty-dependent uniform draws
    float flip_xy_rng, flip_xy_lo, flip_lin_rng, flip_lin_lo, dr_rng, dr_lo, tau_rng, tau_lo, noise_rng, noise_lo;
    // graph mode only (else null): device copy of [difficulty, flip_xy_rng, flip_xy_lo, flip_lin_rng, flip_lin_lo, dr_rng, dr_lo,
    // noise_rng, noise_lo], rewritten by taco_env_set_difficulty -- a launch captured in a CUDA graph freezes the by-value
    // fields above, and the trainer changes the difficulty every epoch (ppo_asymmetry.py:173-175)
    const float* diff_dev;
    float lag_gain_fixed;          // 0.001 / rotor_response_time (or 1.0 when rotor_response is off)
    int has_dr;                    // per-env DR planes are live
    // inputs / state / outputs (device)
    const float4* actions;
    float4* S[8];
    int* progress;
    uint32_t* qmeta;
    float4* qact;                  // [kQueueCap][n_pad]
    uint16_t* qend;                // [kQueueCap][n_pad]
    float4* D[4];
    long long* reset_buf;
    uint8_t* time_outs;
    float* rew;
    const float* obs_in;
    float* obs_out;
    const float* states_in;        // attached rollout ring: slot k (read) and slot k + 1 (written), contiguous (n, len_states, 26)
    float* states_out;
    float* states_strip;           // else the env's own history strip (see write_strip in fpv_step_kernel.cuh), null while a ring is attached
    int strip_frames, strip_period;   // frames per env row of the strip, and the period K of the window offset
    float* roll_rew;               // row of the attached rollout buffer for this step (or null): rew, done as f32, time-outs
    float* roll_done;
    uint8_t* roll_tout;
    float* host_rew;               // taco_env_step_host, mapped mode: the caller's pinned host buffers (device-visible addresses,
    long long* host_reset;         // or null); the kernel posts rew / reset / time-outs across PCIe itself
    uint8_t* host_tout;
    uint8_t* host_flags;           // taco_env_step_host_compact: one byte per env, bit 0 = reset, bit 1 = time-out
    double* stats;                 // [kStatSlots][kStatStride]
    float4* dbg_delay;             // [cfi][n_pad] or null
};

void launch_fpv_step_fast(const StepParams& p, cudaStream_t stream);
void launch_fpv_step_strict(const StepParams& p, cudaStream_t stream);

}  // namespace taco
