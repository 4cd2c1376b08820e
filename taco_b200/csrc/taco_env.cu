// Host side of the C ABI (include/taco_b200.h): owns every device buffer of one env shard and
// launches the fused step kernel.  No torch types, no exceptions across the boundary.
//
// Mirrors, for buffer ownership and layout, VecTask.allocate_buffers
// (IsaacGymEnvs/isaacgymenvs/tasks/base/vec_task_asymmetry.py:231-254) and the state tensors of
// FpvBase.__init__ (IsaacGymEnvs/isaacgymenvs/tasks/fpv_asymmetry.py:124-200).
#include "launch_count.h"
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <new>
#include <string>
#include <vector>

#include "host_common.h"
#include "philox.cuh"
#include "fpv_math.cuh"
#include "step_params.h"
#include "episode_log.cuh"
#include "rollout_episodes.cuh"

namespace taco {

std::atomic<unsigned long long> g_launches{0};
static thread_local std::string g_err;
int fail(int code, const std::string& msg) { g_err = msg; return code; }

}  // namespace taco

struct TacoEnv {
    TacoCfg cfg;
    int device;
    int n, n_pad;
    taco::StepParams p;          // pointers + constants (step_index / ping-pong patched per step)
    void* arena = nullptr;       // one cudaMalloc for everything
    size_t arena_bytes = 0;
    float* obs_ab[2] = {nullptr, nullptr};
    float* strip = nullptr;      // state history: strip_frames frames per env, window at offset step_index % strip_period (write_strip)
    int strip_frames = 0, strip_period = 0;
    int cur = 0;                 // index of the obs buffer holding the latest observation history
    // caller-owned rollout ring (taco_env_attach_rollout): slot k of obs / states, row k of rew / done / time-outs
    float* ring_obs = nullptr;
    float* ring_states = nullptr;
    float* ring_rew = nullptr;
    float* ring_done = nullptr;
    uint8_t* ring_tout = nullptr;
    int ring_slots = 0, ring_cur = 0;
    float4* actions_stage = nullptr;   // device staging for taco_env_step_host
    double* stats_out = nullptr;       // 8 doubles, device
    float* export_stage = nullptr;     // n * TACO_STATE_WORDS floats, device
    float4* dbg_delay = nullptr;
    // episode log (taco_env_attach_episode_log): one allocation = counter, two accumulator planes, records
    void* log_mem = nullptr;
    unsigned long long* log_count = nullptr;
    float4* log_acc[2] = {nullptr, nullptr};
    TacoEpisode* log_rec = nullptr;
    unsigned long long log_cap = 0;
    // rollout episodes (taco_env_attach_rollout_episodes): one allocation = counters, per-env ret / len / live planes, block
    // partials, records; rep_scanned = the first ring row the next scan reads
    void* rep_mem = nullptr;
    unsigned long long* rep_count = nullptr;
    unsigned int* rep_blocks_done = nullptr;
    float* rep_ret = nullptr;
    int* rep_len = nullptr;
    uint8_t* rep_live = nullptr;
    double* rep_partial = nullptr;
    TacoRolloutEpisode* rep_rec = nullptr;
    unsigned long long rep_cap = 0;
    int rep_scanned = 0;
    uint32_t step_index = 0;
    // graph mode (taco_env_graph_begin .. _end): the step index of a launch = *step_counter (device) + its offset since
    // graph_begin, so a CUDA graph captured over a rollout replays with fresh Philox counters / queue time slots
    uint32_t* step_counter = nullptr;   // device, one word
    float* diff_dev = nullptr;          // device, 9 floats (upload_derived)
    bool graph_mode = false;
    uint32_t graph_origin = 0;
    // host-buffer pipeline (taco_env_step_host): copy-in / kernel / copy-out of successive env chunks overlap
    static constexpr int kMaxChunks = 16;
    static constexpr int kKernelStreams = 3;     // chunk kernels rotate over these so that a chunk's tail wave overlaps the next chunk
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr, s_k[kKernelStreams] = {};
    cudaEvent_t ev_h2d[kMaxChunks] = {}, ev_k[kMaxChunks] = {}, ev_begin = nullptr, ev_end = nullptr;
    bool pipe_ready = false;
};

namespace taco {

static void refresh_derived(TacoEnv* e) {
    // bounds of the difficulty-dependent uniform draws, evaluated in double like the python
    // expressions they replace (fpv_asymmetry.py:856,870,405; thrust_dynamics.py:118,136), then cast to f32
    StepParams& p = e->p;
    const double d = (double)e->cfg.difficulty;
    const double lim = 0.5 + 1.5 * d;
    p.flip_xy_rng = (float)(lim - (-lim)); p.flip_xy_lo = (float)(-lim);
    p.flip_lin_rng = (float)(3 * d - (-3 * d)); p.flip_lin_lo = (float)(-3 * d);
    const double lo = 1 - 0.05 * d, hi = 1 + 0.05 * d;
    p.dr_rng = (float)(hi - lo); p.dr_lo = (float)lo;
    const double tau0 = (double)e->cfg.rotor_response_time;
    p.tau_rng = (float)((tau0 + 0.001) - (tau0 - 0.001)); p.tau_lo = (float)(tau0 - 0.001);
    const double nl = d * 0.05;
    p.noise_rng = (float)(nl - (-nl)); p.noise_lo = (float)(-nl);
    p.difficulty = e->cfg.difficulty;
}

// the device copy of the difficulty-dependent scalars that launches captured in a CUDA graph read (StepParams::diff_dev)
static cudaError_t upload_derived(TacoEnv* e) {
    if (!e->diff_dev) return cudaSuccess;
    const StepParams& p = e->p;
    const float v[9] = {p.difficulty, p.flip_xy_rng, p.flip_xy_lo, p.flip_lin_rng, p.flip_lin_lo, p.dr_rng, p.dr_lo, p.noise_rng, p.noise_lo};
    return cudaMemcpy(e->diff_dev, v, sizeof(v), cudaMemcpyHostToDevice);
}

// ---- small utility kernels -----------------------------------------------------------------
__global__ void init_state_kernel(StepParams p) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_pad) return;
    // default pose (0,0,4), identity attitude, at rest (fpv_asymmetry.py:264-266); reset_buf = 1 (vec_task_asymmetry.py:246-247)
    p.S[0][i] = make_float4(0.f, 0.f, 4.f, 0.f);
    p.S[1][i] = make_float4(0.f, 0.f, 1.f, 0.f);
    p.S[2][i] = make_float4(0.f, 0.f, 0.f, 0.f);
    p.S[3][i] = make_float4(0.f, 0.f, 0.f, 4.f);
    p.S[4][i] = make_float4(0.f, 1.f, 0.f, 0.f);
    p.S[5][i] = make_float4(0.f, 0.f, 0.f, 0.f);
    p.S[6][i] = make_float4(0.f, 0.f, 0.f, 0.f);
    p.S[7][i] = make_float4(0.f, 0.f, 0.f, 0.f);
    p.progress[i] = 0;
    p.qmeta[i] = qm_pack(0, (uint32_t)p.delay_time, 0);
    p.reset_buf[i] = 1;
    p.time_outs[i] = 0;
    p.rew[i] = 0.f;
    if (p.has_dr) {
        p.D[0][i] = make_float4(kPolyNom[0], kPolyNom[1], kPolyNom[2], kPolyNom[3]);
        p.D[1][i] = make_float4(kPolyNom[4], kAeroNom[0], kAeroNom[1], kAeroNom[2]);
        p.D[2][i] = make_float4(kAeroNom[3], kAeroNom[4], 0.f, 0.f);
        p.D[3][i] = make_float4(p.lag_gain_fixed, p.lag_gain_fixed, p.lag_gain_fixed, p.lag_gain_fixed);
    }
}

__global__ void fill_actions_kernel(float4* out, int n, long long env_offset, uint32_t step, uint32_t k0, uint32_t k1) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint4 r = philox4x32_10((uint32_t)(env_offset + i), step, 0, STREAM_ACTIONS, k0, k1);
    out[i] = make_float4(2.0f * u01(r.x) - 1.0f, 2.0f * u01(r.y) - 1.0f, 2.0f * u01(r.z) - 1.0f, 2.0f * u01(r.w) - 1.0f);
}

__global__ void reduce_stats_kernel(double* partial, double* out) {
    // kStatSlots x kNumStats partial sums -> out[kNumStats]; clears the partials
    const int j = threadIdx.x;
    if (j >= kNumStats) return;
    double acc = 0.0;
    for (int s = 0; s < kStatSlots; ++s) { acc += partial[s * kStatStride + j]; partial[s * kStatStride + j] = 0.0; }
    out[j] = acc;
}

// SoA planes <-> TACO_STATE_WORDS floats per env (layout documented in DESIGN.md "state export").  Row j of `out` is env ids[j]
// (ids = null: env j) for j < count; an id outside [0, n) gives a row of NaN (taco_env_record_state takes device ids unchecked)
__global__ void export_state_kernel(StepParams p, const int32_t* ids, int count, float* out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const int i = ids ? ids[j] : j;
    float* o = out + (size_t)j * TACO_STATE_WORDS;
    if (i < 0 || i >= p.n) {
        for (int w = 0; w < TACO_STATE_WORDS; ++w) o[w] = __int_as_float(0x7fc00000);
        return;
    }
    const float4 s0 = p.S[0][i], s1 = p.S[1][i], s2 = p.S[2][i], s3 = p.S[3][i], s4 = p.S[4][i], s5 = p.S[5][i], s6 = p.S[6][i], s7 = p.S[7][i];
    o[0] = s0.x; o[1] = s0.y; o[2] = s0.z;                    // pos
    o[3] = s0.w; o[4] = s1.x; o[5] = s1.y; o[6] = s1.z;       // quat xyzw
    o[7] = s1.w; o[8] = s2.x; o[9] = s2.y;                    // linvel (world)
    o[10] = s2.z; o[11] = s2.w; o[12] = s3.x;                 // angvel (world)
    o[13] = s3.y; o[14] = s3.z; o[15] = s3.w;                 // target pos
    o[16] = 0.f; o[17] = 0.f; o[18] = s4.x; o[19] = s4.y;     // target quat
    o[20] = s4.z; o[21] = s4.w;                               // roll_old, roll_continuous
    o[22] = s5.x; o[23] = s5.y; o[24] = s5.z; o[25] = s5.w;   // rotor speed
    o[26] = s6.x; o[27] = s6.y; o[28] = s6.z;                 // PID previous error
    o[29] = s6.w;                                             // command state (rotate speed / flip_radian)
    o[30] = s7.x; o[31] = s7.y; o[32] = s7.z;                 // battery u_1, E_c, time
    o[33] = s7.w;                                             // running episode return
    const uint32_t qm = p.qmeta[i];
    o[34] = (float)p.progress[i];
    o[35] = (float)qm_len(qm);                                // actions_remained_length
    o[36] = (float)qm_runs(qm);                               // live runs in the action queue
    o[37] = (float)qm_ovf(qm);                                // delay overflow flag
    o[38] = (float)p.reset_buf[i];
    o[39] = 0.f;                                              // (was: queue head; the head is implied by the step clock)
    if (p.has_dr) {
        const float4 d0 = p.D[0][i], d1 = p.D[1][i], d2 = p.D[2][i], d3 = p.D[3][i];
        o[40] = d0.x; o[41] = d0.y; o[42] = d0.z; o[43] = d0.w; o[44] = d1.x;             // omega polynomial
        o[45] = d1.y; o[46] = d1.z; o[47] = d1.w; o[48] = d2.x; o[49] = d2.y;             // aero k_f,k_tau,d_x,d_y,k_th
        o[50] = d3.x; o[51] = d3.y; o[52] = d3.z; o[53] = d3.w;                           // lag gains
    } else {
        for (int j = 0; j < 5; ++j) { o[40 + j] = kPolyNom[j]; o[45 + j] = kAeroNom[j]; }
        o[50] = o[51] = o[52] = o[53] = p.lag_gain_fixed;
    }
    for (int j = 54; j < TACO_STATE_WORDS; ++j) o[j] = 0.f;
}

__global__ void import_state_kernel(StepParams p, const float* in) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const float* o = in + (size_t)i * TACO_STATE_WORDS;
    p.S[0][i] = make_float4(o[0], o[1], o[2], o[3]);
    p.S[1][i] = make_float4(o[4], o[5], o[6], o[7]);
    p.S[2][i] = make_float4(o[8], o[9], o[10], o[11]);
    p.S[3][i] = make_float4(o[12], o[13], o[14], o[15]);
    p.S[4][i] = make_float4(o[18], o[19], o[20], o[21]);
    p.S[5][i] = make_float4(o[22], o[23], o[24], o[25]);
    p.S[6][i] = make_float4(o[26], o[27], o[28], o[29]);
    p.S[7][i] = make_float4(o[30], o[31], o[32], o[33]);
    // the pending-action runs themselves are not imported (only their scalar meta: length / counts), but their end slots are kept
    // on the absolute clock 10 * progress (fpv_step_kernel.cuh): a changed progress counter rebases them
    const int shift = 10 * ((int)o[34] - p.progress[i]);
    if (shift != 0)
        for (int k = 0; k < kQueueCap; ++k) {
            const size_t j = (size_t)k * p.n_pad + i;
            const int e = (int)p.qend[j] + shift;
            p.qend[j] = (uint16_t)(e < 0 ? 0 : (e > 65535 ? 65535 : e));
        }
    p.progress[i] = (int)o[34];
    p.reset_buf[i] = (long long)o[38];
    p.qmeta[i] = qm_pack((uint32_t)o[36], (uint32_t)o[35], (uint32_t)o[37]);
    if (p.has_dr) {
        p.D[0][i] = make_float4(o[40], o[41], o[42], o[43]);
        p.D[1][i] = make_float4(o[44], o[45], o[46], o[47]);
        p.D[2][i] = make_float4(o[48], o[49], 0.f, 0.f);
        p.D[3][i] = make_float4(o[50], o[51], o[52], o[53]);
    }
}

// exhaustive check of the constant-division sequence against IEEE division: every float bit pattern whose magnitude
// is in [2^-60, 2^60] (and +-0), for every divisor the step kernel uses
template <int K>
__device__ __forceinline__ bool divc_case(float x, float c) {
    const float a = divc_impl(x, c, 1.0f / c), b = x / c;
    return __float_as_uint(a) == __float_as_uint(b) || (a == 0.0f && b == 0.0f);   // -0 / C gives +0 (sign of zero only)
}
__global__ void selftest_divc_kernel(unsigned long long* bad, float dt, uint32_t* rec) {
    const float cs[11] = {4500.0f, 0.75f, 9000.0f, 3.3f, 3.0f, 1000.0f, kPi, 6.0f, 100.0f, dt, 2.0f};
    unsigned long long local = 0;
    for (unsigned long long b = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; b < (1ull << 32); b += (unsigned long long)gridDim.x * blockDim.x) {
        const float x = __uint_as_float((uint32_t)b);
        const float ax = fabsf(x);
        if (!(ax == 0.0f || (ax >= 8.673617379884035e-19f && ax <= 1.152921504606847e18f))) continue;
#pragma unroll
        for (int k = 0; k < 11; ++k)
            if (!divc_case<0>(x, cs[k])) {
                local += 1;
                const unsigned long long slot = atomicAdd(bad + 1, 1ull);
                if (slot < 32) { rec[2 * slot] = (uint32_t)b; rec[2 * slot + 1] = (uint32_t)k; }
            }
    }
    if (local) atomicAdd(bad, local);
}

// atan2_poly (fpv_math.cuh) against double-precision atan2 on a dense sweep of the circle at many radii, plus the axes and the
// origin: out[0] = max error in ulp of the exact result (as float bits of the largest value seen), out[1] = non-finite results
__global__ void selftest_atan2_kernel(uint32_t* out, uint32_t n_angles) {
    float worst = 0.0f;
    uint32_t nonfinite = 0;
    for (uint32_t a = blockIdx.x * blockDim.x + threadIdx.x; a < n_angles; a += gridDim.x * blockDim.x) {
        const double ang = -3.14159265358979323846 + 6.28318530717958647692 * ((double)a + 0.5) / (double)n_angles;
#pragma unroll 1
        for (int e = -12; e <= 4; e += 2) {                    // radii 2^-12 .. 2^4: the roll arguments have radius <= 2
            const double rad = exp2((double)e) * (1.0 + 0.37 * (double)(a & 7u) / 8.0);
            const float y = (float)(rad * sin(ang)), x = (float)(rad * cos(ang));
            const float got = atan2_poly(y, x);
            const double ref = atan2((double)y, (double)x);
            const float ulp = __uint_as_float(__float_as_uint(fabsf((float)ref)) + 1u) - fabsf((float)ref);
            if (!isfinite(got)) nonfinite += 1;
            else worst = fmaxf(worst, (float)(fabs((double)got - ref) / (double)ulp));
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {                  // axes and origin: exact values expected
        const float ys[5] = {0.0f, 1.0f, 0.0f, -1.0f, 0.0f}, xs[5] = {1.0f, 0.0f, -1.0f, 0.0f, 0.0f};
        const float want[5] = {0.0f, kHalfPi, kPi, -kHalfPi, 0.0f};
        for (int k = 0; k < 5; ++k) {
            const float got = atan2_poly(ys[k], xs[k]);
            if (!isfinite(got)) nonfinite += 1;
            else worst = fmaxf(worst, fabsf(got - want[k]) / 1.1920929e-7f);
        }
    }
    atomicMax(out, __float_as_uint(worst));                     // non-negative floats order like their bit patterns
    if (nonfinite) atomicAdd(out + 1, nonfinite);
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace taco

using namespace taco;

extern "C" {

const char* taco_last_error(void) { return g_err.c_str(); }

int taco_selftest_divc(int device, float dt, uint64_t* n_mismatch) {
    if (!n_mismatch) return fail(TACO_E_INVALID, "taco_selftest_divc: null argument");
    DevGuard guard(device);
    unsigned long long* d = nullptr;
    TACO_CUDA(cudaMalloc(&d, 2 * sizeof(unsigned long long) + 64 * sizeof(uint32_t)));
    TACO_CUDA(cudaMemset(d, 0, 2 * sizeof(unsigned long long) + 64 * sizeof(uint32_t)));
    selftest_divc_kernel<<<148 * 8, 256>>>(d, dt, (uint32_t*)(d + 2)); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    unsigned long long h[2 + 32] = {0};
    TACO_CUDA(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
    cudaFree(d);
    *n_mismatch = h[0];
    if (h[0]) {
        std::string msg = "divc mismatches (x bits, divisor index):";
        const uint32_t* rec = (const uint32_t*)(h + 2);
        for (unsigned long long i = 0; i < h[0] && i < 32; ++i) { char buf[64]; snprintf(buf, sizeof(buf), " (0x%08x,%u)", rec[2 * i], rec[2 * i + 1]); msg += buf; }
        g_err = msg;
    }
    return TACO_OK;
}
int taco_selftest_atan2(int device, uint32_t n_angles, float* max_ulp, uint32_t* n_nonfinite) {
    if (!max_ulp || !n_nonfinite || n_angles == 0) return fail(TACO_E_INVALID, "taco_selftest_atan2: null / empty argument");
    DevGuard guard(device);
    uint32_t* d = nullptr;
    TACO_CUDA(cudaMalloc(&d, 2 * sizeof(uint32_t)));
    TACO_CUDA(cudaMemset(d, 0, 2 * sizeof(uint32_t)));
    selftest_atan2_kernel<<<148 * 4, 256>>>(d, n_angles); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    uint32_t h[2] = {0, 0};
    TACO_CUDA(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
    cudaFree(d);
    memcpy(max_ulp, &h[0], sizeof(float));
    *n_nonfinite = h[1];
    return TACO_OK;
}
int taco_abi_version(void) { return TACO_ABI_VERSION; }
int taco_launch_count(uint64_t* out) {
    if (!out) return fail(TACO_E_INVALID, "taco_launch_count: null argument");
    *out = (uint64_t)taco::g_launches.load(std::memory_order_relaxed);
    return TACO_OK;
}

int taco_env_create(const TacoCfg* cfg, int device, TacoEnv** out) {
    if (!cfg || !out) return fail(TACO_E_INVALID, "taco_env_create: null argument");
    *out = nullptr;
    if (cfg->abi_version != TACO_ABI_VERSION) return fail(TACO_E_INVALID, "taco_env_create: ABI version mismatch");
    if (cfg->num_envs <= 0) return fail(TACO_E_INVALID, "num_envs must be positive");
    if (cfg->task_mode < TACO_TASK_POS || cfg->task_mode > TACO_TASK_MIX) return fail(TACO_E_INVALID, "unknown task_mode");
    if (cfg->len_obs < 1 || cfg->len_states < 1 || cfg->len_obs > 64 || cfg->len_states > 64)
        return fail(TACO_E_INVALID, "len_obs / len_states must be in [1, 64]");
    if (cfg->control_freq_inv < 1) return fail(TACO_E_INVALID, "control_freq_inv must be >= 1");
    if (cfg->control_freq_inv != 10)
        return fail(TACO_E_INVALID, "control_freq_inv must be 10: the delay buffer advances 10 slots per RL step (fpv_asymmetry.py:326,378)");
    if (cfg->substeps < 1 || cfg->substeps > 16) return fail(TACO_E_INVALID, "substeps must be in [1, 16]");
    if (cfg->delay_time < 0 || cfg->delay_time > 100) return fail(TACO_E_INVALID, "delay_time must be in [0, 100] ms (delay_time_max is 100, fpv_asymmetry.py:329)");
    if (cfg->max_episode_length < 2 || (long long)cfg->max_episode_length * 10 + 200 >= 65536)
        return fail(TACO_E_INVALID, "max_episode_length must be in [2, 6500]");
    if (!(cfg->dt > 0.f) || !(cfg->rotor_response_time > 0.f)) return fail(TACO_E_INVALID, "dt and rotor_response_time must be positive");
    if (cfg->env_offset < 0 || cfg->num_envs_global < cfg->env_offset + cfg->num_envs || cfg->num_envs_global > 0xFFFFFFFFll)
        return fail(TACO_E_INVALID, "env_offset / num_envs_global inconsistent");
    int ndev = 0;
    TACO_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(TACO_E_INVALID, "no such CUDA device");
    DevGuard guard(device);

    TacoEnv* e = new (std::nothrow) TacoEnv();
    if (!e) return fail(TACO_E_NOMEM, "host allocation failed");
    e->cfg = *cfg;
    e->device = device;
    e->n = cfg->num_envs;
    e->n_pad = (int)align_up((size_t)cfg->num_envs, kBlock);
    const size_t np = (size_t)e->n_pad;
    StepParams& p = e->p;
    memset(&p, 0, sizeof(p));
    p.n = e->n; p.n_pad = e->n_pad;
    p.env_offset = cfg->env_offset;
    // python: int(num_envs / 3 * 1), int(num_envs / 3 * 2) in double (fpv_asymmetry.py:924-925)
    p.mix_n1 = (long long)((double)cfg->num_envs_global / 3 * 1);
    p.mix_n2 = (long long)((double)cfg->num_envs_global / 3 * 2);
    p.task_mode = cfg->task_mode; p.len_obs = cfg->len_obs; p.len_states = cfg->len_states;
    p.max_len = cfg->max_episode_length; p.cfi = cfg->control_freq_inv; p.substeps = cfg->substeps; p.delay_time = cfg->delay_time;
    p.flags = cfg->flags;
    p.seed_lo = (uint32_t)(cfg->seed & 0xFFFFFFFFull); p.seed_hi = (uint32_t)(cfg->seed >> 32);
    p.dt = cfg->dt;
    p.inv_dt = 1.0f / cfg->dt;
    p.h = (float)((double)cfg->dt / cfg->substeps);
    p.half_h = (float)(0.5 * ((double)cfg->dt / cfg->substeps));
    {   // python evaluates hh*hh, -1/6, 1/120, 1/24 in double and casts at the tensor op (oracle/rigid_body.py)
        const double hh = 0.5 * ((double)cfg->dt / cfg->substeps);
        p.half_h2 = (float)(hh * hh); p.c_sin3 = (float)(-1.0 / 6.0); p.c_sin5 = (float)(1.0 / 120.0); p.c_cos4 = (float)(1.0 / 24.0);
    }
    p.inv_mass = (float)(1.0 / (0.46 + 8 * 1e-7));            // fpv_without_duct.xml:6,11-13
    p.clip_actions = cfg->clip_actions;
    // thrust_dynamics.py:84 `sample_time / response_time` is python-float / tensor = tensor.reciprocal() * float
    p.lag_gain_fixed = (cfg->flags & TACO_F_ROTOR_RESPONSE) ? (1.0f / cfg->rotor_response_time) * 0.001f : (1.0f / 0.001f) * 0.001f;
    p.has_dr = (cfg->flags & (TACO_F_RANDOM_ROTORDYNAMIC_COE | TACO_F_RANDOM_ROTOR_RESPONSE | TACO_F_RANDOM_AERODYNAMIC_COE)) ? 1 : 0;
    refresh_derived(e);
    if (cudaMalloc(&e->diff_dev, 9 * sizeof(float)) != cudaSuccess) { delete e; return fail(TACO_E_NOMEM, "cudaMalloc of the difficulty block failed"); }
    if (upload_derived(e) != cudaSuccess) { cudaFree(e->diff_dev); delete e; return fail(TACO_E_CUDA, "upload of the difficulty block failed"); }

    // ---- one arena, every plane 512-byte aligned
    const size_t A = 512;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, A); return o; };
    size_t oS[8], oD[4];
    for (int k = 0; k < 8; ++k) oS[k] = take(np * sizeof(float4));
    for (int k = 0; k < 4; ++k) oD[k] = p.has_dr ? take(np * sizeof(float4)) : 0;
    const size_t oProg = take(np * sizeof(int)), oMeta = take(np * sizeof(uint32_t));
    const size_t oQact = take((size_t)kQueueCap * np * sizeof(float4)), oQend = take((size_t)kQueueCap * np * sizeof(uint16_t));
    const size_t oReset = take(np * sizeof(long long)), oTout = take(np), oRew = take(np * sizeof(float));
    // state history strip: L + K - 1 frames per env with K = max(16, L) (K >= L keeps the rebase of write_strip free of overlap;
    // at L = 5 an env's row is 20 frames = 2080 B, a multiple of the 32-byte sector)
    e->strip_period = cfg->len_states > 16 ? cfg->len_states : 16;
    e->strip_frames = cfg->len_states + e->strip_period - 1;
    const size_t obs_bytes = np * cfg->len_obs * kObs * sizeof(float), st_bytes = np * e->strip_frames * kObs * sizeof(float);
    const size_t oObs0 = take(obs_bytes), oObs1 = take(obs_bytes), oSt = take(st_bytes);
    const size_t oStats = take((size_t)kStatSlots * kStatStride * sizeof(double)), oStatsOut = take(kNumStats * sizeof(double));
    const size_t oStage = take(np * sizeof(float4));
    const size_t oDbg = (cfg->flags & TACO_F_DEBUG_DELAY) ? take((size_t)cfg->control_freq_inv * np * sizeof(float4)) : 0;
    e->arena_bytes = off;
    cudaError_t ce = cudaMalloc(&e->arena, e->arena_bytes);
    if (ce != cudaSuccess) { delete e; return fail(TACO_E_NOMEM, std::string("cudaMalloc of env arena failed: ") + cudaGetErrorString(ce)); }
    char* base = (char*)e->arena;
    ce = cudaMemset(base, 0, e->arena_bytes);
    if (ce != cudaSuccess) { cudaFree(e->arena); delete e; return fail(TACO_E_CUDA, cudaGetErrorString(ce)); }
    for (int k = 0; k < 8; ++k) p.S[k] = (float4*)(base + oS[k]);
    for (int k = 0; k < 4; ++k) p.D[k] = p.has_dr ? (float4*)(base + oD[k]) : nullptr;
    p.progress = (int*)(base + oProg); p.qmeta = (uint32_t*)(base + oMeta);
    p.qact = (float4*)(base + oQact); p.qend = (uint16_t*)(base + oQend);
    p.reset_buf = (long long*)(base + oReset); p.time_outs = (uint8_t*)(base + oTout); p.rew = (float*)(base + oRew);
    e->obs_ab[0] = (float*)(base + oObs0); e->obs_ab[1] = (float*)(base + oObs1);
    e->strip = (float*)(base + oSt);
    p.strip_frames = e->strip_frames; p.strip_period = e->strip_period;
    p.stats = (double*)(base + oStats); e->stats_out = (double*)(base + oStatsOut);
    e->actions_stage = (float4*)(base + oStage);
    e->dbg_delay = (cfg->flags & TACO_F_DEBUG_DELAY) ? (float4*)(base + oDbg) : nullptr;
    p.dbg_delay = e->dbg_delay;
    e->cur = 0;
    e->step_index = 0;
    init_state_kernel<<<(e->n_pad + 255) / 256, 256>>>(p); TACO_LAUNCHED();
    ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) { cudaFree(e->arena); delete e; return fail(TACO_E_CUDA, std::string("init kernel: ") + cudaGetErrorString(ce)); }
    *out = e;
    return TACO_OK;
}

int taco_env_destroy(TacoEnv* env) {
    if (!env) return TACO_OK;
    DevGuard guard(env->device);
    if (env->pipe_ready) {
        cudaStreamDestroy(env->s_h2d); cudaStreamDestroy(env->s_d2h);
        for (int k = 0; k < TacoEnv::kKernelStreams; ++k) cudaStreamDestroy(env->s_k[k]);
        for (int c = 0; c < TacoEnv::kMaxChunks; ++c) { cudaEventDestroy(env->ev_h2d[c]); cudaEventDestroy(env->ev_k[c]); }
        cudaEventDestroy(env->ev_begin); cudaEventDestroy(env->ev_end);
    }
    if (env->export_stage) cudaFree(env->export_stage);
    if (env->log_mem) cudaFree(env->log_mem);
    if (env->rep_mem) cudaFree(env->rep_mem);
    if (env->arena) cudaFree(env->arena);
    if (env->step_counter) cudaFree(env->step_counter);
    if (env->diff_dev) cudaFree(env->diff_dev);
    delete env;
    return TACO_OK;
}

// first frame of the current window of the state history strip (rows of strip_frames frames: not a contiguous (n, L, 26) array)
static float* strip_window(TacoEnv* env) {
    return env->strip + (size_t)(env->step_index % (uint32_t)env->strip_period) * kObs;
}
static size_t strip_row_bytes(TacoEnv* env) { return (size_t)env->strip_frames * kObs * sizeof(float); }

int taco_env_buffers(TacoEnv* env, TacoBuffers* out) {
    if (!env || !out) return fail(TACO_E_INVALID, "taco_env_buffers: null argument");
    if (env->ring_slots) {
        out->obs = env->ring_obs + (size_t)env->n * env->cfg.len_obs * kObs * env->ring_cur;
        out->states = env->ring_states + (size_t)env->n * env->cfg.len_states * kObs * env->ring_cur;
    } else {
        out->obs = env->obs_ab[env->cur];
        out->states = strip_window(env);
    }
    out->rew = env->p.rew;
    out->reset = (int64_t*)env->p.reset_buf;
    out->time_outs = env->p.time_outs;
    out->progress = env->p.progress;
    for (int k = 0; k < 2; ++k) out->obs_ab[k] = env->obs_ab[k];
    out->states_ab[0] = env->strip; out->states_ab[1] = nullptr;
    out->num_envs = env->n; out->len_obs = env->cfg.len_obs; out->len_states = env->cfg.len_states; out->num_obs = kObs;
    return TACO_OK;
}

// history buffers of the next step: the env's own ping-pong pair, or consecutive slots of the attached rollout ring
static int bind_history(TacoEnv* env) {
    StepParams& p = env->p;
    if (env->ring_slots) {
        if (env->ring_cur + 1 >= env->ring_slots)
            return fail(TACO_E_INVALID, "rollout ring is full: call taco_env_rewind_rollout before stepping again");
        const size_t so = (size_t)env->n * env->cfg.len_obs * kObs, ss = (size_t)env->n * env->cfg.len_states * kObs;
        p.obs_in = env->ring_obs + so * env->ring_cur; p.obs_out = env->ring_obs + so * (env->ring_cur + 1);
        p.states_in = env->ring_states + ss * env->ring_cur; p.states_out = env->ring_states + ss * (env->ring_cur + 1);
        p.states_strip = nullptr;
        p.roll_rew = env->ring_rew ? env->ring_rew + (size_t)env->n * env->ring_cur : nullptr;
        p.roll_done = env->ring_rew ? env->ring_done + (size_t)env->n * env->ring_cur : nullptr;
        p.roll_tout = env->ring_rew ? env->ring_tout + (size_t)env->n * env->ring_cur : nullptr;
    } else {
        const int nxt = env->cur ^ 1;
        p.obs_in = env->obs_ab[env->cur]; p.obs_out = env->obs_ab[nxt];
        p.states_in = nullptr; p.states_out = nullptr; p.states_strip = env->strip;
        p.roll_rew = nullptr; p.roll_done = nullptr; p.roll_tout = nullptr;
    }
    return TACO_OK;
}
static void advance_history(TacoEnv* env) {
    if (env->ring_slots) env->ring_cur += 1; else env->cur ^= 1;
    env->step_index += 1;
}

// the step index of the next launch: absolute, or an offset to the device counter in graph mode
static void bind_step_index(TacoEnv* env) {
    StepParams& p = env->p;
    if (env->graph_mode) { p.step_base = env->step_counter; p.step_index = env->step_index - env->graph_origin; }
    else { p.step_base = nullptr; p.step_index = env->step_index; }
}

__global__ void step_counter_kernel(uint32_t* c, uint32_t value, int add) { *c = add ? *c + value : value; }

// the episode log's update for the step just taken (after advance_history): a launch of its own, never part of the step kernel
static int log_after_step(TacoEnv* env, cudaStream_t s) {
    if (!env->log_mem) return TACO_OK;
    const uint32_t t = env->step_index - 1u;
    const uint32_t step = env->graph_mode ? t - env->graph_origin : t;
    episode_log_update_kernel<<<(env->n + 255) / 256, 256, 0, s>>>(env->p, env->log_acc[0], env->log_acc[1], env->log_rec, env->log_count,
                                                                  env->log_cap, step, env->graph_mode ? env->step_counter : nullptr);
    TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

// the attach initialisation of an attached log (a no-op without one): the episodes in progress are discarded
static int log_restart(TacoEnv* env, cudaStream_t s) {
    if (!env->log_mem) return TACO_OK;
    episode_log_init_kernel<<<(env->n_pad + 255) / 256, 256, 0, s>>>(env->p, env->log_acc[0], env->log_acc[1]); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

// the start rule of attached rollout episodes (a no-op without them): the episodes in progress are discarded, and the ring rows
// written so far count as scanned
static int rep_restart(TacoEnv* env, cudaStream_t s) {
    if (!env->rep_mem) return TACO_OK;
    rollout_episodes_init_kernel<<<(env->n + 255) / 256, 256, 0, s>>>(env->p.reset_buf, env->n, env->rep_ret, env->rep_len, env->rep_live);
    TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    env->rep_scanned = env->ring_slots ? env->ring_cur : 0;
    return TACO_OK;
}

// the step kernel of the env's build (-fmad=false or FMA contraction) with the bound StepParams
static void launch_step(TacoEnv* env, cudaStream_t s) {
    if (env->cfg.flags & TACO_F_STRICT_FP) launch_fpv_step_strict(env->p, s);
    else launch_fpv_step_fast(env->p, s);
}

// The step as one launch over the whole shard.  actions and the host_* result buffers (null, or device-visible addresses of the
// caller's pinned host memory) are bound for this launch only: the host pointers are cleared whatever the launch returns, and a
// failed launch leaves the history and the step index where they were.  sync: return after the step has finished.
static int step_single(TacoEnv* env, const void* actions, float* host_rew, long long* host_reset, uint8_t* host_tout, uint8_t* host_flags,
                       cudaStream_t s, bool sync) {
    StepParams& p = env->p;
    int rc = bind_history(env);
    if (rc != TACO_OK) return rc;
    p.actions = (const float4*)actions;
    p.host_rew = host_rew; p.host_reset = host_reset; p.host_tout = host_tout; p.host_flags = host_flags;
    bind_step_index(env);
    launch_step(env, s);
    const cudaError_t launch = cudaGetLastError();
    p.host_rew = nullptr; p.host_reset = nullptr; p.host_tout = nullptr; p.host_flags = nullptr;
    TACO_CUDA(launch);
    advance_history(env);
    rc = log_after_step(env, s);
    if (rc != TACO_OK) return rc;
    if (sync) TACO_CUDA(cudaStreamSynchronize(s));
    return TACO_OK;
}

int taco_env_step(TacoEnv* env, const float* actions_dev, void* stream) {
    if (!env || !actions_dev) return fail(TACO_E_INVALID, "taco_env_step: null argument");
    if (((uintptr_t)actions_dev & 15u) != 0) return fail(TACO_E_INVALID, "actions must be 16-byte aligned (contiguous (N,4) float32)");
    DevGuard guard(env->device);
    return step_single(env, actions_dev, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream, false);
}

// device-visible address of a pinned (cudaHostAlloc / cudaHostRegister) host buffer, or null for pageable memory
static void* mapped_ptr(const void* host) {
    if (!host) return nullptr;
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, const_cast<void*>(host), 0) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return d;
}

static int pipe_init(TacoEnv* env) {
    if (env->pipe_ready) return TACO_OK;
    TACO_CUDA(cudaStreamCreateWithFlags(&env->s_h2d, cudaStreamNonBlocking));
    TACO_CUDA(cudaStreamCreateWithFlags(&env->s_d2h, cudaStreamNonBlocking));
    for (int k = 0; k < TacoEnv::kKernelStreams; ++k) TACO_CUDA(cudaStreamCreateWithFlags(&env->s_k[k], cudaStreamNonBlocking));
    for (int c = 0; c < TacoEnv::kMaxChunks; ++c) {
        TACO_CUDA(cudaEventCreateWithFlags(&env->ev_h2d[c], cudaEventDisableTiming));
        TACO_CUDA(cudaEventCreateWithFlags(&env->ev_k[c], cudaEventDisableTiming));
    }
    TACO_CUDA(cudaEventCreateWithFlags(&env->ev_begin, cudaEventDisableTiming));
    TACO_CUDA(cudaEventCreateWithFlags(&env->ev_end, cudaEventDisableTiming));
    env->pipe_ready = true;
    return TACO_OK;
}

// The step through HOST buffers.  Envs are independent, so the shard is cut into chunks of whole CTAs and the three
// legs of successive chunks overlap: chunk c+1's actions cross PCIe while chunk c steps and chunk c-1's results return
// (H2D and D2H use opposite directions of the link).  Chunk kernels rotate over a few internal streams, so the partial
// last wave of one chunk overlaps the first wave of the next; everything is ordered after the work already queued on
// the caller's stream, which in turn waits for the last copy before the call synchronises it.
// Compact result format of the host-buffer step (opt-in; the reference dtypes stay the default): rew f32 + ONE flag byte per env
// (bit 0 = reset_buf != 0, bit 1 = time_outs) = 5 bytes of device->host traffic per env instead of 13 (8 of which are an int64
// reset).  Mapped mode only: every buffer must be pinned (cudaHostAlloc / cudaHostRegister / torch pin_memory).
int taco_env_step_host_compact(TacoEnv* env, const float* actions_host, float* rew_host, uint8_t* flags_host, void* stream) {
    if (!env || !actions_host || !flags_host) return fail(TACO_E_INVALID, "taco_env_step_host_compact: null argument");
    if (((uintptr_t)actions_host & 15u) != 0) return fail(TACO_E_INVALID, "taco_env_step_host_compact: actions must be 16-byte aligned");
    DevGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    void* d_act = mapped_ptr(actions_host);
    void* d_rew = mapped_ptr(rew_host);
    void* d_flags = mapped_ptr(flags_host);
    if (!d_act || (rew_host && !d_rew) || !d_flags)
        return fail(TACO_E_INVALID, "taco_env_step_host_compact: the host buffers must be pinned (device-mapped); use taco_env_step_host for pageable memory");
    return step_single(env, d_act, (float*)d_rew, nullptr, nullptr, (uint8_t*)d_flags, s, true);
}

int taco_env_step_host(TacoEnv* env, const float* actions_host, float* rew_host, int64_t* reset_host, uint8_t* time_outs_host,
                       void* stream) {
    if (!env || !actions_host) return fail(TACO_E_INVALID, "taco_env_step_host: null argument");
    DevGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = pipe_init(env);
    if (rc != TACO_OK) return rc;
    StepParams& p = env->p;
    // Mapped mode (default whenever the caller's buffers are pinned, i.e. have a device-visible address): ONE launch; the
    // kernel loads each env's action from host memory and posts rew / reset / time-outs into host memory itself, so the
    // PCIe transfers of a CTA overlap the arithmetic of the ~890 other resident CTAs and there is no fill / drain phase of
    // a copy pipeline.  TACO_HOST_MODE=copy forces the chunked copy pipeline below (also the path for pageable memory).
    const char* hm = getenv("TACO_HOST_MODE");                      // read per call: tests and tuning runs switch it
    const int host_mode = (hm && !strcmp(hm, "copy")) ? 1 : 0;
    if (host_mode == 0 && ((uintptr_t)actions_host & 15u) == 0) {
        void* d_act = mapped_ptr(actions_host);
        void* d_rew = mapped_ptr(rew_host); void* d_reset = mapped_ptr(reset_host); void* d_tout = mapped_ptr(time_outs_host);
        if (d_act && (!rew_host || d_rew) && (!reset_host || d_reset) && (!time_outs_host || d_tout))
            return step_single(env, d_act, (float*)d_rew, (long long*)d_reset, (uint8_t*)d_tout, nullptr, s, true);
    }
    const int total_blocks = env->n_pad / kBlock;
    // 4 equal chunks of at least 512 CTAs (64 Ki envs): measured best of 4 / 8 / 12 / 16 equal chunks and of a graded
    // 1-2-4-5-3-1 schedule at 2 Mi envs (per-copy and per-launch overheads outweigh shorter fill / drain phases; the call
    // is bound by the 16 B/env action upload at ~50 GB/s).  TACO_HOST_CHUNKS=<n> overrides (tuning aid).
    static const int forced_chunks = [] { const char* e = getenv("TACO_HOST_CHUNKS"); const int v = e ? atoi(e) : 0; return v > 0 ? v : 0; }();
    int bounds[TacoEnv::kMaxChunks + 1];
    int nchunks = 0;
    bounds[0] = 0;
    {
        int want = forced_chunks ? forced_chunks : 4;
        if (want > TacoEnv::kMaxChunks) want = TacoEnv::kMaxChunks;
        int per = (total_blocks + want - 1) / want;
        if (per < 512) per = 512;
        for (int b = per; nchunks < TacoEnv::kMaxChunks; b += per) { bounds[++nchunks] = b < total_blocks ? b : total_blocks; if (b >= total_blocks) break; }
    }
    bounds[nchunks] = total_blocks;
    rc = bind_history(env);
    if (rc != TACO_OK) return rc;
    p.actions = (const float4*)env->actions_stage;
    bind_step_index(env);
    const bool want_out = rew_host || reset_host || time_outs_host;
    TACO_CUDA(cudaEventRecord(env->ev_begin, s));                    // work already queued on the caller's stream comes first
    TACO_CUDA(cudaStreamWaitEvent(env->s_h2d, env->ev_begin, 0));
    for (int k = 0; k < TacoEnv::kKernelStreams; ++k) TACO_CUDA(cudaStreamWaitEvent(env->s_k[k], env->ev_begin, 0));
    for (int c = 0; c < nchunks; ++c) {
        const int b0 = bounds[c], b1 = bounds[c + 1];
        if (b0 >= b1) continue;
        const size_t e0 = (size_t)b0 * kBlock;
        const size_t e1 = ((size_t)b1 * kBlock < (size_t)env->n) ? (size_t)b1 * kBlock : (size_t)env->n;
        const size_t cnt = e1 - e0;
        cudaStream_t sk = env->s_k[c % TacoEnv::kKernelStreams];
        TACO_CUDA(cudaMemcpyAsync(env->actions_stage + e0, actions_host + e0 * 4, cnt * 4 * sizeof(float), cudaMemcpyHostToDevice, env->s_h2d));
        TACO_CUDA(cudaEventRecord(env->ev_h2d[c], env->s_h2d));
        TACO_CUDA(cudaStreamWaitEvent(sk, env->ev_h2d[c], 0));
        p.block0 = b0; p.nblocks = b1 - b0;
        launch_step(env, sk);
        TACO_CUDA(cudaGetLastError());
        TACO_CUDA(cudaEventRecord(env->ev_k[c], sk));
        if (want_out) {
            TACO_CUDA(cudaStreamWaitEvent(env->s_d2h, env->ev_k[c], 0));
            if (reset_host) TACO_CUDA(cudaMemcpyAsync(reset_host + e0, p.reset_buf + e0, cnt * sizeof(int64_t), cudaMemcpyDeviceToHost, env->s_d2h));
            if (rew_host) TACO_CUDA(cudaMemcpyAsync(rew_host + e0, p.rew + e0, cnt * sizeof(float), cudaMemcpyDeviceToHost, env->s_d2h));
            if (time_outs_host) TACO_CUDA(cudaMemcpyAsync(time_outs_host + e0, p.time_outs + e0, cnt, cudaMemcpyDeviceToHost, env->s_d2h));
        } else {
            TACO_CUDA(cudaStreamWaitEvent(s, env->ev_k[c], 0));
        }
    }
    p.block0 = 0; p.nblocks = 0;
    advance_history(env);
    if (want_out) {
        TACO_CUDA(cudaEventRecord(env->ev_end, env->s_d2h));         // s_d2h has waited for every chunk kernel
        TACO_CUDA(cudaStreamWaitEvent(s, env->ev_end, 0));
    }
    rc = log_after_step(env, s);                                     // s has waited for every chunk kernel
    if (rc != TACO_OK) return rc;
    TACO_CUDA(cudaStreamSynchronize(s));
    return TACO_OK;
}

int taco_env_graph_begin(TacoEnv* env, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_graph_begin: null argument");
    DevGuard guard(env->device);
    if (!env->step_counter) TACO_CUDA(cudaMalloc(&env->step_counter, sizeof(uint32_t)));
    step_counter_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(env->step_counter, env->step_index, 0); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    env->graph_mode = true;
    env->graph_origin = env->step_index;
    env->p.diff_dev = env->diff_dev;
    return TACO_OK;
}

int taco_env_graph_advance(TacoEnv* env, uint32_t steps, void* stream) {
    if (!env || !env->graph_mode) return fail(TACO_E_INVALID, "taco_env_graph_advance: call taco_env_graph_begin first");
    DevGuard guard(env->device);
    step_counter_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(env->step_counter, steps, 1); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

int taco_env_graph_end(TacoEnv* env, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_graph_end: null argument");
    if (!env->graph_mode) return TACO_OK;
    DevGuard guard(env->device);
    uint32_t v = 0;
    TACO_CUDA(cudaMemcpyAsync(&v, env->step_counter, sizeof(v), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    TACO_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    env->step_index = v;
    env->graph_mode = false;
    env->p.diff_dev = nullptr;
    return TACO_OK;
}

int taco_env_step_counter(TacoEnv* env, uint32_t** counter_dev, uint32_t* step_index_host) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_step_counter: null argument");
    if (counter_dev) *counter_dev = env->graph_mode ? env->step_counter : nullptr;
    if (step_index_host) *step_index_host = env->step_index;
    return TACO_OK;
}

int taco_env_attach_rollout(TacoEnv* env, float* obs_ring, float* states_ring, int32_t slots, float* rew_rows, float* done_rows,
                            uint8_t* time_out_rows, void* stream) {
    if (!env || !obs_ring || !states_ring) return fail(TACO_E_INVALID, "taco_env_attach_rollout: null argument");
    if (slots < 2) return fail(TACO_E_INVALID, "taco_env_attach_rollout: need at least 2 slots (horizon + 1)");
    if ((rew_rows || done_rows || time_out_rows) && !(rew_rows && done_rows && time_out_rows))
        return fail(TACO_E_INVALID, "taco_env_attach_rollout: rew / done / time-out rows must be given together (or all NULL)");
    if (((uintptr_t)obs_ring | (uintptr_t)states_ring) & 7u) return fail(TACO_E_INVALID, "taco_env_attach_rollout: rings must be 8-byte aligned");
    if (env->ring_slots) return fail(TACO_E_INVALID, "taco_env_attach_rollout: a ring is already attached");
    if (env->log_mem) return fail(TACO_E_INVALID, "taco_env_attach_rollout: an episode log is attached (evaluation only; detach it first)");
    DevGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    // the newest observation / state history moves into slot 0
    TACO_CUDA(cudaMemcpyAsync(obs_ring, env->obs_ab[env->cur], (size_t)env->n * env->cfg.len_obs * kObs * sizeof(float), cudaMemcpyDeviceToDevice, s));
    const size_t win = (size_t)env->cfg.len_states * kObs * sizeof(float);
    TACO_CUDA(cudaMemcpy2DAsync(states_ring, win, strip_window(env), strip_row_bytes(env), win, env->n, cudaMemcpyDeviceToDevice, s));
    env->ring_obs = obs_ring; env->ring_states = states_ring;
    env->ring_rew = rew_rows; env->ring_done = done_rows; env->ring_tout = time_out_rows;
    env->ring_slots = slots; env->ring_cur = 0;
    return rep_restart(env, s);
}

int taco_env_rewind_rollout(TacoEnv* env, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_rewind_rollout: null argument");
    if (!env->ring_slots) return fail(TACO_E_INVALID, "taco_env_rewind_rollout: no ring attached");
    DevGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    if (env->rep_scanned < env->ring_cur) {                          // unscanned rows: their episodes would be lost half-seen
        const int rc = rep_restart(env, s);
        if (rc != TACO_OK) return rc;
    }
    env->rep_scanned = 0;
    if (env->ring_cur > 0) {
        const size_t so = (size_t)env->n * env->cfg.len_obs * kObs, ss = (size_t)env->n * env->cfg.len_states * kObs;
        TACO_CUDA(cudaMemcpyAsync(env->ring_obs, env->ring_obs + so * env->ring_cur, so * sizeof(float), cudaMemcpyDeviceToDevice, s));
        TACO_CUDA(cudaMemcpyAsync(env->ring_states, env->ring_states + ss * env->ring_cur, ss * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    env->ring_cur = 0;
    return TACO_OK;
}

int taco_env_detach_rollout(TacoEnv* env, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_detach_rollout: null argument");
    if (!env->ring_slots) return TACO_OK;
    DevGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t so = (size_t)env->n * env->cfg.len_obs * kObs, ss = (size_t)env->n * env->cfg.len_states * kObs;
    TACO_CUDA(cudaMemcpyAsync(env->obs_ab[env->cur], env->ring_obs + so * env->ring_cur, so * sizeof(float), cudaMemcpyDeviceToDevice, s));
    const size_t win = (size_t)env->cfg.len_states * kObs * sizeof(float);
    TACO_CUDA(cudaMemcpy2DAsync(strip_window(env), strip_row_bytes(env), env->ring_states + ss * env->ring_cur, win, win, env->n, cudaMemcpyDeviceToDevice, s));
    env->ring_obs = env->ring_states = env->ring_rew = env->ring_done = nullptr; env->ring_tout = nullptr;
    env->ring_slots = 0; env->ring_cur = 0;
    env->rep_scanned = 0;
    return TACO_OK;
}

int taco_env_states_strip(TacoEnv* env, float** base, int32_t* frames, int32_t* period) {
    if (!env || !base || !frames || !period) return fail(TACO_E_INVALID, "taco_env_states_strip: null argument");
    *base = env->strip; *frames = env->strip_frames; *period = env->strip_period;
    return TACO_OK;
}

int taco_env_rollout_cursor(TacoEnv* env) { return (env && env->ring_slots) ? env->ring_cur : -1; }

int taco_env_reset_all(TacoEnv* env, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_reset_all: null argument");
    DevGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t np = (size_t)env->n_pad;
    for (int k = 0; k < 2; ++k) TACO_CUDA(cudaMemsetAsync(env->obs_ab[k], 0, np * env->cfg.len_obs * kObs * sizeof(float), s));
    TACO_CUDA(cudaMemsetAsync(env->strip, 0, np * strip_row_bytes(env), s));
    if (env->ring_slots) {                                           // restart the attached ring from a zeroed slot 0
        TACO_CUDA(cudaMemsetAsync(env->ring_obs, 0, (size_t)env->n * env->cfg.len_obs * kObs * sizeof(float), s));
        TACO_CUDA(cudaMemsetAsync(env->ring_states, 0, (size_t)env->n * env->cfg.len_states * kObs * sizeof(float), s));
        env->ring_cur = 0;
    }
    TACO_CUDA(cudaMemsetAsync(env->p.stats, 0, (size_t)kStatSlots * kStatStride * sizeof(double), s));
    init_state_kernel<<<(env->n_pad + 255) / 256, 256, 0, s>>>(env->p); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    int rc = log_restart(env, s);
    if (rc != TACO_OK) return rc;
    rc = rep_restart(env, s);
    if (rc != TACO_OK) return rc;
    env->step_index = 0;
    env->graph_mode = false;                                         // host-side counting again; taco_env_graph_begin re-arms
    env->p.diff_dev = nullptr;
    return TACO_OK;
}

int taco_env_set_difficulty(TacoEnv* env, float difficulty) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_set_difficulty: null argument");
    env->cfg.difficulty = difficulty;
    refresh_derived(env);
    DevGuard guard(env->device);
    TACO_CUDA(upload_derived(env));       // captured launches (graph mode) read the device copy
    return TACO_OK;
}

int taco_env_get_difficulty(TacoEnv* env, float* out) {
    if (!env || !out) return fail(TACO_E_INVALID, "taco_env_get_difficulty: null argument");
    *out = env->cfg.difficulty;
    return TACO_OK;
}

int taco_env_set_seed(TacoEnv* env, uint64_t seed) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_set_seed: null argument");
    env->cfg.seed = seed;
    env->p.seed_lo = (uint32_t)(seed & 0xFFFFFFFFull); env->p.seed_hi = (uint32_t)(seed >> 32);
    return TACO_OK;
}

int taco_env_stats(TacoEnv* env, double* out_dev, double* out_host, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_stats: null argument");
    DevGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    double* dst = out_dev ? out_dev : env->stats_out;
    reduce_stats_kernel<<<1, 32, 0, s>>>(env->p.stats, dst); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    if (out_host) {
        TACO_CUDA(cudaMemcpyAsync(out_host, dst, kNumStats * sizeof(double), cudaMemcpyDeviceToHost, s));
        TACO_CUDA(cudaStreamSynchronize(s));
    }
    return TACO_OK;
}

int taco_env_fill_random_actions(TacoEnv* env, float* actions_dev, uint32_t step_index, void* stream) {
    if (!env || !actions_dev) return fail(TACO_E_INVALID, "taco_env_fill_random_actions: null argument");
    DevGuard guard(env->device);
    fill_actions_kernel<<<(env->n + 255) / 256, 256, 0, (cudaStream_t)stream>>>((float4*)actions_dev, env->n, env->p.env_offset, step_index,
                                                                               env->p.seed_lo, env->p.seed_hi); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

int taco_env_export_state(TacoEnv* env, float* out_host) {
    if (!env || !out_host) return fail(TACO_E_INVALID, "taco_env_export_state: null argument");
    DevGuard guard(env->device);
    const size_t bytes = (size_t)env->n * TACO_STATE_WORDS * sizeof(float);
    if (!env->export_stage) TACO_CUDA(cudaMalloc(&env->export_stage, bytes));
    TACO_CUDA(cudaDeviceSynchronize());
    export_state_kernel<<<(env->n + 255) / 256, 256>>>(env->p, nullptr, env->n, env->export_stage); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    TACO_CUDA(cudaMemcpy(out_host, env->export_stage, bytes, cudaMemcpyDeviceToHost));
    return TACO_OK;
}

int taco_env_import_state(TacoEnv* env, const float* in_host) {
    if (!env || !in_host) return fail(TACO_E_INVALID, "taco_env_import_state: null argument");
    DevGuard guard(env->device);
    const size_t bytes = (size_t)env->n * TACO_STATE_WORDS * sizeof(float);
    if (!env->export_stage) TACO_CUDA(cudaMalloc(&env->export_stage, bytes));
    TACO_CUDA(cudaDeviceSynchronize());
    TACO_CUDA(cudaMemcpy(env->export_stage, in_host, bytes, cudaMemcpyHostToDevice));
    import_state_kernel<<<(env->n + 255) / 256, 256>>>(env->p, env->export_stage); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    int rc = log_restart(env, 0);
    if (rc != TACO_OK) return rc;
    rc = rep_restart(env, 0);
    if (rc != TACO_OK) return rc;
    TACO_CUDA(cudaDeviceSynchronize());
    return TACO_OK;
}

// ---- env-state checkpoint: the whole device arena (SoA state planes, DR planes, pending-action ring, reward / reset / time-out
// buffers, both observation history buffers, the state history strip, statistics partials) + a header.  The reference never checkpoints the env
// (SURVEY.md section 5); here a resumed run continues bit-identically.
struct CkptHeader {
    char magic[8];              // "TACOENV1"
    uint64_t arena_bytes;
    TacoCfg cfg;                // must match the env's (difficulty and seed are restored from the checkpoint)
    uint32_t step_index;
    int32_t cur;
};

int taco_env_checkpoint_size(TacoEnv* env, uint64_t* bytes) {
    if (!env || !bytes) return fail(TACO_E_INVALID, "taco_env_checkpoint_size: null argument");
    *bytes = sizeof(CkptHeader) + env->arena_bytes;
    return TACO_OK;
}

int taco_env_checkpoint_save(TacoEnv* env, void* out_host, uint64_t bytes) {
    if (!env || !out_host) return fail(TACO_E_INVALID, "taco_env_checkpoint_save: null argument");
    if (bytes != sizeof(CkptHeader) + env->arena_bytes) return fail(TACO_E_INVALID, "taco_env_checkpoint_save: wrong buffer size (taco_env_checkpoint_size)");
    if (env->ring_slots || env->graph_mode) return fail(TACO_E_INVALID, "taco_env_checkpoint_save: detach the rollout ring / leave graph mode first");
    DevGuard guard(env->device);
    CkptHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, "TACOENV1", 8);
    h.arena_bytes = env->arena_bytes; h.cfg = env->cfg; h.step_index = env->step_index; h.cur = env->cur;
    memcpy(out_host, &h, sizeof(h));
    TACO_CUDA(cudaDeviceSynchronize());
    TACO_CUDA(cudaMemcpy((char*)out_host + sizeof(h), env->arena, env->arena_bytes, cudaMemcpyDeviceToHost));
    return TACO_OK;
}

int taco_env_checkpoint_load(TacoEnv* env, const void* in_host, uint64_t bytes) {
    if (!env || !in_host) return fail(TACO_E_INVALID, "taco_env_checkpoint_load: null argument");
    if (bytes < sizeof(CkptHeader)) return fail(TACO_E_INVALID, "taco_env_checkpoint_load: truncated checkpoint");
    if (env->ring_slots || env->graph_mode) return fail(TACO_E_INVALID, "taco_env_checkpoint_load: detach the rollout ring / leave graph mode first");
    CkptHeader h;
    memcpy(&h, in_host, sizeof(h));
    if (memcmp(h.magic, "TACOENV1", 8) != 0) return fail(TACO_E_INVALID, "taco_env_checkpoint_load: not a taco env checkpoint");
    if (h.arena_bytes != env->arena_bytes || bytes != sizeof(CkptHeader) + h.arena_bytes)
        return fail(TACO_E_INVALID, "taco_env_checkpoint_load: checkpoint size does not match this env");
    TacoCfg a = h.cfg, b = env->cfg;
    a.difficulty = b.difficulty = 0.f; a.seed = b.seed = 0;
    if (memcmp(&a, &b, sizeof(TacoCfg)) != 0) return fail(TACO_E_INVALID, "taco_env_checkpoint_load: the checkpoint was written by an env with another configuration");
    DevGuard guard(env->device);
    TACO_CUDA(cudaDeviceSynchronize());
    TACO_CUDA(cudaMemcpy(env->arena, (const char*)in_host + sizeof(h), env->arena_bytes, cudaMemcpyHostToDevice));
    env->step_index = h.step_index; env->cur = h.cur;
    env->cfg.difficulty = h.cfg.difficulty;
    refresh_derived(env);
    TACO_CUDA(upload_derived(env));
    taco_env_set_seed(env, h.cfg.seed);
    if (env->log_mem) {
        const int rc = log_restart(env, 0);
        if (rc != TACO_OK) return rc;
        TACO_CUDA(cudaDeviceSynchronize());
    }
    return TACO_OK;
}

int taco_env_attach_episode_log(TacoEnv* env, int64_t capacity, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_attach_episode_log: null argument");
    if (capacity < 1) return fail(TACO_E_INVALID, "taco_env_attach_episode_log: capacity must be >= 1");
    if (env->log_mem) return fail(TACO_E_INVALID, "taco_env_attach_episode_log: a log is already attached");
    if (env->ring_slots) return fail(TACO_E_INVALID, "taco_env_attach_episode_log: a rollout ring is attached (the log reads the env's own result buffers)");
    DevGuard guard(env->device);
    const size_t acc_bytes = (size_t)env->n_pad * sizeof(float4);
    const size_t bytes = 256 + 2 * acc_bytes + (size_t)capacity * sizeof(TacoEpisode);
    void* mem = nullptr;
    const cudaError_t ce = cudaMalloc(&mem, bytes);
    if (ce != cudaSuccess) { cudaGetLastError(); return fail(TACO_E_NOMEM, std::string("cudaMalloc of the episode log failed: ") + cudaGetErrorString(ce)); }
    char* base = (char*)mem;
    env->log_mem = mem;
    env->log_count = (unsigned long long*)base;
    env->log_acc[0] = (float4*)(base + 256);
    env->log_acc[1] = (float4*)(base + 256 + acc_bytes);
    env->log_rec = (TacoEpisode*)(base + 256 + 2 * acc_bytes);
    env->log_cap = (unsigned long long)capacity;
    cudaStream_t s = (cudaStream_t)stream;
    TACO_CUDA(cudaMemsetAsync(env->log_count, 0, sizeof(unsigned long long), s));
    return log_restart(env, s);
}

int taco_env_detach_episode_log(TacoEnv* env) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_detach_episode_log: null argument");
    if (!env->log_mem) return TACO_OK;
    DevGuard guard(env->device);
    TACO_CUDA(cudaDeviceSynchronize());
    cudaFree(env->log_mem);
    env->log_mem = nullptr; env->log_count = nullptr; env->log_acc[0] = env->log_acc[1] = nullptr; env->log_rec = nullptr;
    env->log_cap = 0;
    return TACO_OK;
}

int taco_env_episode_log_buffers(TacoEnv* env, TacoEpisode** records_dev, uint64_t** count_dev, int64_t* capacity) {
    if (!env || !records_dev || !count_dev) return fail(TACO_E_INVALID, "taco_env_episode_log_buffers: null argument");
    if (!env->log_mem) return fail(TACO_E_INVALID, "taco_env_episode_log_buffers: no episode log attached");
    *records_dev = env->log_rec;
    *count_dev = (uint64_t*)env->log_count;
    if (capacity) *capacity = (int64_t)env->log_cap;
    return TACO_OK;
}

int taco_env_episode_log_clear(TacoEnv* env, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_episode_log_clear: null argument");
    if (!env->log_mem) return fail(TACO_E_INVALID, "taco_env_episode_log_clear: no episode log attached");
    DevGuard guard(env->device);
    TACO_CUDA(cudaMemsetAsync(env->log_count, 0, sizeof(unsigned long long), (cudaStream_t)stream));
    return TACO_OK;
}

int taco_env_record_state(TacoEnv* env, const int32_t* ids_dev, int32_t k, float* out_dev, void* stream) {
    if (!env || !ids_dev || !out_dev) return fail(TACO_E_INVALID, "taco_env_record_state: null argument");
    if (k < 1) return fail(TACO_E_INVALID, "taco_env_record_state: k must be >= 1");
    DevGuard guard(env->device);
    export_state_kernel<<<(k + 255) / 256, 256, 0, (cudaStream_t)stream>>>(env->p, ids_dev, k, out_dev); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

int taco_env_attach_rollout_episodes(TacoEnv* env, int64_t capacity, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_attach_rollout_episodes: null argument");
    if (capacity < 1) return fail(TACO_E_INVALID, "taco_env_attach_rollout_episodes: capacity must be >= 1");
    if (env->rep_mem) return fail(TACO_E_INVALID, "taco_env_attach_rollout_episodes: rollout episodes are already attached");
    DevGuard guard(env->device);
    const size_t n = (size_t)env->n, blocks = (n + kScanBlock - 1) / kScanBlock;
    size_t off = 256;                                                // counter at 0, blocks_done at 8
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t oRet = take(n * sizeof(float)), oLen = take(n * sizeof(int)), oLive = take(n);
    const size_t oPart = take(blocks * kSummaryStride * sizeof(double)), oRec = take((size_t)capacity * sizeof(TacoRolloutEpisode));
    void* mem = nullptr;
    const cudaError_t ce = cudaMalloc(&mem, off);
    if (ce != cudaSuccess) { cudaGetLastError(); return fail(TACO_E_NOMEM, std::string("cudaMalloc of the rollout episodes failed: ") + cudaGetErrorString(ce)); }
    char* base = (char*)mem;
    env->rep_mem = mem;
    env->rep_count = (unsigned long long*)base;
    env->rep_blocks_done = (unsigned int*)(base + 8);
    env->rep_ret = (float*)(base + oRet);
    env->rep_len = (int*)(base + oLen);
    env->rep_live = (uint8_t*)(base + oLive);
    env->rep_partial = (double*)(base + oPart);
    env->rep_rec = (TacoRolloutEpisode*)(base + oRec);
    env->rep_cap = (unsigned long long)capacity;
    cudaStream_t s = (cudaStream_t)stream;
    TACO_CUDA(cudaMemsetAsync(base, 0, 256, s));
    return rep_restart(env, s);
}

int taco_env_detach_rollout_episodes(TacoEnv* env) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_detach_rollout_episodes: null argument");
    if (!env->rep_mem) return TACO_OK;
    DevGuard guard(env->device);
    TACO_CUDA(cudaDeviceSynchronize());
    cudaFree(env->rep_mem);
    env->rep_mem = nullptr; env->rep_count = nullptr; env->rep_blocks_done = nullptr;
    env->rep_ret = nullptr; env->rep_len = nullptr; env->rep_live = nullptr; env->rep_partial = nullptr; env->rep_rec = nullptr;
    env->rep_cap = 0; env->rep_scanned = 0;
    return TACO_OK;
}

int taco_env_rollout_episodes_buffers(TacoEnv* env, TacoRolloutEpisode** records_dev, uint64_t** count_dev, int64_t* capacity) {
    if (!env || !records_dev || !count_dev) return fail(TACO_E_INVALID, "taco_env_rollout_episodes_buffers: null argument");
    if (!env->rep_mem) return fail(TACO_E_INVALID, "taco_env_rollout_episodes_buffers: no rollout episodes attached");
    *records_dev = env->rep_rec;
    *count_dev = (uint64_t*)env->rep_count;
    if (capacity) *capacity = (int64_t)env->rep_cap;
    return TACO_OK;
}

int taco_env_rollout_episodes_clear(TacoEnv* env, void* stream) {
    if (!env) return fail(TACO_E_INVALID, "taco_env_rollout_episodes_clear: null argument");
    if (!env->rep_mem) return fail(TACO_E_INVALID, "taco_env_rollout_episodes_clear: no rollout episodes attached");
    DevGuard guard(env->device);
    TACO_CUDA(cudaMemsetAsync(env->rep_count, 0, sizeof(unsigned long long), (cudaStream_t)stream));
    return TACO_OK;
}

int taco_env_scan_rollout_episodes(TacoEnv* env, double* summary_dev, void* stream) {
    if (!env || !summary_dev) return fail(TACO_E_INVALID, "taco_env_scan_rollout_episodes: null argument");
    if (!env->rep_mem) return fail(TACO_E_INVALID, "taco_env_scan_rollout_episodes: no rollout episodes attached");
    if (!env->ring_slots || !env->ring_rew)
        return fail(TACO_E_INVALID, "taco_env_scan_rollout_episodes: no rollout ring with rew / done / time-out rows attached");
    DevGuard guard(env->device);
    const int k0 = env->rep_scanned, rows = env->ring_cur - k0;
    const size_t n = (size_t)env->n;
    RolloutScanParams q;
    q.rew = env->ring_rew + n * k0; q.done = env->ring_done + n * k0; q.tout = env->ring_tout + n * k0;
    q.n = env->n; q.rows = rows;
    // step index of row k0: the ring cursor and the step index advance together
    q.step0 = (env->graph_mode ? env->step_index - env->graph_origin : env->step_index) - (uint32_t)rows;
    q.step_base = env->graph_mode ? env->step_counter : nullptr;
    q.env_offset = env->p.env_offset; q.mix_n1 = env->p.mix_n1; q.mix_n2 = env->p.mix_n2; q.task_mode = env->p.task_mode;
    q.ret = env->rep_ret; q.len = env->rep_len; q.live = env->rep_live;
    q.rec = env->rep_rec; q.count = env->rep_count; q.capacity = env->rep_cap;
    q.partial = env->rep_partial; q.blocks_done = env->rep_blocks_done; q.summary = summary_dev;
    rollout_episodes_scan_kernel<<<(env->n + kScanBlock - 1) / kScanBlock, kScanBlock, 0, (cudaStream_t)stream>>>(q); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    env->rep_scanned = env->ring_cur;
    return TACO_OK;
}

int taco_env_debug_delay(TacoEnv* env, float* out_host) {
    if (!env || !out_host) return fail(TACO_E_INVALID, "taco_env_debug_delay: null argument");
    if (!env->dbg_delay) return fail(TACO_E_INVALID, "env was not created with TACO_F_DEBUG_DELAY");
    DevGuard guard(env->device);
    TACO_CUDA(cudaDeviceSynchronize());
    // device layout [cfi][n_pad] float4 -> host (n, cfi, 4)
    const int cfi = env->cfg.control_freq_inv;
    std::vector<float4> tmp((size_t)cfi * env->n_pad);
    TACO_CUDA(cudaMemcpy(tmp.data(), env->dbg_delay, tmp.size() * sizeof(float4), cudaMemcpyDeviceToHost));
    for (int i = 0; i < env->n; ++i)
        for (int k = 0; k < cfi; ++k) {
            const float4 v = tmp[(size_t)k * env->n_pad + i];
            float* o = out_host + ((size_t)i * cfi + k) * 4;
            o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
        }
    return TACO_OK;
}

}  // extern "C"
