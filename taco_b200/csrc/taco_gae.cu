// Rollout-buffer post-processing behind the C ABI (include/taco_b200.h, taco_gae_*).
//
// Mirrors (IsaacGymEnvs/algorithms/):
//   PPOReplayBuffer.compute_returns_and_advantage   buffer_asymmetry.py:93-132   (backward GAE(lambda) scan, ret = adv + value,
//                                                   adv = (adv - mean) / (std + 1e-8) over all horizon x envs samples)
//   the time-out bootstrap of the stored reward     ppo_asymmetry.py:313-324     (rew += gamma * V(pre-step obs) for truncated envs;
//                                                   V(pre-step obs) is the `value` stored for that step)
// The reference runs a Python loop over the horizon (7 small kernels per step) and two full-buffer reductions.  Here one
// thread owns one env and walks the horizon backwards with the recurrence in registers (every access is coalesced over
// envs: the buffers are (H, N, 1)), accumulating [sum adv, sum adv^2, count] in float64 -- the vector a multi-GPU job
// all-reduces -- and a second, purely elementwise launch applies the normalisation from those moments.
//
// Compiled with -fmad=false: the recurrence is op-for-op the reference's float32 expression (bit-exact adv / ret).
#include "launch_count.h"
#include <cstdint>
#include <string>

#include <cuda_runtime.h>

#include "host_common.h"

namespace taco {
namespace gae {

constexpr int kThreads = 128;

__global__ void __launch_bounds__(kThreads) gae_scan_kernel(int H, int N, const float* __restrict__ rew, const float* __restrict__ done,
                                                            const uint8_t* __restrict__ time_outs, const float* __restrict__ value,
                                                            const float* __restrict__ last_value, float gamma, float lam,
                                                            float* __restrict__ adv, float* __restrict__ ret, double* __restrict__ moments) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    double s1 = 0.0, s2 = 0.0;
    if (i < N) {
        float next_value = __ldg(last_value + i);
        float last_gae = 0.0f;
#pragma unroll 4
        for (int s = H - 1; s >= 0; --s) {
            const size_t k = (size_t)s * N + i;
            const float v = __ldg(value + k);
            const float d = __ldg(done + k);
            float r = __ldg(rew + k);
            if (time_outs != nullptr) {                              // ppo_asymmetry.py:313-324
                const float trunc = (float)__ldg(time_outs + k) * d;
                if (trunc != 0.0f) r = r + gamma * v;
            }
            const float nnt = 1.0f - d;                              // buffer_asymmetry.py:118
            const float td_target = r + (nnt * gamma) * next_value;  // :120
            const float delta = td_target - v;                       // :121
            last_gae = delta + ((nnt * gamma) * lam) * last_gae;     // :122
            adv[k] = last_gae;
            ret[k] = last_gae + v;                                   // :127
            s1 += (double)last_gae;
            s2 += (double)last_gae * (double)last_gae;
            next_value = v;
        }
    }
    __shared__ double red[2][kThreads / 32];
    for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s1; red[1][threadIdx.x >> 5] = s2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < kThreads / 32; ++w) { a += red[0][w]; b += red[1][w]; }
        const int nv = min(kThreads, N - (int)blockIdx.x * kThreads);
        atomicAdd(moments + 0, a);
        atomicAdd(moments + 1, b);
        atomicAdd(moments + 2, (double)nv * (double)H);
    }
}

__global__ void gae_normalize_kernel(float* __restrict__ adv, long long count, const double* __restrict__ moments) {
    const double s = moments[0], ss = moments[1], n = moments[2];
    const double mean = s / n;
    const double var = fmax(ss - n * mean * mean, 0.0) / fmax(n - 1.0, 1.0);   // torch.std: unbiased
    const float mean32 = (float)mean;
    const float den = (float)sqrt(var) + 1e-8f;                                 // buffer_asymmetry.py:132
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += (long long)gridDim.x * blockDim.x)
        adv[k] = (adv[k] - mean32) / den;
}

}  // namespace gae
}  // namespace taco

using namespace taco::gae;
using taco::DevGuard;

extern "C" {

int taco_gae_advantages(int device, int32_t horizon, int32_t num_envs, const float* rew_dev, const float* done_dev, const uint8_t* time_outs_dev,
                        const float* value_dev, const float* last_value_dev, float gamma, float lam, float* adv_dev, float* ret_dev,
                        double* moments_dev, void* stream) {
    if (!rew_dev || !done_dev || !value_dev || !last_value_dev || !adv_dev || !ret_dev || !moments_dev)
        return taco::fail(TACO_E_INVALID, "taco_gae_advantages: null argument");
    if (horizon <= 0 || num_envs <= 0) return taco::fail(TACO_E_INVALID, "taco_gae_advantages: horizon and num_envs must be positive");
    DevGuard guard(device);
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(moments_dev, 0, 3 * sizeof(double), s);
    if (e == cudaSuccess) {
        gae_scan_kernel<<<(num_envs + kThreads - 1) / kThreads, kThreads, 0, s>>>(horizon, num_envs, rew_dev, done_dev, time_outs_dev, value_dev,
                                                                                   last_value_dev, gamma, lam, adv_dev, ret_dev, moments_dev); TACO_LAUNCHED();
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return taco::fail(TACO_E_CUDA, std::string("taco_gae_advantages: ") + cudaGetErrorString(e));
    return TACO_OK;
}

int taco_gae_normalize(int device, float* adv_dev, int64_t count, const double* moments_dev, void* stream) {
    if (!adv_dev || !moments_dev) return taco::fail(TACO_E_INVALID, "taco_gae_normalize: null argument");
    if (count <= 0) return taco::fail(TACO_E_INVALID, "taco_gae_normalize: count must be positive");
    DevGuard guard(device);
    const long long blocks = (count + 1023) / 1024;
    const int grid = (int)(blocks < 148 * 8 ? blocks : 148 * 8);
    gae_normalize_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(adv_dev, (long long)count, moments_dev); TACO_LAUNCHED();
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return taco::fail(TACO_E_CUDA, std::string("taco_gae_normalize: ") + cudaGetErrorString(e));
    return TACO_OK;
}

}  // extern "C"
