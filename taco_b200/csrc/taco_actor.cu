// Actor MLP inference behind the C ABI (include/taco_b200.h, taco_actor_*).
//
// Mirrors, for rollout inference only (the PPO update stays in PyTorch):
//   MLP.forward / PPO_ActorCritic.act actor branch   IsaacGymEnvs/algorithms/nets_asymmetry.py:23-39, :326-346
//   PPO.spectral_normalize_actors                    IsaacGymEnvs/algorithms/ppo_asymmetry.py:398-404
//
// Two kernels compute the same function: an FP32 CUDA-core path (op order of a plain dot product; the parity
// path) and the tcgen05 bf16 path in actor_tc.cuh (the throughput path for env counts where the MLP is a real
// dense contraction).  taco_actor_load uploads the weights, applies the spectral projection on the device
// (power iteration in double precision, once per update) and pre-swizzles the bf16 weight images.
#include "launch_count.h"
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "host_common.h"
#include "actor_tc.cuh"

namespace taco {
namespace actor {

constexpr int kMaxLayers = 8;        // linear layers of the FP32 path

struct FpParams {
    const float* obs; float* mean;
    int n_rows, n_layers;
    int sizes[kMaxLayers + 1];
    const float* w[kMaxLayers];       // (out, in) row-major, like nn.Linear.weight
    const float* b[kMaxLayers];
    int stride;                       // smem row stride (max width + 1)
    SampleParams sp;
};

// FP32 reference path: CTA = 32 envs; activations ping-pong in shared memory; lane = env, each warp owns a strip of
// output neurons, kFpTile per pass; the dot product runs over k in order with one FMA per term.
__global__ void __launch_bounds__(kFpThreads) actor_fp32_kernel(const FpParams p) {
    extern __shared__ float s_act[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long row = (long long)blockIdx.x * kFpEnvs + lane;
    const bool valid = row < p.n_rows;
    float* cur = s_act;
    float* nxt = s_act + kFpEnvs * p.stride;
    for (int k = warp; k < p.sizes[0]; k += kFpThreads / 32) cur[lane * p.stride + k] = valid ? __ldg(p.obs + row * p.sizes[0] + k) : 0.0f;
    __syncthreads();
    for (int l = 0; l < p.n_layers; ++l) {
        const int in = p.sizes[l], out = p.sizes[l + 1];
        const float* __restrict__ W = p.w[l];
        const float* __restrict__ B = p.b[l];
        const bool last = (l + 1 == p.n_layers);
        // kFpTile output neurons per pass; when the rows of W are 16-byte aligned (in % 4 == 0) the weights come as float4 along k:
        // 4 LDS + kFpTile LDG.128 per 4 * kFpTile FMAs.  Every dot product still runs over k in ascending order, one FMA per term.
        const bool vec = (in & 3) == 0;
        for (int j0 = warp * kFpTile; j0 < out; j0 += (kFpThreads / 32) * kFpTile) {
            float acc[kFpTile];
            const float* wr[kFpTile];
#pragma unroll
            for (int i = 0; i < kFpTile; ++i) { acc[i] = 0.f; wr[i] = W + (size_t)min(j0 + i, out - 1) * in; }
            const float* a = cur + lane * p.stride;
            if (vec) {
                for (int k = 0; k < in; k += 4) {
                    const float x0 = a[k], x1 = a[k + 1], x2 = a[k + 2], x3 = a[k + 3];
#pragma unroll
                    for (int i = 0; i < kFpTile; ++i) {
                        const float4 w = __ldg(reinterpret_cast<const float4*>(wr[i] + k));
                        acc[i] = fmaf(x3, w.w, fmaf(x2, w.z, fmaf(x1, w.y, fmaf(x0, w.x, acc[i]))));
                    }
                }
            } else {
                for (int k = 0; k < in; ++k) {
                    const float x = a[k];
#pragma unroll
                    for (int i = 0; i < kFpTile; ++i) acc[i] = fmaf(x, __ldg(wr[i] + k), acc[i]);
                }
            }
#pragma unroll
            for (int i = 0; i < kFpTile; ++i) {
                if (j0 + i < out) {
                    const float v = acc[i] + __ldg(B + j0 + i);
                    nxt[lane * p.stride + j0 + i] = last ? v : fmaxf(v, 0.0f);
                }
            }
        }
        __syncthreads();
        float* t = cur; cur = nxt; nxt = t;
    }
    if (warp == 0 && valid) {
        float pre[kOutPad] = {0.f, 0.f, 0.f, 0.f};
        const int out = p.sizes[p.n_layers];
        for (int o = 0; o < out && o < kOutPad; ++o) pre[o] = cur[lane * p.stride + o];
        actor_tail(pre, out, row, p.mean, p.sp);
    }
}

// ---- spectral norm (largest singular value) by power iteration on W^T W, double precision, one CTA per matrix.
// PPO.spectral_normalize_actors uses torch.linalg.matrix_norm(ord=2) (ppo_asymmetry.py:401); the projection itself is
// W *= c / sigma when sigma > c.
constexpr int kSnThreads = 256;
__device__ double block_sum(double v, double* red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    for (int i = 0; i < kSnThreads / 32; ++i) t += red[i];
    return t;
}
__global__ void __launch_bounds__(kSnThreads) spectral_norm_kernel(float* w, int rows, int cols, float lipschitz, double* sigma_out,
                                                                   int max_iter, double tol) {
    extern __shared__ double s_vec[];          // v[cols], u[rows]
    __shared__ double red[kSnThreads / 32];
    double* v = s_vec;
    double* u = s_vec + cols;
    // deterministic start vector with every component non-zero
    for (int c = threadIdx.x; c < cols; c += kSnThreads) v[c] = 1.0 + 0.37 * (double)((c * 2654435761u) >> 24) / 256.0;
    __syncthreads();
    double sigma = 0.0, prev = -1.0;
    for (int it = 0; it < max_iter; ++it) {
        // u = W v   (warp per row, lanes stride the row: coalesced)
        for (int r = threadIdx.x >> 5; r < rows; r += kSnThreads / 32) {
            double acc = 0.0;
            for (int c = threadIdx.x & 31; c < cols; c += 32) acc += (double)w[(size_t)r * cols + c] * v[c];
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if ((threadIdx.x & 31) == 0) u[r] = acc;
        }
        __syncthreads();
        // v = W^T u  (thread per column: coalesced across threads)
        double part = 0.0;
        for (int c = threadIdx.x; c < cols; c += kSnThreads) {
            double acc = 0.0;
            for (int r = 0; r < rows; ++r) acc += (double)w[(size_t)r * cols + c] * u[r];
            v[c] = acc;
            part += acc * acc;
        }
        const double nv = sqrt(block_sum(part, red));       // |W^T W v| with |v| = 1  ->  sigma^2
        sigma = sqrt(nv);
        if (nv > 0.0)
            for (int c = threadIdx.x; c < cols; c += kSnThreads) v[c] /= nv;
        __syncthreads();
        if (it == 0) {                                      // the start vector was not normalised: discard this estimate
            prev = -1.0;
        } else {
            if (fabs(sigma - prev) <= tol * sigma) break;
            prev = sigma;
        }
    }
    if (threadIdx.x == 0) *sigma_out = sigma;
    if (lipschitz > 0.0f && sigma > (double)lipschitz) {
        const float s = (float)((double)lipschitz / sigma);
        for (int i = threadIdx.x; i < rows * cols; i += kSnThreads) w[i] *= s;
    }
}

}  // namespace actor
}  // namespace taco

using namespace taco::actor;
using taco::DevGuard;
using taco::fail;

struct TacoActor {
    int device = 0;
    std::vector<int> sizes;              // [in, h1, ..., hL, out]
    int n_layers = 0;
    MlpF32 f32;                          // all layers, (out, in) row-major each
    double* sigma = nullptr;             // per layer, device
    bool loaded = false;
    // tensor-core path
    bool tc_ok = false;
    std::string tc_why;
    TcImage tc;                          // hidden layers + the output layer (16-row padded image)
    int num_sms = 148;
    int fp_smem = 0;
    // sampling constants [std0..3, logp_const, pad]: device copy read by the kernels, host copy to detect changes
    float* samp_dev = nullptr;
    float samp_host[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    bool samp_set = false;
};

// std = exp(log_std)^2 in float32 (nets_asymmetry.py:338) and the constant of the log-probability; uploads when they changed
static int actor_set_log_std(TacoActor* a, const float* log_std_host, cudaStream_t s) {
    float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const int out = a->sizes.back();
    double lsum = 0.0;
    for (int o = 0; o < out; ++o) {
        const float e = expf(log_std_host[o]);
        v[o] = e * e;
        lsum += std::log((double)v[o]);
    }
    v[4] = (float)(-lsum - 0.5 * out * std::log(2.0 * M_PI));
    if (a->samp_set && memcmp(v, a->samp_host, sizeof(v)) == 0) return TACO_OK;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    TACO_CUDA(cudaStreamIsCapturing(s, &cs));
    if (cs != cudaStreamCaptureStatusNone)
        return fail(TACO_E_INVALID, "taco_actor: log_std changed while the stream is capturing; call taco_actor_set_log_std before the capture");
    memcpy(a->samp_host, v, sizeof(v));
    TACO_CUDA(cudaMemcpyAsync(a->samp_dev, a->samp_host, sizeof(v), cudaMemcpyHostToDevice, s));   // pageable source: staged before the call returns
    a->samp_set = true;
    return TACO_OK;
}

static int actor_run(TacoActor* a, const float* obs_dev, float* mean_dev, int32_t n, int32_t use_tc, const SampleParams& sp, void* stream) {
    if (!a || !obs_dev || !mean_dev) return fail(TACO_E_INVALID, "taco_actor: null argument");
    if (!a->loaded) return fail(TACO_E_INVALID, "taco_actor: call taco_actor_load first");
    if (n <= 0) return fail(TACO_E_INVALID, "taco_actor: n must be positive");
    if (a->sizes.back() == 4 && ((uintptr_t)mean_dev & 15u)) return fail(TACO_E_INVALID, "taco_actor: mean must be 16-byte aligned");
    DevGuard guard(a->device);
    cudaStream_t s = (cudaStream_t)stream;
    if (use_tc) {
        if (!a->tc_ok) return fail(TACO_E_INVALID, "taco_actor: tensor-core path unavailable for this shape: " + a->tc_why);
        TcParams p;
        memset(&p, 0, sizeof(p));
        p.obs = obs_dev; p.mean = mean_dev;
        p.in_dim = a->sizes[0]; p.out_dim = a->sizes.back(); p.n_rows = n; p.num_tiles = (n + kTileM - 1) / kTileM;
        p.n_hidden = a->n_layers - 1;
        p.obs_vec2 = ((p.in_dim & 1) == 0 && ((uintptr_t)obs_dev & 7u) == 0) ? 1 : 0;
        p.obs_bulk = ((p.in_dim & 1) == 0 && p.in_dim <= kObsBulkMaxIn && ((uintptr_t)obs_dev & 15u) == 0 && !getenv("TACO_ACTOR_NO_BULK_OBS")) ? 1 : 0;
        p.wimg = a->tc.wimg; p.bias = a->tc.bias; p.b_out = a->tc.b_out;
        for (int l = 0; l <= p.n_hidden; ++l) p.layer[l] = a->tc.layer[l];
        p.sp = sp;
        const int grid = tc_grid(p.num_tiles, a->num_sms, &p.tiles_per_cta);
        const char* tl = getenv("TACO_ACTOR_TIMELINE");
        if (int rc = timeline_begin(tl, &p.dbg, s)) return rc;
        actor_tc_kernel<<<grid, kTcThreads, kActorSmemBytes, s>>>(p); TACO_LAUNCHED();
        if (int rc = timeline_end(tl, p.dbg, s)) return rc;
    } else {
        FpParams p;
        memset(&p, 0, sizeof(p));
        p.obs = obs_dev; p.mean = mean_dev; p.n_rows = n; p.n_layers = a->n_layers;
        int mx = 0;
        for (int l = 0; l <= a->n_layers; ++l) { p.sizes[l] = a->sizes[l]; mx = a->sizes[l] > mx ? a->sizes[l] : mx; }
        for (int l = 0; l < a->n_layers; ++l) { p.w[l] = a->f32.w + a->f32.w_off[l]; p.b[l] = a->f32.b + a->f32.b_off[l]; }
        p.stride = mx + 1;
        p.sp = sp;
        actor_fp32_kernel<<<(n + kFpEnvs - 1) / kFpEnvs, kFpThreads, a->fp_smem, s>>>(p); TACO_LAUNCHED();
    }
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

extern "C" {

int taco_actor_create(int device, const int32_t* sizes, int32_t n_sizes, TacoActor** out) {
    if (!sizes || !out) return fail(TACO_E_INVALID, "taco_actor_create: null argument");
    *out = nullptr;
    if (n_sizes < 2 || n_sizes > kMaxLayers + 1) return fail(TACO_E_INVALID, "taco_actor_create: need 2..9 layer sizes [in, h1, ..., out]");
    for (int i = 0; i < n_sizes; ++i)
        if (sizes[i] < 1 || sizes[i] > 512) return fail(TACO_E_INVALID, "taco_actor_create: layer sizes must be in [1, 512]");
    if (sizes[n_sizes - 1] > kOutPad) return fail(TACO_E_INVALID, "taco_actor_create: output width must be <= 4 (num_acts, fpv_asymmetry.py:102)");
    int ndev = 0;
    TACO_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(TACO_E_INVALID, "taco_actor_create: no such CUDA device");
    DevGuard guard(device);
    TacoActor* a = new (std::nothrow) TacoActor();
    if (!a) return fail(TACO_E_NOMEM, "host allocation failed");
    a->device = device;
    a->sizes.assign(sizes, sizes + n_sizes);
    a->n_layers = n_sizes - 1;
    int mx = 0;
    for (int i = 0; i < n_sizes; ++i) mx = sizes[i] > mx ? sizes[i] : mx;
    a->fp_smem = 2 * kFpEnvs * (mx + 1) * (int)sizeof(float);
    cudaDeviceProp prop;
    TACO_CUDA(cudaGetDeviceProperties(&prop, device));
    a->num_sms = prop.multiProcessorCount;
    // ---- is the shape eligible for the tcgen05 path?
    const int n_hidden = a->n_layers - 1;
    a->tc_ok = true;
    if (prop.major != 10) { a->tc_ok = false; a->tc_why = "device is not sm_100"; }
    else if (n_hidden < 1 || n_hidden > kMaxHidden) { a->tc_ok = false; a->tc_why = "needs 1..4 hidden layers"; }
    else if (sizes[0] > kMaxN) { a->tc_ok = false; a->tc_why = "input width > 256"; }
    else if (!tc_hidden_widths_ok(sizes, n_hidden)) { a->tc_ok = false; a->tc_why = "hidden widths must be multiples of 64, <= 256"; }
    cudaError_t ce = mlp_f32_alloc(a->f32, sizes, a->n_layers);
    if (ce == cudaSuccess) ce = cudaMalloc(&a->sigma, kMaxLayers * sizeof(double));
    if (ce == cudaSuccess) ce = cudaMemset(a->sigma, 0, kMaxLayers * sizeof(double));
    if (ce == cudaSuccess) ce = cudaMalloc(&a->samp_dev, 8 * sizeof(float));
    if (ce == cudaSuccess && a->tc_ok) {
        ce = tc_image_alloc(a->tc, sizes, n_hidden, 0, 0);
        if (ce == cudaSuccess) ce = cudaFuncSetAttribute(actor_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kActorSmemBytes);
    }
    if (ce == cudaSuccess && a->fp_smem > 48 * 1024)
        ce = cudaFuncSetAttribute(actor_fp32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, a->fp_smem);
    if (ce != cudaSuccess) {
        const std::string msg = std::string("taco_actor_create: ") + cudaGetErrorString(ce);
        taco_actor_destroy(a);
        return fail(ce == cudaErrorMemoryAllocation ? TACO_E_NOMEM : TACO_E_CUDA, msg);
    }
    *out = a;
    return TACO_OK;
}

int taco_actor_destroy(TacoActor* a) {
    if (!a) return TACO_OK;
    DevGuard guard(a->device);
    mlp_f32_free(a->f32); cudaFree(a->sigma); cudaFree(a->samp_dev);
    tc_image_free(a->tc);
    delete a;
    return TACO_OK;
}

int taco_actor_load(TacoActor* a, const float* const* weights_host, const float* const* biases_host, float lipschitz_const, void* stream) {
    if (!a || !weights_host || !biases_host) return fail(TACO_E_INVALID, "taco_actor_load: null argument");
    for (int l = 0; l < a->n_layers; ++l)
        if (!weights_host[l] || !biases_host[l]) return fail(TACO_E_INVALID, "taco_actor_load: null layer pointer");
    DevGuard guard(a->device);
    cudaStream_t s = (cudaStream_t)stream;
    if (int rc = mlp_f32_upload(a->f32, weights_host, biases_host, a->sizes.data(), a->n_layers, s)) return rc;
    // spectral projection of every weight matrix (ppo_asymmetry.py:398-404); also records sigma when lipschitz_const <= 0
    for (int l = 0; l < a->n_layers && lipschitz_const >= 0.0f; ++l) {        // negative: weights are known to be projected, skip the measurement
        const int in = a->sizes[l], out = a->sizes[l + 1];
        spectral_norm_kernel<<<1, kSnThreads, (size_t)(in + out) * sizeof(double), s>>>(a->f32.w + a->f32.w_off[l], out, in, lipschitz_const,
                                                                                         a->sigma + l, 20000, 1e-12); TACO_LAUNCHED();
    }
    TACO_CUDA(cudaGetLastError());
    if (a->tc_ok) {
        TACO_CUDA(cudaMemsetAsync(a->tc.bias, 0, kMaxHidden * kMaxN * sizeof(float), s));
        if (int rc = tc_image_pack(a->tc, a->f32, a->sizes.data(), a->n_layers - 1, s)) return rc;
    }
    TACO_CUDA(cudaStreamSynchronize(s));     // the host weight buffers may be released by the caller on return
    a->loaded = true;
    return TACO_OK;
}

int taco_actor_sigmas(TacoActor* a, double* out_host) {
    if (!a || !out_host) return fail(TACO_E_INVALID, "taco_actor_sigmas: null argument");
    DevGuard guard(a->device);
    TACO_CUDA(cudaDeviceSynchronize());
    TACO_CUDA(cudaMemcpy(out_host, a->sigma, (size_t)a->n_layers * sizeof(double), cudaMemcpyDeviceToHost));
    return TACO_OK;
}

int taco_actor_weights(TacoActor* a, int32_t layer, float* w_host, float* b_host) {
    if (!a || layer < 0 || layer >= a->n_layers) return fail(TACO_E_INVALID, "taco_actor_weights: bad argument");
    DevGuard guard(a->device);
    TACO_CUDA(cudaDeviceSynchronize());
    const int in = a->sizes[layer], out = a->sizes[layer + 1];
    if (w_host) TACO_CUDA(cudaMemcpy(w_host, a->f32.w + a->f32.w_off[layer], (size_t)in * out * sizeof(float), cudaMemcpyDeviceToHost));
    if (b_host) TACO_CUDA(cudaMemcpy(b_host, a->f32.b + a->f32.b_off[layer], (size_t)out * sizeof(float), cudaMemcpyDeviceToHost));
    return TACO_OK;
}

int taco_actor_tc_available(TacoActor* a) { return (a && a->tc_ok) ? 1 : 0; }

// PPO.spectral_normalize_actors for ONE parameter that already lives on the device (e.g. the storage of a torch nn.Linear weight
// during PPO.update, ppo_asymmetry.py:248-249): in place, asynchronous, no SVD and no host round trip.
int taco_spectral_project(int device, float* w_dev, int32_t rows, int32_t cols, float lipschitz_const, double* sigma_dev, void* stream) {
    if (!w_dev || !sigma_dev) return fail(TACO_E_INVALID, "taco_spectral_project: null argument");
    if (rows < 1 || cols < 1 || (size_t)(rows + cols) * sizeof(double) > 200 * 1024)
        return fail(TACO_E_INVALID, "taco_spectral_project: rows + cols must be in [2, 25600]");
    DevGuard guard(device);
    const size_t smem = (size_t)(rows + cols) * sizeof(double);
    if (smem > 48 * 1024) TACO_CUDA(cudaFuncSetAttribute(spectral_norm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    spectral_norm_kernel<<<1, kSnThreads, smem, (cudaStream_t)stream>>>(w_dev, rows, cols, lipschitz_const, sigma_dev, 20000, 1e-12); TACO_LAUNCHED();
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

int taco_actor_forward(TacoActor* a, const float* obs_dev, float* mean_dev, int32_t n, int32_t use_tensor_cores, void* stream) {
    SampleParams sp;
    memset(&sp, 0, sizeof(sp));
    return actor_run(a, obs_dev, mean_dev, n, use_tensor_cores, sp, stream);
}

int taco_actor_act_counter(TacoActor* a, const float* obs_dev, int32_t n, const float* log_std_host, int64_t env_offset, uint64_t seed,
                           uint32_t step_index, const uint32_t* step_base_dev, float* mean_dev, float* action_dev, float* clipped_dev,
                           float* logp_dev, int32_t use_tensor_cores, void* stream) {
    if (!a || !action_dev) return fail(TACO_E_INVALID, "taco_actor_act: null argument");
    if (!log_std_host && !a->samp_set) return fail(TACO_E_INVALID, "taco_actor_act: no log_std given and taco_actor_set_log_std was never called");
    DevGuard guard(a->device);
    if (log_std_host) {
        const int rc = actor_set_log_std(a, log_std_host, (cudaStream_t)stream);
        if (rc != TACO_OK) return rc;
    }
    SampleParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.action = action_dev; sp.clipped = clipped_dev; sp.logp = logp_dev;
    sp.samp = a->samp_dev;
    sp.env_offset = env_offset;
    sp.seed_lo = (uint32_t)(seed & 0xFFFFFFFFull); sp.seed_hi = (uint32_t)(seed >> 32);
    sp.step_index = step_index;
    sp.step_base = step_base_dev;
    return actor_run(a, obs_dev, mean_dev, n, use_tensor_cores, sp, stream);
}

int taco_actor_set_log_std(TacoActor* a, const float* log_std_host, void* stream) {
    if (!a || !log_std_host) return fail(TACO_E_INVALID, "taco_actor_set_log_std: null argument");
    DevGuard guard(a->device);
    return actor_set_log_std(a, log_std_host, (cudaStream_t)stream);
}

int taco_actor_act(TacoActor* a, const float* obs_dev, int32_t n, const float* log_std_host, int64_t env_offset, uint64_t seed,
                   uint32_t step_index, float* mean_dev, float* action_dev, float* clipped_dev, float* logp_dev, int32_t use_tensor_cores,
                   void* stream) {
    return taco_actor_act_counter(a, obs_dev, n, log_std_host, env_offset, seed, step_index, nullptr, mean_dev, action_dev, clipped_dev, logp_dev,
                                  use_tensor_cores, stream);
}

}  // extern "C"
