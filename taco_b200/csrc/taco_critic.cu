// Critic inference behind the C ABI (include/taco_b200.h, taco_critic_*).
//
// Mirrors, for rollout inference only (the PPO update stays in PyTorch), the critic branch of PPO_ActorCritic.act
// (IsaacGymEnvs/algorithms/nets_asymmetry.py:350-352) in the configuration the reference trains with (README.md:60-66:
// --use_critic_encoder=True --critic_encoder_type=LSTM --lenStates=5):
//   LSTMEncoder.forward   nets_asymmetry.py:128-136   nn.LSTM(input, hidden, num_layers, batch_first=True), zero initial state,
//                                                     output = top layer's h after the last time step
//   MLP.forward           nets_asymmetry.py:23-39     [Linear -> ReLU] x L -> Linear -> Identity (:318)
//
// Two kernels compute the same function: an FP32 CUDA-core path (any shape; the parity path) and the tcgen05 bf16 path in
// critic_tc.cuh (1..4 LSTM layers of width <= 64, MLP widths multiples of 64 up to 256).  A stacked LSTM runs on the tcgen05
// path as one launch per layer over a chunk of the batch (kChunkWaves), the layers handing h over through a workspace.
#include "launch_count.h"
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "host_common.h"
#include "critic_tc.cuh"

namespace taco {
namespace critic {

constexpr int kMaxLstmLayers = 4;
constexpr int kMaxMlpLayers = 8;     // linear layers of the FP32 path
// Stacked LSTM on the tensor cores: the batch is walked in chunks of kChunkWaves full waves of tile pairs (2 x SMs tiles each), and
// each chunk runs layer 0 -> top, so that much of a chunk's hand-off between the layers (128 B per row and step and buffer) is read
// back from L2.  Measured on a B200 (DESIGN.md 6c): 4 waves beat 1 and 2 (fewer launches and wave tails outweigh the part of the
// hand-off that no longer fits L2).  TACO_CRITIC_CHUNK_WAVES in the environment at create time overrides it (tuning).
constexpr int kChunkWaves = 4;

struct FpParams {
    const float* states; float* value;
    int n_rows, in_dim, seq_len, hidden, lstm_layers, n_mlp;
    const float* w_ih[kMaxLstmLayers]; const float* w_hh[kMaxLstmLayers];
    const float* b_ih[kMaxLstmLayers]; const float* b_hh[kMaxLstmLayers];
    int mlp_sizes[kMaxMlpLayers + 1];
    const float* w[kMaxMlpLayers]; const float* b[kMaxMlpLayers];
    int stride;                       // floats per env in shared memory (odd)
    int off_lstm, off_mlp, mlp_w;     // offsets inside an env's row: per-layer [h_a | h_b | c], then the MLP ping-pong
};

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

// FP32 reference path: CTA = 32 envs (lane = env); everything an env needs sits in its shared-memory row; each warp owns a
// strip of hidden units / output neurons; dot products run over k in order with one FMA per term, the two matrix products
// of a gate are summed like torch (W_ih x + b_ih) + (W_hh h + b_hh).
__global__ void __launch_bounds__(kFpThreads) critic_fp32_kernel(const FpParams p) {
    extern __shared__ float s_row[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int kWarps = kFpThreads / 32;
    const long long row = (long long)blockIdx.x * kFpEnvs + lane;
    const bool valid = row < p.n_rows;
    float* me = s_row + lane * p.stride;
    const int H = p.hidden, T = p.seq_len, In = p.in_dim;
    for (int k = warp; k < T * In; k += kWarps) me[k] = valid ? __ldg(p.states + row * (long long)(T * In) + k) : 0.0f;
    for (int k = warp; k < p.lstm_layers * 3 * H; k += kWarps) me[p.off_lstm + k] = 0.0f;
    __syncthreads();
    for (int t = 0; t < T; ++t) {
        const int cur = t & 1;
        for (int l = 0; l < p.lstm_layers; ++l) {
            float* hl = me + p.off_lstm + l * 3 * H;
            const float* inp = l == 0 ? me + t * In : me + p.off_lstm + (l - 1) * 3 * H + (cur ^ 1) * H;   // layer below, this step
            const int in_l = l == 0 ? In : H;
            const float* hprev = hl + cur * H;
            float* hnew = hl + (cur ^ 1) * H;
            float* cst = hl + 2 * H;
            const float* __restrict__ Wi = p.w_ih[l];
            const float* __restrict__ Wh = p.w_hh[l];
            // two hidden units per pass = 8 gate rows per product; float4 weights along k when the rows are 16-byte aligned.  Every
            // dot product still runs over k in ascending order with one FMA per term.
            const bool vec_i = (in_l & 3) == 0, vec_h = (H & 3) == 0;
            for (int j0 = warp * 2; j0 < H; j0 += kWarps * 2) {
                float a[8], g[8];
                const float* wi[8];
                const float* wh[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int j = min(j0 + (q >> 2), H - 1), row_ = (q & 3) * H + j;
                    a[q] = 0.f; g[q] = 0.f; wi[q] = Wi + (size_t)row_ * in_l; wh[q] = Wh + (size_t)row_ * H;
                }
                if (vec_i) {
                    for (int k = 0; k < in_l; k += 4) {
                        const float x0 = inp[k], x1 = inp[k + 1], x2 = inp[k + 2], x3 = inp[k + 3];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float4 w = __ldg(reinterpret_cast<const float4*>(wi[q] + k));
                            a[q] = fmaf(x3, w.w, fmaf(x2, w.z, fmaf(x1, w.y, fmaf(x0, w.x, a[q]))));
                        }
                    }
                } else {
                    for (int k = 0; k < in_l; ++k) {
                        const float x = inp[k];
#pragma unroll
                        for (int q = 0; q < 8; ++q) a[q] = fmaf(x, __ldg(wi[q] + k), a[q]);
                    }
                }
                if (vec_h) {
                    for (int k = 0; k < H; k += 4) {
                        const float x0 = hprev[k], x1 = hprev[k + 1], x2 = hprev[k + 2], x3 = hprev[k + 3];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float4 w = __ldg(reinterpret_cast<const float4*>(wh[q] + k));
                            g[q] = fmaf(x3, w.w, fmaf(x2, w.z, fmaf(x1, w.y, fmaf(x0, w.x, g[q]))));
                        }
                    }
                } else {
                    for (int k = 0; k < H; ++k) {
                        const float x = hprev[k];
#pragma unroll
                        for (int q = 0; q < 8; ++q) g[q] = fmaf(x, __ldg(wh[q] + k), g[q]);
                    }
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int j = j0 + u;
                    if (j < H) {
                        float gate[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) gate[q] = (a[u * 4 + q] + __ldg(p.b_ih[l] + q * H + j)) + (g[u * 4 + q] + __ldg(p.b_hh[l] + q * H + j));
                        const float c = sigmoid_f(gate[1]) * cst[j] + sigmoid_f(gate[0]) * tanhf(gate[2]);
                        cst[j] = c;
                        hnew[j] = sigmoid_f(gate[3]) * tanhf(c);
                    }
                }
            }
            __syncthreads();
        }
    }
    // encoder output: top layer's h after the last step
    float* cur = me + p.off_mlp;
    float* nxt = cur + p.mlp_w;
    {
        const float* hT = me + p.off_lstm + (p.lstm_layers - 1) * 3 * H + (T & 1) * H;
        for (int k = warp; k < H; k += kWarps) cur[k] = hT[k];
    }
    __syncthreads();
    for (int l = 0; l < p.n_mlp; ++l) {
        const int in = p.mlp_sizes[l], out = p.mlp_sizes[l + 1];
        const float* __restrict__ W = p.w[l];
        const float* __restrict__ B = p.b[l];
        const bool last = (l + 1 == p.n_mlp);
        const bool vec = (in & 3) == 0;
        for (int j0 = warp * kFpTile; j0 < out; j0 += kWarps * kFpTile) {
            float acc[kFpTile];
            const float* wr[kFpTile];
#pragma unroll
            for (int i = 0; i < kFpTile; ++i) { acc[i] = 0.f; wr[i] = W + (size_t)min(j0 + i, out - 1) * in; }
            if (vec) {
                for (int k = 0; k < in; k += 4) {
                    const float x0 = cur[k], x1 = cur[k + 1], x2 = cur[k + 2], x3 = cur[k + 3];
#pragma unroll
                    for (int i = 0; i < kFpTile; ++i) {
                        const float4 w = __ldg(reinterpret_cast<const float4*>(wr[i] + k));
                        acc[i] = fmaf(x3, w.w, fmaf(x2, w.z, fmaf(x1, w.y, fmaf(x0, w.x, acc[i]))));
                    }
                }
            } else {
                for (int k = 0; k < in; ++k) {
                    const float x = cur[k];
#pragma unroll
                    for (int i = 0; i < kFpTile; ++i) acc[i] = fmaf(x, __ldg(wr[i] + k), acc[i]);
                }
            }
#pragma unroll
            for (int i = 0; i < kFpTile; ++i) {
                if (j0 + i < out) {
                    const float v = acc[i] + __ldg(B + j0 + i);
                    nxt[j0 + i] = last ? v : fmaxf(v, 0.0f);
                }
            }
        }
        __syncthreads();
        float* tsw = cur; cur = nxt; nxt = tsw;
    }
    if (warp == 0 && valid) p.value[row] = cur[0];
}

}  // namespace critic
}  // namespace taco

using namespace taco::critic;
using taco::DevGuard;
using taco::fail;

struct TacoCritic {
    int device = 0;
    int in_dim = 0, seq_len = 0, hidden = 0, lstm_layers = 0;
    std::vector<int> mlp_sizes;          // [hidden, h1, ..., 1]
    int n_mlp = 0;
    std::vector<size_t> lstm_off;        // per layer: float offsets of w_ih, w_hh, b_ih, b_hh (4 per layer)
    float* lstm_f32 = nullptr;
    MlpF32 f32;
    bool loaded = false;
    int fp_smem = 0, fp_stride = 0, off_lstm = 0, off_mlp = 0, mlp_w = 0;
    bool tc_ok = false;
    std::string tc_why;
    TcImage tc;                          // layer[0] / bias row 0: the LSTM step (its image in front of the MLP's), MLP from 1 on
    int num_sms = 148;
    // stacked LSTM on the tensor cores (lstm_layers > 1).  The image of LSTM layer k is at k * lstm_img_bytes in tc.wimg.  Layer k's
    // launch reads its gate biases from row 0 of its bias block: tc.bias for the top layer (whose rows 1.. hold the MLP's; the bottom
    // layer's bias rides in its image), seq_bias[k - 1] for a middle layer.  Everything is allocated at create: a captured graph
    // keeps these addresses across taco_critic_load.
    size_t lstm_img_bytes = 0;
    float* seq_bias = nullptr;           // [lstm_layers - 2][kMaxHidden][kMaxN]
    uint4* seq_ws[2] = {nullptr, nullptr};   // hand-off buffers (two from three layers on: ping-pong), chunk_tiles x seq_len x 16 KB each
    int chunk_tiles = 0;
};

static float* tc_bias_block(const TacoCritic* c, int k) {
    return (k == 0 || k + 1 == c->lstm_layers) ? c->tc.bias : c->seq_bias + (size_t)(k - 1) * kMaxHidden * kMaxN;
}

template <bool kSeqIn, bool kSeqOut>
static void set_tc_smem(cudaError_t& ce) {
    if (ce == cudaSuccess)
        ce = cudaFuncSetAttribute(critic_tc_kernel<kSeqIn, kSeqOut>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  kSeqIn ? kCriticSeqSmemBytes : kCriticSmemBytes);
}
template <bool kSeqIn, bool kSeqOut>
static void launch_tc(const CriticTcParams& p, int grid, cudaStream_t s) {
    critic_tc_kernel<kSeqIn, kSeqOut><<<grid, kTcThreads, kSeqIn ? kCriticSeqSmemBytes : kCriticSmemBytes, s>>>(p); TACO_LAUNCHED();
}

extern "C" {

int taco_critic_destroy(TacoCritic* c);

int taco_critic_create(int device, int32_t in_dim, int32_t seq_len, int32_t lstm_hidden, int32_t lstm_layers, const int32_t* mlp_sizes,
                       int32_t n_mlp_sizes, TacoCritic** out) {
    if (!mlp_sizes || !out) return fail(TACO_E_INVALID, "taco_critic_create: null argument");
    *out = nullptr;
    if (in_dim < 1 || in_dim > 256 || seq_len < 1 || seq_len > 64) return fail(TACO_E_INVALID, "taco_critic_create: in_dim must be in [1, 256], seq_len in [1, 64]");
    if (lstm_hidden < 1 || lstm_hidden > 256 || lstm_layers < 1 || lstm_layers > kMaxLstmLayers)
        return fail(TACO_E_INVALID, "taco_critic_create: lstm_hidden must be in [1, 256], lstm_layers in [1, 4]");
    if (n_mlp_sizes < 2 || n_mlp_sizes > kMaxMlpLayers + 1) return fail(TACO_E_INVALID, "taco_critic_create: need 2..9 MLP sizes [lstm_hidden, h1, ..., 1]");
    if (mlp_sizes[0] != lstm_hidden) return fail(TACO_E_INVALID, "taco_critic_create: mlp_sizes[0] must equal lstm_hidden (the encoder output feeds the MLP)");
    if (mlp_sizes[n_mlp_sizes - 1] != 1) return fail(TACO_E_INVALID, "taco_critic_create: the critic output width is 1");
    for (int i = 0; i < n_mlp_sizes; ++i)
        if (mlp_sizes[i] < 1 || mlp_sizes[i] > 512) return fail(TACO_E_INVALID, "taco_critic_create: layer sizes must be in [1, 512]");
    int ndev = 0;
    TACO_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(TACO_E_INVALID, "taco_critic_create: no such CUDA device");
    DevGuard guard(device);
    TacoCritic* c = new (std::nothrow) TacoCritic();
    if (!c) return fail(TACO_E_NOMEM, "host allocation failed");
    c->device = device; c->in_dim = in_dim; c->seq_len = seq_len; c->hidden = lstm_hidden; c->lstm_layers = lstm_layers;
    c->mlp_sizes.assign(mlp_sizes, mlp_sizes + n_mlp_sizes);
    c->n_mlp = n_mlp_sizes - 1;
    const int H = lstm_hidden;
    size_t lo = 0;
    for (int l = 0; l < lstm_layers; ++l) {
        const int in_l = l == 0 ? in_dim : H;
        const size_t sz[4] = {(size_t)4 * H * in_l, (size_t)4 * H * H, (size_t)4 * H, (size_t)4 * H};
        for (int q = 0; q < 4; ++q) { c->lstm_off.push_back(lo); lo += (sz[q] + 3) & ~(size_t)3; }
    }
    int mx = 0;
    for (int i = 0; i < n_mlp_sizes; ++i) mx = mlp_sizes[i] > mx ? mlp_sizes[i] : mx;
    c->off_lstm = seq_len * in_dim;
    c->off_mlp = c->off_lstm + lstm_layers * 3 * H;
    c->mlp_w = mx;
    c->fp_stride = (c->off_mlp + 2 * mx) | 1;
    c->fp_smem = kFpEnvs * c->fp_stride * (int)sizeof(float);
    cudaDeviceProp prop;
    cudaError_t ce = cudaGetDeviceProperties(&prop, device);
    if (ce == cudaSuccess && (size_t)c->fp_smem > prop.sharedMemPerBlockOptin) {
        delete c;
        return fail(TACO_E_INVALID, "taco_critic_create: shape needs more shared memory per CTA than the device has");
    }
    c->num_sms = prop.multiProcessorCount;
    // ---- is the shape eligible for the tcgen05 path?
    const int n_hidden = c->n_mlp - 1;
    c->tc_ok = true;
    if (prop.major != 10) { c->tc_ok = false; c->tc_why = "device is not sm_100"; }
    else if (H % 16 != 0 || H > kTcMaxLstmHidden) { c->tc_ok = false; c->tc_why = "LSTM width must be a multiple of 16, <= 64"; }
    else if (in_dim > kTcMaxIn || (in_dim & 1)) { c->tc_ok = false; c->tc_why = "input width must be even, <= 30"; }
    else if (seq_len > kMaxSeq) { c->tc_ok = false; c->tc_why = "sequence length > 8"; }
    else if (n_hidden < 1 || n_hidden > kMaxMlpHidden) { c->tc_ok = false; c->tc_why = "needs 1..3 MLP hidden layers"; }
    else if (!tc_hidden_widths_ok(mlp_sizes, n_hidden)) { c->tc_ok = false; c->tc_why = "MLP hidden widths must be multiples of 64, <= 256"; }
    if (ce == cudaSuccess) ce = cudaMalloc(&c->lstm_f32, lo * sizeof(float));
    if (ce == cudaSuccess) ce = mlp_f32_alloc(c->f32, mlp_sizes, c->n_mlp);
    if (ce == cudaSuccess && c->tc_ok) {
        // [0] the LSTM step: n = 4H gate rows, K = [h (64) | x (64)] = 2 chunks; every layer's image in front of the MLP's
        c->tc.layer[0].n = 4 * H; c->tc.layer[0].kchunks = 2; c->tc.layer[0].img_off = 0;
        c->lstm_img_bytes = (size_t)2 * 4 * H * 128;
        ce = tc_image_alloc(c->tc, mlp_sizes, n_hidden, 1, lstm_layers * c->lstm_img_bytes);
        if (lstm_layers == 1) {
            set_tc_smem<false, false>(ce);
        } else {
            const char* e = getenv("TACO_CRITIC_CHUNK_WAVES");
            const int waves = (e && atoi(e) > 0) ? atoi(e) : kChunkWaves;
            c->chunk_tiles = waves * 2 * c->num_sms;
            const size_t ws_bytes = (size_t)c->chunk_tiles * seq_len * kTileM * 128;
            for (int b = 0; b < (lstm_layers > 2 ? 2 : 1); ++b)
                if (ce == cudaSuccess) ce = cudaMalloc(&c->seq_ws[b], ws_bytes);
            if (ce == cudaSuccess && lstm_layers > 2) ce = cudaMalloc(&c->seq_bias, (size_t)(lstm_layers - 2) * kMaxHidden * kMaxN * sizeof(float));
            set_tc_smem<false, true>(ce);
            set_tc_smem<true, true>(ce);
            set_tc_smem<true, false>(ce);
        }
    }
    if (ce == cudaSuccess && c->fp_smem > 48 * 1024)
        ce = cudaFuncSetAttribute(critic_fp32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, c->fp_smem);
    if (ce != cudaSuccess) {
        const std::string msg = std::string("taco_critic_create: ") + cudaGetErrorString(ce);
        taco_critic_destroy(c);
        return fail(ce == cudaErrorMemoryAllocation ? TACO_E_NOMEM : TACO_E_CUDA, msg);
    }
    *out = c;
    return TACO_OK;
}

int taco_critic_destroy(TacoCritic* c) {
    if (!c) return TACO_OK;
    DevGuard guard(c->device);
    cudaFree(c->lstm_f32); mlp_f32_free(c->f32);
    tc_image_free(c->tc);
    cudaFree(c->seq_bias); cudaFree(c->seq_ws[0]); cudaFree(c->seq_ws[1]);
    delete c;
    return TACO_OK;
}

int taco_critic_load(TacoCritic* c, const float* const* lstm_host, const float* const* mlp_weights_host, const float* const* mlp_biases_host,
                     void* stream) {
    if (!c || !lstm_host || !mlp_weights_host || !mlp_biases_host) return fail(TACO_E_INVALID, "taco_critic_load: null argument");
    for (int i = 0; i < 4 * c->lstm_layers; ++i)
        if (!lstm_host[i]) return fail(TACO_E_INVALID, "taco_critic_load: null LSTM parameter pointer");
    for (int l = 0; l < c->n_mlp; ++l)
        if (!mlp_weights_host[l] || !mlp_biases_host[l]) return fail(TACO_E_INVALID, "taco_critic_load: null MLP layer pointer");
    DevGuard guard(c->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int H = c->hidden;
    for (int l = 0; l < c->lstm_layers; ++l) {
        const int in_l = l == 0 ? c->in_dim : H;
        const size_t sz[4] = {(size_t)4 * H * in_l, (size_t)4 * H * H, (size_t)4 * H, (size_t)4 * H};
        for (int q = 0; q < 4; ++q)
            TACO_CUDA(cudaMemcpyAsync(c->lstm_f32 + c->lstm_off[4 * l + q], lstm_host[4 * l + q], sz[q] * sizeof(float), cudaMemcpyDefault, s));
    }
    if (int rc = mlp_f32_upload(c->f32, mlp_weights_host, mlp_biases_host, c->mlp_sizes.data(), c->n_mlp, s)) return rc;
    if (c->tc_ok) {
        TACO_CUDA(cudaMemsetAsync(c->tc.bias, 0, kMaxHidden * kMaxN * sizeof(float), s));
        if (c->seq_bias) TACO_CUDA(cudaMemsetAsync(c->seq_bias, 0, (size_t)(c->lstm_layers - 2) * kMaxHidden * kMaxN * sizeof(float), s));
        pack_lstm_kernel<<<64, 256, 0, s>>>(c->lstm_f32 + c->lstm_off[0], c->lstm_f32 + c->lstm_off[1], c->lstm_f32 + c->lstm_off[2],
                                            c->lstm_f32 + c->lstm_off[3], H, c->in_dim, 4 * H, c->tc.wimg); TACO_LAUNCHED();
        for (int l = 1; l < c->lstm_layers; ++l) {
            pack_lstm_seq_kernel<<<64, 256, 0, s>>>(c->lstm_f32 + c->lstm_off[4 * l], c->lstm_f32 + c->lstm_off[4 * l + 1],
                                                    c->lstm_f32 + c->lstm_off[4 * l + 2], c->lstm_f32 + c->lstm_off[4 * l + 3], H, 4 * H,
                                                    c->tc.wimg + l * c->lstm_img_bytes, tc_bias_block(c, l)); TACO_LAUNCHED();
        }
        if (int rc = tc_image_pack(c->tc, c->f32, c->mlp_sizes.data(), c->n_mlp - 1, s)) return rc;
    }
    TACO_CUDA(cudaStreamSynchronize(s));     // the host buffers may be released by the caller on return
    c->loaded = true;
    return TACO_OK;
}

int taco_critic_tc_available(TacoCritic* c) { return (c && c->tc_ok) ? 1 : 0; }

int taco_critic_forward(TacoCritic* c, const float* states_dev, float* value_dev, int32_t n, int32_t use_tensor_cores, void* stream) {
    if (!c || !states_dev || !value_dev) return fail(TACO_E_INVALID, "taco_critic_forward: null argument");
    if (!c->loaded) return fail(TACO_E_INVALID, "taco_critic_forward: call taco_critic_load first");
    if (n <= 0) return fail(TACO_E_INVALID, "taco_critic_forward: n must be positive");
    DevGuard guard(c->device);
    cudaStream_t s = (cudaStream_t)stream;
    if (use_tensor_cores) {
        if (!c->tc_ok) return fail(TACO_E_INVALID, "taco_critic_forward: tensor-core path unavailable for this shape: " + c->tc_why);
        CriticTcParams p;
        memset(&p, 0, sizeof(p));
        p.states = states_dev; p.value = value_dev;
        p.in_dim = c->in_dim; p.seq_len = c->seq_len; p.n_rows = n; p.num_tiles = (n + kTileM - 1) / kTileM;
        p.lstm_hidden = c->hidden; p.n_hidden = c->n_mlp - 1;
        p.wimg = c->tc.wimg; p.bias = c->tc.bias; p.b_out = c->tc.b_out;
        for (int l = 0; l <= p.n_hidden + 1; ++l) p.layer[l] = c->tc.layer[l];
        static const int stagger = [] { const char* e = getenv("TACO_CRITIC_STAGGER"); return e ? atoi(e) : kCriticStagger; }();
        p.stagger = stagger;
        if (c->lstm_layers == 1) {
            const int grid = tc_grid(p.num_tiles, c->num_sms, &p.tiles_per_cta);
            const char* tl = getenv("TACO_CRITIC_TIMELINE");
            if (int rc = timeline_begin(tl, &p.dbg, s)) return rc;
            launch_tc<false, false>(p, grid, s);
            if (int rc = timeline_end(tl, p.dbg, s)) return rc;
        } else {
            // chunk by chunk, layer 0 -> top on the stream (no timeline); the next layer reads the hand-off of a chunk while much
            // of it is still in L2.  The workspace is the handle's: one forward at a time per handle.
            const int L = c->lstm_layers, T = c->seq_len;
            const long long chunk_rows = (long long)c->chunk_tiles * kTileM;
            for (long long row0 = 0; row0 < n; row0 += chunk_rows) {
                const int rows = (int)(n - row0 < chunk_rows ? n - row0 : chunk_rows);
                p.states = states_dev + row0 * T * c->in_dim; p.value = value_dev + row0;
                p.n_rows = rows; p.num_tiles = (rows + kTileM - 1) / kTileM;
                const int grid = tc_grid(p.num_tiles, c->num_sms, &p.tiles_per_cta);
                for (int k = 0; k < L; ++k) {
                    p.layer[0].img_off = (uint32_t)(k * c->lstm_img_bytes);
                    p.bias = tc_bias_block(c, k);
                    p.seq_in = k > 0 ? c->seq_ws[(k - 1) & 1] : nullptr;
                    p.seq_out = k + 1 < L ? c->seq_ws[k & 1] : nullptr;
                    if (k == 0) launch_tc<false, true>(p, grid, s);
                    else if (k + 1 < L) launch_tc<true, true>(p, grid, s);
                    else launch_tc<true, false>(p, grid, s);
                }
            }
        }
    } else {
        FpParams p;
        memset(&p, 0, sizeof(p));
        p.states = states_dev; p.value = value_dev; p.n_rows = n;
        p.in_dim = c->in_dim; p.seq_len = c->seq_len; p.hidden = c->hidden; p.lstm_layers = c->lstm_layers; p.n_mlp = c->n_mlp;
        for (int l = 0; l < c->lstm_layers; ++l) {
            p.w_ih[l] = c->lstm_f32 + c->lstm_off[4 * l + 0]; p.w_hh[l] = c->lstm_f32 + c->lstm_off[4 * l + 1];
            p.b_ih[l] = c->lstm_f32 + c->lstm_off[4 * l + 2]; p.b_hh[l] = c->lstm_f32 + c->lstm_off[4 * l + 3];
        }
        for (int l = 0; l <= c->n_mlp; ++l) p.mlp_sizes[l] = c->mlp_sizes[l];
        for (int l = 0; l < c->n_mlp; ++l) { p.w[l] = c->f32.w + c->f32.w_off[l]; p.b[l] = c->f32.b + c->f32.b_off[l]; }
        p.stride = c->fp_stride; p.off_lstm = c->off_lstm; p.off_mlp = c->off_mlp; p.mlp_w = c->mlp_w;
        critic_fp32_kernel<<<(n + kFpEnvs - 1) / kFpEnvs, kFpThreads, c->fp_smem, s>>>(p); TACO_LAUNCHED();
    }
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

}  // extern "C"
