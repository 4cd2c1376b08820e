// Native PPO update behind the C ABI (include/taco_b200.h, taco_ppo_*): SURVEY.md section 8f row 4.
//
// Mirrors PPO.update of the reference (IsaacGymEnvs/algorithms/ppo_asymmetry.py:137-258) for the network configuration the
// reference trains with (README.md:60-66; nets_asymmetry.py:270-377): actor = MLP(obs) -> tanh mean, state-independent log_std,
// MultivariateNormal(mean, scale_tril = diag(exp(log_std)^2)); critic = MLP(LSTMEncoder(states)).  Per minibatch:
//
//   gather        obs / states / action / old log-prob / advantage / return rows of the minibatch indices -> bf16 operands
//   forward       actor MLP and critic (5 LSTM steps + MLP) as tcgen05 GEMMs (gemm_tc.cuh), activations saved for the backward pass
//   loss          PPO_ActorCritic.evaluate + the loss terms of :190-212: ratio, clipped surrogate, value MSE, entropy, approx KL
//                 (:218-221); writes d loss / d mean-pre-activation and d loss / d value, accumulates the statistics
//   decide        the KL early stop of :223-226 taken ON THE DEVICE (a flag later launches test), so an update needs no host sync
//   backward      dX / dW GEMMs (split-K partials for the K = batch weight gradients), LSTM backward through time
//   apply         gradient assembly + global norm (clip_grad_norm_, :244), Adam (torch.optim.Adam, eps 1e-5, :117), spectral
//                 projection of the actor weights (:248-249, :398-404), re-pack of the bf16 operand copies
//
// Arithmetic: bf16 operands, fp32 accumulation (tensor memory), fp32 master weights / Adam moments / losses.  Everything
// else on the path (gathers, losses, LSTM point-wise backward, reductions, Adam) is plain fp32 CUDA.
#include "launch_count.h"
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>

#include "host_common.h"
#include "gemm_tc.cuh"

namespace taco {
namespace ppo {

using namespace taco::gemm;
typedef __nv_bfloat16 bf16;

constexpr int kMaxHiddenL = 4;
constexpr int kMaxLstmL = 4;        // stacked LSTM layers of the critic encoder
constexpr int kH = 64;              // LSTM hidden width the LSTM epilogue is written for
constexpr int kG = 4 * kH;          // gate rows
constexpr int kSeqMax = 8;
constexpr int kNumStat = 16;        // accumulators: [0] surrogate, [1] value, [2] kl, [3] count, [4..7] d log_std, [8] grad norm^2
constexpr int kLogCols = 8;         // per minibatch log row: pg, value, entropy, total, kl, grad_norm, stopped, clip_coef

static inline int pad8(int x) { return (x + 7) & ~7; }
static inline int pad16(int x) { return (x + 15) & ~15; }

// ---------------------------------------------------------------------------------------------- tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}
// row-major matrix [rows][cols] of elem_bytes-sized elements, row pitch ld elements, 128-byte swizzle; box = box_cols x box_rows
static bool encode_map(CUtensorMap* tm, CUtensorMapDataType type, size_t elem_bytes, const void* ptr, long long rows, long long cols, long long ld,
                       int box_cols, int box_rows) {
    EncodeTiledFn f = encode_fn();
    if (!f) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * elem_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return f(tm, type, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// bf16 operand: box = 64 columns (one 128-byte swizzle row) x box_rows rows
static bool make_map(CUtensorMap* tm, const bf16* ptr, long long rows, long long cols, long long ld, int box_rows) {
    return encode_map(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, sizeof(bf16), ptr, rows, cols, ld, BK, box_rows);
}
// fp32 output of the split-K GEMMs, stored tile by tile (32 columns x 128 rows) by the TMA store engine
static bool make_map_f32(CUtensorMap* tm, const float* ptr, long long rows, long long cols, long long ld) {
    return encode_map(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sizeof(float), ptr, rows, cols, ld, 32, BM);
}

// ---------------------------------------------------------------------------------------------- small kernels
struct Hyper {
    float lr, clip, target_kl, max_grad, pi_coef, vf_coef, ent_coef, lipschitz;
    int use_lipschitz, world;
};

// minibatch gather: rows idx[i] of the rollout tensors -> bf16 operands (batch-major) + compact fp32 side arrays
struct GatherParams {
    const float* obs; int obs_dim;                  // [N][obs_dim]
    const float* states; int seq, state_dim;        // [N][seq][state_dim]
    const float* act; const float* logp; const float* adv; const float* ret;   // [N][A], [N], [N], [N]
    const long long* idx; int B, act_dim;
    bf16* x0_bm; int ld_x0;                         // [B][ld_x0]
    bf16* u_bm; int ld_u;                           // [seq*B][ld_u]: columns [h(64) | x | 1 1 | 0]
    float* g_act; float* g_logp; float* g_adv; float* g_ret;
    const int* stop;
};
// one operand matrix for the 32 samples of a CTA: features [0, n_src) come from the sample's source row, [n_src, n_src + n_one) are
// the constant 1, the rest up to n_out is 0
__device__ __forceinline__ void gather_matrix(const float* src, long long src_stride, const long long* rows, int n_valid,
                                              int n_src, int n_one, int n_out, bf16* bm, long long ld_bm) {
    for (int e = threadIdx.x; e < n_valid * n_out; e += blockDim.x) {
        const int sidx = e / n_out, f = e % n_out;
        const float v = f < n_src ? __ldg(src + rows[sidx] * src_stride + f) : (f < n_src + n_one ? 1.0f : 0.0f);
        bm[(long long)sidx * ld_bm + f] = __float2bfloat16_rn(v);
    }
}
__global__ void __launch_bounds__(256) gather_kernel(const GatherParams p) {
    pdl_launch_dependents();
    pdl_wait();
    if (p.stop && *p.stop) return;
    __shared__ long long rows[32];
    const int i0 = blockIdx.x * 32;
    const int nv = min(32, p.B - i0);
    if (threadIdx.x < 32) rows[threadIdx.x] = threadIdx.x < nv ? p.idx[i0 + threadIdx.x] : 0;
    __syncthreads();
    gather_matrix(p.obs, p.obs_dim, rows, nv, p.obs_dim, 0, (p.obs_dim + 7) & ~7, p.x0_bm + (long long)i0 * p.ld_x0, p.ld_x0);
    // U_t = [h_{t-1} (64, written by the previous LSTM step; h_0 = 0 stays as allocated) | x_t | 1 1 | 0]: two constant-1 inputs carry the bias
    for (int t = 0; t < p.seq; ++t)
        gather_matrix(p.states + (long long)t * p.state_dim, (long long)p.seq * p.state_dim, rows, nv, p.state_dim, 2, p.ld_u - kH,
                      p.u_bm + ((long long)t * p.B + i0) * p.ld_u + kH, p.ld_u);
    for (int e = threadIdx.x; e < nv * (p.act_dim + 3); e += blockDim.x) {
        const int sidx = e / (p.act_dim + 3), c = e % (p.act_dim + 3);
        const long long r = rows[sidx];
        if (c < p.act_dim) p.g_act[(long long)(i0 + sidx) * p.act_dim + c] = __ldg(p.act + r * p.act_dim + c);
        else if (c == p.act_dim) p.g_logp[i0 + sidx] = __ldg(p.logp + r);
        else if (c == p.act_dim + 1) p.g_adv[i0 + sidx] = __ldg(p.adv + r);
        else p.g_ret[i0 + sidx] = __ldg(p.ret + r);
    }
}

// PPO_ActorCritic.evaluate + losses (nets_asymmetry.py:356-377, ppo_asymmetry.py:190-221), one thread per sample
struct LossParams {
    const float* mean; const float* value;          // [B][A], [B]
    const float* act; const float* old_logp; const float* adv; const float* ret;
    const float* log_std;                           // [A] (master parameter)
    int B, act_dim;
    Hyper h;
    bf16* dz_bm;                                    // actor output-layer pre-activation gradient: [B][16]
    bf16* dv_bm;                                    // critic value gradient: [B][16] (column 0)
    double* acc;                                    // kNumStat accumulators
    const int* stop;
};
__global__ void __launch_bounds__(256) loss_kernel(const LossParams p) {
    pdl_launch_dependents();
    pdl_wait();
    if (p.stop && *p.stop) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float s_sur = 0.f, s_val = 0.f, s_kl = 0.f, dls[4] = {0.f, 0.f, 0.f, 0.f};
    if (i < p.B) {
        const int A = p.act_dim;
        float z[4], mu[4], inv_sd[4];
        float logp = -0.5f * A * 1.8378770664093453f;                  // -k/2 log(2 pi)
        for (int k = 0; k < A; ++k) {
            const float lsd = 2.0f * __ldg(p.log_std + k);              // std = exp(log_std)^2 (nets_asymmetry.py:338)
            inv_sd[k] = __expf(-lsd);
            mu[k] = p.mean[(long long)i * A + k];
            z[k] = (p.act[(long long)i * A + k] - mu[k]) * inv_sd[k];
            logp += -0.5f * z[k] * z[k] - lsd;
        }
        const float adv = p.adv[i];
        const float log_ratio = logp - p.old_logp[i];
        const float ratio = __expf(log_ratio);
        const float rc = fminf(fmaxf(ratio, 1.0f - p.h.clip), 1.0f + p.h.clip);
        const float s1 = adv * ratio, s2 = adv * rc;
        s_sur = -fminf(s1, s2);                                         // :196-199
        // d(-min(s1, s2)) / d logp: the unclipped branch when it is the minimum (ties: clamp passes the gradient inside the range)
        const float dl_dlogp = (s1 <= s2) ? -adv * ratio : 0.0f;
        const float dv = p.value[i] - p.ret[i];
        s_val = dv * dv;                                                // F.mse_loss(ret, value), :206
        s_kl = (ratio - 1.0f) - log_ratio;                              // :219-220
        const float invB = 1.0f / (float)p.B;
        const float gl = p.h.pi_coef * dl_dlogp * invB;
        for (int k = 0; k < 16; ++k) {
            float g = 0.0f;
            if (k < A) {
                g = gl * z[k] * inv_sd[k] * (1.0f - mu[k] * mu[k]);     // through mean = tanh(pre-activation)
                dls[k] = gl * 2.0f * (z[k] * z[k] - 1.0f);              // d logp / d log_std = 2 (z^2 - 1)
            }
            const bf16 b = __float2bfloat16_rn(g);
            p.dz_bm[(long long)i * 16 + k] = b;
            const bf16 bv = __float2bfloat16_rn(k == 0 ? p.h.vf_coef * 2.0f * dv * invB : 0.0f);
            p.dv_bm[(long long)i * 16 + k] = bv;
        }
    }
    __shared__ float red[7][8];
    float vals[7] = {s_sur, s_val, s_kl, dls[0], dls[1], dls[2], dls[3]};
#pragma unroll
    for (int q = 0; q < 7; ++q) {
        float v = vals[q];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 7) {
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += (double)red[threadIdx.x][w];
        const int slot = threadIdx.x < 3 ? threadIdx.x : threadIdx.x + 1;       // 0,1,2 = losses; 4..7 = d log_std
        atomicAdd(p.acc + slot, s);
    }
}

// the per-minibatch bookkeeping of :214-226 on the device: means, log row, KL early stop
struct DecideParams {
    double* acc; float* log; int* n_logged; int* stop; int max_log;
    const float* log_std; int act_dim, B;
    Hyper h;
    float* grad_log_std;                           // flat gradient slot of log_std
};
__global__ void decide_kernel(const DecideParams p) {
    pdl_launch_dependents();
    pdl_wait();
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (*p.stop) return;
    const double w = (double)p.h.world, n = (double)p.B * w;           // under data parallelism acc holds the all-reduced sums
    const double pg = p.acc[0] / n, vl = p.acc[1] / n, kl = p.acc[2] / n;
    double ent = 0.5 * p.act_dim * (1.0 + 1.8378770664093453);
    for (int k = 0; k < p.act_dim; ++k) ent += 2.0 * (double)p.log_std[k];
    const double el = -ent;                                             // entropy_loss = -mean(entropy), :209
    const double total = p.h.pi_coef * pg + p.h.vf_coef * vl + p.h.ent_coef * el;
    const int row = *p.n_logged;
    if (row < p.max_log) {
        float* L = p.log + (size_t)row * kLogCols;
        L[0] = (float)pg; L[1] = (float)vl; L[2] = (float)el; L[3] = (float)total; L[4] = (float)kl; L[5] = 0.f; L[6] = 0.f; L[7] = 1.f;
    }
    *p.n_logged = row + 1;
    if (kl > 1.5 * (double)p.h.target_kl && p.h.pi_coef > 0.0f) {      // :223-226
        *p.stop = 1;
        if (row < p.max_log) p.log[(size_t)row * kLogCols + 6] = 1.f;
    }
    // d loss / d log_std (local sums: the flat gradient is averaged over ranks later like every other gradient)
    for (int k = 0; k < p.act_dim; ++k) p.grad_log_std[k] = (float)(p.acc[4 + k] / w) + p.h.ent_coef * -2.0f;
    for (int k = 0; k < 8; ++k) p.acc[k] = 0.0;
}

// LSTM backward, point-wise part of one time step (the gate math of nn.LSTM): one thread per (sample, unit), lanes along the units
struct LstmBwdParams {
    const float* dh; float* dc;                     // [B][ld_dh], [B][64]: dL/dh_t from this layer's step t+1 or the critic MLP (null: 0),
    int ld_dh;                                      // dL/dc_t carried from step t+1 (in) -> dL/dc_{t-1} (out)
    const float* dh_add; int ld_dh_add;             // [B][ld_dh_add]: dL/dh_t through the LSTM layer above (null: top layer), added to dh
    const bf16* gates; const float* c_prev; const float* c_cur;     // [B][256] activated gates of step t (chunked layout), c_{t-1} (null: 0), c_t
    bf16* dg_bm;                                    // [B][256] gate pre-activation gradients of step t
    int B; int first;                               // first = this is the last time step (dc_in = 0)
    const int* stop;
};
__global__ void __launch_bounds__(256) lstm_bwd_kernel(const LstmBwdParams p) {
    pdl_launch_dependents();
    pdl_wait();
    if (p.stop && *p.stop) return;
    const int j = threadIdx.x & (kH - 1);
    const long long i = (long long)blockIdx.x * 4 + (threadIdx.x >> 6);
    if (i >= p.B) return;
    const bf16* g = p.gates + i * kG + (j >> 4) * 64 + (j & 15);     // [4 chunks][4 gates][16 units] (gemm_tc.cuh LstmEpi::gates_out)
    const float gi = __bfloat162float(g[0]), gf = __bfloat162float(g[16]), gg = __bfloat162float(g[32]), go = __bfloat162float(g[48]);
    const float c = p.c_cur[i * kH + j], cp = p.c_prev ? p.c_prev[i * kH + j] : 0.0f;
    const float tc = tanhf(c);
    float dh = p.dh ? p.dh[i * p.ld_dh + j] : 0.0f;
    if (p.dh_add) dh += p.dh_add[i * p.ld_dh_add + j];
    const float dc = (p.first ? 0.0f : p.dc[i * kH + j]) + dh * go * (1.0f - tc * tc);
    p.dc[i * kH + j] = dc * gf;
    bf16* d = p.dg_bm + i * kG + j;
    d[0] = __float2bfloat16_rn(dc * gg * gi * (1.0f - gi));
    d[kH] = __float2bfloat16_rn(dc * cp * gf * (1.0f - gf));
    d[2 * kH] = __float2bfloat16_rn(dc * gi * (1.0f - gg * gg));
    d[3 * kH] = __float2bfloat16_rn(dh * tc * go * (1.0f - go));
}

// column sums of batch-major bf16 matrices = bias gradients.  A CTA sums kColRows rows of one matrix (lanes along the columns, bf16
// pairs) and writes one partial row; grad_assemble_kernel adds the partial rows in a fixed order (bit-reproducible).
constexpr int kColRows = 512, kColLd = 256;
struct ColSumSeg { const bf16* src; int ld; };      // [B][ld], ld a multiple of 16, <= 256
struct ColSumParams { ColSumSeg seg[2 * (kMaxHiddenL + 1)]; int n_seg; int B; float* partial; const int* stop; };   // partial: [seg][chunk][kColLd]
__global__ void __launch_bounds__(256) colsum_kernel(const ColSumParams p) {
    pdl_launch_dependents();
    pdl_wait();
    if (p.stop && *p.stop) return;
    __shared__ float2 part[256];
    const ColSumSeg sg = p.seg[blockIdx.y];
    const int pairs = sg.ld >> 1;                    // 8 .. 128 column pairs
    const int lanes = 256 / pairs;                   // row lanes
    const int cp = threadIdx.x % pairs, rl = threadIdx.x / pairs;
    const int r0 = blockIdx.x * kColRows, r1 = min(r0 + kColRows, p.B);
    float2 acc = make_float2(0.f, 0.f);
    if (rl < lanes)
        for (int r = r0 + rl; r < r1; r += lanes) {
            const uint32_t u = *reinterpret_cast<const uint32_t*>(sg.src + (long long)r * sg.ld + 2 * cp);
            acc.x += __uint_as_float(u << 16); acc.y += __uint_as_float(u & 0xFFFF0000u);
        }
    part[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < pairs) {
        float2 t = make_float2(0.f, 0.f);
        for (int l = 0; l < lanes; ++l) { t.x += part[l * pairs + threadIdx.x].x; t.y += part[l * pairs + threadIdx.x].y; }
        float* dst = p.partial + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * kColLd + 2 * threadIdx.x;
        dst[0] = t.x; dst[1] = t.y;
    }
}

// gradient assembly: flat_grad[dst + r * cols + c] = sum over splits of partial[s][r][col0 + c]; accumulates the global norm^2
struct GradSeg { const float* partial; int splits; long long split_stride; int ld, col0, rows, cols; long long dst; };
struct GradParams { GradSeg seg[4 * (kMaxHiddenL + 1) + 4 * kMaxLstmL]; int n_seg; float* grad; double* acc; const int* stop; };
__global__ void __launch_bounds__(256) grad_assemble_kernel(const GradParams p) {
    pdl_launch_dependents();
    pdl_wait();
    if (p.stop && *p.stop) return;
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (int s = 0; s < p.n_seg; ++s) {
        const long long cnt = (long long)p.seg[s].rows * p.seg[s].cols;
        if (e < cnt) {
            const GradSeg& g = p.seg[s];
            const int r = (int)(e / g.cols), c = (int)(e % g.cols);
            const float* src = g.partial + (long long)r * g.ld + g.col0 + c;
            float acc = 0.f;
            for (int k = 0; k < g.splits; ++k) acc += src[(long long)k * g.split_stride];
            p.grad[g.dst + e] = acc;
            return;
        }
        e -= cnt;
    }
}
__global__ void __launch_bounds__(256) grad_norm_kernel(const float* grad, long long n, float inv_world, double* acc, const int* stop) {
    pdl_launch_dependents();
    pdl_wait();
    if (stop && *stop) return;
    double s = 0.0;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const double g = (double)grad[e] * inv_world;
        s += g * g;
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
        atomicAdd(acc + 8, t);
    }
}

// clip_grad_norm_ (:244) + torch.optim.Adam (betas 0.9 / 0.999, eps 1e-5, :117): element-wise over the flat parameter vector
__global__ void __launch_bounds__(256) adam_kernel(float* prm, float* m, float* v, const float* grad, long long n, Hyper h, int* step, double* acc,
                                                   float* log, const int* n_logged, int max_log, const int* stop) {
    pdl_launch_dependents();
    pdl_wait();
    if (stop && *stop) return;
    const double norm = sqrt(acc[8]);
    const float coef = fminf((float)((double)h.max_grad / (norm + 1e-6)), 1.0f) / (float)h.world;     // the 1 / world averages the summed gradient
    const int t = *step + 1;
    const float b1 = 0.9f, b2 = 0.999f;
    const float a1 = 0.1f, a2 = 0.001f;             // 1 - beta rounded from the exact value, as torch passes it (1.0f - b2 is 1.3e-5 off)
    const float bc1 = 1.0f - powf(b1, (float)t), bc2 = 1.0f - powf(b2, (float)t);
    const float step_size = h.lr / bc1, inv_sqrt_bc2 = rsqrtf(bc2);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const float g = grad[e] * coef;
        const float mm = b1 * m[e] + a1 * g;
        const float vv = b2 * v[e] + a2 * g * g;
        m[e] = mm; v[e] = vv;
        prm[e] -= step_size * (mm / (sqrtf(vv) * inv_sqrt_bc2 + 1e-5f));
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const int row = *n_logged - 1;
        if (row >= 0 && row < max_log) { log[(size_t)row * kLogCols + 5] = (float)norm; log[(size_t)row * kLogCols + 7] = coef * (float)h.world; }
    }
}
__global__ void finish_step_kernel(int* step, double* acc, const int* stop) {
    pdl_launch_dependents();
    pdl_wait();
    if (stop && *stop) return;
    *step += 1;
    acc[8] = 0.0;
}

// PPO.spectral_normalize_actors (:398-404): sigma = ||W||_2 by power iteration on W^T W, warm-started from the previous optimiser
// step's right singular vector; W *= c / sigma when sigma > c.  One CTA per weight matrix, all matrices in one launch.
//
// A matrix whose `cold` flag is set (a new handle, or weights loaded from outside) starts from the constant vector with the cold
// iteration cap and clears its flag; a launch the early-stop flag turns into a no-op leaves it set.  Power iteration only ever
// underestimates sigma, and the estimate can rise slowly for many iterations (a small top gap, or a start vector with little
// weight on the top singular vector), so a single small change is not convergence: the loop stops once sigma has risen by at
// most kSpecTol over the last kSpecWindow iterations (fp32 rounding moves sigma by ~1e-7, far below what a window may gain).
// sigma is estimated as sqrt(||W^T W v||) for ||v|| = 1: a lower bound like ||W v||, closer to sigma_1, and it needs only the
// norm that normalises v.
constexpr int kSpecWindow = 8, kSpecColdIter = 4000, kSpecWarmIter = 200;
constexpr double kSpecTol = 1e-6;
struct SpecSeg { float* w; int rows, cols; float* v; double* sigma; int* cold; };
struct SpecParams { SpecSeg seg[kMaxHiddenL + 1]; int n_seg; float lipschitz; const int* stop; };
__global__ void __launch_bounds__(512) spectral_kernel(const SpecParams p) {
    pdl_launch_dependents();
    pdl_wait();
    if (p.stop && *p.stop) return;
    const SpecSeg& S = p.seg[blockIdx.x];
    __shared__ float v[256], u[256], part[2][256];
    __shared__ float red[16];
    __shared__ double hist[kSpecWindow], s_norm, s_sigma;
    __shared__ int s_done;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int rows = S.rows, cols = S.cols;
    const float* __restrict__ W = S.w;
    const bool cold = *S.cold != 0;
    const int max_iter = cold ? kSpecColdIter : kSpecWarmIter;
    for (int c = tid; c < cols; c += 512) v[c] = cold ? 1.0f / sqrtf((float)cols) : S.v[c];
    __syncthreads();
    for (int it = 0; it < max_iter; ++it) {
        // u = W v: a warp per row (two rows in flight), lanes along the row: coalesced reads of W from L2
        for (int r0 = warp * 2; r0 < rows; r0 += 32) {
            float a0 = 0.f, a1 = 0.f;
            const bool two = r0 + 1 < rows;
            for (int c = lane; c < cols; c += 32) {
                const float vc = v[c];
                a0 = fmaf(__ldg(W + (long long)r0 * cols + c), vc, a0);
                if (two) a1 = fmaf(__ldg(W + (long long)(r0 + 1) * cols + c), vc, a1);
            }
            for (int o = 16; o > 0; o >>= 1) { a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o); }
            if (lane == 0) { u[r0] = a0; if (two) u[r0 + 1] = a1; }
        }
        __syncthreads();
        // W^T u: thread <-> (column, half of the rows): lanes read consecutive columns of one row, 8 loads in flight
        {
            const int c = tid & 255, half = tid >> 8;
            if (c < cols) {
                const int rb = half * ((rows + 1) >> 1), re = half ? rows : ((rows + 1) >> 1);
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                int r = rb;
                for (; r + 3 < re; r += 4) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[q] = fmaf(__ldg(W + (long long)(r + q) * cols + c), u[r + q], acc[q]);
                }
                for (; r < re; ++r) acc[0] = fmaf(__ldg(W + (long long)r * cols + c), u[r], acc[0]);
                part[half][c] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
            }
        }
        __syncthreads();
        // v = W^T u and ||v||^2; thread 0 takes sigma and the stop test
        {
            float a = 0.f;
            for (int c = tid; c < cols; c += 512) { const float x = part[0][c] + part[1][c]; v[c] = x; a = fmaf(x, x, a); }
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0) red[warp] = a;
            __syncthreads();
            if (tid == 0) {
                double t = 0.0;
                for (int w = 0; w < 16; ++w) t += (double)red[w];
                const double sg = sqrt(sqrt(t));
                const int slot = it % kSpecWindow;
                s_done = it >= kSpecWindow && sg - hist[slot] <= kSpecTol * sg;
                hist[slot] = sg;
                s_norm = t; s_sigma = sg;
            }
            __syncthreads();
        }
        const float inv = s_norm > 0.0 ? (float)(1.0 / sqrt(s_norm)) : 0.f;
        for (int c = tid; c < cols; c += 512) v[c] *= inv;                  // (each thread its own columns, as written above)
        if (s_done) break;
        __syncthreads();
    }
    const float sig = (float)s_sigma;
    for (int c = tid; c < cols; c += 512) S.v[c] = v[c];
    if (tid == 0) { *S.sigma = (double)sig; *S.cold = 0; }
    if (p.lipschitz > 0.0f && sig > p.lipschitz) {
        const float sc = p.lipschitz / sig;                             // param.data *= lipschitz_const / spectral_norm
        for (long long e = tid; e < (long long)rows * cols; e += 512) S.w[e] *= sc;
    }
}

// fp32 master weights -> bf16 operand copies: W [out][ld_w] (K = in) and W^T [in][ld_t] (K = out), zero padded
struct PackSeg { const float* w; int out, in; bf16* wb; int ld_w; bf16* wt; int ld_t; int rows_t; };
struct PackParams { PackSeg seg[2 * (kMaxHiddenL + 1)]; int n_seg; const int* stop; };
__global__ void __launch_bounds__(256) pack_kernel(const PackParams p) {
    pdl_launch_dependents();
    pdl_wait();
    if (p.stop && *p.stop) return;
    const PackSeg& S = p.seg[blockIdx.y];
    const long long nw = (long long)S.out * S.ld_w, ntr = (long long)S.rows_t * S.ld_t;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nw + ntr; e += (long long)gridDim.x * blockDim.x) {
        if (e < nw) {
            const int o = (int)(e / S.ld_w), i = (int)(e % S.ld_w);
            S.wb[e] = __float2bfloat16_rn(i < S.in ? S.w[(long long)o * S.in + i] : 0.0f);
        } else if (S.wt) {
            const long long f = e - nw;
            const int i = (int)(f / S.ld_t), o = (int)(f % S.ld_t);
            S.wt[f] = __float2bfloat16_rn((i < S.in && o < S.out) ? S.w[(long long)o * S.in + i] : 0.0f);
        }
    }
}
// one LSTM layer: Wcat [256][ld_u] = [W_hh | W_ih | b_hi b_lo | 0] and its transpose Wcat^T [t_rows][256]: rows 0..63 W_hh^T, then
// (t_rows = 128, layers above the first) W_ih^T
__global__ void __launch_bounds__(256) pack_lstm_kernel(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, int in_dim, int ld_u,
                                                        bf16* wcat, bf16* wcat_t, int t_rows, const int* stop) {
    pdl_launch_dependents();
    pdl_wait();
    if (stop && *stop) return;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < kG * ld_u + t_rows * kG; e += gridDim.x * blockDim.x) {
        if (e < kG * ld_u) {
            const int r = e / ld_u, c = e % ld_u;
            float v = 0.0f;
            if (c < kH) v = w_hh[r * kH + c];
            else if (c < kH + in_dim) v = w_ih[r * in_dim + (c - kH)];
            else if (c < kH + in_dim + 2) {
                const float b = b_ih[r] + b_hh[r];
                const float hi = __bfloat162float(__float2bfloat16_rn(b));
                v = (c == kH + in_dim) ? hi : b - hi;
            }
            wcat[e] = __float2bfloat16_rn(v);
        } else {
            const int f = e - kG * ld_u;
            const int j = f / kG, r = f % kG;                             // W_hh^T[j][r] = W_hh[r][j], W_ih^T[j - 64][r] = W_ih[r][j - 64]
            wcat_t[f] = __float2bfloat16_rn(j < kH ? w_hh[r * kH + j] : w_ih[r * in_dim + (j - kH)]);
        }
    }
}

}  // namespace ppo
}  // namespace taco

using namespace taco::ppo;
using taco::DevGuard;
using taco::fail;

// ---------------------------------------------------------------------------------------------- the trainer object
// split-K plan of a GEMM of depth k: `splits` work items of kb_per_split k-blocks each, none of them empty
struct SplitK { int splits = 1, kb_per_split = 1; };
static SplitK split_k(int requested, long long k) {
    const int kb_total = (int)((k + BK - 1) / BK);
    SplitK r;
    r.splits = requested < 1 ? 1 : (requested > kb_total ? kb_total : requested);
    r.kb_per_split = (kb_total + r.splits - 1) / r.splits;
    r.splits = (kb_total + r.kb_per_split - 1) / r.kb_per_split;      // merge the splits that would be left empty
    return r;
}

// one linear layer Y = X W^T + b of an MLP (M = batch)
struct MlpLayer {
    int in = 0, out = 0;
    long long w_off = 0, b_off = 0;                 // offsets into the flat parameter vector
    bf16* wb = nullptr; int ld_w = 0;               // [out_pad16][pad8(in)]
    bf16* wt = nullptr; int ld_t = 0;               // [in][pad8(out) (>= 16)]
    bf16* x_bm = nullptr; int ld_x = 0;             // input activation X: [B][pad8(in)]
    uint32_t* mask = nullptr;                       // layers >= 1: ReLU mask of X, [ceil(in / 32)][B] words, bit j = pre-activation (sample, 32 c + j) > 0
    bf16* dz_bm = nullptr; int ld_dz = 0;           // dZ, the gradient of this layer's output pre-activation: [B][pad16(out)]
    float* partial = nullptr; int ld_p = 0;         // dW split-K partials: [split.splits][out][ld_p]
    SplitK split;
    // K-major maps (forward / dX GEMMs) and MN-major maps of the same batch-major tensors (dW = dZ^T X reads both transposed)
    CUtensorMap m_x_bm, m_x_mn, m_w, m_wt, m_dz_bm, m_dz_mn;
    CUtensorMap m_partial;                          // only when out % 128 == 0: the partials are then TMA-stored
};
struct MlpNet {
    int L = 0;                                      // linear layers
    MlpLayer layer[kMaxHiddenL + 1];
};

// one layer k of the stacked LSTM encoder; its operand of step t is U_k[t] = [h^k_{t-1} | x^k_t | 1 1 | 0] with x^0_t = states[:, t] and
// x^k_t = h^{k-1}_t (written by layer k-1's epilogue), so one GEMM U_k[t] Wcat_k^T gives the gate pre-activations with the bias
struct LstmLayer {
    int in = 0, ld_u = 0, t_rows = 0;               // input width (state_dim, or 64 above layer 0), U / Wcat row pitch, rows of Wcat^T
    long long off_wih = 0, off_whh = 0, off_bih = 0, off_bhh = 0;
    bf16 *wcat = nullptr, *wcat_t = nullptr;        // [256][ld_u], [t_rows][256] (W_hh^T, then W_ih^T for k >= 1)
    bf16 *u_bm = nullptr, *gates = nullptr, *dg_bm = nullptr;       // [seq*B][ld_u], [seq*B][256] x 2 (all time steps)
    float *c_state = nullptr, *partial = nullptr;   // [seq*B][64]; dWcat split-K partials [split.splits][256][ld_u]
    float* dhx = nullptr;                           // k >= 1: [seq][B][128] = d[h_{t-1} | x_t] of step t (slot 0: the x half only)
    SplitK split;
    CUtensorMap m_u_bm, m_u_mn, m_wcat, m_wcat_t, m_wih_t, m_dg_bm, m_dg_mn, m_partial;
    CUtensorMap m_dhx[kSeqMax], m_dx0;              // k >= 1: output maps of the d[h | x] GEMM per step, and of the dx-only GEMM of step 0
};

struct TacoPPO {
    int device = 0, num_sms = 148;
    TacoPPOCfg cfg;
    int B = 0, A = 0, seq = 0, sd = 0, n_lstm = 1;
    long long n_params = 0;
    long long off_log_std = 0;
    float *prm = nullptr, *grad = nullptr, *adam_m = nullptr, *adam_v = nullptr;
    MlpNet actor, critic;
    // LSTM: the layers, dL/dh of layer 0's recurrence (and of the top layer's last step, from the critic MLP), dL/dc of the layer in flight
    LstmLayer lstm[kMaxLstmL];
    float *dh = nullptr, *dc = nullptr, *colsum_partial = nullptr;
    CUtensorMap m_dh;
    // heads / side arrays
    float *mean = nullptr, *value = nullptr, *g_act = nullptr, *g_logp = nullptr, *g_adv = nullptr, *g_ret = nullptr;
    // bookkeeping
    double* acc = nullptr; float* log = nullptr; int *n_logged = nullptr, *stop = nullptr, *step = nullptr;
    int max_log = 4096;
    // power iteration state per actor matrix: right singular vector, sigma, cold-start flag (set: the next projection starts over)
    float* spec_v[kMaxHiddenL + 1] = {nullptr}; double* spec_sigma = nullptr; int* spec_cold = nullptr;
    // the spectral projection + re-pack of the ACTOR runs on a side stream under the next minibatch's gather and critic forward
    cudaStream_t side = nullptr;
    cudaEvent_t ev_adam = nullptr, ev_actor = nullptr;
    bool actor_pending = false;
    std::vector<void*> allocs;
};

// zero-filled device allocations owned by t (the h_0 columns and the LSTM rings' zero padding rely on the zero fill).  The first
// failure stays in `err` and turns every later call into a no-op, so a run of allocations is checked once, at its end.
struct DevAlloc {
    TacoPPO* t;
    cudaError_t err = cudaSuccess;
    template <typename T>
    void operator()(T** p, size_t count) {
        if (err != cudaSuccess) return;
        err = cudaMalloc((void**)p, count * sizeof(T));
        if (err == cudaSuccess) { err = cudaMemset(*p, 0, count * sizeof(T)); t->allocs.push_back((void*)*p); }
    }
};

// launch with programmatic stream serialization: the kernel may be scheduled while its predecessor in the stream drains; every
// kernel launched this way starts with pdl_wait() (gemm_tc.cuh)
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    TACO_LAUNCHED();
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// c: tensor map of the output when the epilogue stores through TMA (p.tma_store is set from it); sk: split-K plan (null: one split)
static int launch_gemm(TacoPPO* t, const CUtensorMap& a, const CUtensorMap& b, GemmParams p, cudaStream_t s, const CUtensorMap* c = nullptr,
                       const SplitK* sk = nullptr) {
    const SplitK plan = sk ? *sk : split_k(1, p.k);
    p.splits = plan.splits; p.kb_per_split = plan.kb_per_split;
    p.stop = t->stop;
    const int total = ((p.m + BM - 1) / BM) * p.splits;
    const int grid = total < t->num_sms ? total : t->num_sms;
    p.tma_store = c != nullptr;
    return launch_pdl(gemm_tc_kernel, dim3(grid), dim3(kGemmThreads), kGemmSmem, s, a, b, c ? *c : a, p) == cudaSuccess ? TACO_OK : fail(TACO_E_CUDA, "gemm_tc_kernel launch failed");
}

// weight gradient dW = dY^T X over K = batch rows, both operands batch-major and read transposed (MN-major): M = out, N = in.  Writes
// the fp32 split-K partials [sk.splits][m][ldc], padding columns included, through the TMA store engine when m is a multiple of 128
// (m_partial is only encoded then)
static int launch_wgrad(TacoPPO* t, const CUtensorMap& dy_mn, const CUtensorMap& x_mn, int m, int n, long long k, float* partial, int ldc,
                        const SplitK& sk, const CUtensorMap& m_partial, cudaStream_t s) {
    GemmParams p{};
    p.m = m; p.n = n; p.k = (int)k; p.n_tile = pad16(n); p.mn_major = 1;
    p.epi = EPI_F32; p.n_valid = ldc; p.out_f32 = partial; p.ldc = ldc; p.split_stride = (long long)m * ldc;
    return launch_gemm(t, dy_mn, x_mn, p, s, m % BM == 0 ? &m_partial : nullptr, &sk);
}

static int splits_for(int m, long long k, int num_sms) {
    const int m_tiles = (m + BM - 1) / BM;
    int s = num_sms / m_tiles;
    const long long kb = (k + BK - 1) / BK;
    if (s > kb) s = (int)kb;
    return s < 1 ? 1 : s;
}

// layer sizes (in -> hidden[0 .. n_hidden) -> out), parameter offsets, buffers and tensor maps of one MLP
static int setup_net(TacoPPO* t, MlpNet& n, int in, const int32_t* hidden, int n_hidden, int out, long long& off) {
    const int B = t->B;
    n.L = n_hidden + 1;
    DevAlloc alloc{t};
    for (int l = 0; l < n.L; ++l) {
        MlpLayer& Ly = n.layer[l];
        Ly.in = l == 0 ? in : hidden[l - 1];
        Ly.out = l + 1 < n.L ? hidden[l] : out;
        Ly.w_off = off; off += (long long)Ly.in * Ly.out;
        Ly.b_off = off; off += Ly.out;
        Ly.ld_w = pad8(Ly.in);
        Ly.ld_t = pad8(Ly.out) < 16 ? 16 : pad8(Ly.out);
        alloc(&Ly.wb, (size_t)pad16(Ly.out) * Ly.ld_w);
        alloc(&Ly.wt, (size_t)pad8(Ly.in) * Ly.ld_t);
        Ly.ld_x = pad8(Ly.in);
        alloc(&Ly.x_bm, (size_t)B * Ly.ld_x);
        if (l > 0) alloc(&Ly.mask, (size_t)((Ly.in + 31) / 32) * B);
        Ly.ld_dz = pad16(Ly.out);
        alloc(&Ly.dz_bm, (size_t)B * Ly.ld_dz);
        Ly.split = split_k(splits_for(Ly.out, B, t->num_sms), B);
        Ly.ld_p = pad16(Ly.in);
        alloc(&Ly.partial, (size_t)Ly.split.splits * Ly.out * Ly.ld_p);
        if (alloc.err != cudaSuccess) return TACO_E_NOMEM;
        bool ok = make_map(&Ly.m_x_bm, Ly.x_bm, B, Ly.in, Ly.ld_x, BM);
        ok = ok && make_map(&Ly.m_x_mn, Ly.x_bm, B, Ly.ld_x, Ly.ld_x, BK);                    // B operand of the dW GEMM (MN-major: 64 x 64 boxes)
        ok = ok && make_map(&Ly.m_w, Ly.wb, Ly.out, Ly.in, Ly.ld_w, pad16(Ly.out));           // B operand of the forward GEMM
        ok = ok && make_map(&Ly.m_wt, Ly.wt, Ly.in, pad8(Ly.out) < 16 ? 16 : Ly.out, Ly.ld_t, pad16(Ly.in));   // B operand of the dX GEMM
        ok = ok && make_map(&Ly.m_dz_bm, Ly.dz_bm, B, Ly.ld_dz, Ly.ld_dz, BM);                // A operand of the dX GEMM
        ok = ok && make_map(&Ly.m_dz_mn, Ly.dz_bm, B, Ly.ld_dz, Ly.ld_dz, BK);                // A operand of the dW GEMM (MN-major)
        if (Ly.out % BM == 0) ok = ok && make_map_f32(&Ly.m_partial, Ly.partial, (long long)Ly.split.splits * Ly.out, Ly.ld_p, Ly.ld_p);
        if (!ok) return fail(TACO_E_CUDA, "cuTensorMapEncodeTiled failed");
    }
    return TACO_OK;
}

extern "C" {

int taco_ppo_create(int device, const TacoPPOCfg* cfg, TacoPPO** out) {
    return taco_ppo_create_layers(device, cfg, 1, out);
}

int taco_ppo_create_layers(int device, const TacoPPOCfg* cfg, int32_t lstm_layers, TacoPPO** out) {
    if (!cfg || !out) return fail(TACO_E_INVALID, "taco_ppo_create: null argument");
    *out = nullptr;
    if (lstm_layers < 1 || lstm_layers > kMaxLstmL) return fail(TACO_E_INVALID, "taco_ppo_create_layers: lstm_layers must be in [1, 4]");
    if (cfg->batch < 128 || cfg->batch % 128) return fail(TACO_E_INVALID, "taco_ppo_create: the minibatch size must be a positive multiple of 128");
    if (cfg->lstm_hidden != kH) return fail(TACO_E_INVALID, "taco_ppo_create: lstm_hidden must be 64");
    if (cfg->act_dim < 1 || cfg->act_dim > 4) return fail(TACO_E_INVALID, "taco_ppo_create: act_dim must be in [1, 4]");
    if (cfg->seq_len < 1 || cfg->seq_len > kSeqMax || cfg->state_dim < 1 || kH + cfg->state_dim + 2 > 128 || cfg->obs_dim < 1 || cfg->obs_dim > 256)
        return fail(TACO_E_INVALID, "taco_ppo_create: seq_len <= 8, state_dim <= 62, obs_dim <= 256");
    if (cfg->n_actor_hidden < 1 || cfg->n_actor_hidden > kMaxHiddenL || cfg->n_critic_hidden < 1 || cfg->n_critic_hidden > kMaxHiddenL)
        return fail(TACO_E_INVALID, "taco_ppo_create: 1..4 hidden layers per MLP");
    for (int l = 0; l < cfg->n_actor_hidden; ++l)
        if (cfg->actor_hidden[l] < 16 || cfg->actor_hidden[l] > 256 || cfg->actor_hidden[l] % 16) return fail(TACO_E_INVALID, "taco_ppo_create: hidden widths must be multiples of 16 in [16, 256]");
    for (int l = 0; l < cfg->n_critic_hidden; ++l)
        if (cfg->critic_hidden[l] < 16 || cfg->critic_hidden[l] > 256 || cfg->critic_hidden[l] % 16) return fail(TACO_E_INVALID, "taco_ppo_create: hidden widths must be multiples of 16 in [16, 256]");
    int ndev = 0;
    TACO_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(TACO_E_INVALID, "taco_ppo_create: no such CUDA device");
    DevGuard guard(device);
    cudaDeviceProp prop;
    TACO_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(TACO_E_INVALID, "taco_ppo_create: the native update needs an sm_100 device (tcgen05); there is no fallback");
    if (!encode_fn()) return fail(TACO_E_CUDA, "taco_ppo_create: cuTensorMapEncodeTiled is not available from the driver");
    TacoPPO* t = new (std::nothrow) TacoPPO();
    if (!t) return fail(TACO_E_NOMEM, "host allocation failed");
    t->device = device; t->cfg = *cfg; t->num_sms = prop.multiProcessorCount;
    t->B = cfg->batch; t->A = cfg->act_dim; t->seq = cfg->seq_len; t->sd = cfg->state_dim; t->n_lstm = lstm_layers;
    const int B = t->B;
    int rc = TACO_OK;
    auto bail = [&](int code, const char* msg) { taco_ppo_destroy(t); return fail(code, msg); };
    // ---- flat parameter layout: log_std | actor MLP (W, b per layer) | LSTM W_ih, W_hh, b_ih, b_hh per layer (bottom first) | critic MLP
    long long off = 0;
    t->off_log_std = off; off += t->A;
    if ((rc = setup_net(t, t->actor, cfg->obs_dim, cfg->actor_hidden, cfg->n_actor_hidden, t->A, off)) != TACO_OK)
        return bail(rc, "taco_ppo_create: actor buffers");
    for (int k = 0; k < t->n_lstm; ++k) {
        LstmLayer& Ly = t->lstm[k];
        Ly.in = k == 0 ? t->sd : kH;
        Ly.ld_u = pad8(kH + Ly.in + 2);
        Ly.t_rows = k == 0 ? kH : 2 * kH;
        Ly.off_wih = off; off += (long long)kG * Ly.in;
        Ly.off_whh = off; off += (long long)kG * kH;
        Ly.off_bih = off; off += kG;
        Ly.off_bhh = off; off += kG;
    }
    if ((rc = setup_net(t, t->critic, kH, cfg->critic_hidden, cfg->n_critic_hidden, 1, off)) != TACO_OK)
        return bail(rc, "taco_ppo_create: critic buffers");
    t->n_params = off;
    DevAlloc alloc{t};
    alloc(&t->prm, (size_t)off);
    alloc(&t->grad, (size_t)off);
    alloc(&t->adam_m, (size_t)off);
    alloc(&t->adam_v, (size_t)off);
    // ---- LSTM buffers
    const long long SB = (long long)t->seq * B;
    for (int k = 0; k < t->n_lstm; ++k) {
        LstmLayer& Ly = t->lstm[k];
        alloc(&Ly.wcat, (size_t)kG * Ly.ld_u);
        alloc(&Ly.wcat_t, (size_t)Ly.t_rows * kG);
        alloc(&Ly.u_bm, (size_t)SB * Ly.ld_u);
        alloc(&Ly.gates, (size_t)SB * kG);
        alloc(&Ly.dg_bm, (size_t)SB * kG);
        alloc(&Ly.c_state, (size_t)SB * kH);
        Ly.split = split_k(splits_for(kG, SB, t->num_sms), SB);
        alloc(&Ly.partial, (size_t)Ly.split.splits * kG * Ly.ld_u);
        if (k > 0) alloc(&Ly.dhx, (size_t)SB * 2 * kH);
        if (k > 0 && alloc.err == cudaSuccess) {
            // the constant-1 columns of U_k (layer 0's come with the gather); the h columns of slot 0 (h_0 = 0) stay as allocated
            const uint32_t ones = 0x3F803F80u;                            // two bf16 1.0
            std::vector<uint32_t> col((size_t)SB, ones);
            alloc.err = cudaMemcpy2D(Ly.u_bm + kH + Ly.in, (size_t)Ly.ld_u * sizeof(bf16), col.data(), sizeof(uint32_t), sizeof(uint32_t), (size_t)SB,
                                     cudaMemcpyHostToDevice);
        }
    }
    alloc(&t->colsum_partial, (size_t)2 * (kMaxHiddenL + 1) * ((B + kColRows - 1) / kColRows) * kColLd);
    alloc(&t->dh, (size_t)B * kH);
    alloc(&t->dc, (size_t)B * kH);
    alloc(&t->mean, (size_t)B * t->A);
    alloc(&t->value, (size_t)B);
    alloc(&t->g_act, (size_t)B * t->A);
    alloc(&t->g_logp, (size_t)B);
    alloc(&t->g_adv, (size_t)B);
    alloc(&t->g_ret, (size_t)B);
    alloc(&t->acc, (size_t)kNumStat);
    alloc(&t->log, (size_t)t->max_log * kLogCols);
    alloc(&t->n_logged, 1);
    alloc(&t->stop, 1);
    alloc(&t->step, 1);
    alloc(&t->spec_sigma, (size_t)(kMaxHiddenL + 1));
    alloc(&t->spec_cold, (size_t)(kMaxHiddenL + 1));
    if (alloc.err == cudaSuccess) alloc.err = cudaMemset(t->spec_cold, 1, (kMaxHiddenL + 1) * sizeof(int));
    for (int l = 0; l < t->actor.L; ++l) alloc(&t->spec_v[l], (size_t)t->actor.layer[l].in);
    if (alloc.err != cudaSuccess)
        return bail(alloc.err == cudaErrorMemoryAllocation ? TACO_E_NOMEM : TACO_E_CUDA, "taco_ppo_create: device allocation failed");
    bool ok = true;
    for (int k = 0; k < t->n_lstm; ++k) {
        LstmLayer& Ly = t->lstm[k];
        ok = ok && make_map(&Ly.m_u_bm, Ly.u_bm, SB, Ly.ld_u, Ly.ld_u, BM);
        ok = ok && make_map(&Ly.m_u_mn, Ly.u_bm, SB, Ly.ld_u, Ly.ld_u, BK);
        ok = ok && make_map(&Ly.m_wcat, Ly.wcat, kG, Ly.ld_u, Ly.ld_u, kG);
        ok = ok && make_map(&Ly.m_wcat_t, Ly.wcat_t, Ly.t_rows, kG, kG, Ly.t_rows);      // B operand of d[h | x] (k >= 1) or dh (k = 0)
        ok = ok && make_map(&Ly.m_dg_bm, Ly.dg_bm, SB, kG, kG, BM);
        ok = ok && make_map(&Ly.m_dg_mn, Ly.dg_bm, SB, kG, kG, BK);
        ok = ok && make_map_f32(&Ly.m_partial, Ly.partial, (long long)Ly.split.splits * kG, Ly.ld_u, Ly.ld_u);
        if (k > 0) {
            ok = ok && make_map(&Ly.m_wih_t, Ly.wcat_t + (size_t)kH * kG, kH, kG, kG, kH);   // W_ih^T alone: the dx-only GEMM of step 0
            for (int s = 0; s < t->seq; ++s) ok = ok && make_map_f32(&Ly.m_dhx[s], Ly.dhx + (size_t)s * B * 2 * kH, B, 2 * kH, 2 * kH);
            ok = ok && make_map_f32(&Ly.m_dx0, Ly.dhx + kH, B, kH, 2 * kH);                  // the x half of slot 0
        }
    }
    ok = ok && make_map_f32(&t->m_dh, t->dh, B, kH, kH);
    if (!ok) return bail(TACO_E_CUDA, "taco_ppo_create: cuTensorMapEncodeTiled failed");
    if (cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGemmSmem) != cudaSuccess)
        return bail(TACO_E_CUDA, "taco_ppo_create: cudaFuncSetAttribute failed");
    if (cudaStreamCreateWithFlags(&t->side, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&t->ev_adam, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&t->ev_actor, cudaEventDisableTiming) != cudaSuccess)
        return bail(TACO_E_CUDA, "taco_ppo_create: stream / event creation failed");
    *out = t;
    return TACO_OK;
}

int taco_ppo_destroy(TacoPPO* t) {
    if (!t) return TACO_OK;
    DevGuard guard(t->device);
    for (void* p : t->allocs) cudaFree(p);
    if (t->side) cudaStreamDestroy(t->side);
    if (t->ev_adam) cudaEventDestroy(t->ev_adam);
    if (t->ev_actor) cudaEventDestroy(t->ev_actor);
    delete t;
    return TACO_OK;
}

int taco_ppo_num_params(TacoPPO* t, int64_t* n) {
    if (!t || !n) return fail(TACO_E_INVALID, "taco_ppo_num_params: null argument");
    *n = t->n_params;
    return TACO_OK;
}

// offsets of the parameter tensors inside the flat vector, in this order: log_std; actor (W, b) x layers; LSTM weight_ih_lk,
// weight_hh_lk, bias_ih_lk, bias_hh_lk for k = 0 .. lstm_layers - 1; critic (W, b) x layers.  `count` = capacity of `offsets`;
// returns the number written.
int taco_ppo_param_offsets(TacoPPO* t, int64_t* offsets, int32_t count, int32_t* n_out) {
    if (!t || !offsets || !n_out) return fail(TACO_E_INVALID, "taco_ppo_param_offsets: null argument");
    std::vector<int64_t> v;
    v.push_back(t->off_log_std);
    for (int l = 0; l < t->actor.L; ++l) { v.push_back(t->actor.layer[l].w_off); v.push_back(t->actor.layer[l].b_off); }
    for (int k = 0; k < t->n_lstm; ++k) {
        const LstmLayer& Ly = t->lstm[k];
        v.push_back(Ly.off_wih); v.push_back(Ly.off_whh); v.push_back(Ly.off_bih); v.push_back(Ly.off_bhh);
    }
    for (int l = 0; l < t->critic.L; ++l) { v.push_back(t->critic.layer[l].w_off); v.push_back(t->critic.layer[l].b_off); }
    if ((int)v.size() > count) return fail(TACO_E_INVALID, "taco_ppo_param_offsets: buffer too small");
    for (size_t i = 0; i < v.size(); ++i) offsets[i] = v[i];
    *n_out = (int32_t)v.size();
    return TACO_OK;
}

// device addresses of the flat fp32 vectors (each n_params floats): parameters, gradient of the last backward, Adam m, Adam v;
// and of the int32 optimiser step counter.  Any pointer may be NULL.
int taco_ppo_buffers(TacoPPO* t, float** params, float** grad, float** adam_m, float** adam_v, int32_t** step) {
    if (!t) return fail(TACO_E_INVALID, "taco_ppo_buffers: null argument");
    if (params) *params = t->prm;
    if (grad) *grad = t->grad;
    if (adam_m) *adam_m = t->adam_m;
    if (adam_v) *adam_v = t->adam_v;
    if (step) *step = t->step;
    return TACO_OK;
}

// the caller's stream waits for the actor's projection / re-pack still running on the side stream
static int join_actor(TacoPPO* t, cudaStream_t s) {
    if (t->actor_pending) {
        TACO_CUDA(cudaStreamWaitEvent(s, t->ev_actor, 0));
        t->actor_pending = false;
    }
    return TACO_OK;
}

// the networks whose bf16 operand copies repack() refreshes; the critic's include its LSTM
enum PackNets { kPackActor = 1, kPackCritic = 2, kPackBoth = kPackActor | kPackCritic };

static int repack(TacoPPO* t, cudaStream_t s, bool honour_stop, PackNets nets) {
    PackParams pp;
    memset(&pp, 0, sizeof(pp));
    auto add = [&](const MlpNet& n) {
        for (int l = 0; l < n.L; ++l) {
            const MlpLayer& Ly = n.layer[l];
            PackSeg& S = pp.seg[pp.n_seg++];
            S.w = t->prm + Ly.w_off; S.out = Ly.out; S.in = Ly.in;
            S.wb = Ly.wb; S.ld_w = Ly.ld_w; S.wt = Ly.wt; S.ld_t = Ly.ld_t; S.rows_t = pad8(Ly.in);
        }
    };
    if (nets & kPackActor) add(t->actor);
    if (nets & kPackCritic) add(t->critic);
    pp.stop = honour_stop ? t->stop : nullptr;
    launch_pdl(pack_kernel, dim3(32, pp.n_seg), dim3(256), 0, s, pp);
    if (nets & kPackCritic) {
        for (int k = 0; k < t->n_lstm; ++k) {
            const LstmLayer& Ly = t->lstm[k];
            launch_pdl(pack_lstm_kernel, dim3(64), dim3(256), 0, s, (const float*)(t->prm + Ly.off_wih), (const float*)(t->prm + Ly.off_whh),
                       (const float*)(t->prm + Ly.off_bih), (const float*)(t->prm + Ly.off_bhh), Ly.in, Ly.ld_u, Ly.wcat, Ly.wcat_t, Ly.t_rows,
                       (const int*)(honour_stop ? t->stop : nullptr));
        }
    }
    return cudaGetLastError() == cudaSuccess ? TACO_OK : fail(TACO_E_CUDA, "pack kernels failed");
}

// call after writing the parameter vector (taco_ppo_buffers) from outside: refreshes the bf16 operand copies, and the next
// projection starts its power iteration over (the stored singular vectors belong to the old weights)
int taco_ppo_params_changed(TacoPPO* t, void* stream) {
    if (!t) return fail(TACO_E_INVALID, "taco_ppo_params_changed: null argument");
    DevGuard guard(t->device);
    const int rcj = join_actor(t, (cudaStream_t)stream);
    if (rcj != TACO_OK) return rcj;
    TACO_CUDA(cudaMemsetAsync(t->spec_cold, 1, (kMaxHiddenL + 1) * sizeof(int), (cudaStream_t)stream));
    return repack(t, (cudaStream_t)stream, false, kPackBoth);
}

// start of one PPO.update: clears the early-stop flag and the log
int taco_ppo_begin_update(TacoPPO* t, void* stream) {
    if (!t) return fail(TACO_E_INVALID, "taco_ppo_begin_update: null argument");
    DevGuard guard(t->device);
    cudaStream_t s = (cudaStream_t)stream;
    TACO_CUDA(cudaMemsetAsync(t->stop, 0, sizeof(int), s));
    TACO_CUDA(cudaMemsetAsync(t->n_logged, 0, sizeof(int), s));
    TACO_CUDA(cudaMemsetAsync(t->acc, 0, kNumStat * sizeof(double), s));
    return TACO_OK;
}

static Hyper to_hyper(const TacoPPOHyper* h) {
    Hyper r;
    r.lr = h->lr; r.clip = h->clip; r.target_kl = h->target_kl; r.max_grad = h->max_grad; r.pi_coef = h->pi_coef; r.vf_coef = h->vf_coef;
    r.ent_coef = h->ent_coef; r.lipschitz = h->lipschitz; r.use_lipschitz = h->use_lipschitz; r.world = h->world < 1 ? 1 : h->world;
    return r;
}

static int mlp_forward(TacoPPO* t, MlpNet& n, bool actor, cudaStream_t s) {
    for (int l = 0; l < n.L; ++l) {
        const MlpLayer& Ly = n.layer[l];
        const MlpLayer* next = l + 1 < n.L ? &n.layer[l + 1] : nullptr;
        GemmParams p{};
        p.m = t->B; p.n = Ly.out; p.k = Ly.in; p.n_tile = pad16(Ly.out);
        p.bias = t->prm + Ly.b_off;
        if (next) {
            p.epi = EPI_BIAS_RELU; p.n_valid = pad8(Ly.out);
            p.mask_out = next->mask; p.ld_mask = t->B;
        } else if (actor) {
            p.epi = EPI_TANH_F32; p.n_valid = t->A; p.out_f32 = t->mean; p.ldc = t->A;
        } else {
            p.epi = EPI_F32; p.n_valid = 1; p.out_f32 = t->value; p.ldc = 1;
        }
        const int rc = launch_gemm(t, Ly.m_x_bm, Ly.m_w, p, s, next ? &next->m_x_bm : nullptr);   // the next layer's X leaves through its own (operand) map
        if (rc != TACO_OK) return rc;
    }
    return TACO_OK;
}

// backward of an MLP whose last layer's dZ (both layouts) is already written.  dx_out != null: also d loss / d input as fp32 [B][in]
// (critic -> LSTM), stored through dx_map when that is not null
static int mlp_backward(TacoPPO* t, MlpNet& n, float* dx_out, const CUtensorMap* dx_map, cudaStream_t s) {
    for (int l = n.L - 1; l >= 0; --l) {
        const MlpLayer& Ly = n.layer[l];
        // dW = dZ^T X: M = out, N = in, K = batch
        int rc = launch_wgrad(t, Ly.m_dz_mn, Ly.m_x_mn, Ly.out, Ly.in, t->B, Ly.partial, Ly.ld_p, Ly.split, Ly.m_partial, s);
        if (rc != TACO_OK) return rc;
        if (l > 0 || dx_out) {   // dX = dZ W, through the ReLU mask of X into the dZ of layer l - 1: M = batch, N = in, K = out
            GemmParams p{};
            p.m = t->B; p.n = Ly.in; p.k = Ly.ld_dz < Ly.ld_t ? Ly.ld_dz : Ly.ld_t; p.n_tile = pad16(Ly.in);
            if (l > 0) {
                p.epi = EPI_RELUBWD; p.n_valid = pad8(Ly.in);
                p.mask_in = Ly.mask; p.ld_mask = t->B;
            } else {
                p.epi = EPI_F32; p.n_valid = Ly.in; p.out_f32 = dx_out; p.ldc = Ly.in;
            }
            rc = launch_gemm(t, Ly.m_dz_bm, Ly.m_wt, p, s, l > 0 ? &n.layer[l - 1].m_dz_bm : dx_map);
            if (rc != TACO_OK) return rc;
        }
    }
    return TACO_OK;
}

// phase 1: gather + forward + loss.  The rollout tensors are flat views [N_total][...] on the device; idx_dev = B int64 row indices.
int taco_ppo_forward_loss(TacoPPO* t, const TacoPPOHyper* hyper, const float* obs, const float* states, const float* act, const float* old_logp,
                          const float* adv, const float* ret, const int64_t* idx_dev, void* stream) {
    if (!t || !hyper || !obs || !states || !act || !old_logp || !adv || !ret || !idx_dev) return fail(TACO_E_INVALID, "taco_ppo_forward_loss: null argument");
    DevGuard guard(t->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int B = t->B;
    GatherParams g;
    memset(&g, 0, sizeof(g));
    g.obs = obs; g.obs_dim = t->cfg.obs_dim; g.states = states; g.seq = t->seq; g.state_dim = t->sd;
    g.act = act; g.logp = old_logp; g.adv = adv; g.ret = ret; g.idx = (const long long*)idx_dev; g.B = B; g.act_dim = t->A;
    g.x0_bm = t->actor.layer[0].x_bm; g.ld_x0 = t->actor.layer[0].ld_x;
    g.u_bm = t->lstm[0].u_bm; g.ld_u = t->lstm[0].ld_u;
    g.g_act = t->g_act; g.g_logp = t->g_logp; g.g_adv = t->g_adv; g.g_ret = t->g_ret; g.stop = t->stop;
    launch_pdl(gather_kernel, dim3((B + 31) / 32), dim3(256), 0, s, g);
    int rc = TACO_OK;
    // critic first: seq LSTM steps per layer, bottom layer first, each one GEMM [h_{t-1} | x_t | 1 1] Wcat^T with the gate math in the
    // epilogue, then its MLP.  A layer below the top also writes h_t into the x columns of the next layer's operand of step t.  The
    // previous optimiser step's projection + re-pack of the ACTOR may still be running on the side stream under these launches.
    for (int l = 0; l < t->n_lstm; ++l) {
        const LstmLayer& Ly = t->lstm[l];
        const LstmLayer* up = l + 1 < t->n_lstm ? &t->lstm[l + 1] : nullptr;
        for (int k = 0; k < t->seq; ++k) {
            GemmParams p{};
            p.m = B; p.n = kG; p.k = Ly.ld_u; p.n_tile = kG; p.a_row0 = k * B; p.epi = EPI_LSTM; p.n_valid = kG;
            p.lstm.c_prev = k > 0 ? Ly.c_state + (size_t)(k - 1) * B * kH : nullptr;
            p.lstm.c_out = Ly.c_state + (size_t)k * B * kH;
            p.lstm.gates_out = Ly.gates + (size_t)k * B * kG;
            bf16* h_up = up ? up->u_bm + (size_t)k * B * up->ld_u + kH : nullptr;      // x columns of U_{l+1}[k]
            if (k + 1 < t->seq) {
                p.lstm.h_bm = Ly.u_bm + (size_t)(k + 1) * B * Ly.ld_u; p.lstm.ld_h_bm = Ly.ld_u;
                if (up) { p.lstm.h2_bm = h_up; p.lstm.ld_h2_bm = up->ld_u; }
            } else if (up) {
                p.lstm.h_bm = h_up; p.lstm.ld_h_bm = up->ld_u;
            } else {
                p.lstm.h_bm = t->critic.layer[0].x_bm; p.lstm.ld_h_bm = t->critic.layer[0].ld_x;
            }
            rc = launch_gemm(t, Ly.m_u_bm, Ly.m_wcat, p, s);
            if (rc != TACO_OK) return rc;
        }
    }
    rc = mlp_forward(t, t->critic, false, s);
    if (rc != TACO_OK) return rc;
    rc = join_actor(t, s);
    if (rc != TACO_OK) return rc;
    rc = mlp_forward(t, t->actor, true, s);
    if (rc != TACO_OK) return rc;
    LossParams L;
    memset(&L, 0, sizeof(L));
    L.mean = t->mean; L.value = t->value; L.act = t->g_act; L.old_logp = t->g_logp; L.adv = t->g_adv; L.ret = t->g_ret;
    L.log_std = t->prm + t->off_log_std; L.B = B; L.act_dim = t->A; L.h = to_hyper(hyper);
    L.dz_bm = t->actor.layer[t->actor.L - 1].dz_bm;
    L.dv_bm = t->critic.layer[t->critic.L - 1].dz_bm;
    L.acc = t->acc; L.stop = t->stop;
    launch_pdl(loss_kernel, dim3((B + 255) / 256), dim3(256), 0, s, L);
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

// device address of the 8 float64 loss accumulators [sum surrogate, sum value, sum kl, -, d log_std x 4]: a data-parallel job
// all-reduces (SUM) them between taco_ppo_forward_loss and taco_ppo_decide and passes world > 1 in the hyper-parameters
int taco_ppo_loss_sums(TacoPPO* t, double** acc_dev) {
    if (!t || !acc_dev) return fail(TACO_E_INVALID, "taco_ppo_loss_sums: null argument");
    *acc_dev = t->acc;
    return TACO_OK;
}

// phase 2: log row + KL early-stop decision (device side)
int taco_ppo_decide(TacoPPO* t, const TacoPPOHyper* hyper, void* stream) {
    if (!t || !hyper) return fail(TACO_E_INVALID, "taco_ppo_decide: null argument");
    DevGuard guard(t->device);
    DecideParams d;
    memset(&d, 0, sizeof(d));
    d.acc = t->acc; d.log = t->log; d.n_logged = t->n_logged; d.stop = t->stop; d.max_log = t->max_log;
    d.log_std = t->prm + t->off_log_std; d.act_dim = t->A; d.B = t->B; d.h = to_hyper(hyper);
    d.grad_log_std = t->grad + t->off_log_std;
    launch_pdl(decide_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, d);
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

// phase 3: backward -> flat gradient (local; a data-parallel job all-reduces (SUM) it before taco_ppo_apply)
int taco_ppo_backward(TacoPPO* t, void* stream) {
    if (!t) return fail(TACO_E_INVALID, "taco_ppo_backward: null argument");
    DevGuard guard(t->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int B = t->B;
    int rc = mlp_backward(t, t->actor, nullptr, nullptr, s);
    if (rc != TACO_OK) return rc;
    rc = mlp_backward(t, t->critic, t->dh, &t->m_dh, s);
    if (rc != TACO_OK) return rc;
    const long long SB = (long long)t->seq * B;
    // LSTM backward through time, top layer first.  Layer 0 back-propagates dh_{t-1} = dgates_t W_hh (N = 64) into t->dh; a layer
    // l >= 1 computes d[h_{t-1} | x_t] = dgates_t [W_hh | W_ih] (N = 128) into its dhx slot t, whose x half the layer below adds to
    // its dh at step t
    for (int l = t->n_lstm - 1; l >= 0; --l) {
        LstmLayer& Ly = t->lstm[l];
        const LstmLayer* up = l + 1 < t->n_lstm ? &t->lstm[l + 1] : nullptr;
        const bool top = up == nullptr;
        for (int k = t->seq - 1; k >= 0; --k) {
            LstmBwdParams b;
            memset(&b, 0, sizeof(b));
            if (l == 0 || k == t->seq - 1) {        // the critic MLP's dh (top layer, last step) or layer 0's recurrence
                b.dh = (k < t->seq - 1 || top) ? t->dh : nullptr; b.ld_dh = kH;
            } else {
                b.dh = Ly.dhx + (size_t)(k + 1) * B * 2 * kH; b.ld_dh = 2 * kH;
            }
            if (up) { b.dh_add = up->dhx + (size_t)k * B * 2 * kH + kH; b.ld_dh_add = 2 * kH; }
            b.dc = t->dc; b.gates = Ly.gates + (size_t)k * B * kG;
            b.c_prev = k > 0 ? Ly.c_state + (size_t)(k - 1) * B * kH : nullptr; b.c_cur = Ly.c_state + (size_t)k * B * kH;
            b.dg_bm = Ly.dg_bm + (size_t)k * B * kG; b.B = B; b.first = (k == t->seq - 1); b.stop = t->stop;
            launch_pdl(lstm_bwd_kernel, dim3((B + 3) / 4), dim3(256), 0, s, b);
            GemmParams p{};
            p.m = B; p.k = kG; p.a_row0 = k * B; p.epi = EPI_F32;
            if (l == 0) {
                if (k == 0) continue;
                // dh_{t-1} = dgates_t W_hh: M = batch, N = 64, K = 256
                p.n = kH; p.n_tile = kH; p.n_valid = kH; p.out_f32 = t->dh; p.ldc = kH;
                rc = launch_gemm(t, Ly.m_dg_bm, Ly.m_wcat_t, p, s, &t->m_dh);
            } else if (k > 0) {
                // d[h_{t-1} | x_t] = dgates_t [W_hh | W_ih]: M = batch, N = 128, K = 256
                p.n = 2 * kH; p.n_tile = 2 * kH; p.n_valid = 2 * kH; p.out_f32 = Ly.dhx + (size_t)k * B * 2 * kH; p.ldc = 2 * kH;
                rc = launch_gemm(t, Ly.m_dg_bm, Ly.m_wcat_t, p, s, &Ly.m_dhx[k]);
            } else {
                // step 0 has no h_{-1} to differentiate: dx_0 = dgates_0 W_ih alone (N = 64)
                p.n = kH; p.n_tile = kH; p.n_valid = kH; p.out_f32 = Ly.dhx + kH; p.ldc = 2 * kH;
                rc = launch_gemm(t, Ly.m_dg_bm, Ly.m_wih_t, p, s, &Ly.m_dx0);
            }
            if (rc != TACO_OK) return rc;
        }
        // dWcat = dgates^T [h | x | 1 1] over all time steps: M = 256, N = ld_u, K = seq * batch
        rc = launch_wgrad(t, Ly.m_dg_mn, Ly.m_u_mn, kG, Ly.ld_u, SB, Ly.partial, Ly.ld_u, Ly.split, Ly.m_partial, s);
        if (rc != TACO_OK) return rc;
    }
    // the flat gradient: weight gradients from the split-K partials, and MLP bias gradients = column sums of the batch-major dZ (partial
    // rows from colsum_kernel, summed by the assembly kernel)
    ColSumParams cs;
    memset(&cs, 0, sizeof(cs));
    GradParams gp;
    memset(&gp, 0, sizeof(gp));
    const int col_chunks = (B + kColRows - 1) / kColRows;
    long long elems = 0;
    auto add = [&](const float* partial, int splits, long long stride, int ld, int col0, int rows, int cols, long long dst) {
        GradSeg& S = gp.seg[gp.n_seg++];
        S.partial = partial; S.splits = splits; S.split_stride = stride; S.ld = ld; S.col0 = col0; S.rows = rows; S.cols = cols; S.dst = dst;
        elems += (long long)rows * cols;
    };
    for (const MlpNet* n : {&t->actor, &t->critic}) {
        for (int l = 0; l < n->L; ++l) {
            const MlpLayer& Ly = n->layer[l];
            const int c = cs.n_seg++;
            cs.seg[c].src = Ly.dz_bm; cs.seg[c].ld = Ly.ld_dz;
            add(Ly.partial, Ly.split.splits, (long long)Ly.out * Ly.ld_p, Ly.ld_p, 0, Ly.out, Ly.in, Ly.w_off);
            add(t->colsum_partial + (long long)c * col_chunks * kColLd, col_chunks, kColLd, kColLd, 0, 1, Ly.out, Ly.b_off);
        }
    }
    for (int l = 0; l < t->n_lstm; ++l) {
        const LstmLayer& Ly = t->lstm[l];
        const int sp = Ly.split.splits;
        const long long stride = (long long)kG * Ly.ld_u;
        add(Ly.partial, sp, stride, Ly.ld_u, 0, kG, kH, Ly.off_whh);
        add(Ly.partial, sp, stride, Ly.ld_u, kH, kG, Ly.in, Ly.off_wih);
        add(Ly.partial, sp, stride, Ly.ld_u, kH + Ly.in, kG, 1, Ly.off_bih);
        add(Ly.partial, sp, stride, Ly.ld_u, kH + Ly.in, kG, 1, Ly.off_bhh);
    }
    cs.B = B; cs.partial = t->colsum_partial; cs.stop = t->stop;
    launch_pdl(colsum_kernel, dim3(col_chunks, cs.n_seg), dim3(256), 0, s, cs);
    gp.grad = t->grad; gp.acc = t->acc; gp.stop = t->stop;
    launch_pdl(grad_assemble_kernel, dim3((unsigned)((elems + 255) / 256)), dim3(256), 0, s, gp);
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}

// phase 4: clip_grad_norm_ + Adam + spectral projection + re-pack of the bf16 operand copies
int taco_ppo_apply(TacoPPO* t, const TacoPPOHyper* hyper, void* stream) {
    if (!t || !hyper) return fail(TACO_E_INVALID, "taco_ppo_apply: null argument");
    DevGuard guard(t->device);
    cudaStream_t s = (cudaStream_t)stream;
    const Hyper h = to_hyper(hyper);
    launch_pdl(grad_norm_kernel, dim3(64), dim3(256), 0, s, (const float*)t->grad, t->n_params, 1.0f / (float)h.world, t->acc, (const int*)t->stop);
    launch_pdl(adam_kernel, dim3(t->num_sms), dim3(256), 0, s, t->prm, t->adam_m, t->adam_v, (const float*)t->grad, t->n_params, h, t->step, t->acc, t->log, (const int*)t->n_logged,
               t->max_log, (const int*)t->stop);
    launch_pdl(finish_step_kernel, dim3(1), dim3(1), 0, s, t->step, t->acc, (const int*)t->stop);
    if (h.use_lipschitz) {
        SpecParams sp;
        memset(&sp, 0, sizeof(sp));
        for (int l = 0; l < t->actor.L; ++l) {
            SpecSeg& S = sp.seg[sp.n_seg++];
            const MlpLayer& Ly = t->actor.layer[l];
            S.w = t->prm + Ly.w_off; S.rows = Ly.out; S.cols = Ly.in; S.v = t->spec_v[l]; S.sigma = t->spec_sigma + l; S.cold = t->spec_cold + l;
        }
        sp.lipschitz = h.lipschitz; sp.stop = t->stop;
        // actor: projection, then the bf16 copies of the projected matrices, on the side stream (4 CTAs of latency-bound power
        // iteration); the caller's stream goes on with the critic's copies and the next minibatch until it needs the actor
        TACO_CUDA(cudaEventRecord(t->ev_adam, s));
        TACO_CUDA(cudaStreamWaitEvent(t->side, t->ev_adam, 0));
        spectral_kernel<<<sp.n_seg, 512, 0, t->side>>>(sp); TACO_LAUNCHED();
        TACO_CUDA(cudaGetLastError());
        int rc = repack(t, t->side, true, kPackActor);
        if (rc != TACO_OK) return rc;
        TACO_CUDA(cudaEventRecord(t->ev_actor, t->side));
        t->actor_pending = true;
        return repack(t, s, true, kPackCritic);
    }
    TACO_CUDA(cudaGetLastError());
    return repack(t, s, true, kPackBoth);
}

// end of an update: synchronises and returns the log rows (n_rows x 8 floats: policy-gradient loss, value loss, entropy loss,
// total loss, approx KL, gradient norm, stopped-here flag, clip coefficient), the number of optimiser steps taken overall and
// whether the KL early stop fired.  log_host may be NULL.
int taco_ppo_end_update(TacoPPO* t, float* log_host, int32_t max_rows, int32_t* n_rows, int32_t* optim_steps, int32_t* early_stop, void* stream) {
    if (!t) return fail(TACO_E_INVALID, "taco_ppo_end_update: null argument");
    DevGuard guard(t->device);
    cudaStream_t s = (cudaStream_t)stream;
    {
        const int rcj = join_actor(t, s);
        if (rcj != TACO_OK) return rcj;
    }
    int h[3] = {0, 0, 0};
    TACO_CUDA(cudaMemcpyAsync(&h[0], t->n_logged, sizeof(int), cudaMemcpyDeviceToHost, s));
    TACO_CUDA(cudaMemcpyAsync(&h[1], t->step, sizeof(int), cudaMemcpyDeviceToHost, s));
    TACO_CUDA(cudaMemcpyAsync(&h[2], t->stop, sizeof(int), cudaMemcpyDeviceToHost, s));
    TACO_CUDA(cudaStreamSynchronize(s));
    int rows = h[0] < t->max_log ? h[0] : t->max_log;
    if (rows > max_rows) rows = max_rows;
    if (log_host && rows > 0) TACO_CUDA(cudaMemcpy(log_host, t->log, (size_t)rows * kLogCols * sizeof(float), cudaMemcpyDeviceToHost));
    if (n_rows) *n_rows = rows;
    if (optim_steps) *optim_steps = h[1];
    if (early_stop) *early_stop = h[2];
    return TACO_OK;
}

// sigma of every actor weight matrix as measured by the last projection (n_actor_layers doubles, host)
int taco_ppo_sigmas(TacoPPO* t, double* out_host) {
    if (!t || !out_host) return fail(TACO_E_INVALID, "taco_ppo_sigmas: null argument");
    DevGuard guard(t->device);
    TACO_CUDA(cudaDeviceSynchronize());
    TACO_CUDA(cudaMemcpy(out_host, t->spec_sigma, (size_t)t->actor.L * sizeof(double), cudaMemcpyDeviceToHost));
    return TACO_OK;
}

// test hook: device addresses of the forward results of the last taco_ppo_forward_loss: action mean (batch, act_dim) and value (batch)
int taco_ppo_debug_outputs(TacoPPO* t, float** mean_dev, float** value_dev) {
    if (!t) return fail(TACO_E_INVALID, "taco_ppo_debug_outputs: null argument");
    if (mean_dev) *mean_dev = t->mean;
    if (value_dev) *value_dev = t->value;
    return TACO_OK;
}

// test hook: D[M][N] (fp32, ld = N) = A[M][K] B[N][K]^T for bf16 row-major device matrices (ld = K, K multiple of 8) through
// gemm_tc_kernel with `splits` split-K partials summed on the host side of the call
static int gemm_selftest_impl(int device, const void* a_bf16, const void* b_bf16, float* d_f32, int32_t m, int32_t n, int32_t k, int32_t splits, bool mn, void* stream) {
    if (!a_bf16 || !b_bf16 || !d_f32 || m < 1 || n < 1 || n > 256 || k < 8 || (k & 7)) return fail(TACO_E_INVALID, "taco_gemm_selftest: bad argument");
    DevGuard guard(device);
    cudaStream_t s = (cudaStream_t)stream;
    if (!encode_fn()) return fail(TACO_E_CUDA, "cuTensorMapEncodeTiled unavailable");
    CUtensorMap ma, mb;
    const bool ok = mn ? make_map(&ma, (const bf16*)a_bf16, k, m, m, BK) && make_map(&mb, (const bf16*)b_bf16, k, n, n, BK)
                       : make_map(&ma, (const bf16*)a_bf16, m, k, k, BM) && make_map(&mb, (const bf16*)b_bf16, n, k, k, pad16(n));
    if (!ok) return fail(TACO_E_CUDA, "tensor map");
    TACO_CUDA(cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGemmSmem));
    const SplitK sk = split_k(splits, k);
    const int sp = sk.splits;
    float* part = nullptr;
    TACO_CUDA(cudaMalloc(&part, (size_t)sp * m * n * sizeof(float)));
    // (compute-sanitizer's initcheck does not observe writes made by cp.async.bulk.tensor stores: without this the partials the
    // TMA-store epilogue writes read as uninitialised in the assembly kernel below)
    TACO_CUDA(cudaMemsetAsync(part, 0, (size_t)sp * m * n * sizeof(float), s));
    GemmParams p{};
    p.m = m; p.n = n; p.k = k; p.n_tile = pad16(n); p.splits = sp; p.kb_per_split = sk.kb_per_split; p.epi = EPI_F32; p.n_valid = n; p.mn_major = mn ? 1 : 0;
    p.out_f32 = part; p.ldc = n; p.split_stride = (long long)m * n;
    cudaDeviceProp prop;
    TACO_CUDA(cudaGetDeviceProperties(&prop, device));
    const int total = ((m + BM - 1) / BM) * sp;
    CUtensorMap mc = ma;
    p.tma_store = (m % BM == 0 && n % 4 == 0) ? 1 : 0;      // exercise the TMA-store epilogue where its shape rule holds
    if (p.tma_store && !make_map_f32(&mc, part, (long long)sp * m, n, n)) return fail(TACO_E_CUDA, "tensor map");
    gemm_tc_kernel<<<total < prop.multiProcessorCount ? total : prop.multiProcessorCount, kGemmThreads, kGemmSmem, s>>>(ma, mb, mc, p); TACO_LAUNCHED();
    GradParams gp;
    memset(&gp, 0, sizeof(gp));
    gp.n_seg = 1;
    gp.seg[0].partial = part; gp.seg[0].splits = sp; gp.seg[0].split_stride = (long long)m * n; gp.seg[0].ld = n; gp.seg[0].rows = m; gp.seg[0].cols = n;
    gp.grad = d_f32;
    grad_assemble_kernel<<<(unsigned)(((long long)m * n + 255) / 256), 256, 0, s>>>(gp); TACO_LAUNCHED();
    const cudaError_t e = cudaStreamSynchronize(s);
    cudaFree(part);
    if (e != cudaSuccess) return fail(TACO_E_CUDA, std::string("taco_gemm_selftest: ") + cudaGetErrorString(e));
    return TACO_OK;
}

// D[m][n] = A[m][k] B[n][k]^T with both operands K-major (k contiguous)
int taco_gemm_selftest(int device, const void* a_bf16, const void* b_bf16, float* d_f32, int32_t m, int32_t n, int32_t k, int32_t splits, void* stream) {
    return gemm_selftest_impl(device, a_bf16, b_bf16, d_f32, m, n, k, splits, false, stream);
}
// the same product from TRANSPOSED operands: at[k][m], bt[k][n] (m, n multiples of 8)
int taco_gemm_selftest_mn(int device, const void* at_bf16, const void* bt_bf16, float* d_f32, int32_t m, int32_t n, int32_t k, int32_t splits, void* stream) {
    if ((m & 7) || (n & 7)) return fail(TACO_E_INVALID, "taco_gemm_selftest_mn: m and n must be multiples of 8");
    return gemm_selftest_impl(device, at_bf16, bt_bf16, d_f32, m, n, k, splits, true, stream);
}

}  // extern "C"
