// What the actor and the critic (taco_actor.cu / actor_tc.cuh, taco_critic.cu / critic_tc.cuh) share: the tile, weight-ring
// and TMEM geometry of their tcgen05 kernels, the MLP weight-image format and its packer, and the host code that sets these up.
#pragma once
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "host_common.h"
#include "launch_count.h"
#include "tc_ptx.cuh"

namespace taco {
namespace mlp {

constexpr int kTileM = 128;                    // envs per tile = TMEM lanes
constexpr int kKC = 64;                        // bf16 per K chunk: one 128-byte swizzle row
constexpr int kMaxN = 256;                     // widest hidden layer
constexpr int kPartN = 128;                    // rows of W per stage = columns of D per part
constexpr int kSlots = 3;                      // weight ring: slots of one part (all K chunks)
constexpr int kChunkBytes = kPartN * 128;      // 16 KB: 128 rows x 64 bf16
constexpr int kSlotBytes = kChunkBytes * (kMaxN / kKC);   // 64 KB
constexpr int kMaxHidden = 4;
constexpr int kOutPad = 4;                     // num_acts = 4
constexpr int kOutN = 16;                      // output layer as an MMA part: N padded to the instruction minimum
constexpr int kEpiWarps = 16;
constexpr int kTcThreads = (2 + kEpiWarps) * 32;   // 576
constexpr int kTmemCols = 512;
constexpr int kTmemSlot = 256;                 // columns per tile slot: A (128, packed bf16 pairs) + D (128, fp32)
constexpr int kTmemD = 128;                    // offset of D inside a slot
constexpr int kFpEnvs = 32;                    // envs per CTA of the FP32 kernels (one warp lane per env)
constexpr int kFpThreads = 128;
constexpr int kFpTile = 8;                     // output neurons per warp pass of an FP32 kernel's MLP layer

struct TcLayer {
    int n;               // output width of the layer (multiple of 64, <= 256)
    int kchunks;         // ceil(K / 64)
    uint32_t img_off;    // byte offset of the layer's first chunk image; chunk c is at img_off + c * n * 128
};

// optional timeline of CTA 0 (TACO_ACTOR_TIMELINE / TACO_CRITIC_TIMELINE=<file>, see timeline_begin): 3 regions of kDbgCap
// (clock << 8 | code) words in p.dbg
constexpr int kDbgCap = 4096;
#define TACO_DBG(region, cnt, code)                                                                         \
    do {                                                                                                    \
        if (p.dbg && blockIdx.x == 0 && (cnt) < kDbgCap)                                                    \
            p.dbg[(region) * kDbgCap + (cnt)++] = ((unsigned long long)clock64() << 8) | (unsigned)(code);  \
    } while (0)

constexpr int kSmemBias = kMaxHidden * kMaxN * 4;          // 4 KB
constexpr int kTcSmemBytes = 1024 /*alignment slack*/ + kSlots * kSlotBytes + kSmemBias + 256;

// relu(D + bias) of 32 accumulator columns -> 16 packed bf16 pairs (column 2j in the low half)
__device__ __forceinline__ void relu_pack32(const uint32_t (&v)[32], const float* bias, uint32_t* pk) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 b = *reinterpret_cast<const float4*>(bias + q * 4);
        pk[q * 2 + 0] = pack_bf16x2(fmaxf(__uint_as_float(v[q * 4 + 0]) + b.x, 0.0f), fmaxf(__uint_as_float(v[q * 4 + 1]) + b.y, 0.0f));
        pk[q * 2 + 1] = pack_bf16x2(fmaxf(__uint_as_float(v[q * 4 + 2]) + b.z, 0.0f), fmaxf(__uint_as_float(v[q * 4 + 3]) + b.w, 0.0f));
    }
}

// fp32 (out, in) row-major weights -> bf16 K-chunk images in the SWIZZLE_128B K-major layout the kernel copies verbatim:
// chunk c holds W[:, 64c .. 64c+63] as n rows of 128 bytes (rows >= n_real are zero); the 16-byte piece q of row r sits
// at r*128 + ((q ^ (r&7)) << 4).
static __global__ void pack_weights_kernel(const float* __restrict__ w, int n_real, int n, int k, uint8_t* __restrict__ img) {
    const int kchunks = (k + kKC - 1) / kKC;
    const int total = kchunks * n * 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int q = i & 7, r = (i >> 3) % n, c = (i >> 3) / n;
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int kk = c * kKC + q * 8 + j;
            f[j] = (kk < k && r < n_real) ? w[(size_t)r * k + kk] : 0.0f;
        }
        const uint4 pk = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
        *reinterpret_cast<uint4*>(img + (size_t)c * n * 128 + sw128_off(r, q)) = pk;
    }
}

// ---------------------------------------------------------------------------------------------- host side
// fp32 weights of an MLP as nn.Linear holds them: layer l = a (sizes[l + 1], sizes[l]) row-major weight and a bias, each starting
// on a 16-byte boundary (the FP32 kernels read weight rows as float4)
struct MlpF32 {
    std::vector<size_t> w_off, b_off;    // float offsets into w / b
    float* w = nullptr;
    float* b = nullptr;
};
static inline cudaError_t mlp_f32_alloc(MlpF32& m, const int* sizes, int n_layers) {
    size_t wo = 0, bo = 0;
    for (int l = 0; l < n_layers; ++l) {
        m.w_off.push_back(wo); m.b_off.push_back(bo);
        wo += ((size_t)sizes[l] * sizes[l + 1] + 3) & ~(size_t)3;
        bo += (size_t)((sizes[l + 1] + 3) & ~3);
    }
    cudaError_t ce = cudaMalloc(&m.w, wo * sizeof(float));
    if (ce == cudaSuccess) ce = cudaMalloc(&m.b, bo * sizeof(float));
    return ce;
}
// w_host[l] / b_host[l]: host or device pointers, copied on stream s
static inline int mlp_f32_upload(const MlpF32& m, const float* const* w_host, const float* const* b_host, const int* sizes, int n_layers,
                                 cudaStream_t s) {
    for (int l = 0; l < n_layers; ++l) {
        const int in = sizes[l], out = sizes[l + 1];
        TACO_CUDA(cudaMemcpyAsync(m.w + m.w_off[l], w_host[l], (size_t)in * out * sizeof(float), cudaMemcpyDefault, s));
        TACO_CUDA(cudaMemcpyAsync(m.b + m.b_off[l], b_host[l], (size_t)out * sizeof(float), cudaMemcpyDefault, s));
    }
    return TACO_OK;
}
static inline void mlp_f32_free(MlpF32& m) { cudaFree(m.w); cudaFree(m.b); }

// The tensor-core kernels' copy of an MLP [in, h1, ..., hL, out]: the bf16 K-chunk images of its layers back to back in wimg (the
// output layer as a kOutN-row part), the hidden biases as rows of a [kMaxHidden][kMaxN] block, the output bias padded to kOutPad.
// MLP layer l is layer[first + l] and its bias row first + l; the slots before `first` (and the image bytes before the MLP's)
// belong to the caller: the critic's LSTM step and its unused bias row 0.
struct TcImage {
    uint8_t* wimg = nullptr;
    float* bias = nullptr;               // [kMaxHidden][kMaxN]; cleared on the stream by the caller before tc_image_pack
    float* b_out = nullptr;              // [kOutPad]
    TcLayer layer[kMaxHidden + 1];
    int first = 0;
};
// the layout of an MLP with n_hidden hidden layers behind `lead` bytes of the caller's images, and the device buffers
static inline cudaError_t tc_image_alloc(TcImage& t, const int* sizes, int n_hidden, int first, size_t lead) {
    t.first = first;
    size_t img = lead;
    for (int l = 0; l <= n_hidden; ++l) {
        const int k = sizes[l], nn = l < n_hidden ? sizes[l + 1] : kOutN;
        const int kch = (k + kKC - 1) / kKC;
        TcLayer& L = t.layer[first + l];
        L.n = nn; L.kchunks = kch; L.img_off = (uint32_t)img;
        img += (size_t)kch * nn * 128;
    }
    cudaError_t ce = cudaMalloc(&t.wimg, img);
    if (ce == cudaSuccess) ce = cudaMalloc(&t.bias, kMaxHidden * kMaxN * sizeof(float));
    if (ce == cudaSuccess) ce = cudaMalloc(&t.b_out, kOutPad * sizeof(float));
    return ce;
}
// packs the fp32 weights into the images and copies the biases, on stream s
static inline int tc_image_pack(const TcImage& t, const MlpF32& m, const int* sizes, int n_hidden, cudaStream_t s) {
    for (int l = 0; l <= n_hidden; ++l) {
        const int in = sizes[l], out = sizes[l + 1];
        const TcLayer& L = t.layer[t.first + l];
        pack_weights_kernel<<<64, 256, 0, s>>>(m.w + m.w_off[l], out, L.n, in, t.wimg + L.img_off); TACO_LAUNCHED();
        if (l < n_hidden)
            TACO_CUDA(cudaMemcpyAsync(t.bias + (size_t)(t.first + l) * kMaxN, m.b + m.b_off[l], (size_t)out * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    TACO_CUDA(cudaMemsetAsync(t.b_out, 0, kOutPad * sizeof(float), s));
    TACO_CUDA(cudaMemcpyAsync(t.b_out, m.b + m.b_off[n_hidden], (size_t)sizes[n_hidden + 1] * sizeof(float), cudaMemcpyDeviceToDevice, s));
    TACO_CUDA(cudaGetLastError());
    return TACO_OK;
}
static inline void tc_image_free(TcImage& t) { cudaFree(t.wimg); cudaFree(t.bias); cudaFree(t.b_out); }

// hidden widths sizes[1 .. n_hidden] the tensor-core kernels take: whole 64-wide K chunks, at most one 256-column accumulator
static inline bool tc_hidden_widths_ok(const int* sizes, int n_hidden) {
    for (int l = 1; l <= n_hidden; ++l)
        if (sizes[l] % 64 != 0 || sizes[l] > kMaxN) return false;
    return true;
}

// CTAs of a tensor-core launch over num_tiles tiles; *tiles_per_cta = 2 (a CTA keeps a pair of tiles in flight) unless every tile
// can have its own SM (small batches: one tile per CTA halves the latency)
static inline int tc_grid(int num_tiles, int num_sms, int* tiles_per_cta) {
    *tiles_per_cta = num_tiles <= num_sms ? 1 : 2;
    const int num_pairs = (num_tiles + *tiles_per_cta - 1) / *tiles_per_cta;
    return num_pairs < num_sms ? num_pairs : num_sms;
}

// Developer aid: with `path` (TACO_ACTOR_TIMELINE / TACO_CRITIC_TIMELINE) set, the launch between timeline_begin and timeline_end
// records clock64 stamps of CTA 0's MMA issuer and epilogue into *dbg (TACO_DBG; tools/actor_timeline.py decodes them) and
// timeline_end writes them to that file.  Synchronous.
static inline int timeline_begin(const char* path, unsigned long long** dbg, cudaStream_t s) {
    if (path && *path) {
        TACO_CUDA(cudaMalloc(dbg, 3 * kDbgCap * sizeof(unsigned long long)));
        TACO_CUDA(cudaMemsetAsync(*dbg, 0, 3 * kDbgCap * sizeof(unsigned long long), s));
    }
    return TACO_OK;
}
static inline int timeline_end(const char* path, unsigned long long* dbg, cudaStream_t s) {
    if (dbg) {
        std::vector<unsigned long long> h(3 * kDbgCap);
        TACO_CUDA(cudaStreamSynchronize(s));
        TACO_CUDA(cudaMemcpy(h.data(), dbg, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        cudaFree(dbg);
        if (FILE* f = fopen(path, "wb")) { fwrite(h.data(), sizeof(unsigned long long), h.size(), f); fclose(f); }
    }
    return TACO_OK;
}

}  // namespace mlp
}  // namespace taco
