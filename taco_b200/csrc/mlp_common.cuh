// What the actor and the critic (taco_actor.cu / actor_tc.cuh, taco_critic.cu / critic_tc.cuh) share: the tile, weight-ring
// and TMEM geometry of their tcgen05 kernels and the pipeline both kernels run, the MLP weight-image format and its packer, and
// the host code that sets these up.
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
// (clock << 8 | code) words in dbg; TACO_DBG writes to the kernel's p.dbg
constexpr int kDbgCap = 4096;
#define TACO_DBG_AT(dbg, region, cnt, code)                                                                 \
    do {                                                                                                    \
        if ((dbg) && blockIdx.x == 0 && (cnt) < kDbgCap)                                                    \
            (dbg)[(region) * kDbgCap + (cnt)++] = ((unsigned long long)clock64() << 8) | (unsigned)(code);  \
    } while (0)
#define TACO_DBG(region, cnt, code) TACO_DBG_AT(p.dbg, region, cnt, code)

constexpr int kSmemBias = kMaxHidden * kMaxN * 4;          // 4 KB
constexpr int kTcSmemBytes = 1024 /*alignment slack*/ + kSlots * kSlotBytes + kSmemBias + 256;

// ---------------------------------------------------------------------------------------------- the tcgen05 MLP pipeline
// One persistent CTA per SM keeps two 128-env tiles in flight.  Warp 0 streams the weights through a ring of 64 KB slots in shared
// memory, one 128-row part of a layer per slot; warp 1 issues the MMAs of every part for both tiles and releases the slot after the
// last tile's; the 16 epilogue warps drain D(t) and write the next layer's A(t) in tensor memory.  Producer and issuer are
// warp-uniform loops with one elected lane issuing, so that every descriptor stays in uniform registers (issuing from inside
// `if (lane == 0)` halved the MMA issue rate).  The kernels keep the slot and phase counters in their own loops.

// Shared memory from its 1024-byte aligned base (SWIZZLE_128B atoms need that alignment): the weight ring, the bias block, the
// barriers, the TMEM address word, then the kernel's own barriers from bar_own on.  The kernel's own buffers start at
// base + kTcSmemBytes - 1024.
struct TcSmem {
    uint8_t* base;
    uint32_t ring;        // kSlots x 64 KB weight ring
    float* bias;          // [kMaxHidden][kMaxN]
    uint32_t bar_full;    // [kSlots] producer -> MMA
    uint32_t bar_empty;   // [kSlots] MMA -> producer
    uint32_t bar_a;       // [2] epilogue(t) -> MMA: D(t) drained (and, for a new layer, A(t) written)
    uint32_t bar_d;       // [2] MMA -> epilogue(t): the part of D(t) is complete
    uint32_t* tmem;       // written by tcgen05.alloc
    uint32_t bar_own;

    __device__ __forceinline__ explicit TcSmem(uint8_t* smem_raw) {
        const uint32_t raw = smem_u32(smem_raw);
        const uint32_t aligned = (raw + 1023u) & ~1023u;
        base = smem_raw + (aligned - raw);
        ring = aligned;
        bias = reinterpret_cast<float*>(base + kSlots * kSlotBytes);
        uint64_t* bars = reinterpret_cast<uint64_t*>(bias + kMaxHidden * kMaxN);
        bar_full = smem_u32(bars);
        bar_empty = bar_full + 8 * kSlots;
        bar_a = bar_empty + 8 * kSlots;
        bar_d = bar_a + 16;
        tmem = reinterpret_cast<uint32_t*>(bars + 2 * kSlots + 4);
        bar_own = bar_d + 16 + 8;
    }

    // copies the biases, initialises the barriers (own_init() adds the kernel's own, on the same thread before the init fence) and
    // allocates all of tensor memory; returns its base address
    template <class OwnInit>
    __device__ __forceinline__ uint32_t setup(int warp, const float* bias_src, OwnInit own_init) const {
        for (int i = threadIdx.x; i < kMaxHidden * kMaxN; i += kTcThreads) bias[i] = bias_src[i];
        if (threadIdx.x == 0) {
            for (int s = 0; s < kSlots; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
            for (int t = 0; t < 2; ++t) { mbar_init(bar_a + 8 * t, (kEpiWarps / 2) * 32); mbar_init(bar_d + 8 * t, 1); }
            own_init();
            fence_barrier_init();
        }
        if (warp == 1) tmem_alloc(smem_u32(tmem), kTmemCols);
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        return *tmem;
    }

    __device__ __forceinline__ void teardown(int warp, uint32_t tmem0) const {
        tc_fence_before();
        __syncthreads();
        if (warp == 1) {
            tc_fence_after();
            tmem_dealloc(tmem0, kTmemCols);
        }
    }
};

// producer: every 128-row part of layer L, all its K chunks, into the next slot of a ring of ring_slots slots once the MMAs have
// released that slot
__device__ __forceinline__ void produce_layer(const TcSmem& s, const uint8_t* wimg, const TcLayer& L, int ring_slots, uint32_t& slot,
                                              uint32_t& phase) {
    const int n = L.n, kch = L.kchunks;
    const uint8_t* img = wimg + L.img_off;
    for (int h0 = 0; h0 < n; h0 += kPartN) {
        const uint32_t bytes = (uint32_t)min(kPartN, n - h0) * 128u;
        mbar_wait(s.bar_empty + 8 * slot, phase ^ 1u);
        if (elect_one_sync()) {
            mbar_arrive_expect_tx(s.bar_full + 8 * slot, bytes * (uint32_t)kch);
            for (int c = 0; c < kch; ++c)
                bulk_g2s(s.ring + slot * kSlotBytes + c * kChunkBytes, img + ((size_t)c * n + h0) * 128u, bytes, s.bar_full + 8 * slot);
        }
        __syncwarp();
        if (++slot == ring_slots) { slot = 0; phase ^= 1u; }
    }
}

// issuer: the MMAs of one part for one tile, D = A * B^T over kch K chunks of 64 (A at a_addr, D next to it), then a commit to
// bar_free if `release` (the ring slot may be refilled once the last tile's MMAs have read it) and to bar_done.  lstm: an LSTM step,
// whose second chunk (x_t: 26 features, 2 bias columns, padding) holds only 32 K values.
__device__ __forceinline__ void issue_part(uint32_t a_addr, uint64_t bdesc, uint32_t idesc, int kch, bool lstm, bool release,
                                           uint32_t bar_free, uint32_t bar_done) {
    if (elect_one_sync()) {
        const uint32_t d_addr = a_addr + (uint32_t)kTmemD;
        for (int c = 0; c < kch; ++c) {
            const uint64_t b_c = bdesc + (uint64_t)(c * (kChunkBytes >> 4));
            const uint32_t a_c = a_addr + (uint32_t)(c * (kKC / 2));
            // 16 bf16 along K = 8 packed TMEM columns of A = 32 bytes inside the B swizzle atom
            umma_bf16_ts(d_addr, a_c, b_c, idesc, (uint32_t)(c != 0));
            umma_bf16_ts(d_addr, a_c + 8u, b_c + 2u, idesc, 1u);
            if (!lstm || c == 0) {
                umma_bf16_ts(d_addr, a_c + 16u, b_c + 4u, idesc, 1u);
                umma_bf16_ts(d_addr, a_c + 24u, b_c + 6u, idesc, 1u);
            }
        }
        if (release) umma_commit(bar_free);
        umma_commit(bar_done);
    }
    __syncwarp();
}

// An epilogue thread (warps 2..17): tile slot t, 64-column half ch of a part, TMEM lane quadrant quad (a warp may only touch TMEM
// lanes 32 (warp % 4) .. + 31); thread <-> TMEM lane <-> env row r of the tile.  t_a / t_d: the thread's lane of A(t) and of its half
// of D(t).  `tile` is the slot's first tile (num_tiles: slot 1 idles with one tile per CTA), tile_step the stride to its next.
struct EpiThread {
    int e, t, ch, quad, r;
    uint32_t t_a, t_d;
    int tile, tile_step;

    __device__ __forceinline__ EpiThread(int warp, int lane, uint32_t tmem0, int tps, int num_tiles) {
        e = warp - 2;
        t = e >> 3; ch = (e >> 2) & 1; quad = warp & 3;
        r = (quad << 5) | lane;
        t_a = tmem0 + ((uint32_t)(quad << 5) << 16) + (uint32_t)(t * kTmemSlot);
        t_d = t_a + (uint32_t)kTmemD + (uint32_t)(ch * 64);
        tile = t < tps ? tps * (int)blockIdx.x + t : num_tiles;
        tile_step = tps * (int)gridDim.x;
    }
};

// relu(D + bias) of 32 accumulator columns -> 16 packed bf16 pairs (column 2j in the low half)
__device__ __forceinline__ void relu_pack32(const uint32_t (&v)[32], const float* bias, uint32_t* pk) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 b = *reinterpret_cast<const float4*>(bias + q * 4);
        pk[q * 2 + 0] = pack_bf16x2(fmaxf(__uint_as_float(v[q * 4 + 0]) + b.x, 0.0f), fmaxf(__uint_as_float(v[q * 4 + 1]) + b.y, 0.0f));
        pk[q * 2 + 1] = pack_bf16x2(fmaxf(__uint_as_float(v[q * 4 + 2]) + b.z, 0.0f), fmaxf(__uint_as_float(v[q * 4 + 3]) + b.w, 0.0f));
    }
}

// Epilogue of hidden layer l (width n, bias row l of the bias block) on tile slot ep.t: relu(D + bias) as bf16 pairs, held in
// registers until every MMA of the layer has read A(t), then written over A(t) as the next layer's operand (feature k -> packed
// column k / 2).  With two parts, D is released as soon as part 0 is in registers, so part 1's MMAs overlap the rest of the drain.
// bar_a / bar_d: the [2] barrier arrays of TcSmem.  kMark: timeline markers 0x02..0x05 in region 1 + t of dbg.
template <bool kMark>
__device__ __forceinline__ void hidden_layer(const EpiThread& ep, const float* bias, int l, int n, uint32_t bar_a, uint32_t bar_d, uint32_t& d_phase,
                                             unsigned long long* dbg, int& dbg_n) {
    const int ch = ep.ch, t = ep.t;
    const uint32_t t_a = ep.t_a, t_d = ep.t_d;
    const float* bl = bias + l * kMaxN;
    const bool two_parts = n > kPartN;
    uint32_t pk0[32];
    const bool mine0 = ch * 64 < min(n, kPartN);                 // this warp has columns in part 0
    const bool mine1 = two_parts && (kPartN + ch * 64 < n);      // ... in part 1
    mbar_wait(bar_d + 8 * t, d_phase); d_phase ^= 1u;
    tc_fence_after();
    if (kMark) TACO_DBG_AT(dbg, 1 + t, dbg_n, 0x02);
    if (mine0) {
        uint32_t v[32];
        tmem_ld32(t_d, v); tmem_ld_wait();
        relu_pack32(v, bl + ch * 64, pk0);
        tmem_ld32(t_d + 32u, v); tmem_ld_wait();
        if (two_parts) { tc_fence_before(); mbar_arrive(bar_a + 8 * t); if (kMark) TACO_DBG_AT(dbg, 1 + t, dbg_n, 0x03); }
        relu_pack32(v, bl + ch * 64 + 32, pk0 + 16);
    } else if (two_parts) { tc_fence_before(); mbar_arrive(bar_a + 8 * t); }
    if (two_parts) {
        mbar_wait(bar_d + 8 * t, d_phase); d_phase ^= 1u;
        tc_fence_after();
        if (kMark) TACO_DBG_AT(dbg, 1 + t, dbg_n, 0x04);
    }
    if (mine0) { tmem_st16(t_a + (uint32_t)(ch * 32), pk0); tmem_st16(t_a + (uint32_t)(ch * 32 + 16), pk0 + 16); }
    if (mine1) {
        uint32_t v[32], pk1[16];
        tmem_ld32(t_d, v); tmem_ld_wait();
        relu_pack32(v, bl + kPartN + ch * 64, pk1);
        tmem_st16(t_a + (uint32_t)(64 + ch * 32), pk1);
        tmem_ld32(t_d + 32u, v); tmem_ld_wait();
        relu_pack32(v, bl + kPartN + ch * 64 + 32, pk1);
        tmem_st16(t_a + (uint32_t)(64 + ch * 32 + 16), pk1);
    }
    tmem_st_wait();
    tc_fence_before();
    mbar_arrive(bar_a + 8 * t);
    if (kMark) TACO_DBG_AT(dbg, 1 + t, dbg_n, 0x05);
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
// belong to the caller: the critic's LSTM step and bias row 0 (the gate biases of a stacked critic's top layer, unused otherwise).
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
