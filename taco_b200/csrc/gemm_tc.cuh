// General tcgen05 GEMM of the native PPO update (taco_ppo.cu):  D[M, N] = A[M, K] * B[N, K]^T, bf16 operands, fp32 accumulation
// in tensor memory.  Operands reach shared memory through TMA tensor maps (cp.async.bulk.tensor.2d, SWIZZLE_128B, out-of-bounds
// boxes zero-filled, so ragged M / N / K need no padding code) in one of two forms:
//   K-major    A as [M][K], B as [N][K] row-major (K contiguous): forward and dX GEMMs (K = features)
//   MN-major   A as [K][M], B as [K][N] row-major (M / N contiguous): the weight-gradient GEMMs dW = dZ^T X (K = batch) read the
//              batch-major gradients and activations exactly as the other GEMMs wrote them -- no transposed copies anywhere
//
//   tile       128 (M) x n_tile (N <= 256, multiple of 16) per work item; K in blocks of 64, 16 per MMA
//   work item  (m_tile, k_split): split-K gives the K = batch GEMMs of the weight gradients (2 output tiles) enough CTAs; every
//              split writes its own fp32 partial, which the assembly kernel sums in a fixed order (bit-reproducible)
//   pipeline   persistent CTAs; warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warps 2..9 = epilogue (two per
//              TMEM lane quarter, alternating 32-column chunks: the epilogue is latency-bound, so two warps per scheduler);
//              3 smem stages (full / empty mbarriers), 2 accumulators of 256 TMEM columns (tmem_full / tmem_empty), so the
//              epilogue of one work item overlaps the MMAs of the next
//   epilogues  EPI_F32            out_f32[split][m][n] = acc (+ bias[n])
//              EPI_BIAS_RELU      y = relu(acc + bias[n]) as bf16 [m][n]; one 32-bit word per (row, 32-column chunk) records which
//                                 pre-activations were > 0
//              EPI_RELUBWD        g = acc * (pre-activation > 0) as bf16 [m][n] (the ReLU backward of the layer below), from those
//                                 mask words
//              EPI_TANH_F32       out_f32[m][n] = tanh(acc + bias[n])     (actor mean, nets_asymmetry.py:32-39)
//              EPI_LSTM           one LSTM time step from the gate pre-activations (nets_asymmetry.py:128-136), see LstmEpi
// A thread of an epilogue warp owns one accumulator row (= TMEM lane), so anything it reads or writes in a row-major tensor
// directly costs one cache line per lane and instruction: the LSU, not DRAM, then bounds the kernel (measured: ~2.4 cycles per
// line and SM).  Outputs therefore leave through a shared-memory staging tile of 128 rows x 128 bytes in the SWIZZLE_128B
// pattern: a thread writes its row with conflict-free 16-byte stores and one elected thread hands the tile to the TMA store
// engine (cp.async.bulk.tensor, clipped at the tensor's edges), which keeps the copy-out off the LSU altogether.  Row-major
// INPUTS of the LSTM step cross with lanes along the row's bytes; the ReLU mask is one word per lane, lanes along the rows.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "tc_ptx.cuh"

namespace taco {
namespace gemm {

constexpr int BM = 128, BK = 64;
constexpr int kStages = 3;
constexpr int kGemmThreads = 320;           // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (2 column halves x 4 TMEM lane quarters)
constexpr int kStageA = BM * BK * 2;          // 16 KB
constexpr int kStageB = 256 * BK * 2;         // 32 KB (n_tile <= 256)
constexpr int kStageBm = BM * 128;            // epilogue staging tile: 128 rows x up to 128 bytes, 16-byte pieces XOR-swizzled
constexpr int kGemmSmem = 1024 + kStages * (kStageA + kStageB) + 256 + 1024 + 2 * 2 * kStageBm;
constexpr int kAccCols = 256;

enum : int { EPI_F32 = 0, EPI_BIAS_RELU = 1, EPI_RELUBWD = 2, EPI_TANH_F32 = 3, EPI_LSTM = 4 };

struct LstmEpi {
    // gates = [i | f | g | o] pre-activations of H = 64 units each (torch nn.LSTM row blocks), bias already inside the GEMM
    const float* c_prev;              // [m][64] fp32 (null: zero)
    float* c_out;                     // [m][64] fp32
    __nv_bfloat16* gates_out;         // [m][4 chunks][4 gates][16 units] bf16: sigmoid(i), sigmoid(f), tanh(g), sigmoid(o) of units 16 c .. 16 c + 15
                                      // (saved for the backward pass; a chunk's 128 bytes are what one epilogue round produces per row)
    __nv_bfloat16* h_bm;              // destination of h: row stride ld_h_bm elements (the next step's operand [h | x | 1 1])
    long long ld_h_bm;
    __nv_bfloat16* h2_bm;             // second destination of h (null: none): the x columns of the next LSTM layer's operand
    long long ld_h2_bm;
};

struct GemmParams {
    int m, n, k;                      // rows of A, rows of B, depth
    int n_tile;                       // UMMA N: multiple of 16, >= n, <= 256
    int splits, kb_per_split;         // split-K: work item (m_tile, split) covers k blocks [split * kb_per_split, ...)
    int a_row0, b_row0;               // row offsets into the tensor maps (views of larger buffers)
    int mn_major;                     // 1: both operands are stored TRANSPOSED, A as [K][M] and B as [K][N] (M / N contiguous): the K = batch
                                      // GEMMs of the weight gradients read the batch-major activations and gradients as they are.  The
                                      // tensor maps then have 64 x 64 boxes (64 M- or N-elements x 64 k-rows, one 8 KB SWIZZLE_128B block
                                      // per 64 columns) and the MMAs use MN-major shared-memory descriptors
    int epi;
    int n_valid;                      // columns written by the epilogue (<= n_tile)
    float* out_f32; long long ldc, split_stride;
    int tma_store;                    // the output leaves through the third tensor map (tmC): bf16 [m][n] (EPI_BIAS_RELU / EPI_RELUBWD, boxes of
                                      // 64 columns x 128 rows) or, with EPI_F32, fp32 [splits * m][n] (32 columns x 128 rows; needs m % 128 == 0)
    const float* bias;
    const uint32_t* mask_in;          // EPI_RELUBWD: [ceil(n / 32)][ld_mask] words, bit j of word (c, m) = pre-activation (m, 32 c + j) > 0
    uint32_t* mask_out;               // EPI_BIAS_RELU: the same array, written (may be null)
    long long ld_mask;
    const int* stop;                  // device flag (may be null): non-zero = the update stopped early (KL), the launch is a no-op
    LstmEpi lstm;
};

// 8 bf16 = 4 packed pairs -> one 16-byte store
__device__ __forceinline__ void st_u4(__nv_bfloat16* dst, const uint32_t* pk) {
    *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}
// the 128 epilogue threads of one column half (named barrier 1 + half); all 256 epilogue threads (barrier 3)
__device__ __forceinline__ void epi_barrier(int half) { asm volatile("bar.sync %0, 128;" ::"r"(1 + half) : "memory"); }
__device__ __forceinline__ void epi_barrier_all() { asm volatile("bar.sync 3, 256;" ::: "memory"); }
// gate non-linearities from ex2.approx + rcp.approx (2 MUFU each, ~1e-6 accurate): close enough to the exact functions that the
// bf16 roundings downstream agree with the emulation oracle (tanh.approx.f32 is 2^-11 accurate: measurably more ReLU-mask flips)
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_fast(float x) { return 1.0f - __fdividef(2.0f, __expf(2.0f * x) + 1.0f); }

__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw_u32 = smem_u32(smem_raw);
    uint8_t* smem = smem_raw + (((raw_u32 + 1023u) & ~1023u) - raw_u32);      // offset arithmetic keeps the pointer in the shared state space (STS / LDS, not generic ST / LD)
    const uint32_t s_a = smem_u32(smem), s_b = s_a + kStages * kStageA;
    uint8_t* s_stage_bm = smem + kStages * (kStageA + kStageB);                                            // [half][2][128][128 B], 1024-aligned: epilogue staging
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_stage_bm + 2 * 2 * kStageBm);
    const uint32_t bar_full = smem_u32(bars), bar_empty = bar_full + 8 * kStages, bar_tfull = bar_empty + 8 * kStages, bar_tempty = bar_tfull + 16;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);
    float* s_bias = reinterpret_cast<float*>(s_stage_bm + 2 * 2 * kStageBm + 256);                         // [256]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 8); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(smem_u32(s_tmem), 2 * kAccCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem0 = *s_tmem;
    // everything above is on-chip set-up and may overlap the tail of the previous kernel in the stream
    pdl_launch_dependents();
    pdl_wait();

    const int m_tiles = (p.m + BM - 1) / BM;
    const int total = (p.stop != nullptr && __ldg(p.stop) != 0) ? 0 : m_tiles * p.splits;
    const int kb_total = (p.k + BK - 1) / BK;
    const uint32_t stage_bytes = (uint32_t)(kStageA + p.n_tile * BK * 2);

    if (warp == 0) {
        // ===================== TMA producer
        uint32_t stage = 0, phase = 0;
        for (int w = blockIdx.x; w < total; w += gridDim.x) {
            const int mt = w % m_tiles, sp = w / m_tiles;
            const int kb0 = sp * p.kb_per_split, kb1 = min(kb0 + p.kb_per_split, kb_total);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(bar_empty + 8 * stage, phase ^ 1u);
                if (elect_one_sync()) {
                    if (!p.mn_major) {
                        mbar_arrive_expect_tx(bar_full + 8 * stage, stage_bytes);
                        tma_load_2d(s_a + stage * kStageA, &tmA, kb * BK, p.a_row0 + mt * BM, bar_full + 8 * stage);
                        tma_load_2d(s_b + stage * kStageB, &tmB, kb * BK, p.b_row0, bar_full + 8 * stage);
                    } else {
                        const int nb = (p.n_tile + 63) >> 6;
                        mbar_arrive_expect_tx(bar_full + 8 * stage, (uint32_t)(2 + nb) * kMnBlock);
                        for (int i = 0; i < 2; ++i) tma_load_2d(s_a + stage * kStageA + i * kMnBlock, &tmA, mt * BM + 64 * i, p.a_row0 + kb * BK, bar_full + 8 * stage);
                        for (int i = 0; i < nb; ++i) tma_load_2d(s_b + stage * kStageB + i * kMnBlock, &tmB, 64 * i, p.b_row0 + kb * BK, bar_full + 8 * stage);
                    }
                }
                __syncwarp();
                if (++stage == kStages) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer
        uint32_t stage = 0, phase = 0, buf = 0, acc_phase = 0;
        const uint32_t idesc = umma_idesc_bf16(BM, p.n_tile) | (p.mn_major ? (1u << 15) | (1u << 16) : 0u);     // a_major / b_major = MN
        for (int w = blockIdx.x; w < total; w += gridDim.x) {
            const int sp = w / m_tiles;
            const int kb0 = sp * p.kb_per_split, kb1 = min(kb0 + p.kb_per_split, kb_total);
            mbar_wait(bar_tempty + 8 * buf, acc_phase ^ 1u);           // the epilogue has drained this accumulator
            tc_fence_after();
            const uint32_t d_addr = tmem0 + buf * kAccCols;
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(bar_full + 8 * stage, phase);
                tc_fence_after();
                if (elect_one_sync()) {
                    const int ksteps = min(BK / 16, (p.k - kb * BK + 15) / 16);      // the zero-filled tail of K costs no MMAs
                    if (!p.mn_major) {
                        const uint64_t adesc = umma_desc_sw128(s_a + stage * kStageA), bdesc = umma_desc_sw128(s_b + stage * kStageB);
                        for (int ks = 0; ks < ksteps; ++ks)          // 16 k = 32 bytes along the swizzled rows
                            umma_bf16(d_addr, adesc + (uint64_t)(2 * ks), bdesc + (uint64_t)(2 * ks), idesc, (uint32_t)(kb != kb0 || ks != 0));
                    } else {
                        const uint64_t adesc = umma_desc_sw128_mn(s_a + stage * kStageA), bdesc = umma_desc_sw128_mn(s_b + stage * kStageB);
                        for (int ks = 0; ks < ksteps; ++ks)          // 16 k = two 8-row atoms = 2048 bytes
                            umma_bf16(d_addr, adesc + (uint64_t)(128 * ks), bdesc + (uint64_t)(128 * ks), idesc, (uint32_t)(kb != kb0 || ks != 0));
                    }
                    umma_commit(bar_empty + 8 * stage);                 // stage free once these MMAs have read it
                    if (kb == kb1 - 1) umma_commit(bar_tfull + 8 * buf);
                }
                __syncwarp();
                if (++stage == kStages) { stage = 0; phase ^= 1u; }
            }
            if (kb1 <= kb0 && elect_one_sync()) umma_commit(bar_tfull + 8 * buf);   // empty split (cannot happen with the host's partition)
            buf ^= 1u;
            if (buf == 0) acc_phase ^= 1u;
        }
    } else {
        // ===================== epilogue: thread <-> accumulator row (TMEM lane)
        const int quad = warp & 3;                                        // a warp may only touch TMEM lanes 32 * (warp % 4) .. + 31
        const int r = (quad << 5) | lane;
        const int half = (warp - 2) >> 2;                                 // warps 2..5 take the even 32-column chunks, 6..9 the odd ones
        const int te = (((warp - 2) & 3) << 5) | lane;                    // 0..127: linear index inside the half's thread group
        uint8_t* const s_bm_h = s_stage_bm + half * (2 * kStageBm);
        uint32_t buf = 0, acc_phase = 0, sb = 0;
        // column-wise constants once per CTA (the bias of the layer)
        if (p.bias != nullptr)
            for (int c = (int)threadIdx.x - 64; c < p.n_tile; c += 256) s_bias[c] = c < p.n ? __ldg(p.bias + c) : 0.0f;
        epi_barrier_all();
        for (int w = blockIdx.x; w < total; w += gridDim.x) {
            const int mt = w % m_tiles, sp = w / m_tiles;
            const long long m = (long long)mt * BM + r;
            const bool row_ok = m < p.m;
            mbar_wait(bar_tfull + 8 * buf, acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem0 + ((uint32_t)(quad << 5) << 16) + buf * kAccCols;
            if (p.epi == EPI_LSTM) {
                // Per 16-unit chunk a row reads 64 B of c_{t-1} and writes 64 B of c_t, 32 B of h_t and 128 B of gates.  All of it
                // crosses global memory with lanes along the row's bytes (3 staging rounds: c in; c + h out; gates out).
                const LstmEpi& L = p.lstm;
                const bool full = (long long)(mt + 1) * BM <= p.m;
                const long long m0 = (long long)mt * BM;
                const int row4 = te >> 2, pc4 = te & 3;                   // 4 lanes per row (64-byte runs): rows row4 + 32 q
                const int row8 = te >> 3, pc8 = te & 7;                   // 8 lanes per row (128-byte runs): rows row8 + 16 q
                const int row2 = te >> 1, pc2 = te & 1;                   // 2 lanes per row (32-byte runs): rows row2 + 64 q
                const uint32_t own = (uint32_t)(r * 128), key = (uint32_t)(r & 7);
#pragma unroll 1
                for (int j0 = 32 * half; j0 < 32 * half + 32; j0 += 16) {
                    uint32_t vi[16], vf[16], vg[16], vo[16];
                    tmem_ld16(t_row + j0, vi); tmem_ld16(t_row + 64 + j0, vf); tmem_ld16(t_row + 128 + j0, vg); tmem_ld16(t_row + 192 + j0, vo);
                    float cp[16];
                    if (L.c_prev) {                                       // round 1: c_{t-1}, 4 lanes per row -> staging -> own row
                        uint8_t* sa = s_bm_h + sb * kStageBm;
                        uint4 in[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int row = row4 + 32 * q;
                            in[q] = (full || m0 + row < p.m) ? __ldg(reinterpret_cast<const uint4*>(L.c_prev + (m0 + row) * 64 + j0 + 4 * pc4)) : make_uint4(0u, 0u, 0u, 0u);
                        }
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int row = row4 + 32 * q;
                            *reinterpret_cast<uint4*>(sa + row * 128 + ((pc4 ^ (row & 7)) << 4)) = in[q];
                        }
                        epi_barrier(half);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float4 c4 = *reinterpret_cast<const float4*>(sa + own + ((q ^ key) << 4));
                            cp[4 * q] = c4.x; cp[4 * q + 1] = c4.y; cp[4 * q + 2] = c4.z; cp[4 * q + 3] = c4.w;
                        }
                        sb ^= 1u;
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) cp[j] = 0.0f;
                    }
                    tmem_ld_wait();
                    uint32_t pg4[4][8], ph[8];                            // packed gates i, f, g, o and h
                    float cc[16];
#pragma unroll
                    for (int j = 0; j < 16; j += 2) {
                        float gi[2], gf[2], gg[2], go[2], hh[2];
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            gi[e] = sigmoid_fast(__uint_as_float(vi[j + e])); gf[e] = sigmoid_fast(__uint_as_float(vf[j + e]));
                            gg[e] = tanh_fast(__uint_as_float(vg[j + e])); go[e] = sigmoid_fast(__uint_as_float(vo[j + e]));
                            cc[j + e] = gf[e] * cp[j + e] + gi[e] * gg[e];
                            hh[e] = go[e] * tanh_fast(cc[j + e]);
                        }
                        pg4[0][j >> 1] = pack_bf16x2(gi[0], gi[1]); pg4[1][j >> 1] = pack_bf16x2(gf[0], gf[1]);
                        pg4[2][j >> 1] = pack_bf16x2(gg[0], gg[1]); pg4[3][j >> 1] = pack_bf16x2(go[0], go[1]);
                        ph[j >> 1] = pack_bf16x2(hh[0], hh[1]);
                    }
                    {                                                     // round 2: c_t (pieces 0..3) and h_t (pieces 4, 5) of the own row -> staging
                        uint8_t* sa = s_bm_h + sb * kStageBm;
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            *reinterpret_cast<float4*>(sa + own + ((q ^ key) << 4)) = make_float4(cc[4 * q], cc[4 * q + 1], cc[4 * q + 2], cc[4 * q + 3]);
                        *reinterpret_cast<uint4*>(sa + own + ((4u ^ key) << 4)) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
                        *reinterpret_cast<uint4*>(sa + own + ((5u ^ key) << 4)) = make_uint4(ph[4], ph[5], ph[6], ph[7]);
                        epi_barrier(half);
                        uint4 oc[4], oh[2];
#pragma unroll
                        for (int q = 0; q < 4; ++q) { const int row = row4 + 32 * q; oc[q] = *reinterpret_cast<const uint4*>(sa + row * 128 + ((pc4 ^ (row & 7)) << 4)); }
#pragma unroll
                        for (int q = 0; q < 2; ++q) { const int row = row2 + 64 * q; oh[q] = *reinterpret_cast<const uint4*>(sa + row * 128 + (((4 + pc2) ^ (row & 7)) << 4)); }
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int row = row4 + 32 * q;
                            if (full || m0 + row < p.m) *reinterpret_cast<uint4*>(L.c_out + (m0 + row) * 64 + j0 + 4 * pc4) = oc[q];
                        }
                        if (L.h_bm) {
#pragma unroll
                            for (int q = 0; q < 2; ++q) {
                                const int row = row2 + 64 * q;
                                if (full || m0 + row < p.m) *reinterpret_cast<uint4*>(L.h_bm + (m0 + row) * L.ld_h_bm + j0 + 8 * pc2) = oh[q];
                            }
                        }
                        if (L.h2_bm) {
#pragma unroll
                            for (int q = 0; q < 2; ++q) {
                                const int row = row2 + 64 * q;
                                if (full || m0 + row < p.m) *reinterpret_cast<uint4*>(L.h2_bm + (m0 + row) * L.ld_h2_bm + j0 + 8 * pc2) = oh[q];
                            }
                        }
                        sb ^= 1u;
                    }
                    {                                                     // round 3: the chunk's 4 x 16 gates = 128 bytes of the own row -> staging
                        uint8_t* sa = s_bm_h + sb * kStageBm;
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            *reinterpret_cast<uint4*>(sa + own + (((uint32_t)q ^ key) << 4)) = make_uint4(pg4[q >> 1][4 * (q & 1)], pg4[q >> 1][4 * (q & 1) + 1], pg4[q >> 1][4 * (q & 1) + 2], pg4[q >> 1][4 * (q & 1) + 3]);
                        epi_barrier(half);
                        uint4 og[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) { const int row = row8 + 16 * q; og[q] = *reinterpret_cast<const uint4*>(sa + row * 128 + ((pc8 ^ (row & 7)) << 4)); }
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const int row = row8 + 16 * q;
                            if (full || m0 + row < p.m) *reinterpret_cast<uint4*>(L.gates_out + (m0 + row) * 256 + (j0 >> 4) * 64 + 8 * pc8) = og[q];
                        }
                        sb ^= 1u;
                    }
                }
            } else if (p.epi == EPI_BIAS_RELU || p.epi == EPI_RELUBWD) {
                // 64 columns (128 bytes of bf16 per row) per round; the two halves take alternating rounds
                const uint32_t own = (uint32_t)(r * 128), key = (uint32_t)(r & 7);
                int c0 = 64 * half;
                uint32_t v[32];
                if (c0 < p.n_valid) tmem_ld32(t_row + c0, v);
#pragma unroll 1
                for (; c0 < p.n_valid; c0 += 128) {
                    uint8_t* sa = s_bm_h + sb * kStageBm;
                    if (te == 0) tma_store_wait_read();                   // the store issued from this buffer two rounds ago has drained it
#pragma unroll 1
                    for (int h2 = 0; h2 < 2; ++h2) {
                        const int cc = c0 + 32 * h2;
                        if (cc >= p.n_valid) break;                       // (n_valid is a multiple of 8; columns past it in a stored box are clipped or zero)
                        uint32_t mw = 0u;                                // ReLU mask word of (row, 32 columns): one coalesced word per lane
                        if (p.epi == EPI_RELUBWD && row_ok) mw = __ldg(p.mask_in + (long long)(cc >> 5) * p.ld_mask + m);
                        tmem_ld_wait();
                        uint32_t pk[16];
                        if (p.epi == EPI_BIAS_RELU) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                                const float4 b4 = *reinterpret_cast<const float4*>(s_bias + cc + 4 * q);
                                const float z0 = __uint_as_float(v[4 * q]) + b4.x, z1 = __uint_as_float(v[4 * q + 1]) + b4.y;
                                const float z2 = __uint_as_float(v[4 * q + 2]) + b4.z, z3 = __uint_as_float(v[4 * q + 3]) + b4.w;
                                mw |= (z0 > 0.0f ? 1u : 0u) << (4 * q) | (z1 > 0.0f ? 2u : 0u) << (4 * q) | (z2 > 0.0f ? 4u : 0u) << (4 * q) | (z3 > 0.0f ? 8u : 0u) << (4 * q);
                                pk[2 * q] = pack_bf16x2(fmaxf(z0, 0.0f), fmaxf(z1, 0.0f));
                                pk[2 * q + 1] = pack_bf16x2(fmaxf(z2, 0.0f), fmaxf(z3, 0.0f));
                            }
                            if (p.mask_out && row_ok) p.mask_out[(long long)(cc >> 5) * p.ld_mask + m] = mw;
                        } else {
#pragma unroll
                            for (int i = 0; i < 16; ++i)
                                pk[i] = pack_bf16x2((mw >> (2 * i)) & 1u ? __uint_as_float(v[2 * i]) : 0.0f, (mw >> (2 * i + 1)) & 1u ? __uint_as_float(v[2 * i + 1]) : 0.0f);
                        }
                        // the next 32 accumulator columns fly under the staging stores
                        const int cn = h2 == 0 ? cc + 32 : c0 + 128;
                        if (cn < p.n_valid) tmem_ld32(t_row + cn, v);
#pragma unroll
                        for (int q = 0; q < 4; ++q)                       // own row, pieces 4 h2 .. 4 h2 + 3 (XOR-swizzled: conflict-free, and the TMA's SWIZZLE_128B)
                            *reinterpret_cast<uint4*>(sa + own + (((uint32_t)(4 * h2 + q) ^ key) << 4)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
                    }
                    fence_proxy_async_smem();
                    epi_barrier(half);
                    if (te == 0) tma_store_2d(&tmC, smem_u32(sa), c0, mt * BM);
                    sb ^= 1u;
                }
            } else if (p.epi == EPI_F32 && p.tma_store) {
                // fp32 tile (split-K partial of a weight gradient): 32 columns = 128 bytes per row and round
                const uint32_t own = (uint32_t)(r * 128), key = (uint32_t)(r & 7);
                int c0 = 32 * half;
                uint32_t v[32];
                if (c0 < p.n_valid) tmem_ld32(t_row + c0, v);
#pragma unroll 1
                for (; c0 < p.n_valid; c0 += 64) {
                    uint8_t* sa = s_bm_h + sb * kStageBm;
                    if (te == 0) tma_store_wait_read();
                    tmem_ld_wait();
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<uint4*>(sa + own + (((uint32_t)q ^ key) << 4)) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                    if (c0 + 64 < p.n_valid) tmem_ld32(t_row + c0 + 64, v);
                    fence_proxy_async_smem();
                    epi_barrier(half);
                    if (te == 0) tma_store_2d(&tmC, smem_u32(sa), c0, sp * p.m + mt * BM);
                    sb ^= 1u;
                }
            } else {
                for (int c0 = 32 * half; c0 < p.n_valid; c0 += 64) {
                    uint32_t v[32];
                    tmem_ld32(t_row + c0, v);
                    tmem_ld_wait();
                    if (!row_ok) continue;
                    const int nv = min(32, p.n_valid - c0);
                    if (p.epi == EPI_F32) {
                        float* o = p.out_f32 + (long long)sp * p.split_stride + m * p.ldc + c0;
                        if (nv == 32 && ((reinterpret_cast<uintptr_t>(o) & 15u) == 0)) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                                if (p.bias) b4 = *reinterpret_cast<const float4*>(s_bias + c0 + 4 * q);
                                *reinterpret_cast<float4*>(o + 4 * q) = make_float4(__uint_as_float(v[4 * q]) + b4.x, __uint_as_float(v[4 * q + 1]) + b4.y,
                                                                                    __uint_as_float(v[4 * q + 2]) + b4.z, __uint_as_float(v[4 * q + 3]) + b4.w);
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < nv) o[j] = __uint_as_float(v[j]) + (p.bias ? s_bias[c0 + j] : 0.0f);
                        }
                    } else {                                              // EPI_TANH_F32
                        float* o = p.out_f32 + m * p.ldc + c0;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (j < nv) o[j] = tanhf(__uint_as_float(v[j]) + s_bias[c0 + j]);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty + 8 * buf);
            buf ^= 1u;
            if (buf == 0) acc_phase ^= 1u;
        }
        if (te == 0) tma_store_wait_all();                                // the staging tiles must outlive the bulk stores reading them
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem0, 2 * kAccCols);
}

}  // namespace gemm
}  // namespace taco
