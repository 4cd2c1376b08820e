// Actor MLP on the 5th-generation tensor cores (tcgen05 + TMEM), one persistent CTA per SM.
//
// Replaces, for rollout inference, MLP.forward + the actor branch of PPO_ActorCritic.act
// (IsaacGymEnvs/algorithms/nets_asymmetry.py:23-39, :326-346):  mean = tanh(W_L relu(... relu(W_1 x + b_1) ...) + b_L).
//
// Shape of the work: a tile is 128 envs (rows = TMEM lanes); a CTA keeps TWO tiles in flight (a pair).  Every hidden
// layer is D[128 x N] = A[128 x K] * W[N x K]^T by tcgen05.mma (bf16 operands, fp32 accumulation, M=128, N = one
// 128-row part of W, K=16 per instruction).  The activations never touch shared memory: A lives in TENSOR MEMORY as
// packed bf16 pairs (the "TS" form of the instruction, A from TMEM), D in the neighbouring 128 TMEM columns, and the
// tile's epilogue warps turn D into the next layer's A register-side (tcgen05.ld -> +bias, ReLU -> bf16x2 ->
// tcgen05.st).  Shared memory holds only the weight ring: W streams from L2 through 64 KB slots (one 128-row part of a
// layer = up to four 16 KB K-chunks, K-major SWIZZLE_128B) filled by the bulk async-copy engine (cp.async.bulk + mbarrier
// complete_tx) from images that taco_actor_load pre-swizzled once per update; every slot is consumed by BOTH tiles of the
// pair before it is released (half the L2 traffic per env), and the two tiles alternate part by part, so while the tensor core works
// on one tile the epilogue warps of the other drain its accumulator.  The 4-wide output layer rides the same chain as
// one more (N = 16, zero-padded) MMA part; tanh and the optional Gaussian sampling are CUDA-core work in its epilogue.
//
// This pipeline is shared with the critic kernel (mlp_common.cuh); this header adds the observation staging, the output part and the
// tail.  TMEM map (512 columns): tile slot t owns columns [256 t, 256 t + 256): A = first 128 (K <= 256 as bf16 pairs),
// D = last 128 (one part of N).
// Warp roles (576 threads): warp 0 = weight producer, warp 1 = TMEM allocator + MMA issuer (both warp-uniform loops
// with one elected lane issuing, so that every operand stays in uniform registers),
// warps 2..17 = epilogue: tile slot t = (warp-2)/8, column half of the part = ((warp-2)/4)&1, TMEM lane quadrant =
// warp%4 (thread <-> TMEM lane <-> env row).
#pragma once
#include "mlp_common.cuh"
#include "philox.cuh"

namespace taco {
namespace actor {
using namespace taco::mlp;

constexpr uint32_t STREAM_ACTOR = 6;           // Philox stream of the action noise

struct SampleParams {    // PPO_ActorCritic.act sampling (nets_asymmetry.py:336-346); enabled when action != nullptr
    float* action;       // (n, out) mean + std * eps
    float* clipped;      // (n, out) clamp(action, -1, 1)   (ppo_asymmetry.py:310)
    float* logp;         // (n)
    const float* samp;   // device, owned by the TacoActor: [0..3] std = exp(log_std)^2 (scale_tril = diag(exp(log_std)^2),
                         // nets_asymmetry.py:338), [4] logp_const = -sum(log std) - out/2 * log(2 pi).  In device memory, not by
                         // value, so that a launch captured in a CUDA graph follows taco_actor_set_log_std between replays
    long long env_offset;
    uint32_t seed_lo, seed_hi, step_index;
    const uint32_t* step_base;   // device word added to step_index (null: none), see taco_actor_act_counter
};

struct TcParams {
    const float* obs;    // (n_rows, in_dim) f32
    float* mean;         // (n_rows, out_dim) f32
    int in_dim, out_dim, n_rows, num_tiles, n_hidden;
    int tiles_per_cta;   // 2 (a CTA keeps a pair of tiles in flight) or 1
    int obs_bulk;        // in_dim <= 26, even, 16-byte aligned base: whole tiles of observations are staged by the bulk-copy engine
    int obs_vec2;        // rows of obs are 8-byte aligned (even in_dim, aligned base): observation loads use 8-byte accesses
    const uint8_t* wimg; // pre-swizzled bf16 chunk images of the hidden layers and of the (16-row padded) output layer
    const float* bias;   // [kMaxHidden][kMaxN] f32
    const float* b_out;  // [kOutPad]
    TcLayer layer[kMaxHidden + 1];   // hidden layers, then the output layer (n = kOutN)
    SampleParams sp;
    unsigned long long* dbg;   // optional timeline of CTA 0 (TACO_ACTOR_TIMELINE=<file>): 3 regions of kDbgCap (clock << 8 | code) words
};

constexpr int kObsBulkMaxIn = 26;              // widest observation row the bulk-staged path takes (26 x len_obs = 1)
constexpr int kObsStageBytes = kTileM * kObsBulkMaxIn * 4;        // one tile's observation block, fp32, as it lies in global memory
constexpr int kActorSmemBytes = kTcSmemBytes + 2 * kObsStageBytes;

// tanh output + optional sampling, shared by the tensor-core and the FP32 kernels (one thread = one env row)
__device__ __forceinline__ void actor_tail(const float* pre, int out_dim, long long row, float* mean, const SampleParams& sp) {
    float mu[kOutPad];
#pragma unroll
    for (int o = 0; o < kOutPad; ++o) mu[o] = tanhf(pre[o]);
    if (out_dim == 4) {
        *reinterpret_cast<float4*>(mean + row * 4) = make_float4(mu[0], mu[1], mu[2], mu[3]);
    } else {
        for (int o = 0; o < out_dim; ++o) mean[row * out_dim + o] = mu[o];
    }
    if (sp.action) {
        const uint4 r = philox4x32_10((uint32_t)(sp.env_offset + row), sp.step_index + (sp.step_base ? __ldg(sp.step_base) : 0u), 0, STREAM_ACTOR,
                                      sp.seed_lo, sp.seed_hi);
        float z[4];
        box_muller(r.x, r.y, z[0], z[1]);
        box_muller(r.z, r.w, z[2], z[3]);
        float lp = __ldg(sp.samp + 4);
        float a[kOutPad] = {0.f, 0.f, 0.f, 0.f};
        for (int o = 0; o < out_dim; ++o) {
            a[o] = mu[o] + __ldg(sp.samp + o) * z[o];
            lp += -0.5f * (z[o] * z[o]);
        }
        if (out_dim == 4 && ((reinterpret_cast<uintptr_t>(sp.action) | reinterpret_cast<uintptr_t>(sp.clipped)) & 15u) == 0) {
            *reinterpret_cast<float4*>(sp.action + row * 4) = make_float4(a[0], a[1], a[2], a[3]);
            if (sp.clipped)
                *reinterpret_cast<float4*>(sp.clipped + row * 4) = make_float4(fminf(fmaxf(a[0], -1.0f), 1.0f), fminf(fmaxf(a[1], -1.0f), 1.0f),
                                                                               fminf(fmaxf(a[2], -1.0f), 1.0f), fminf(fmaxf(a[3], -1.0f), 1.0f));
        } else {
            for (int o = 0; o < out_dim; ++o) {
                sp.action[row * out_dim + o] = a[o];
                if (sp.clipped) sp.clipped[row * out_dim + o] = fminf(fmaxf(a[o], -1.0f), 1.0f);
            }
        }
        if (sp.logp) sp.logp[row] = lp;
    }
}

// ---------------------------------------------------------------------------------------------- the kernel
// the observation features [32 g, 32 g + 32) of one row as 16 packed bf16 pairs (zero beyond in_dim / for invalid rows).  Rows of an
// even width are 8-byte aligned ((N, in_dim) float32 contiguous): one 8-byte load per pair halves the L1 wavefronts of this
// row-per-thread access pattern (every lane touches its own row, i.e. its own cache line).
__device__ __forceinline__ void load_obs_group(const float* x, int g, int in_dim, bool valid, uint32_t* pk, bool vec2) {
    if (vec2) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int k = g * 32 + 2 * j;
            const float2 f = (valid && k < in_dim) ? __ldg(reinterpret_cast<const float2*>(x + k)) : make_float2(0.0f, 0.0f);
            pk[j] = pack_bf16x2(f.x, f.y);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int k = g * 32 + 2 * j;
            const float f0 = (valid && k < in_dim) ? __ldg(x + k) : 0.0f;
            const float f1 = (valid && k + 1 < in_dim) ? __ldg(x + k + 1) : 0.0f;
            pk[j] = pack_bf16x2(f0, f1);
        }
    }
}

// features [0, 32) of row r of a bulk-staged observation block (rows of in_dim floats, as in global memory) as 16 packed bf16
// pairs; 8-byte reads at a row stride of in_dim * 4 bytes (26 words: conflict-free per half-warp)
__device__ __forceinline__ void read_staged_obs(const float* stage, int r, int in_dim, uint32_t* pk) {
    const float2* row = reinterpret_cast<const float2*>(stage + r * in_dim);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float2 f = (2 * j < in_dim) ? row[j] : make_float2(0.0f, 0.0f);
        pk[j] = pack_bf16x2(f.x, f.y);
    }
}

__global__ void __launch_bounds__(kTcThreads, 1) actor_tc_kernel(const TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    const TcSmem sm(smem_raw);
    const uint32_t bar_obs = sm.bar_own;                             // [2] a tile's observation block has landed in the staging buffer
    float* s_obs = reinterpret_cast<float*>(sm.base + kTcSmemBytes - 1024);   // [2 tiles][128 rows x in_dim] (only with p.obs_bulk)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tps = p.tiles_per_cta;                                 // 2, or 1 when there are fewer tiles than SMs (small batches: one tile per CTA halves the latency)
    const int num_pairs = (p.num_tiles + tps - 1) / tps;
    const int n_layers = p.n_hidden + 1;                             // hidden layers + the output layer as a 16-wide part

    const uint32_t tmem0 = sm.setup(warp, p.bias, [&] { for (int t = 0; t < 2; ++t) mbar_init(bar_obs + 8 * t, 1); });

    if (warp == 0) {
        // ===================== weight producer: per pair, per layer, per 128-row part one slot
        uint32_t slot = 0, phase = 0;
        for (int pair = blockIdx.x; pair < num_pairs; pair += gridDim.x)
            for (int l = 0; l < n_layers; ++l) produce_layer(sm, p.wimg, p.layer[l], kSlots, slot, phase);
    } else if (warp == 1) {
        // ===================== MMA issuer: tiles A (slot 0) and B (slot 1) of the pair alternate part by part and share every weight slot
        uint32_t slot = 0, phase = 0, a_phase = 0;
        int dbg_n = lane == 0 ? 0 : kDbgCap;
        const uint64_t bdesc0 = umma_desc_sw128(sm.ring);
        for (int pair = blockIdx.x; pair < num_pairs; pair += gridDim.x) {
            const int nt = min(tps, p.num_tiles - tps * pair);
            for (int l = 0; l < n_layers; ++l) {
                const int n = p.layer[l].n, kch = p.layer[l].kchunks;
                for (int h0 = 0; h0 < n; h0 += kPartN) {
                    const uint32_t idesc = umma_idesc_bf16(kTileM, min(kPartN, n - h0));
                    const uint64_t bdesc = bdesc0 + (uint64_t)(slot * (kSlotBytes >> 4));
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        if (t < nt) {
                            mbar_wait(sm.bar_a + 8 * t, (a_phase >> t) & 1u); a_phase ^= (1u << t);   // D(t) free; A(t) of this layer in TMEM
                            if (t == 0) mbar_wait(sm.bar_full + 8 * slot, phase);
                            tc_fence_after();
                            TACO_DBG(0, dbg_n, 0x20 | t);
                            issue_part(tmem0 + (uint32_t)(t * kTmemSlot), bdesc, idesc, kch, false, t == nt - 1, sm.bar_empty + 8 * slot,
                                       sm.bar_d + 8 * t);
                            TACO_DBG(0, dbg_n, 0x30 | t);
                        }
                    }
                    if (++slot == kSlots) { slot = 0; phase ^= 1u; }
                }
            }
        }
    } else {
        // ===================== epilogue warps
        const EpiThread ep(warp, lane, tmem0, tps, p.num_tiles);
        const int e = ep.e, t = ep.t, ch = ep.ch, r = ep.r;
        const uint32_t t_a = ep.t_a, t_d = ep.t_d;
        uint32_t d_phase = 0;
        const int kc0 = p.layer[0].kchunks;
        int dbg_n = (ch == 0 && ep.quad == 0 && lane == 0) ? 0 : kDbgCap;
        int tile = ep.tile;
        const int tile_step = ep.tile_step;
        // Bulk-staged observations (p.obs_bulk): a FULL tile's rows are one contiguous block of global memory (128 x in_dim floats), so
        // one elected thread of the tile has the bulk-copy engine fetch the block of the tile AFTER the one being staged; the
        // 128 x 26 row-per-thread scalar loads (one cache line per lane and instruction) leave the LSU.  Partial last tiles use loads.
        float* s_obs_t = s_obs + t * (kTileM * kObsBulkMaxIn);
        const uint32_t obs_bytes = (uint32_t)(kTileM * p.in_dim * 4);
        uint32_t o_phase = 0;
        const bool staged_first = p.obs_bulk && (long long)(tile + 1) * kTileM <= p.n_rows;
        auto fetch_obs = [&](int tl) {                               // all 256 threads of the tile call this; one issues the copy
            asm volatile("bar.sync %0, %1;" ::"r"(1 + t), "r"((kEpiWarps / 2) * 32) : "memory");     // every reader of the buffer is done
            if (e % 8 == 0 && elect_one_sync()) {
                fence_proxy_async_smem();
                mbar_arrive_expect_tx(bar_obs + 8 * t, obs_bytes);
                bulk_g2s(smem_u32(s_obs_t), p.obs + (size_t)tl * kTileM * p.in_dim, obs_bytes, bar_obs + 8 * t);
            }
        };
        auto bulk_tile = [&](int tl) { return p.obs_bulk && tl < p.num_tiles && (long long)(tl + 1) * kTileM <= p.n_rows; };
        if (tile < p.num_tiles) {
            // ---- the first tile's observation row as packed bf16 into A(t), K padded with zeros to kc0 * 64; groups of 32
            // features (16 TMEM columns) alternate between ch 0 / 1
            const long long row0 = (long long)tile * kTileM + r;
            if (staged_first) {
                fetch_obs(tile);
                mbar_wait(bar_obs + 8 * t, o_phase); o_phase ^= 1u;
                uint32_t pk[16];
                if (ch == 0) read_staged_obs(s_obs_t, r, p.in_dim, pk);
                else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) pk[j] = 0u;
                }
                tmem_st16(t_a + (uint32_t)(ch * 16), pk);
                if (bulk_tile(tile + tile_step)) fetch_obs(tile + tile_step);
            } else {
                for (int g = ch; g < kc0 * 2; g += 2) {
                    uint32_t pk[16];
                    load_obs_group(p.obs + row0 * p.in_dim, g, p.in_dim, row0 < p.n_rows, pk, p.obs_vec2 != 0);
                    tmem_st16(t_a + (uint32_t)(g * 16), pk);
                }
                if (bulk_tile(tile + tile_step)) fetch_obs(tile + tile_step);
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(sm.bar_a + 8 * t);
            TACO_DBG(1 + t, dbg_n, 0x01);
        }
        for (; tile < p.num_tiles; tile += tile_step) {
            const long long row = (long long)tile * kTileM + r;
            const bool valid = row < p.n_rows;
            const bool has_next = tile + tile_step < p.num_tiles;
            const long long row_next = row + (long long)tile_step * kTileM;
            const float* x_next = p.obs + row_next * p.in_dim;
            if (has_next && row_next < p.n_rows) prefetch_l2(x_next + ch * 32);   // this thread's first group of the next tile
            for (int l = 0; l < p.n_hidden; ++l)
                hidden_layer<true>(ep, sm.bias, l, p.layer[l].n, sm.bar_a, sm.bar_d, d_phase, p.dbg, dbg_n);
            // ---- output layer (columns 0..3 of its 16-wide part).  The next tile's first observation group is fetched while the
            // output MMAs run; once D is in registers the next A(t) is written and the issuer released, and only then the tanh /
            // sampling tail of this tile runs (overlapping the next tile's first MMAs).
            uint32_t pkn[16];
            const bool next_staged = has_next && bulk_tile(tile + tile_step);
            if (next_staged) {                                       // the block was fetched a whole tile ago: no load latency to hide
                mbar_wait(bar_obs + 8 * t, o_phase); o_phase ^= 1u;
                if (ch == 0) read_staged_obs(s_obs_t, r, p.in_dim, pkn);
                else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) pkn[j] = 0u;
                }
                if (bulk_tile(tile + 2 * tile_step)) fetch_obs(tile + 2 * tile_step);
            } else if (has_next) load_obs_group(x_next, ch, p.in_dim, row_next < p.n_rows, pkn, p.obs_vec2 != 0);
            mbar_wait(sm.bar_d + 8 * t, d_phase); d_phase ^= 1u;
            tc_fence_after();
            TACO_DBG(1 + t, dbg_n, 0x06);
            uint32_t v[4];
            if (ch == 0) { tmem_ld4(t_d, v); tmem_ld_wait(); }
            if (has_next) {
                tmem_st16(t_a + (uint32_t)(ch * 16), pkn);
                for (int g = ch + 2; g < kc0 * 2 && !next_staged; g += 2) {
                    load_obs_group(x_next, g, p.in_dim, row_next < p.n_rows, pkn, p.obs_vec2 != 0);
                    tmem_st16(t_a + (uint32_t)(g * 16), pkn);
                }
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(sm.bar_a + 8 * t);
                TACO_DBG(1 + t, dbg_n, 0x01);
            }
            if (ch == 0 && valid) {
                float pre[kOutPad];
#pragma unroll
                for (int o = 0; o < kOutPad; ++o) pre[o] = __uint_as_float(v[o]) + __ldg(p.b_out + o);
                actor_tail(pre, p.out_dim, row, p.mean, p.sp);
            }
            TACO_DBG(1 + t, dbg_n, 0x07);
        }
    }
    sm.teardown(warp, tmem0);
}

}  // namespace actor
}  // namespace taco
