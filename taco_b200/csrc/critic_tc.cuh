// Critic (LSTM encoder over the state history + MLP -> value) on the 5th-generation tensor cores, one persistent CTA per SM.
//
// Replaces, for rollout inference, the critic branch of PPO_ActorCritic.act
// (IsaacGymEnvs/algorithms/nets_asymmetry.py:350-352): value = critic_mlp(critic_encoder(states)) with
//   LSTMEncoder.forward   nets_asymmetry.py:128-136   nn.LSTM(26, H, 1, batch_first=True) over (N, len_states, 26), output h_T
//   MLP.forward           nets_asymmetry.py:23-39     [Linear -> ReLU] x L -> Linear(-> 1), Identity output (:318)
//
// Runs the tcgen05 MLP pipeline of mlp_common.cuh, as the actor kernel does: two 128-env tiles in flight per CTA, the A operand in
// TENSOR MEMORY, weights streamed through a shared-memory ring by the bulk-copy engine and shared by both tiles, MMA parts of the
// two tiles interleaved so that one tile's accumulator is drained while the tensor core works on the other.  The critic's own
// parts are the schedule and the LSTM epilogue:
//   * one LSTM time step is ONE layer of the chain: gates[128 x 4H] = [h_{t-1} | x_t] (K = 64 + 64, zero padded) * Wcat^T,
//     Wcat = [W_hh | W_ih] with its rows permuted so that every 16 accumulator columns hold the four gates (i, f, g, o; 4
//     columns each) of the same 4 hidden units -- an epilogue thread reads 16 columns and owns those 4 units outright;
//   * the cell state c lives in tensor memory too (fp32, in the 64 columns of the tile's A region the K = 128 LSTM operand leaves
//     free), read and rewritten by the thread that owns (env row, hidden unit); h_t is written back over the A operand as
//     packed bf16 pairs next to the freshly staged x_{t+1};
//   * the T = len_states steps reuse one weight image; then come the MLP layers and the 16-wide output part.
// A stacked LSTM (nn.LSTM(.., H, L), L = 2..4) runs its layers one after another as launches of the same kernel, one
// instantiation per role (critic_tc_kernel<kSeqIn, kSeqOut>): the layers below the top stop after the T steps and write h^k_t of
// every step to a workspace (kSeqOut), the layers above the bottom read their x_t = h^{k-1}_t from it instead of the state frames
// (kSeqIn).  The hand-off is in "owner order" (seq_idx), so that no transpose is needed on either side.
// Gate non-linearities use MUFU.TANH (tanh.approx.f32; sigmoid(x) = 0.5 + 0.5 tanh(x / 2)): five per (env, unit, step) -- the
// LSTM phase is bound by the 16 MUFU lanes of the SM, not by the tensor core.
#pragma once
#include <cuda_fp16.h>
#include "mlp_common.cuh"

namespace taco {
namespace critic {
using namespace taco::mlp;

constexpr int kMaxSeq = 8;             // len_states of the reference runs is 5 (README.md:60-66)
constexpr int kTcMaxLstmHidden = 64;   // the cell state lives in the 64 spare TMEM columns of the tile's A operand
constexpr int kTcMaxIn = 30;           // features per frame (26) + two constant-1 bias columns, padded to 32 = 16 packed TMEM columns
constexpr int kMaxMlpHidden = 3;       // bias rows: LSTM gates + up to 3 hidden layers
static_assert(1 + kMaxMlpHidden <= kMaxHidden, "the LSTM step and the MLP's hidden layers share the kMaxHidden bias rows / TcImage layers");
constexpr int kRing = kSlots - 1;        // ring slots of the MLP weights; the last 64 KB slot holds the LSTM image for the whole kernel
constexpr int kAColH = 0;              // A operand columns (packed bf16 pairs): h in [0, 32), x_t in [32, 48), zero pad [48, 64)
                                       // (the layers above the bottom of a stack: x_t = h^{k-1}_t in all of [32, 64))
constexpr int kAColX = 32;
constexpr int kAColC = 64;              // cell state, fp32, one column per hidden unit (LSTM phase only)

struct CriticTcParams {
    const float* states;   // (n_rows, seq_len, in_dim) f32
    float* value;          // (n_rows) f32
    int in_dim, seq_len, n_rows, num_tiles;
    int tiles_per_cta;     // 2 (a CTA keeps a pair of tiles in flight) or 1
    int stagger;           // cycles by which tile 1's LSTM chain trails tile 0's (0 = strictly alternating issue order)
    int lstm_hidden;       // H: multiple of 16, <= 64
    int n_hidden;          // MLP hidden layers, 1..3
    const uint8_t* wimg;   // pre-swizzled bf16 chunk images: LSTM [W_hh | W_ih] (gate-permuted rows), MLP layers, output (16 rows)
    const float* bias;     // [kMaxHidden][kMaxN]: row 0 = the gate biases of a layer above the bottom (kSeqIn; the bottom layer's
                           // bias rides in the MMA and leaves row 0 unused), rows 1.. = MLP hidden biases
    const float* b_out;    // [kOutPad]
    TcLayer layer[2 + kMaxMlpHidden];   // [0] one LSTM step, [1 .. n_hidden] MLP hidden layers, [n_hidden + 1] output layer
    unsigned long long* dbg;            // optional timeline of CTA 0 (TACO_CRITIC_TIMELINE=<file>), see TACO_DBG in mlp_common.cuh
    const uint4* seq_in;   // kSeqIn: h of the layer below for every step (seq_idx layout); bias row 0 = this layer's gate biases
    uint4* seq_out;        // kSeqOut: this layer's h for every step, same layout
};

constexpr int kCriticStagger = 1200;      // default of CriticTcParams::stagger (TACO_CRITIC_STAGGER in the environment overrides it: tuning)

// TACO_CRITIC_GATES (tuning builds): 0 (default) = tanh.approx.f32; 1 = MUFU.TANH on packed half pairs (tanh.approx.f16x2: the same
// 16.4 results per clock and SM as the f32 form, tools/probes/mufu_probe.cu, plus conversions -- no faster, twice the error);
// 2 = no transcendentals at all (timing experiment only, wrong values)
#ifndef TACO_CRITIC_GATES
#define TACO_CRITIC_GATES 0
#endif
// tanh of two floats
__device__ __forceinline__ float2 tanh_pair(float a, float b) {
#if TACO_CRITIC_GATES == 1
    return __half22float2(h2tanh_approx(__floats2half2_rn(a, b)));
#elif TACO_CRITIC_GATES == 0
    return make_float2(tanh_mufu(a), tanh_mufu(b));
#else
    return make_float2(fminf(fmaxf(a, -1.0f), 1.0f), fminf(fmaxf(b, -1.0f), 1.0f));
#endif
}
// 16 accumulator columns = [i(4) f(4) g(4) o(4)] of 4 hidden units.  The rows of the sigmoid gates are pre-scaled by 1/2
// (exact in bf16), sigmoid(x) = 0.5 + 0.5 tanh(x / 2).  In the bottom layer the accumulator already holds the complete argument
// of each tanh: the bias rides in the MMA (two constant-1 input columns against bf16 hi / lo halves of b_ih + b_hh).  The layers
// above have no room for those columns (kBias): their bias b (the 16 columns' values, scaled like the rows) is added here.
// c' = sig(f) c + sig(i) tanh(g), h' = sig(o) tanh(c'); h' leaves as 2 packed bf16 pairs (unit 2j in the low half)
template <bool kBias>
__device__ __forceinline__ void lstm_group(uint32_t (&v)[16], uint32_t (&c)[4], uint32_t* hp, const float* b) {
    if constexpr (kBias) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 bb = *reinterpret_cast<const float4*>(b + q * 4);
            v[q * 4 + 0] = __float_as_uint(__uint_as_float(v[q * 4 + 0]) + bb.x);
            v[q * 4 + 1] = __float_as_uint(__uint_as_float(v[q * 4 + 1]) + bb.y);
            v[q * 4 + 2] = __float_as_uint(__uint_as_float(v[q * 4 + 2]) + bb.z);
            v[q * 4 + 3] = __float_as_uint(__uint_as_float(v[q * 4 + 3]) + bb.w);
        }
    }
#pragma unroll
    for (int u = 0; u < 4; u += 2) {
        const float2 ti = tanh_pair(__uint_as_float(v[u]), __uint_as_float(v[u + 1]));
        const float2 tf = tanh_pair(__uint_as_float(v[4 + u]), __uint_as_float(v[5 + u]));
        const float2 tg = tanh_pair(__uint_as_float(v[8 + u]), __uint_as_float(v[9 + u]));
        const float2 to = tanh_pair(__uint_as_float(v[12 + u]), __uint_as_float(v[13 + u]));
        const float c0 = fmaf(fmaf(0.5f, tf.x, 0.5f), __uint_as_float(c[u]), fmaf(0.5f, ti.x, 0.5f) * tg.x);
        const float c1 = fmaf(fmaf(0.5f, tf.y, 0.5f), __uint_as_float(c[u + 1]), fmaf(0.5f, ti.y, 0.5f) * tg.y);
        c[u] = __float_as_uint(c0); c[u + 1] = __float_as_uint(c1);
        const float2 tc = tanh_pair(c0, c1);
        hp[u >> 1] = pack_bf16x2(fmaf(0.5f, to.x, 0.5f) * tc.x, fmaf(0.5f, to.y, 0.5f) * tc.y);
    }
}
// one 64-column half of a gate part = 4 groups = 16 hidden units of this thread's env row; t_c = TMEM address of their cell
// states; `early` = arrive on the tile's A/D barrier as soon as the last accumulator columns are in registers (the next part of
// the layer may then overwrite D); b = the half's 64 gate biases (kBias)
template <bool kBias>
__device__ __forceinline__ void lstm_half(uint32_t t_d, uint32_t t_c, uint32_t* hp, bool early, uint32_t bar, const float* b) {
#pragma unroll
    for (int g = 0; g < 4; ++g) {                    // (two groups per TMEM round trip, LDTM.x32 + x8, measured no faster)
        uint32_t v[16], c[4];
        tmem_ld16(t_d + (uint32_t)(g * 16), v);
        tmem_ld4(t_c + (uint32_t)(g * 4), c);
        tmem_ld_wait();
        if (g == 3 && early) { tc_fence_before(); mbar_arrive(bar); }
        lstm_group<kBias>(v, c, hp + g * 2, b + g * 16);
        tmem_st4(t_c + (uint32_t)(g * 4), c);
    }
}

// One state frame x_t of a whole tile (128 rows x in_dim floats) crosses from global memory COALESCED: the 256 epilogue threads
// of the tile walk the (row, feature pair) grid in memory order with 8-byte loads, so a warp-wide request touches ~3 cache
// lines.  (One thread reading its own row's 26 floats costs 32 L1 wavefronts per load instruction -- measured, that alone was
// 80 % of an LSTM step; 4-byte cp.async copies are no better, the LSU serialises them per lane.  And with 220 KB of the SM's
// 228 KB configured as shared memory there is no L1 left to absorb register spills, so this kernel must not spill: that is why
// the cell state lives in tensor memory.)  The values wait in registers while the step's MMAs and gate math run, then go through
// a shared-memory transpose (packed bf16 pairs, row stride kXStride words) to the thread that owns the row.  Pair in_dim / 2 of
// every row is the constant (1, 1) the two bias columns of the weight image multiply; the rest of the 16 pairs is zero (written
// once at kernel start).
constexpr int kXRaw = 8;                       // ceil(128 * 15 / 256) feature pairs per thread
constexpr int kXStride = 20;                   // words per row in shared memory: 16 used, 80-byte rows keep LDS.128 conflict-free
constexpr int kXBytes = 2 * kTileM * kXStride * 4;
constexpr int kCriticSmemBytes = kTcSmemBytes + kXBytes;
constexpr int kCriticSeqSmemBytes = kTcSmemBytes;   // layers above the bottom stage no frames

// idx = tt + 256 k -> (row, pair), walked incrementally (256 = q pairs + rem)
struct FrameWalk {
    int row, j, q, rem, pairs;
    __device__ __forceinline__ FrameWalk(int tt, int pairs_, float inv_pairs) : pairs(pairs_) {
        row = (int)(((float)tt + 0.5f) * inv_pairs); j = tt - row * pairs;
        q = (int)(256.5f * inv_pairs); rem = 256 - q * pairs;
    }
    __device__ __forceinline__ void next() { row += q; j += rem; if (j >= pairs) { j -= pairs; row += 1; } }
};
// loads this thread's feature pairs of frame ts and packs them to bf16 at once (8 registers stay live across the gate math; the
// load latency overlaps the wait for the step's accumulator); also pulls frame ts + 1 into L2
__device__ __forceinline__ void frame_load(const float* states, long long tile_row0, int ts, int T, int in_dim, size_t row_floats, int n_rows,
                                           int tt, float inv_pairs, uint32_t (&xp)[kXRaw]) {
    FrameWalk w(tt, in_dim >> 1, inv_pairs);
    const float* base = states + tile_row0 * row_floats + (size_t)ts * in_dim;
    const int rows_left = (int)min((long long)kTileM, (long long)n_rows - tile_row0);
    float2 raw[kXRaw];
#pragma unroll
    for (int k = 0; k < kXRaw; ++k) {
        const float2* src = reinterpret_cast<const float2*>(base + (size_t)w.row * row_floats) + w.j;
        raw[k] = make_float2(0.f, 0.f);
        if (w.row < rows_left) {
            raw[k] = __ldcg(src);               // read once: no point allocating in the ~10 KB of L1 left next to 217 KB of shared memory
            if (ts + 1 < T && (k & 1) == 0) prefetch_l2(reinterpret_cast<const float*>(src) + in_dim);
        }
        w.next();
    }
#pragma unroll
    for (int k = 0; k < kXRaw; ++k) xp[k] = pack_bf16x2(raw[k].x, raw[k].y);
}
__device__ __forceinline__ void frame_store(uint32_t* s_xt, int in_dim, int tt, float inv_pairs, const uint32_t (&xp)[kXRaw]) {
    FrameWalk w(tt, in_dim >> 1, inv_pairs);
#pragma unroll
    for (int k = 0; k < kXRaw; ++k) {
        if (w.row < kTileM) s_xt[w.row * kXStride + w.j] = xp[k];
        w.next();
    }
}
// all 256 epilogue threads of tile slot t
__device__ __forceinline__ void tile_barrier(int t) { asm volatile("bar.sync %0, %1;" ::"r"(1 + t), "r"(256) : "memory"); }
// features [16 ch, 16 ch + 16) of row r as 8 packed bf16 pairs
__device__ __forceinline__ void frame_read(const uint32_t* s_xt, int r, int ch, uint32_t* pk) {
    const uint4 a = *reinterpret_cast<const uint4*>(s_xt + r * kXStride + ch * 8);
    const uint4 b = *reinterpret_cast<const uint4*>(s_xt + r * kXStride + ch * 8 + 4);
    pk[0] = a.x; pk[1] = a.y; pk[2] = a.z; pk[3] = a.w; pk[4] = b.x; pk[5] = b.y; pk[6] = b.z; pk[7] = b.w;
}

// Hand-off between stacked layers: thread (r, ch) of layer k - 1 produces hp[16] = the 16 hidden units it owns in gate part 0,
// then the 16 of part 1 (zero where the part has no columns for it), as packed bf16 pairs; thread (r, ch) of layer k reads exactly
// these 64 bytes as its 16 packed columns of x_t (the W_ih columns of layer k are permuted to match, seq_unit).  Per (tile, step,
// ch) they are 4 x 16 bytes, each a 128-row array: a warp's 16-byte access covers 512 contiguous bytes.  seq_idx is the uint4
// index of access 0; access i is kTileM further on.
__device__ __forceinline__ size_t seq_idx(int tile, int ts, int T, int ch, int r) {
    return (size_t)(((tile * T + ts) * 2 + ch) * 4) * kTileM + r;
}
__device__ __forceinline__ void seq_load(const uint4* ws, int tile, int ts, int T, int ch, int r, uint32_t (&x)[16]) {
    const uint4* src = ws + seq_idx(tile, ts, T, ch, r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint4 v = __ldcg(src + i * kTileM);
        x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
    }
}
__device__ __forceinline__ void seq_store(uint4* ws, int tile, int ts, int T, int ch, int r, const uint32_t (&h)[16]) {
    uint4* dst = ws + seq_idx(tile, ts, T, ch, r);
#pragma unroll
    for (int i = 0; i < 4; ++i) __stcg(dst + i * kTileM, make_uint4(h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]));
}

// c_0 = 0 for a fresh tile (fp32, unit k -> column kAColC + k).  Before the first tile, or after the MLP, the two halves of a row
// may split the 64 columns any way: every cell access of the previous tile is ordered before by the bar_a arrivals the MLP's MMAs
// waited for and the bar_d wait on them.  kOwnCells: only the columns of
// the units lstm_half gives this half (16 ch .. + 15 and 32 + 16 ch .. + 15), for staging right after the tile's last gate math,
// while the row's other half may still read and write its own cells.
template <bool kOwnCells>
__device__ __forceinline__ void stage_zero_cells(uint32_t t_a, int ch, const uint32_t (&z)[16]) {
    if constexpr (kOwnCells) {
        tmem_st16(t_a + (uint32_t)(kAColC + ch * 16), z);
        tmem_st16(t_a + (uint32_t)(kAColC + 32 + ch * 16), z);
    } else {
        tmem_st16(t_a + (uint32_t)(kAColC + ch * 32), z);
        tmem_st16(t_a + (uint32_t)(kAColC + ch * 32 + 16), z);
    }
}
// A operand of a fresh tile: h_0 = 0 in columns [0, 32), x_0 in [32, 48), zeros in [48, 64) (TMEM is never read uninitialised:
// the weight rows of the padding are zero, but 0 * NaN is NaN), and the cell state c_0 = 0 as fp32 in the columns [64, 128) the
// LSTM phase does not use as an operand (stage_zero_cells)
template <bool kOwnCells = false>
__device__ __forceinline__ void stage_new_tile(uint32_t t_a, int ch, const uint32_t* x0) {
    uint32_t z[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) z[j] = 0u;
    tmem_st16(t_a + (uint32_t)(kAColH + ch * 16), z);
    tmem_st8(t_a + (uint32_t)(kAColX + ch * 8), x0);
    tmem_st8(t_a + (uint32_t)(kAColX + 16 + ch * 8), z);
    stage_zero_cells<kOwnCells>(t_a, ch, z);
}
// the same for a layer above the bottom: x_0 = h^{k-1}_0 fills the whole x chunk [32, 64), 16 packed columns per thread
template <bool kOwnCells = false>
__device__ __forceinline__ void stage_new_tile_seq(uint32_t t_a, int ch, const uint32_t (&x0)[16]) {
    uint32_t z[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) z[j] = 0u;
    tmem_st16(t_a + (uint32_t)(kAColH + ch * 16), z);
    tmem_st16(t_a + (uint32_t)(kAColX + ch * 16), x0);
    stage_zero_cells<kOwnCells>(t_a, ch, z);
}

// kSeqIn: x_t is h^{k-1}_t from p.seq_in (an LSTM layer above the bottom) instead of the state frames; its bias is added in the
// epilogue.  kSeqOut: h_t of every step goes to p.seq_out and the kernel stops after the T steps (a layer below the top: no MLP, no
// output part).  <false, false> is the one-layer critic.
template <bool kSeqIn, bool kSeqOut>
__global__ void __launch_bounds__(kTcThreads, 1) critic_tc_kernel(const CriticTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    const TcSmem sm(smem_raw);
    const uint32_t bar_lstm = sm.bar_own;                             // the resident LSTM weight image has landed
    uint32_t* s_x = reinterpret_cast<uint32_t*>(sm.base + kTcSmemBytes - 1024);     // [2 tiles][128 rows][kXStride] staged state frames (bf16 pairs)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tps = p.tiles_per_cta;                                 // 2, or 1 when there are fewer tiles than SMs (small batches: one tile per CTA halves the latency)
    const int num_pairs = (p.num_tiles + tps - 1) / tps;
    const int T = p.seq_len;
    const int n_sched = kSeqOut ? T : T + p.n_hidden + 1;            // T LSTM steps, the MLP hidden layers, the output part

    // constant part of the staged frames: pair in_dim / 2 = (1, 1) (the bias columns), zero elsewhere
    if constexpr (!kSeqIn)
        for (int i = threadIdx.x; i < 2 * kTileM * kXStride; i += kTcThreads) s_x[i] = (i % kXStride == (p.in_dim >> 1)) ? 0x3F803F80u : 0u;
    const uint32_t tmem0 = sm.setup(warp, p.bias, [&] { mbar_init(bar_lstm, 1); });

    if (warp == 0) {
        // ===================== weight producer.  The LSTM image (<= 64 KB: [W_hh | W_ih] for 4H <= 256 gate rows) is the same for
        // every time step of every tile: it is loaded ONCE into the last 64 KB slot and stays there instead of being re-streamed five
        // times per pair (5x less L2 -> SM traffic in the LSTM phase; time-neutral at the measured sizes).  The MLP layers
        // stream through the remaining kRing slots: per pair, per layer, per 128-row part one slot.
        {
            const int n = p.layer[0].n;
            const uint8_t* img = p.wimg + p.layer[0].img_off;
            if (elect_one_sync()) {
                mbar_arrive_expect_tx(bar_lstm, (uint32_t)n * 128u * 2u);
                for (int h0 = 0, part = 0; h0 < n; h0 += kPartN, ++part)
                    for (int c = 0; c < 2; ++c)
                        bulk_g2s(sm.ring + kRing * kSlotBytes + (part * 2 + c) * kChunkBytes, img + ((size_t)c * n + h0) * 128u,
                                 (uint32_t)min(kPartN, n - h0) * 128u, bar_lstm);
            }
            __syncwarp();
        }
        if constexpr (!kSeqOut) {
            uint32_t slot = 0, phase = 0;
            for (int pair = blockIdx.x; pair < num_pairs; pair += gridDim.x)
                for (int l = 1; l <= p.n_hidden + 1; ++l) produce_layer(sm, p.wimg, p.layer[l], kRing, slot, phase);
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: the two tiles alternate part by part and share every weight slot.  An LSTM part of the
        // bottom layer reads 32 K values of x_t (issue_part's `lstm`), one of the layers above reads all 64.
        uint32_t slot = 0, phase = 0, a_phase = 0;
        int dbg_n = lane == 0 ? 0 : kDbgCap;
        const uint64_t bdesc0 = umma_desc_sw128(sm.ring);
        mbar_wait(bar_lstm, 0u);                                       // the resident LSTM image
        for (int pair = blockIdx.x; pair < num_pairs; pair += gridDim.x) {
            const int nt = min(tps, p.num_tiles - tps * pair);
            // ---- LSTM steps: the weights are resident, so the two tiles' chains need not advance in lock step.  Their parts are
            // issued as the tiles become ready (the epilogue side is unchanged: per tile, wait bar_d / arrive bar_a), and tile 1's
            // chain is started p.stagger cycles after tile 0's, so that one tile's gate math (MUFU-bound: 4 warps per
            // scheduler when both tiles are in it) falls into the other's accumulator / frame-load / staging waits.
            int s_first = 0;
            if (p.stagger > 0 && nt == 2) {
                const int n = p.layer[0].n, parts = (n + kPartN - 1) / kPartN, total_parts = T * parts;
                int done0 = 0, done1 = 0;
                long long t0_start = 0;
                while (done0 < total_parts || done1 < total_parts) {
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        const int dn = t == 0 ? done0 : done1;
                        if (dn >= total_parts) continue;
                        if (t == 1 && dn == 0 && (done0 == 0 || clock64() - t0_start < (long long)p.stagger)) continue;
                        if (!mbar_test(sm.bar_a + 8 * t, (a_phase >> t) & 1u)) continue;
                        a_phase ^= (1u << t);
                        const int h0 = (dn % parts) * kPartN;
                        const uint32_t idesc = umma_idesc_bf16(kTileM, min(kPartN, n - h0));
                        const uint64_t bdesc = bdesc0 + (uint64_t)((kRing * kSlotBytes + (h0 / kPartN) * 2 * kChunkBytes) >> 4);
                        tc_fence_after();
                        TACO_DBG(0, dbg_n, 0x20 | t);
                        issue_part(tmem0 + (uint32_t)(t * kTmemSlot), bdesc, idesc, p.layer[0].kchunks, !kSeqIn, false, 0u, sm.bar_d + 8 * t);
                        TACO_DBG(0, dbg_n, 0x30 | t);
                        if (t == 0) { if (done0 == 0) t0_start = clock64(); ++done0; } else ++done1;
                    }
                    __nanosleep(20);
                }
                s_first = T;
            }
            for (int s = s_first; s < n_sched; ++s) {
                const int l = s < T ? 0 : s - T + 1;
                const int n = p.layer[l].n, kch = p.layer[l].kchunks;
                for (int h0 = 0; h0 < n; h0 += kPartN) {
                    const uint32_t idesc = umma_idesc_bf16(kTileM, min(kPartN, n - h0));
                    const bool ring = l != 0;                              // LSTM parts sit in the resident slot
                    const uint64_t bdesc = ring ? bdesc0 + (uint64_t)(slot * (kSlotBytes >> 4))
                                                : bdesc0 + (uint64_t)((kRing * kSlotBytes + (h0 / kPartN) * 2 * kChunkBytes) >> 4);
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        if (t < nt) {
                            mbar_wait(sm.bar_a + 8 * t, (a_phase >> t) & 1u); a_phase ^= (1u << t);
                            if (t == 0 && ring) mbar_wait(sm.bar_full + 8 * slot, phase);
                            tc_fence_after();
                            TACO_DBG(0, dbg_n, 0x20 | t);
                            issue_part(tmem0 + (uint32_t)(t * kTmemSlot), bdesc, idesc, kch, !ring && !kSeqIn, t == nt - 1 && ring, sm.bar_empty + 8 * slot,
                                       sm.bar_d + 8 * t);
                            TACO_DBG(0, dbg_n, 0x30 | t);
                        }
                    }
                    if (ring && ++slot == kRing) { slot = 0; phase ^= 1u; }
                }
            }
        }
    } else {
        // ===================== epilogue warps
        const EpiThread ep(warp, lane, tmem0, tps, p.num_tiles);
        const int t = ep.t, ch = ep.ch, r = ep.r;
        const uint32_t t_a = ep.t_a, t_d = ep.t_d;
        uint32_t d_phase = 0;
        int dbg_n = (ch == 0 && ep.quad == 0 && lane == 0) ? 0 : kDbgCap;
        const size_t row_floats = (size_t)T * p.in_dim;
        int tile = ep.tile;
        const int tile_step = ep.tile_step;
        const int tt = ((ep.e & 7) << 5) | lane;                       // index among the 256 epilogue threads of this tile
        const float inv_in = 1.0f / (float)(p.in_dim >> 1);           // 1 / feature pairs per frame
        uint32_t* s_xt = s_x + t * (kTileM * kXStride);
        if (tile < p.num_tiles) {
            if constexpr (kSeqIn) {
                uint32_t x0[16];
                seq_load(p.seq_in, tile, 0, T, ch, r, x0);
                stage_new_tile_seq(t_a, ch, x0);
            } else {
                uint32_t x0[8];
                uint32_t raw[kXRaw];
                frame_load(p.states, (long long)tile * kTileM, 0, T, p.in_dim, row_floats, p.n_rows, tt, inv_in, raw);
                frame_store(s_xt, p.in_dim, tt, inv_in, raw);
                tile_barrier(t);
                frame_read(s_xt, r, ch, x0);
                stage_new_tile(t_a, ch, x0);
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(sm.bar_a + 8 * t);
        }
        // the LSTM layer: n = 4H accumulator columns in parts of 128; this thread owns 16 hidden units of every part it has columns in
        const int n_g = p.layer[0].n;
        const bool g_two = n_g > kPartN;
        const bool g_mine0 = ch * 64 < min(n_g, kPartN);
        const bool g_mine1 = g_two && (kPartN + ch * 64 < n_g);
        const float* b_g = sm.bias + ch * 64;                           // kSeqIn: bias row 0, this thread's columns of gate part 0
        for (; tile < p.num_tiles; tile += tile_step) {
            const long long row = (long long)tile * kTileM + r;
            const bool valid = row < p.n_rows;
            const bool has_next = tile + tile_step < p.num_tiles;
            const long long row_next = row + (long long)tile_step * kTileM;
            const float* xs_next = p.states + row_next * row_floats;
            if (!kSeqIn && has_next && row_next < p.n_rows) prefetch_l2(xs_next + ch * 16);
            // ---- T LSTM steps
            for (int ts = 0; ts < T; ++ts) {
                // kSeqOut: nothing reads this tile's A operand after its last step, so that step stages the slot's next tile
                const bool next_tile = kSeqOut && ts + 1 == T;
                const bool have_x = ts + 1 < T || (next_tile && has_next);
                const int x_tile = next_tile ? tile + tile_step : tile, x_ts = next_tile ? 0 : ts + 1;
                uint32_t hp[16];
                uint32_t raw[kSeqIn ? 16 : kXRaw];
                TACO_DBG(1 + t, dbg_n, 0x08);
                // x_{t+1}: with one gate part the loads fly while the step's MMAs run; with two they are issued between the parts
                // (their latency then overlaps part 1's MMAs instead of delaying the drain of part 0)
                if (have_x && !g_two) {
                    if constexpr (kSeqIn) seq_load(p.seq_in, x_tile, x_ts, T, ch, r, raw);
                    else frame_load(p.states, (long long)x_tile * kTileM, x_ts, T, p.in_dim, row_floats, p.n_rows, tt, inv_in, raw);
                }
                mbar_wait(sm.bar_d + 8 * t, d_phase); d_phase ^= 1u;
                tc_fence_after();
                TACO_DBG(1 + t, dbg_n, 0x02);
                if (g_mine0) lstm_half<kSeqIn>(t_d, t_a + (uint32_t)(kAColC + ch * 16), hp, g_two, sm.bar_a + 8 * t, b_g);      // D drained: part 1 may start
                else if (g_two) { tc_fence_before(); mbar_arrive(sm.bar_a + 8 * t); }
                TACO_DBG(1 + t, dbg_n, 0x0A);
                if (have_x && g_two) {
                    if constexpr (kSeqIn) seq_load(p.seq_in, x_tile, x_ts, T, ch, r, raw);
                    else frame_load(p.states, (long long)x_tile * kTileM, x_ts, T, p.in_dim, row_floats, p.n_rows, tt, inv_in, raw);
                }
                TACO_DBG(1 + t, dbg_n, 0x09);
                if (g_two) {
                    mbar_wait(sm.bar_d + 8 * t, d_phase); d_phase ^= 1u;
                    tc_fence_after();
                    TACO_DBG(1 + t, dbg_n, 0x04);
                }
                if (g_mine1) lstm_half<kSeqIn>(t_d, t_a + (uint32_t)(kAColC + 32 + ch * 16), hp + 8, false, 0u, b_g + kPartN);
                if constexpr (kSeqOut) {                              // h_t to the layer above, zero for the units this thread lacks
                    if (!g_mine0)
#pragma unroll
                        for (int j = 0; j < 8; ++j) hp[j] = 0u;
                    if (!g_mine1)
#pragma unroll
                        for (int j = 8; j < 16; ++j) hp[j] = 0u;
                    seq_store(p.seq_out, tile, ts, T, ch, r, hp);
                }
                // every MMA of this step on this tile is complete: h_t over h_{t-1} (unit k -> packed column k / 2), x_{t+1} over x_t
                if (!next_tile) {
                    if (g_mine0) tmem_st8(t_a + (uint32_t)(kAColH + ch * 8), hp);
                    if (g_mine1) tmem_st8(t_a + (uint32_t)(kAColH + 16 + ch * 8), hp + 8);
                }
                TACO_DBG(1 + t, dbg_n, 0x0B);
                if (have_x) {
                    if (next_tile) tmem_st_wait();                    // this thread's cell stores of the step land before its c_0 = 0
                    if constexpr (kSeqIn) {                           // x_{t+1} is already in owner order
                        if (next_tile) stage_new_tile_seq<true>(t_a, ch, raw);
                        else tmem_st16(t_a + (uint32_t)(kAColX + ch * 16), raw);
                    } else {                                          // x_{t+1}: registers -> shared-memory transpose -> own row -> A operand
                        // every thread of the tile read x_t out of the staging buffer before it arrived on bar_a at the end of the
                        // previous step, and this step's MMAs needed all those arrivals: the buffer is free
                        uint32_t xn[8];
                        frame_store(s_xt, p.in_dim, tt, inv_in, raw);
                        tile_barrier(t);
                        frame_read(s_xt, r, ch, xn);
                        if (next_tile) stage_new_tile<true>(t_a, ch, xn);
                        else tmem_st8(t_a + (uint32_t)(kAColX + ch * 8), xn);
                    }
                }
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(sm.bar_a + 8 * t);
                TACO_DBG(1 + t, dbg_n, 0x05);
            }
            if constexpr (!kSeqOut) {
                // ---- MLP hidden layers
                for (int l = 1; l <= p.n_hidden; ++l)
                    hidden_layer<false>(ep, sm.bias, l, p.layer[l].n, sm.bar_a, sm.bar_d, d_phase, nullptr, dbg_n);
                // ---- output part (column 0 of 16): the next tile's A operand is staged before the value leaves
                uint32_t raw[kSeqIn ? 16 : kXRaw];
                if (has_next) {
                    if constexpr (kSeqIn) seq_load(p.seq_in, tile + tile_step, 0, T, ch, r, raw);
                    else frame_load(p.states, (long long)(tile + tile_step) * kTileM, 0, T, p.in_dim, row_floats, p.n_rows, tt, inv_in, raw);
                }
                mbar_wait(sm.bar_d + 8 * t, d_phase); d_phase ^= 1u;
                tc_fence_after();
                uint32_t v[4];
                if (ch == 0) { tmem_ld4(t_d, v); tmem_ld_wait(); }
                if (has_next) {
                    if constexpr (kSeqIn) {
                        stage_new_tile_seq(t_a, ch, raw);
                    } else {
                        uint32_t x0[8];
                        frame_store(s_xt, p.in_dim, tt, inv_in, raw);
                        tile_barrier(t);
                        frame_read(s_xt, r, ch, x0);
                        stage_new_tile(t_a, ch, x0);
                    }
                    tmem_st_wait();
                    tc_fence_before();
                    mbar_arrive(sm.bar_a + 8 * t);
                }
                if (ch == 0 && valid) p.value[row] = __uint_as_float(v[0]) + __ldg(p.b_out);
            }
        }
    }
    sm.teardown(warp, tmem0);
}

// LSTM weights (torch layout: w_ih (4H, In), w_hh (4H, H), gate row blocks i, f, g, o) -> two bf16 K-chunk images of n = 4H
// rows each in the SWIZZLE_128B K-major layout: chunk 0 = W_hh (K padded to 64), chunk 1 = W_ih (K padded to 64).  Image row
// r = 128 part + j holds gate (j % 16) / 4 of hidden unit 32 part + 4 (j / 16) + j % 4.  Columns in_dim / in_dim + 1 of the W_ih chunk
// hold b_ih + b_hh split into two bf16 halves (the kernel feeds 1.0 there); rows of the i, f, o gates are scaled by 1/2.
__device__ __forceinline__ int lstm_src_row(int r, int hidden) {
    const int part = r >> 7, j = r & 127;
    const int unit = part * 32 + (j >> 4) * 4 + (j & 3), gate = (j & 15) >> 2;
    return unit < hidden ? gate * hidden + unit : -1;
}
__global__ void pack_lstm_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, const float* __restrict__ b_ih,
                                 const float* __restrict__ b_hh, int hidden, int in_dim, int n, uint8_t* __restrict__ img) {
    const int total = 2 * n * 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int q = i & 7, r = (i >> 3) % n, c = (i >> 3) / n;
        const int src = lstm_src_row(r, hidden);
        const float* w = c == 0 ? w_hh : w_ih;
        const int k = c == 0 ? hidden : in_dim;
        const float scale = (src >= 0 && src / hidden == 2) ? 1.0f : 0.5f;      // i, f, o rows: sigmoid(x) = 0.5 + 0.5 tanh(x / 2)
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int kk = q * 8 + j;
            f[j] = (src >= 0 && kk < k) ? scale * w[(size_t)src * k + kk] : 0.0f;
            if (c == 1 && src >= 0 && (kk == in_dim || kk == in_dim + 1)) {     // bias columns: bf16 hi part, then the bf16 of the rest
                const float b = scale * (b_ih[src] + b_hh[src]);
                const float hi = __bfloat162float(__float2bfloat16_rn(b));
                f[j] = kk == in_dim ? hi : b - hi;
            }
        }
        const uint4 pk = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
        *reinterpret_cast<uint4*>(img + (size_t)c * n * 128 + sw128_off(r, q)) = pk;
    }
}
// hidden unit of the layer below whose h sits at K position k of the x chunk in the hand-off order (seq_idx): thread half
// ch = k / 32 holds its 16 units of gate part 0, then its 16 of part 1
__device__ __forceinline__ int seq_unit(int k) {
    const int q = k & 31;
    return 16 * (k >> 5) + (q < 16 ? q : q + 16);
}
// An LSTM layer k >= 1 (w_ih and w_hh both (4H, H)): the rows as in pack_lstm_kernel, chunk 0 = W_hh, chunk 1 = W_ih with its
// columns in the hand-off order, no bias columns; bias[r] = the scaled b_ih + b_hh of image row r (accumulator column r), which
// the epilogue adds (bias row 0 of the layer's launch).
__global__ void pack_lstm_seq_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, const float* __restrict__ b_ih,
                                     const float* __restrict__ b_hh, int hidden, int n, uint8_t* __restrict__ img, float* __restrict__ bias) {
    const int total = 2 * n * 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int q = i & 7, r = (i >> 3) % n, c = (i >> 3) / n;
        const int src = lstm_src_row(r, hidden);
        const float* w = c == 0 ? w_hh : w_ih;
        const float scale = (src >= 0 && src / hidden == 2) ? 1.0f : 0.5f;
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int kk = c == 0 ? q * 8 + j : seq_unit(q * 8 + j);
            f[j] = (src >= 0 && kk < hidden) ? scale * w[(size_t)src * hidden + kk] : 0.0f;
        }
        const uint4 pk = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
        *reinterpret_cast<uint4*>(img + (size_t)c * n * 128 + sw128_off(r, q)) = pk;
        if (c == 0 && q == 0) bias[r] = src >= 0 ? scale * (b_ih[src] + b_hh[src]) : 0.0f;
    }
}

}  // namespace critic
}  // namespace taco
