// Episode records and per-task summaries of training rollouts (taco_env_attach_rollout_episodes, include/taco_b200.h): one launch
// per rollout walks the rollout ring's result rows (rew_rows / done_rows / time_out_rows, written by the step kernel) that have not
// been scanned yet.  No launch is added to the step loop and the step kernel is not touched.
//
// Per-env planes carried from one scan to the next: ret (f32, the running return), len (i32, steps of the running episode) and
// live (u8).  live = 1: the scans saw the running episode start (attach / reset_all / ring attach / rewind over unscanned rows:
// the env had reset_buf != 0; afterwards: every episode after one the scans saw end), so no record holds a partial sum.
#pragma once
#include <stdint.h>

#include "../../include/taco_b200.h"

namespace taco {

static_assert(sizeof(TacoRolloutEpisode) == 24, "TacoRolloutEpisode is written as three 8-byte words");
static_assert(TACO_EPISODE_SUMMARY_WORDS == 15, "3 tasks x [episodes, time-outs, sum length, sum ret, sum ret^2]");

constexpr int kScanBlock = 256;
constexpr int kSummaryStride = 16;   // doubles per block partial (15 used; 128 B)
constexpr int kRowBatch = 8;         // rows whose loads a thread issues together (one 4-byte load per row in flight is latency-bound)

struct RolloutScanParams {
    const float* rew;                // row k0 of the ring's rows; row k of env i at [k * n + i]
    const float* done;
    const uint8_t* tout;
    int n, rows;
    uint32_t step0;                  // step index of row k0 (absolute, or the offset to *step_base in graph mode)
    const uint32_t* step_base;
    long long env_offset, mix_n1, mix_n2;
    int task_mode;
    float* ret;
    int* len;
    uint8_t* live;
    TacoRolloutEpisode* rec;
    unsigned long long* count;
    unsigned long long capacity;
    double* partial;                 // gridDim.x x kSummaryStride
    unsigned int* blocks_done;       // 0 between launches
    double* summary;                 // TACO_EPISODE_SUMMARY_WORDS
};

// the start rule: an env starts a whole episode with its next step exactly when reset_buf != 0 now (lazy reset, DESIGN.md 3.4)
__global__ void rollout_episodes_init_kernel(const long long* reset_buf, int n, float* ret, int* len, uint8_t* live) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ret[i] = 0.f;
    len[i] = 0;
    live[i] = reset_buf[i] != 0 ? 1 : 0;
}

// the 15 summary words of one block in fixed order: a shuffle-down tree per warp, then the warps in order; valid in threads 0..14.
// s: (kScanBlock / 32) x kSummaryStride doubles
__device__ __forceinline__ double block_summary_word(const double (&v)[TACO_EPISODE_SUMMARY_WORDS], double (*s)[kSummaryStride]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int w = 0; w < TACO_EPISODE_SUMMARY_WORDS; ++w) {
        double x = v[w];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        if (lane == 0) s[warp][w] = x;
    }
    __syncthreads();
    double r = 0.0;
    if (threadIdx.x < TACO_EPISODE_SUMMARY_WORDS)
        for (int k = 0; k < kScanBlock / 32; ++k) r += s[k][threadIdx.x];
    return r;
}

// One thread per env, kScanBlock threads per block.
// Pass 1 counts the records each thread will append (done rows only), a block scan gives every thread its offset and one 64-bit
// atomicAdd per block its base: slots at or past `capacity` are dropped but counted.  Pass 2 walks the rows in step order with
// ret = __fadd_rn(ret, rew) (the step kernel's ep_ret order) and writes the records; it loads kRowBatch rows at a time.
// Summary: each thread sums its own episodes in step order in float64, the block reduces in a fixed tree order into a partial, and
// the last block to finish reduces the partials in block order, so the summary is bit-identical for the same rows whatever the
// launch timing or the record order.
__global__ void __launch_bounds__(kScanBlock) rollout_episodes_scan_kernel(const RolloutScanParams p) {
    __shared__ double s_red[kScanBlock / 32][kSummaryStride];
    __shared__ int s_warp[kScanBlock / 32];
    __shared__ unsigned long long s_base;
    __shared__ bool s_last;
    const int i = blockIdx.x * kScanBlock + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool active = i < p.n;
    const size_t n = (size_t)p.n;

    // ---- pass 1: records of this thread
    bool live = active && p.live[i] != 0;
    int emits = 0;
    if (active) {
        int nd = 0;
#pragma unroll kRowBatch
        for (int k = 0; k < p.rows; ++k) nd += p.done[k * n + i] != 0.f ? 1 : 0;
        emits = nd - ((!live && nd > 0) ? 1 : 0);
    }
    int incl = emits;                                          // inclusive warp scan
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int w = 0; w < kScanBlock / 32; ++w) { const int c = s_warp[w]; s_warp[w] = tot; tot += c; }
        s_base = tot ? atomicAdd(p.count, (unsigned long long)tot) : 0ull;
    }
    __syncthreads();
    unsigned long long slot = s_base + (unsigned long long)(s_warp[warp] + incl - emits);

    // ---- pass 2: returns, lengths, records, per-thread summary
    int task = p.task_mode;
    double c_ep = 0.0, c_to = 0.0, c_len = 0.0, c_ret = 0.0, c_ret2 = 0.0;
    if (active) {
        const long long gid = p.env_offset + i;
        if (task == TACO_TASK_MIX) task = gid < p.mix_n1 ? TACO_TASK_POS : (gid < p.mix_n2 ? TACO_TASK_ROTATE : TACO_TASK_FLIP);
        const uint32_t step0 = p.step0 + (p.step_base ? __ldg(p.step_base) : 0u);
        float ret = p.ret[i];
        int len = p.len[i];
        for (int kb = 0; kb < p.rows; kb += kRowBatch) {
            float rw[kRowBatch], dn[kRowBatch];
#pragma unroll
            for (int u = 0; u < kRowBatch; ++u) {
                const bool in = kb + u < p.rows;
                rw[u] = in ? p.rew[(kb + u) * n + i] : 0.f;
                dn[u] = in ? p.done[(kb + u) * n + i] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < kRowBatch; ++u) {
                const int k = kb + u;
                if (k >= p.rows) break;
                ret = __fadd_rn(ret, rw[u]);
                len += 1;
                if (dn[u] != 0.f) {
                    if (live) {
                        const int tout = p.tout[k * n + i] != 0 ? 1 : 0;
                        if (slot < p.capacity) {
                            long long* o = reinterpret_cast<long long*>(p.rec + slot);
                            o[0] = gid;
                            o[1] = (long long)(((unsigned long long)(uint32_t)len << 32) | (step0 + (uint32_t)k));
                            o[2] = (long long)(((unsigned long long)__float_as_uint(ret) << 32) |
                                               ((uint32_t)task | ((uint32_t)tout << 16)));
                        }
                        slot += 1;
                        c_ep += 1.0;
                        c_to += (double)tout;
                        c_len += (double)len;
                        c_ret += (double)ret;
                        c_ret2 += (double)ret * (double)ret;
                    }
                    ret = 0.f;
                    len = 0;
                    live = true;
                }
            }
        }
        p.ret[i] = ret;
        p.len[i] = len;
        p.live[i] = live ? 1 : 0;
    }

    // ---- block partial: 3 tasks x 5 sums
    double v[TACO_EPISODE_SUMMARY_WORDS];
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        v[t * 5 + 0] = task == t ? c_ep : 0.0;
        v[t * 5 + 1] = task == t ? c_to : 0.0;
        v[t * 5 + 2] = task == t ? c_len : 0.0;
        v[t * 5 + 3] = task == t ? c_ret : 0.0;
        v[t * 5 + 4] = task == t ? c_ret2 : 0.0;
    }
    const double part = block_summary_word(v, s_red);
    if (threadIdx.x < TACO_EPISODE_SUMMARY_WORDS) p.partial[(size_t)blockIdx.x * kSummaryStride + threadIdx.x] = part;

    // ---- the last block reduces the partials in block order
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(p.blocks_done, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
#pragma unroll
    for (int w = 0; w < TACO_EPISODE_SUMMARY_WORDS; ++w) {
        double acc = 0.0;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += kScanBlock) acc += __ldcg(p.partial + (size_t)b * kSummaryStride + w);
        v[w] = acc;
    }
    __syncthreads();                                           // s_red is reused
    const double total = block_summary_word(v, s_red);
    if (threadIdx.x < TACO_EPISODE_SUMMARY_WORDS) p.summary[threadIdx.x] = total;
    if (threadIdx.x == 0) *p.blocks_done = 0u;                 // ready for the next launch (graph replays included)
}

}  // namespace taco
