// mortal_b200 — action selection for engines on the device path (mortal/engine.py MortalEngine._react_batch after the network,
// with mortal/model.py DQN.forward's dueling combination), written straight into the environment's per-row buffers.
//
// k_select_actions: one warp per decision row i of an engine's batch, environment row r = rows[i] (or i). Lane l owns actions l and
// l + 32 (< 46). q = v + a - mean(a over legal), -inf on illegal actions; greedy = argmax q, lowest index on ties (torch.argmax).
// With epsilon > 0 the row is greedy with probability 1 - epsilon, otherwise an action is drawn from softmax(q / temp) over the legal
// actions restricted to the top-p nucleus (engine.py sample_top_p): an action is kept when the probability mass ranked strictly above
// it (probability descending, lower index first on ties) is <= top_p; top_p >= 1 keeps every legal action, top_p <= 0 is the argmax.
// The randomness is Philox4x32-10 keyed by the engine's seed with the counter (table, step of the table, seat byte): rows are appended
// to the environment through an atomic counter, so their order changes between runs, but each decision's draw does not.
//
// k_split_rows: stable compaction of a step's rows into one index list per agent (agent_of[table * 4 + seat] = 0 or 1), one CTA.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace mjx_sel {

constexpr int NA = 46;

struct U4 { uint32_t x, y, z, w; };

__device__ __forceinline__ U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
        const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
        c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }  // [0, 1)

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

struct SelectArgs {
    const float* v; long long v_stride;   // [n] value, f32
    const float* a; long long a_stride;   // [n, 46] advantage, f32
    const int* rows;                      // [n] environment row of batch row i (nullptr: i)
    const int* count;                     // device: rows i < *count are live
    int n_max;
    const uint8_t* masks;                 // [row_cap, 46] legal-action mask of the environment
    const int* row_table; const uint32_t* row_step; const uint8_t* row_seat;
    uint32_t seed_lo, seed_hi;
    int table_offset;
    float epsilon, inv_temp, top_p;
    int64_t* actions;                     // [row_cap] written at rows[i]
    float* q_out;                         // [row_cap, 46]
    uint8_t* greedy;                      // [row_cap] (optional)
};

__global__ void __launch_bounds__(256) k_select_actions(SelectArgs A) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int n = min(*A.count, A.n_max);
    const int j1 = lane + 32;
    const bool has1 = j1 < NA;
    const float NEG_INF = __int_as_float(0xff800000);
    for (int i = warp; i < n; i += nwarps) {
        const int r = A.rows ? A.rows[i] : i;
        const bool m0 = A.masks[(size_t)r * NA + lane] != 0, m1 = has1 && A.masks[(size_t)r * NA + j1] != 0;
        const float* ai = A.a + (size_t)i * A.a_stride;
        const float a0 = ai[lane], a1 = has1 ? ai[j1] : 0.f;
        const float vv = A.v[(size_t)i * A.v_stride];
        const int n_legal = __popc(__ballot_sync(0xffffffffu, m0)) + __popc(__ballot_sync(0xffffffffu, m1));
        const float mean = warp_sum((m0 ? a0 : 0.f) + (m1 ? a1 : 0.f)) / (float)n_legal;
        const float q0 = m0 ? (vv + a0) - mean : NEG_INF, q1 = m1 ? (vv + a1) - mean : NEG_INF;
        // argmax, lowest index on ties
        float best = q0;
        int bi = lane;
        if (q1 > best) { best = q1; bi = j1; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        int action = bi;
        bool is_greedy = true;
        if (A.epsilon > 0.f) {
            const U4 rnd = philox4x32_10(U4{(uint32_t)(A.table_offset + A.row_table[r]), A.row_step[r], (uint32_t)A.row_seat[r], 0u},
                                         A.seed_lo, A.seed_hi);
            is_greedy = u01(rnd.x) < 1.f - A.epsilon;
            if (!is_greedy && A.top_p > 0.f) {
                // softmax(q / temp) over the legal actions, the row max subtracted first (temp = 0.05 scales q by 20)
                const float lmax = best * A.inv_temp;
                const float w0 = m0 ? expf(q0 * A.inv_temp - lmax) : 0.f, w1 = m1 ? expf(q1 * A.inv_temp - lmax) : 0.f;
                const float z = warp_sum(w0 + w1);
                const float p0 = w0 / z, p1 = w1 / z;
                float k0 = p0, k1 = p1;
                if (A.top_p < 1.f) {
                    // mass ranked strictly above each action: probability descending, lower index first on ties
                    float b0 = 0.f, b1 = 0.f;
                    for (int k = 0; k < NA; k++) {
                        const float pk = __shfl_sync(0xffffffffu, k < 32 ? p0 : p1, k & 31);
                        if (pk > p0 || (pk == p0 && k < lane)) b0 += pk;
                        if (pk > p1 || (pk == p1 && k < j1)) b1 += pk;
                    }
                    if (!(m0 && b0 <= A.top_p)) k0 = 0.f;
                    if (!(m1 && b1 <= A.top_p)) k1 = 0.f;
                }
                // inverse-CDF draw over the kept mass in action order
                float s0 = k0, s1 = k1;  // inclusive prefix sums over lanes, first then second half
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const float t0 = __shfl_up_sync(0xffffffffu, s0, o), t1 = __shfl_up_sync(0xffffffffu, s1, o);
                    if (lane >= o) { s0 += t0; s1 += t1; }
                }
                const float half = __shfl_sync(0xffffffffu, s0, 31);
                s1 += half;
                const float total = __shfl_sync(0xffffffffu, s1, 31);
                const float target = u01(rnd.y) * total;
                const unsigned hit0 = __ballot_sync(0xffffffffu, k0 > 0.f && s0 > target);
                const unsigned hit1 = __ballot_sync(0xffffffffu, k1 > 0.f && s1 > target);
                if (hit0) action = __ffs(hit0) - 1;
                else if (hit1) action = 32 + __ffs(hit1) - 1;
                else {  // target rounded up to the total: the last kept action
                    const unsigned kept0 = __ballot_sync(0xffffffffu, k0 > 0.f), kept1 = __ballot_sync(0xffffffffu, k1 > 0.f);
                    action = kept1 ? 32 + 31 - __clz(kept1) : (kept0 ? 31 - __clz(kept0) : bi);
                }
            }
        }
        float* qo = A.q_out + (size_t)r * NA;
        qo[lane] = q0;
        if (has1) qo[j1] = q1;
        if (lane == 0) {
            A.actions[r] = action;
            if (A.greedy) A.greedy[r] = is_greedy;
        }
    }
}

constexpr int SPLIT_THREADS = 1024;
__global__ void __launch_bounds__(SPLIT_THREADS) k_split_rows(const int* __restrict__ row_table, const uint8_t* __restrict__ row_seat,
                                                             const int* __restrict__ count, const uint8_t* __restrict__ agent_of,
                                                             int* __restrict__ rows0, int* __restrict__ rows1, int* __restrict__ counts) {
    __shared__ int warp_ones[SPLIT_THREADS / 32];
    __shared__ int base_ones;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int n = *count;
    int done_ones = 0;  // rows of agent 1 in earlier chunks
    for (int base = 0; base < n; base += SPLIT_THREADS) {
        const int i = base + threadIdx.x;
        const bool live = i < n;
        const bool one = live && agent_of[row_table[i] * 4 + (row_seat[i] & 3)] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, one);
        if (lane == 0) warp_ones[w] = __popc(bal);
        __syncthreads();
        if (w == 0) {
            const int x = warp_ones[lane];
            int s = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, s, o);
                if (lane >= o) s += t;
            }
            warp_ones[lane] = s - x;  // exclusive prefix over the warps
            if (lane == 31) base_ones = s;
        }
        __syncthreads();
        const int ones_before = done_ones + warp_ones[w] + __popc(bal & ((1u << lane) - 1u));
        if (live) {
            if (one) rows1[ones_before] = i;
            else rows0[i - ones_before] = i;
        }
        done_ones += base_ones;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        counts[0] = n - done_ones;
        counts[1] = done_ones;
    }
}

}  // namespace mjx_sel
