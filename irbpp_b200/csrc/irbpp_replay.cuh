// irbpp_replay.cuh -- prioritized n-step replay for N bins on the device (SURVEY.md 8(f)2).
//
// Reference: main.py:61-63 builds one ReplayMemory (memory.py:95-208) per bin and trainer.py:184-186 appends to each
// of them from a Python loop.  Here the N memories are N banks of one device allocation (include/irbpp.h
// irbpp_replay_banks) and every operation is one launch over all banks:
//   append  memory.py:58-69,110-113  one CTA per bank: the state row, the slot's action / reward / nonterminal, the
//           new leaf (= the bank's running max) and its ancestors, index / full / t;
//   sample  memory.py:162-203       one CTA per sampled bank, one warp per stratified draw: lane 0 descends and
//           retries, the warp gathers the n-step window; the CTA normalises the weights by the bank's maximum;
//   update  memory.py:206-208,53-56 one CTA: leaf writes in batch order (a later duplicate wins), then the
//           ancestors of every touched leaf and the bank maxima.
// Sum trees keep the reference's heap of 2C-1 float32 nodes for any C (leaves C-1 .. 2C-2, no padding to a power of
// two): every internal node is fl(left + right), so a tree is a function of its leaves and recomputing ancestors in any
// order reproduces the reference's nodes bit for bit.  Precision of the reference's sample path, as measured on it:
//   segment = p_total / batch and i * segment are float32 (0-d float32 tensors);
//   np.random.uniform(lo, hi) is lo + (hi - lo) * u in float64 (NumPy's legacy uniform);
//   `value <= sum_tree[left]` rounds the Python float to float32 before comparing, and `value - sum_tree[left]` is
//   float32, so the whole descent runs on fl32(value);
//   weights: `np.array(probs) / p_total` dispatches to Tensor.__rtruediv__, i.e. probs * (1 / p_total) in float32;
//   capacity * probs and ** -beta are float32 tensor ops (beta = 1 is a reciprocal).
// The library is built -fmad=false, so none of these is contracted into an FMA.
#pragma once
#include <stdint.h>

#include "../../include/irbpp.h"

namespace irbpp {

constexpr int REPLAY_APPEND_THREADS = 256;
constexpr int REPLAY_UPDATE_THREADS = 256;
constexpr int REPLAY_MAX_WARPS = 32;

// Kernel view of irbpp_replay_sample_args: the launch-time part only.
struct ReplaySampleParams {
    int32_t per;                   // draws per sampled bank (batch // N, or 1 when N > batch)
    int32_t n;                     // multi_step
    float scale[IRBPP_REPLAY_MAX_STEPS];   // n_step_scaling (memory.py:107) as float32
    float neg_beta;                // -priority_weight
    int32_t beta_is_one;
    uint64_t seed, counter;
    const double* u_table; int32_t max_attempts;
    int32_t* banks;                // [rows / per] the sampled banks: chosen beforehand, or written here (bank = CTA)
    int32_t choose;
    int64_t* tree_index; float* states; int64_t* actions; float* returns; float* next_states; float* nonterminals;
    float* weights; int32_t* error;
};

__host__ __device__ __forceinline__ uint64_t replay_mix(uint64_t seed, uint64_t a, uint64_t b, uint64_t c) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (a + 1) + 0xC2B2AE3D27D4EB4Full * (b + 1) + 0x165667B19E3779F9ull * (c + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;                         // splitmix64 finaliser
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// the 53-bit double in [0, 1) NumPy's random_standard_uniform builds from 64 random bits
__host__ __device__ __forceinline__ double replay_u01(uint64_t seed, uint64_t counter, uint32_t row, uint32_t attempt) {
    return (double)(replay_mix(seed, counter, row, attempt) >> 11) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ int replay_mod(int a, int c) { const int r = a % c; return r < 0 ? r + c : r; }

// memory.py:110-113 + SegmentTree.append (:58-69) for every bank whose `valid` is set (trainer.py:184-186).
__global__ void __launch_bounds__(REPLAY_APPEND_THREADS)
irbpp_replay_append_kernel(const irbpp_replay_banks Bk, const float* __restrict__ state, int64_t state_stride,
                           const int64_t* __restrict__ action, const float* __restrict__ reward,
                           const uint8_t* __restrict__ done, const uint8_t* __restrict__ valid, float reward_clip) {
    const int b = blockIdx.x;
    if (valid && !valid[b]) return;                                   // uniform in the CTA
    const int C = Bk.capacity, L = Bk.obs_len;
    const int slot = Bk.index[b];
    const float* src = state + (int64_t)b * state_stride;
    float* dst = Bk.states + ((int64_t)b * C + slot) * Bk.row_stride;     // row_stride % 4 == 0: 16-byte aligned rows
    const bool src_aligned = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0);
    const int nvec = Bk.row_stride >> 2;
    for (int v = threadIdx.x; v < nvec; v += blockDim.x) {
        const int e = v * 4;
        float4 q;
        if (src_aligned && e + 3 < L) {
            q = *reinterpret_cast<const float4*>(src + e);
        } else {
            q.x = e < L ? src[e] : 0.0f;         q.y = e + 1 < L ? src[e + 1] : 0.0f;
            q.z = e + 2 < L ? src[e + 2] : 0.0f; q.w = e + 3 < L ? src[e + 3] : 0.0f;
        }
        *reinterpret_cast<float4*>(dst + e) = q;
    }
    __syncthreads();                                                  // every thread has read index[b]
    if (threadIdx.x == 0) {
        const int64_t s = (int64_t)b * C + slot;
        Bk.actions[s] = (int64_t)(float)action[b];                    // stored in a float32 tensor (memory.py:32,63)
        float r = reward[b];
        if (reward_clip > 0.0f) { r = r < reward_clip ? r : reward_clip; r = r > -reward_clip ? r : -reward_clip; }  // trainer.py:181-182
        Bk.rewards[s] = r;
        Bk.nonterminals[s] = done[b] ? 0 : 1;
        float* tree = Bk.tree + (int64_t)b * (2 * C - 1);
        int node = slot + C - 1;
        tree[node] = Bk.max_priority[b];                              // memory.py:112: the bank's current max
        while (node > 0) {                                            // _propagate (memory.py:45-50)
            node = (node - 1) >> 1;
            tree[node] = tree[2 * node + 1] + tree[2 * node + 2];
        }
        const int next = (slot + 1) % C;
        Bk.index[b] = next;
        if (next == 0) Bk.full[b] = 1;
        Bk.timestep[b] = done[b] ? 0 : Bk.timestep[b] + 1;
    }
}

// Banks for N > batch: `m` of `N` uniformly without replacement (Floyd's algorithm, one warp).
__global__ void irbpp_replay_choose_kernel(int32_t* banks, int32_t m, int32_t N, uint64_t seed, uint64_t counter) {
    const int lane = threadIdx.x & 31;
    for (int k = 0; k < m; ++k) {
        const int j = N - m + k;
        const int t = (int)(replay_mix(seed, counter, 0xFFFFFFFFu, (uint64_t)j) % (uint64_t)(j + 1));
        bool hit = false;
        for (int i = lane; i < k; i += 32) hit |= banks[i] == t;
        hit = __any_sync(0xffffffffu, hit);
        if (lane == 0) banks[k] = hit ? j : t;
        __syncwarp();
    }
}

// ReplayMemory.sample (memory.py:191-203) of `per` draws from bank blockIdx.x (or banks[blockIdx.x]); output rows
// blockIdx.x * per .. + per - 1, laid out as agent.learn concatenates them (agent.py:72-82).
__global__ void __launch_bounds__(REPLAY_MAX_WARPS * 32)
irbpp_replay_sample_kernel(const irbpp_replay_banks Bk, const ReplaySampleParams S) {
    __shared__ float s_max[REPLAY_MAX_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int bank = S.choose ? S.banks[blockIdx.x] : (int)blockIdx.x;
    if (!S.choose && threadIdx.x == 0) S.banks[blockIdx.x] = bank;
    const int C = Bk.capacity, L = Bk.obs_len, n = S.n;
    const float* tree = Bk.tree + (int64_t)bank * (2 * C - 1);
    const float total = tree[0];
    const int widx = Bk.index[bank];
    const int cap = Bk.full[bank] ? C : widx;                         // memory.py:200
    const float segment = total / (float)S.per;                        // memory.py:193
    float wmax = 0.0f;
    for (int i = warp; i < S.per; i += nwarps) {
        const int row = blockIdx.x * S.per + i;
        int node = 0, ok = 0;
        if (lane == 0) {                                              // _get_sample_from_segment (memory.py:163-170)
            const float lo = (float)i * segment, hi = (float)(i + 1) * segment;
            for (int a = 0; a < S.max_attempts && !ok; ++a) {
                const double u = S.u_table ? S.u_table[(int64_t)row * S.max_attempts + a]
                                           : replay_u01(S.seed, S.counter, (uint32_t)row, (uint32_t)a);
                const double v = (double)lo + ((double)hi - (double)lo) * u;
                float x = (float)v;
                node = 0;
                while (2 * node + 1 < 2 * C - 1) {                    // _retrieve (memory.py:72-79)
                    const int left = 2 * node + 1;
                    if (x <= tree[left]) node = left;
                    else { x = x - tree[left]; node = left + 1; }
                }
                const int idx = node - C + 1;
                ok = replay_mod(widx - idx, C) > n && replay_mod(idx - widx, C) >= 1 && tree[node] != 0.0f;
            }
        }
        node = __shfl_sync(0xffffffffu, node, 0);
        ok = __shfl_sync(0xffffffffu, ok, 0);
        const int idx = ok ? node - C + 1 : 0;                        // a row out of attempts reads slot 0 (and is flagged)
        // n-step window (memory.py:115-130): position t is real while the previous one was nonterminal
        const int64_t base = (int64_t)bank * C;
        bool live = ok != 0;
        float R = 0.0f;
        for (int t = 0; t < n; ++t) {
            const int p = (idx + t) % C;
            if (t > 0) live = live && Bk.nonterminals[base + (idx + t - 1) % C] != 0;
            R = R + (live ? Bk.rewards[base + p] : 0.0f) * S.scale[t];
        }
        if (n > 0) live = live && Bk.nonterminals[base + (idx + n - 1) % C] != 0;
        const int pn = (idx + n) % C;
        const float* st = Bk.states + (base + idx) * Bk.row_stride;
        const float* nx = Bk.states + (base + pn) * Bk.row_stride;
        float* so = S.states + (int64_t)row * L;
        float* no = S.next_states + (int64_t)row * L;
        for (int e = lane; e < L; e += 32) {
            so[e] = ok ? st[e] : 0.0f;
            no[e] = live ? nx[e] : 0.0f;
        }
        if (lane == 0) {
            S.tree_index[row] = (int64_t)bank * (2 * C - 1) + node;
            S.actions[row] = ok ? Bk.actions[base + idx] : 0;
            S.returns[row] = R;
            S.nonterminals[row] = live && Bk.nonterminals[base + pn] ? 1.0f : 0.0f;
            S.error[row] = ok ? 0 : 1;
            float w = 0.0f;
            if (ok) {
                const float x = (float)cap * (tree[node] * (1.0f / total));   // memory.py:199-201
                w = S.beta_is_one ? 1.0f / x : powf(x, S.neg_beta);
                wmax = w > wmax ? w : wmax;
            }
            S.weights[row] = w;
        }
    }
    if (lane == 0) s_max[warp] = wmax;
    __syncthreads();
    float m = s_max[0];
    for (int w = 1; w < nwarps; ++w) m = s_max[w] > m ? s_max[w] : m;
    for (int i = warp; i < S.per; i += nwarps) {                      // memory.py:202: normalised by the draw's maximum
        const int row = blockIdx.x * S.per + i;
        if (lane == 0 && !S.error[row]) S.weights[row] = S.weights[row] / m;
    }
}

// update_priorities (memory.py:206-208) for `count` (tree node, priority) pairs in batch order.
__global__ void __launch_bounds__(REPLAY_UPDATE_THREADS)
irbpp_replay_update_kernel(const irbpp_replay_banks Bk, const int64_t* __restrict__ gidx,
                           const float* __restrict__ priority, int32_t count) {
    const int C = Bk.capacity, T = 2 * C - 1;
    const int64_t nodes = (int64_t)Bk.num_banks * T;
    auto leaf_ok = [&](int64_t g) { return g >= 0 && g < nodes && (int)(g % T) >= C - 1; };
    for (int j = threadIdx.x; j < count; j += blockDim.x) {          // SegmentTree.update (:54): the last write wins
        const int64_t g = gidx[j];
        if (!leaf_ok(g)) continue;
        bool later = false;
        for (int k = j + 1; k < count && !later; ++k) later = gidx[k] == g;
        if (!later) Bk.tree[g] = priority[j];
    }
    __syncthreads();
    for (int j = threadIdx.x; j < count; j += blockDim.x) {          // the first row of each bank owns that bank
        const int64_t g = gidx[j];
        if (!leaf_ok(g)) continue;
        const int64_t bank = g / T;
        bool first = true;
        for (int k = 0; k < j && first; ++k) first = !(leaf_ok(gidx[k]) && gidx[k] / T == bank);
        if (!first) continue;
        float* tree = Bk.tree + bank * T;
        float mx = Bk.max_priority[bank];
        for (int k = j; k < count; ++k) {
            if (!leaf_ok(gidx[k]) || gidx[k] / T != bank) continue;
            const float v = priority[k];
            mx = v > mx ? v : mx;                                     // max(value, self.max) (:56)
            int node = (int)(gidx[k] - bank * T);
            while (node > 0) {                                        // _propagate (:45-50)
                node = (node - 1) >> 1;
                tree[node] = tree[2 * node + 1] + tree[2 * node + 2];
            }
        }
        Bk.max_priority[bank] = mx;
    }
}

}  // namespace irbpp
