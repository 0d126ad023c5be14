// per.cuh — proportional prioritized replay (Schaul et al., ICLR 2016) on the device: a sum tree over the replay ring.
//
// Leaves: one f32 priority per physical transition slot, in the record ring's layout [time_slots][n_envs] (leaf of time T,
// env e = (T % time_slots) * n_envs + e); non-zero exactly for the transitions in the replay. Internal nodes: f64, fan-out 32,
// node j of level k = the sum of children 32j .. 32j + 31 of level k - 1, added one after another from child 0 (starting from
// 0.0; padding children are 0). Every array is padded to a multiple of 32 with zeros, so a node always reads 32 children. No
// float atomics touch the sums: the tree equals a rebuild from its leaves bit for bit after any sequence of calls.
// DESIGN.md §13 has the rules (sync, sampling arithmetic, importance weights, update).
#pragma once
#include "physics.cuh"
#include "qnet_conv.cuh"     // pdl_wait / pdl_launch_dependents

namespace qlc {
namespace per {

using qnet::pdl_launch_dependents;
using qnet::pdl_wait;

constexpr uint32_t LOG_FAN = 5, FAN = 1u << LOG_FAN, MAX_LEVELS = 16;

struct Tree {
    float* leaves;                    // [count[0]] padded to a multiple of 32
    double* node[MAX_LEVELS];         // node[k], k = 1 .. depth; node[depth][0] = the root (total priority)
    uint64_t count[MAX_LEVELS];       // unpadded counts; count[0] = time_slots * n_envs
    uint32_t depth;
    uint32_t n_envs, time_slots;
    unsigned int* max_bits;           // running maximum priority (f32 bits; positive floats order like their bits)
};

// up to 4 index intervals [lo, hi) of one tree level (a lazy sync: the rows that entered and left, each split at the wrap)
struct Intervals {
    uint64_t lo[4], hi[4];
    uint32_t n;
};

__device__ __forceinline__ double child_value(const Tree& t, uint32_t level, uint64_t i) {
    return level == 0 ? (double)t.leaves[i] : t.node[level][i];
}

// node j of `level` (>= 1) = children summed left to right
__device__ __forceinline__ void resum_node(const Tree& t, uint32_t level, uint64_t j) {
    const uint64_t c0 = j << LOG_FAN;
    double s = 0.0;
    if (level == 1) {
        const float4* p = reinterpret_cast<const float4*>(t.leaves + c0);
        #pragma unroll
        for (int v = 0; v < 8; ++v) { const float4 x = p[v]; s += (double)x.x; s += (double)x.y; s += (double)x.z; s += (double)x.w; }
    } else {
        const double2* p = reinterpret_cast<const double2*>(t.node[level - 1] + c0);
        #pragma unroll
        for (int v = 0; v < 16; ++v) { const double2 x = p[v]; s += x.x; s += x.y; }
    }
    t.node[level][j] = s;
}

// the time whose transitions occupy ring slot `slot` at time t_now (the latest T < t_now with T % time_slots == slot);
// false: the slot has not been written yet
__device__ __forceinline__ bool slot_owner(uint64_t t_now, uint32_t time_slots, uint32_t slot, uint64_t& T) {
    if (t_now == 0) return false;
    const uint32_t r = (uint32_t)((t_now - 1) % time_slots);
    const uint64_t d = r >= slot ? r - slot : (uint64_t)r + time_slots - slot;
    if (d > t_now - 1) return false;
    T = t_now - 1 - d;
    return true;
}

__device__ __forceinline__ uint64_t leaf_of(const Tree& t, uint64_t t_oldest, uint32_t idx) {
    const uint64_t T = t_oldest + idx / t.n_envs;
    return (T % t.time_slots) * t.n_envs + idx % t.n_envs;
}

__device__ __forceinline__ bool interval_item(const Intervals& iv, uint64_t j, uint64_t& out) {
    #pragma unroll
    for (uint32_t k = 0; k < 4; ++k) {              // unrolled: the intervals stay in parameter space
        if (k >= iv.n) break;
        const uint64_t w = iv.hi[k] - iv.lo[k];
        if (j < w) { out = iv.lo[k] + j; return true; }
        j -= w;
    }
    return false;
}

// p = (|delta| + epsilon)^alpha in f64, rounded to f32 once; never 0 (a zero leaf would drop a transition from the replay)
__device__ __forceinline__ float priority(float delta, float alpha, float epsilon) {
    const float p = (float)pow(fabs((double)delta) + (double)epsilon, (double)alpha);
    return fmaxf(p, 1.17549435e-38f);
}

// ---- lazy sync: the leaves of the slot intervals `iv` (leaf indices) get the running max if their owner time is in
// [t_oldest, t_now), else 0 ----
__global__ void __launch_bounds__(256) per_sync_leaves_kernel(Tree t, Intervals iv, uint64_t total, uint64_t t_now, uint64_t t_oldest) {
    pdl_launch_dependents(); pdl_wait();
    const float maxp = __uint_as_float(*t.max_bits);
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t leaf;
        interval_item(iv, j, leaf);
        uint64_t T;
        const bool valid = slot_owner(t_now, t.time_slots, (uint32_t)(leaf / t.n_envs), T) && T >= t_oldest;
        t.leaves[leaf] = valid ? maxp : 0.0f;
    }
}

// re-sum the nodes of `level` in the node intervals `iv` (overlapping intervals recompute a node twice, to the same value)
__global__ void __launch_bounds__(256) per_resum_intervals_kernel(Tree t, uint32_t level, Intervals iv, uint64_t total) {
    pdl_launch_dependents(); pdl_wait();
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t node;
        interval_item(iv, j, node);
        resum_node(t, level, node);
    }
}

// ---- priority update: zero the leaves of the valid indices and raise the running max by the finite priorities ... ----
__global__ void __launch_bounds__(256) per_update_clear_kernel(Tree t, const uint32_t* __restrict__ idx, const float* __restrict__ td, uint32_t n,
                                                               uint32_t len, uint64_t t_oldest, float alpha, float epsilon) {
    pdl_launch_dependents(); pdl_wait();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || idx[i] >= len) return;
    t.leaves[leaf_of(t, t_oldest, idx[i])] = 0.0f;
    const float d = td[i];
    if (isfinite(d)) atomicMax(t.max_bits, __float_as_uint(priority(d, alpha, epsilon)));
}
// ... then set them: the largest priority among an index's duplicates wins (atomicMax on positive f32 bits: order-independent);
// a non-finite delta gives the running max as raised by this update's finite ones
__global__ void __launch_bounds__(256) per_update_set_kernel(Tree t, const uint32_t* __restrict__ idx, const float* __restrict__ td, uint32_t n,
                                                             uint32_t len, uint64_t t_oldest, float alpha, float epsilon) {
    pdl_launch_dependents(); pdl_wait();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || idx[i] >= len) return;
    const float d = td[i];
    const float p = isfinite(d) ? priority(d, alpha, epsilon) : __uint_as_float(*t.max_bits);
    atomicMax(reinterpret_cast<unsigned int*>(t.leaves) + leaf_of(t, t_oldest, idx[i]), __float_as_uint(p));
}
// ... and re-sum each updated leaf's ancestor on `level` (duplicates recompute the same node to the same value)
__global__ void __launch_bounds__(256) per_resum_items_kernel(Tree t, uint32_t level, const uint32_t* __restrict__ idx, uint32_t n, uint32_t len, uint64_t t_oldest) {
    pdl_launch_dependents(); pdl_wait();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || idx[i] >= len) return;
    resum_node(t, level, leaf_of(t, t_oldest, idx[i]) >> (LOG_FAN * level));
}

// ---- stratified proportional sampling with replacement: item i of minibatch m (c = call0 + m) takes
// u = (i + (w32 + 0.5) * 2^-32) * total / batch, w32 = word i & 3 of philox({i >> 2, c_lo, c_hi, 'PRIO'}, seed), and walks down
// from the root subtracting children in summation order; rounding past the last child takes the last non-zero one.
// Writes the logical replay index and (p_out != NULL) the item's leaf priority. ----
__global__ void __launch_bounds__(128) per_sample_kernel(Tree t, uint32_t batch, uint32_t n_items, uint64_t call0, uint64_t seed, uint64_t t_now,
                                                         uint64_t t_oldest, uint32_t* __restrict__ idx_out, float* __restrict__ p_out) {
    pdl_launch_dependents(); pdl_wait();
    const uint32_t item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= n_items) return;
    const uint32_t m = item / batch, i = item - m * batch;
    const uint64_t c = call0 + m;
    const uint4 r = philox4x32_10(make_uint4(i >> 2, (uint32_t)c, (uint32_t)(c >> 32), STREAM_PRIORITY), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t w32 = (i & 3u) == 0 ? r.x : (i & 3u) == 1 ? r.y : (i & 3u) == 2 ? r.z : r.w;
    const double total = t.node[t.depth][0];
    double u = ((double)i + ((double)w32 + 0.5) * 0x1p-32) * total / (double)batch;
    uint64_t node = 0;
    for (uint32_t level = t.depth; level >= 1; --level) {
        const uint64_t c0 = node << LOG_FAN;
        int pick = -1, last_nz = 0;
        #pragma unroll 4
        for (int k = 0; k < (int)FAN; ++k) {
            const double v = child_value(t, level - 1, c0 + (uint64_t)k);
            if (v > 0.0) last_nz = k;
            if (pick < 0) { if (u < v) pick = k; else u -= v; }
        }
        node = c0 + (uint64_t)(pick < 0 ? last_nz : pick);
    }
    const uint32_t slot = (uint32_t)(node / t.n_envs), e = (uint32_t)(node - (uint64_t)slot * t.n_envs);
    uint64_t T = t_oldest;
    slot_owner(t_now, t.time_slots, slot, T);                                 // a non-zero leaf always has an owner in the replay
    idx_out[item] = (uint32_t)((T - t_oldest) * t.n_envs + e);
    if (p_out) p_out[item] = t.leaves[node];
}

// importance weights of one minibatch per CTA, in place: w = (p_min / p)^beta in f64, rounded to f32; p_min = the smallest
// priority among the minibatch's items (= (len * P(i))^-beta normalised by the minibatch's largest weight)
__global__ void __launch_bounds__(256) per_weight_kernel(float* __restrict__ pw, uint32_t batch, float beta) {
    pdl_launch_dependents(); pdl_wait();
    __shared__ float wmin[8];
    float* p = pw + (size_t)blockIdx.x * batch;
    float mn = __int_as_float(0x7f800000);
    for (uint32_t i = threadIdx.x; i < batch; i += blockDim.x) mn = fminf(mn, p[i]);
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
    if ((threadIdx.x & 31) == 0) wmin[threadIdx.x >> 5] = mn;
    __syncthreads();
    mn = wmin[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) mn = fminf(mn, wmin[w]);
    const double pmin = (double)mn;
    for (uint32_t i = threadIdx.x; i < batch; i += blockDim.x) p[i] = (float)pow(pmin / (double)p[i], (double)beta);
}

}  // namespace per
}  // namespace qlc
