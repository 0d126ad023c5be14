// qnet_train.cuh — one DQN update of the Q-network on the device: the training half of the reference's DeepQLearningModel
// (Keras Huber loss on Q(s)[a], per-variable clipnorm, Adam; DESIGN §11).
//
// The forward pass is the inference chain itself (conv_sw_kernel x 3, dense_tc_kernel with the dense-1 activations kept):
// the bf16 post-ReLU activations it leaves in the plane buffers a1p / a2p / a3p / a4 are the saved tensors, the ReLU mask is
// act > 0. Every GEMM of the backward runs on gemm_tc_kernel (tcgen05, bf16 operands, f32 accumulation in TMEM) with the
// loaders below; weight gradients split their long K (batch x output pixels) over blockIdx.z into f32 slices that
// reduce_splits_kernel adds in slice order. All other sums (bias gradients, the head, norms, the loss) are fixed-order
// two-level reductions: no float atomics anywhere, so an update is bit-reproducible.
#pragma once
#include "qnet_conv.cuh"

namespace qlc {
namespace qnet {

// ---- parameter block: the f32 masters (and gradients, Adam moments) of the 10 Keras variables, back to back ----
constexpr int NVARS = 10;
__host__ __device__ constexpr uint32_t var_size(int v) {
    return v == 0 ? 8 * 8 * 4 * 32 : v == 1 ? 32 : v == 2 ? 4 * 4 * 32 * 64 : v == 3 ? 64 : v == 4 ? 3 * 3 * 64 * 64 : v == 5 ? 64 : v == 6 ? 3136 * 512 : v == 7 ? 512 : v == 8 ? 512 * 3 : 3;
}
__host__ __device__ constexpr uint32_t var_offset(int v) { return v == 0 ? 0 : var_offset(v - 1) + var_size(v - 1); }
constexpr uint32_t N_PARAMS = var_offset(NVARS);   // 1,685,667
static_assert(N_PARAMS == 1685667u, "parameter count");
constexpr int NORM_CHUNKS = 32;                     // partial sums of squares per variable

__device__ __forceinline__ uint16_t bf16_bits(float x) { const __nv_bfloat16 b = __float2bfloat16_rn(x); return *reinterpret_cast<const uint16_t*>(&b); }
__device__ __forceinline__ uint4 pack8_bits(const uint16_t (&h)[8]) {
    return make_uint4(h[0] | ((uint32_t)h[1] << 16), h[2] | ((uint32_t)h[3] << 16), h[4] | ((uint32_t)h[5] << 16), h[6] | ((uint32_t)h[7] << 16));
}
__device__ __forceinline__ float bf16_at(const __nv_bfloat16* p, size_t i) { return __bfloat162float(p[i]); }

// saved activations, read back from the forward's operand layouts (x = Keras' first spatial axis)
__device__ __forceinline__ size_t a1_index(uint32_t b, uint32_t x, uint32_t y, uint32_t c) {       // conv1 out 20x20x32 (OutConv2Planes)
    const uint32_t plane = (((y & 1u) * 2u + (x & 1u)) * 32u + c) >> 3, row = (y >> 1) * 10u + (x >> 1);
    return plane_elem_offset<Conv2Geom>(b, plane, row) + (c & 7u);
}
__device__ __forceinline__ size_t a2_index(uint32_t b, uint32_t x, uint32_t y, uint32_t c) {       // conv2 out 9x9x64 (OutConv3Planes)
    return plane_elem_offset<Conv3Geom>(b, c >> 3, y * 9u + x) + (c & 7u);
}
__device__ __forceinline__ size_t a3_index(uint32_t b, uint32_t k) {                                // conv3 out, Flatten k (OutDensePlanes)
    return (((size_t)(b >> 7) * DenseGeom::PLANES + (k >> 3)) * TILE_M + (b & 127u)) * 8 + (k & 7u);
}

// ---- A-operand loaders of the backward GEMMs (same prepare / load8 interface as qnet.cuh) ----
// Weight gradients: rows = weight index in the Keras order, K = (item, output pixel) of this K split (blockIdx.z * kc + k),
// zero beyond k_valid. dW = im2col(act)^T * dZ.
struct LoadA3T {                     // dense 1: rows k of Flatten, K = item
    const __nv_bfloat16* a3p; uint32_t k_valid, kc;
    struct Row { uint32_t k; };
    __device__ __forceinline__ Row prepare(uint32_t row) const { return Row{row}; }
    __device__ __forceinline__ uint4 load8(const Row& r, uint32_t kchunk) const {
        const uint32_t k0 = blockIdx.z * kc + kchunk * 8u;
        uint16_t h[8];
        #pragma unroll
        for (int e = 0; e < 8; ++e) { const uint32_t b = k0 + e; h[e] = b < k_valid ? __ldg(reinterpret_cast<const uint16_t*>(a3p) + a3_index(b, r.k)) : 0; }
        return pack8_bits(h);
    }
};
struct LoadIm2colT3 {                // conv3: rows (kx, ky, ci), K = item*49 + ox*7 + oy
    const __nv_bfloat16* a2p; uint32_t k_valid, kc;
    struct Row { uint32_t kx, ky, ci; };
    __device__ __forceinline__ Row prepare(uint32_t row) const { return Row{row / 192u, (row / 64u) % 3u, row % 64u}; }
    __device__ __forceinline__ uint4 load8(const Row& r, uint32_t kchunk) const {
        const uint32_t k0 = blockIdx.z * kc + kchunk * 8u;
        uint16_t h[8];
        #pragma unroll
        for (int e = 0; e < 8; ++e) {
            const uint32_t kk = k0 + e, b = kk / 49u, p = kk % 49u, ox = p / 7u, oy = p % 7u;
            h[e] = kk < k_valid ? __ldg(reinterpret_cast<const uint16_t*>(a2p) + a2_index(b, ox + r.kx, oy + r.ky, r.ci)) : 0;
        }
        return pack8_bits(h);
    }
};
struct LoadIm2colT2 {                // conv2 (stride 2): rows (kx, ky, ci), K = item*81 + ox*9 + oy
    const __nv_bfloat16* a1p; uint32_t k_valid, kc;
    struct Row { uint32_t kx, ky, ci; };
    __device__ __forceinline__ Row prepare(uint32_t row) const { return Row{row / 128u, (row / 32u) % 4u, row % 32u}; }
    __device__ __forceinline__ uint4 load8(const Row& r, uint32_t kchunk) const {
        const uint32_t k0 = blockIdx.z * kc + kchunk * 8u;
        uint16_t h[8];
        #pragma unroll
        for (int e = 0; e < 8; ++e) {
            const uint32_t kk = k0 + e, b = kk / 81u, p = kk % 81u, ox = p / 9u, oy = p % 9u;
            h[e] = kk < k_valid ? __ldg(reinterpret_cast<const uint16_t*>(a1p) + a1_index(b, 2u * ox + r.kx, 2u * oy + r.ky, r.ci)) : 0;
        }
        return pack8_bits(h);
    }
};
struct LoadIm2colT1 {                // conv1 (stride 4) straight from the u8 ring: rows (kx, ky, slot), K = item*400 + ox*20 + oy
    const uint8_t* frames; const uint32_t* slot_frame; uint32_t k_valid, kc;
    struct Row { uint32_t kx, ky, slot; };
    __device__ __forceinline__ Row prepare(uint32_t row) const { return Row{row / 32u, (row / 4u) % 8u, row % 4u}; }
    __device__ __forceinline__ uint4 load8(const Row& r, uint32_t kchunk) const {
        const uint32_t k0 = blockIdx.z * kc + kchunk * 8u;
        uint16_t h[8];
        #pragma unroll
        for (int e = 0; e < 8; ++e) {
            const uint32_t kk = k0 + e, b = kk / 400u, p = kk % 400u, ox = p / 20u, oy = p % 20u;
            uint32_t px = 0;
            if (kk < k_valid) {
                const uint32_t fi = __ldg(slot_frame + b * 4u + r.slot);
                if (fi != 0xFFFFFFFFu) px = __ldg(frames + (size_t)fi * FRAME_BYTES + (4u * oy + r.ky) * FRAME_W + 4u * ox + r.kx);
            }
            h[e] = bf16_bits((float)px);                                    // u8 -> bf16 is exact
        }
        return pack8_bits(h);
    }
};
// Data gradients: rows = (item, input pixel), K = (kx, ky, cout) with cout fastest: 8 consecutive K are 16 contiguous bytes of
// dZ [item][ox][oy][cout] (bf16), or zero where the tap falls outside the output.
struct LoadDz3Taps {                 // conv3: dA2 = full correlation of dZ3 with W3; rows item*81 + x*9 + y, K = 9 taps x 64
    const __nv_bfloat16* dz3;
    struct Row { uint32_t b, x, y; };
    __device__ __forceinline__ Row prepare(uint32_t row) const { const uint32_t b = row / 81u, p = row % 81u; return Row{b, p / 9u, p % 9u}; }
    __device__ __forceinline__ uint4 load8(const Row& r, uint32_t kchunk) const {
        const uint32_t tap = kchunk >> 3, co = (kchunk & 7u) * 8u, kx = tap / 3u, ky = tap % 3u;
        const uint32_t ox = r.x - kx, oy = r.y - ky;                                     // wraps (huge) when negative
        if (ox >= 7u || oy >= 7u) return make_uint4(0u, 0u, 0u, 0u);
        return __ldg(reinterpret_cast<const uint4*>(dz3 + (((size_t)r.b * 7u + ox) * 7u + oy) * 64u + co));
    }
};
struct LoadDz2Taps {                 // conv2 (stride 2): dA1; rows item*400 + x*20 + y, K = 16 taps x 64
    const __nv_bfloat16* dz2;
    struct Row { uint32_t b, x, y; };
    __device__ __forceinline__ Row prepare(uint32_t row) const { const uint32_t b = row / 400u, p = row % 400u; return Row{b, p / 20u, p % 20u}; }
    __device__ __forceinline__ uint4 load8(const Row& r, uint32_t kchunk) const {
        const uint32_t tap = kchunk >> 3, co = (kchunk & 7u) * 8u, kx = tap / 4u, ky = tap % 4u;
        const uint32_t dx = r.x - kx, dy = r.y - ky;
        if (((dx | dy) & 1u) || dx >= 18u || dy >= 18u) return make_uint4(0u, 0u, 0u, 0u);
        return __ldg(reinterpret_cast<const uint4*>(dz2 + (((size_t)r.b * 9u + dx / 2u) * 9u + dy / 2u) * 64u + co));
    }
};

// ---- B operands ------------------------------------------------------------------------------------------------
// data-gradient weights: Keras [kx][ky][ci][co] (f32 master) -> bf16 [ci][(kx, ky, co)]; TAPS = kx*ky count
template <int TAPS, int CI, int CO>
__global__ void prep_dgrad_weights_kernel(const float* __restrict__ kernel, __nv_bfloat16* __restrict__ w) {
    pdl_launch_dependents(); pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= TAPS * CI * CO) return;
    const int ci = i / (TAPS * CO), t = (i / CO) % TAPS, co = i % CO;
    w[i] = __float2bfloat16_rn(kernel[((size_t)t * CI + ci) * CO + co]);
}
// dZ f32 [rows][c] -> bf16 K slices [S][c][kc] (K = row; zero beyond rows): the B operand of a split-K weight gradient
__global__ void pack_splits_kernel(const float* __restrict__ src, uint32_t rows, uint32_t c, uint32_t kc, uint32_t n_splits, __nv_bfloat16* __restrict__ dst) {
    pdl_launch_dependents(); pdl_wait();
    const size_t total = (size_t)n_splits * c * kc;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t z = i / ((size_t)c * kc), rem = i % ((size_t)c * kc), col = rem / kc, kr = rem % kc;
        const size_t k = z * kc + kr;
        dst[i] = __float2bfloat16_rn(k < rows ? src[k * c + col] : 0.0f);
    }
}
// out[i] = sum over the split slices in slice order
__global__ void reduce_splits_kernel(const float* __restrict__ part, uint32_t n_splits, uint32_t n, float* __restrict__ out) {
    pdl_launch_dependents(); pdl_wait();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float s = 0.0f;
        for (uint32_t z = 0; z < n_splits; ++z) s += part[(size_t)z * n + i];
        out[i] = s;
    }
}

// ---- fixed-order column sums of a row-major f32 matrix [rows][c]: blocks (32 columns x 8 row lanes) x row splits ----
__global__ void __launch_bounds__(256) colsum_partial_kernel(const float* __restrict__ x, uint32_t rows, uint32_t c, uint32_t rows_per_split, float* __restrict__ partial) {
    pdl_launch_dependents(); pdl_wait();
    __shared__ float s[8][33];
    const uint32_t col = blockIdx.x * 32u + threadIdx.x;
    const uint32_t r0 = blockIdx.y * rows_per_split, r1 = min(rows, r0 + rows_per_split);
    float acc = 0.0f;
    if (col < c)
        for (uint32_t r = r0 + threadIdx.y; r < r1; r += 8u) acc += x[(size_t)r * c + col];
    s[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0 && col < c) {
        float t = 0.0f;
        #pragma unroll
        for (int i = 0; i < 8; ++i) t += s[i][threadIdx.x];
        partial[(size_t)blockIdx.y * c + col] = t;
    }
}
// out[col] = (sum of the partials in split order) / div
__global__ void colsum_final_kernel(const float* __restrict__ partial, uint32_t n_splits, uint32_t c, float div, float* __restrict__ out) {
    pdl_launch_dependents(); pdl_wait();
    const uint32_t col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= c) return;
    float t = 0.0f;
    for (uint32_t z = 0; z < n_splits; ++z) t += partial[(size_t)z * c + col];
    out[col] = t / div;
}

// ---- target: y [n] = G where the record of g.indices [i] is done, else G + Q_boot * d (-fmad=false: the multiply rounds first).
// One-step TD target (learner.py): g.indices = the items, ret = disc = NULL, so G = r of their record and d = gamma. n-step
// (nstep.cuh, DESIGN §14): g.indices = boot, whose record's done bit is R_{m-1}'s (terminal), G = ret [n], d = disc [n].
// Q_boot is max_q [n], or q [n][3] of the target network at the online network's greedy action [n] (double DQN, max_q NULL). ----
__global__ void target_kernel(GatherParams g, const float* __restrict__ ret, const float* __restrict__ disc, float gamma, const float* __restrict__ max_q,
                              const float* __restrict__ q, const uint8_t* __restrict__ action, float* __restrict__ y) {
    pdl_launch_dependents(); pdl_wait();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n_items) return;
    uint64_t T; uint32_t e, k, rec;
    locate(g, i, g.indices[i], T, e, k, rec);
    const float G = ret ? ret[i] : (float)((rec >> 8) & 0xFFu);
    const float d = disc ? disc[i] : gamma;
    const float qb = max_q ? max_q[i] : q[(size_t)i * 3 + action[i]];
    const float fut = qb * d;
    y[i] = ((rec >> 2) & 1u) ? G : G + fut;
}

// ---- head backward (CUDA cores, one warp per item): Huber(delta 1) on Q(s)[a], weighted by w [B] (NULL = 1), averaged over
// the batch ----
// dq [B][3] (only column a is non-zero), loss_i [B], dH = (dq . W5^T) masked by h > 0: f32 [B][512] and bf16 [B][512];
// td [B] (optional) = Q(s)[a] - y. A weight of 1.0 multiplies exactly, so the unweighted update keeps its bits.
__global__ void __launch_bounds__(256) head_backward_kernel(GatherParams g, const float* __restrict__ q, const float* __restrict__ y,
                                                            const float* __restrict__ w, const __nv_bfloat16* __restrict__ h,
                                                            const float* __restrict__ w5 /*Keras [512][3]*/, float* __restrict__ dq, float* __restrict__ loss_i,
                                                            float* __restrict__ dh, __nv_bfloat16* __restrict__ dh_bf, float* __restrict__ td) {
    pdl_launch_dependents(); pdl_wait();
    const uint32_t b = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
    if (b >= g.n_items) return;
    uint64_t T; uint32_t e, k, rec;
    locate(g, b, g.indices[b], T, e, k, rec);
    const uint32_t a = rec & 3u;
    const float d = q[(size_t)b * 3 + a] - y[b];
    const float ad = fabsf(d);
    const float wb = w ? w[b] : 1.0f;
    const float g_a = (fminf(fmaxf(d, -1.0f), 1.0f) * wb) / (float)g.n_items;
    if (lane == 0) {
        loss_i[b] = wb * (ad <= 1.0f ? 0.5f * (d * d) : ad - 0.5f);
        if (td) td[b] = d;
        #pragma unroll
        for (uint32_t j = 0; j < 3; ++j) dq[(size_t)b * 3 + j] = j == a ? g_a : 0.0f;
    }
    for (uint32_t n = lane; n < 512u; n += 32u) {
        const float v = bf16_at(h, (size_t)b * 512 + n) > 0.0f ? g_a * w5[n * 3 + a] : 0.0f;
        dh[(size_t)b * 512 + n] = v;
        dh_bf[(size_t)b * 512 + n] = __float2bfloat16_rn(v);
    }
}
// dW5[n][j] partial sums: blocks (32 hidden units x 8 row lanes) x row splits; partial [split][512][3]
__global__ void __launch_bounds__(256) head_wgrad_partial_kernel(const __nv_bfloat16* __restrict__ h, const float* __restrict__ dq, uint32_t rows,
                                                                 uint32_t rows_per_split, float* __restrict__ partial) {
    pdl_launch_dependents(); pdl_wait();
    __shared__ float s[3][8][33];
    const uint32_t n = blockIdx.x * 32u + threadIdx.x;
    const uint32_t r0 = blockIdx.y * rows_per_split, r1 = min(rows, r0 + rows_per_split);
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f;
    for (uint32_t r = r0 + threadIdx.y; r < r1; r += 8u) {
        const float hv = bf16_at(h, (size_t)r * 512 + n);
        a0 += hv * dq[(size_t)r * 3]; a1 += hv * dq[(size_t)r * 3 + 1]; a2 += hv * dq[(size_t)r * 3 + 2];
    }
    s[0][threadIdx.y][threadIdx.x] = a0; s[1][threadIdx.y][threadIdx.x] = a1; s[2][threadIdx.y][threadIdx.x] = a2;
    __syncthreads();
    if (threadIdx.y < 3) {
        float t = 0.0f;
        #pragma unroll
        for (int i = 0; i < 8; ++i) t += s[threadIdx.y][i][threadIdx.x];
        partial[((size_t)blockIdx.y * 512 + n) * 3 + threadIdx.y] = t;
    }
}

// ---- ReLU masks of the saved activations; f32 in place, plus a bf16 copy where a data-gradient GEMM reads it ----
__global__ void mask_conv3_kernel(float* __restrict__ d /*[B][3136]*/, const __nv_bfloat16* __restrict__ a3p, __nv_bfloat16* __restrict__ d_bf, uint32_t n_items) {
    pdl_launch_dependents(); pdl_wait();
    const size_t total = (size_t)n_items * 3136;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t b = (uint32_t)(i / 3136), k = (uint32_t)(i % 3136);
        const float v = bf16_at(a3p, a3_index(b, k)) > 0.0f ? d[i] : 0.0f;
        d[i] = v; d_bf[i] = __float2bfloat16_rn(v);
    }
}
__global__ void mask_conv2_kernel(float* __restrict__ d /*[B][9][9][64]*/, const __nv_bfloat16* __restrict__ a2p, __nv_bfloat16* __restrict__ d_bf, uint32_t n_items) {
    pdl_launch_dependents(); pdl_wait();
    const size_t total = (size_t)n_items * 5184;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t b = (uint32_t)(i / 5184), p = (uint32_t)(i % 5184), x = p / 576u, y = (p / 64u) % 9u, c = p % 64u;
        const float v = bf16_at(a2p, a2_index(b, x, y, c)) > 0.0f ? d[i] : 0.0f;
        d[i] = v; d_bf[i] = __float2bfloat16_rn(v);
    }
}
__global__ void mask_conv1_kernel(float* __restrict__ d /*[B][20][20][32]*/, const __nv_bfloat16* __restrict__ a1p, uint32_t n_items) {
    pdl_launch_dependents(); pdl_wait();
    const size_t total = (size_t)n_items * 12800;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t b = (uint32_t)(i / 12800), p = (uint32_t)(i % 12800), x = p / 640u, y = (p / 32u) % 20u, c = p % 32u;
        if (!(bf16_at(a1p, a1_index(b, x, y, c)) > 0.0f)) d[i] = 0.0f;
    }
}

// ---- per-variable clipnorm + Adam (Keras 2.12) ----
__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ g, float* __restrict__ partial /*[NVARS][NORM_CHUNKS]*/) {
    pdl_launch_dependents(); pdl_wait();
    __shared__ float s[256];
    const int v = blockIdx.x;
    const uint32_t n = var_size(v), per = (n + NORM_CHUNKS - 1) / NORM_CHUNKS;
    const uint32_t i0 = blockIdx.y * per, i1 = min(n, i0 + per);
    const float* p = g + var_offset(v);
    float acc = 0.0f;
    for (uint32_t i = i0 + threadIdx.x; i < i1; i += 256u) acc += p[i] * p[i];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) s[threadIdx.x] += s[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[v * NORM_CHUNKS + blockIdx.y] = s[0];
}
struct AdamStep { float alpha, one_minus_beta1, one_minus_beta2, epsilon, clipnorm; };   // 1 - beta as Keras forms them (double, then f32)
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ w, float* __restrict__ m, float* __restrict__ v, const float* __restrict__ g,
                                                   const float* __restrict__ sumsq, AdamStep p) {
    pdl_launch_dependents(); pdl_wait();
    __shared__ float s_norm[NVARS];
    if (threadIdx.x < NVARS) {
        float t = 0.0f;
        for (int c = 0; c < NORM_CHUNKS; ++c) t += sumsq[threadIdx.x * NORM_CHUNKS + c];
        s_norm[threadIdx.x] = sqrtf(t);
    }
    __syncthreads();
    const float one_b1 = p.one_minus_beta1, one_b2 = p.one_minus_beta2;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < N_PARAMS; i += gridDim.x * blockDim.x) {
        int var = 0;
        #pragma unroll
        for (int k = 1; k < NVARS; ++k) var += i >= var_offset(k);
        float gi = g[i];
        if (p.clipnorm > 0.0f) gi = (gi * p.clipnorm) / fmaxf(s_norm[var], p.clipnorm);     // tf.clip_by_norm
        const float mi = m[i] + (gi - m[i]) * one_b1;
        const float vi = v[i] + (gi * gi - v[i]) * one_b2;
        m[i] = mi; v[i] = vi;
        w[i] = w[i] - (mi * p.alpha) / (sqrtf(vi) + p.epsilon);
    }
}

}  // namespace qnet
}  // namespace qlc
