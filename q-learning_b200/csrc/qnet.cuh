// qnet.cuh — tcgen05 (5th-generation tensor core) helpers and gemm_tc_kernel, the GEMM engine of the Q-network's backward
// pass (qnet_train.cuh: weight gradients with split K, data gradients) and of the qlc_debug_gemm_bf16 test hook. The forward
// runs on the shifted-window convolutions and the bulk-copy fed dense layer of qnet_conv.cuh, which share the helpers.
// Architecture = the reference's Keras model (/root/reference/src/ql-with-tensorflow/python_model/create_ql_model_breakout_84x84x4_3_32.py:17-33):
//   Conv(32, 8x8, stride 4) -> Conv(64, 4x4, stride 2) -> Conv(64, 3x3, stride 1) -> Dense 512 -> Dense 3, ReLU between.
// gemm_tc_kernel: C[M x N] = A[M x K] * W[N x K]^T, bf16 operands, f32 accumulation in TMEM:
//   * one CTA (128 threads) owns a 128-row tile of M and one N tile of NT <= 256 columns;
//   * the threads gather A through a loader policy, and W, into the canonical K-major, non-swizzled core-matrix layout
//     (8 rows x 16 bytes per core matrix);
//   * one elected thread issues tcgen05.mma (cta_group::1, kind::f16, M = 128) from shared-memory descriptors, completion
//     via tcgen05.commit -> mbarrier; the epilogue reads TMEM with tcgen05.ld (32x32b) and hands the f32 accumulators to an
//     epilogue policy.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include "kernels.cuh"

namespace qlc {
namespace qnet {

constexpr int TILE_M = 128;      // UMMA M (cta_group::1)
constexpr int KC = 64;           // K elements staged per pipeline step (4 MMAs of K = 16)
constexpr int CORE_BYTES = 128;  // one core matrix: 8 rows x 16 bytes

// ---- tcgen05 / TMEM helpers (PTX as in CUTLASS' cute/arch/{mma_sm100_umma,copy_sm100,tmem_allocator_sm100}.hpp) ----
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> f32
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// shared-memory matrix descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor): start address [0,14), leading-dimension
// byte offset [16,30) = distance between the two K core matrices of one MMA, stride byte offset [32,46) = distance between
// 8-row groups, version [46,48) = 1, layout type [61,64) = 0. All offsets without their 4 LSBs.
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) |
           ((uint64_t)1 << 46);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 [4,6) = 1, a/b_format BF16 [7,10),[10,13) = 1, both
// K-major, n_dim [17,23) = N >> 3, m_dim [24,29) = M >> 4
__host__ __device__ constexpr uint32_t instr_desc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// mbarrier wait that gives up (returns false) instead of hanging the GPU if the tensor core never signals
__device__ __forceinline__ bool mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
    for (uint32_t i = 0; i < (1u << 22); ++i) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (ok) return true;
    }
    return false;
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&v);
}

// ---- A-operand loaders: prepare(row) hoists the per-row index math, load8() returns 8 consecutive K elements (16 B) ----
struct LoadRowMajorBf16 {            // plain GEMM: A bf16 [M][K] row-major (dH of the dA3 GEMM, the debug hook)
    const __nv_bfloat16* a; uint32_t k_total;
    struct Row { const __nv_bfloat16* p; };
    __device__ __forceinline__ Row prepare(uint32_t row) const { return Row{a + (size_t)row * k_total}; }
    __device__ __forceinline__ uint4 load8(const Row& r, uint32_t kchunk) const { return __ldg(reinterpret_cast<const uint4*>(r.p + (size_t)kchunk * 8)); }
};
// which frame of the ring holds ring-slot h of item b's state (obs mode: indices == NULL, item = env at the current time;
// replay mode: logical transition index, which = 0 state / 1 next) — same rules as the gather kernels (locate()).
__global__ void qnet_locate_kernel(GatherParams g, uint32_t which, uint32_t* slot_frame) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");      // programmatic dependent launch (see qnet_conv.cuh)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= g.n_items) return;
    reinterpret_cast<uint4*>(slot_frame)[b] = slot_frames(g, b, which);
}

// the head weights of the dense epilogue: Keras [512][3] -> [3][512] f32
__global__ void prep_head_kernel(const float* __restrict__ kernel /*[512][3]*/, float* __restrict__ w /*[3][512]*/) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 3 * 512) return;
    w[i] = kernel[(i % 512) * 3 + i / 512];
}

// ---------------------------------------------------------------------------------------------------------
// C[M x N_TOTAL] = act(A * W^T + bias). Persistent CTAs (128 threads): blockIdx.y picks an N tile of NT columns, the CTA
// walks the 128-row M tiles blockIdx.x, +gridDim.x, ... K is consumed in 64-element chunks through a 2-stage shared-memory
// ring that runs on across tile boundaries: while the tensor core works on chunk g the threads already gather chunk g+1
// (global loads in flight) and chunk g-1's stage is being refilled; completion per stage via tcgen05.commit -> mbarrier.
// W: bf16 [N_TOTAL][K] (K-major). The epilogue policy stores the accumulators. NT in {32, 64, 128, 256}; K % 64 == 0.
// ---------------------------------------------------------------------------------------------------------
// Epilogue policies: store8(row, n, v) receives the f32 accumulators of columns n .. n+7 of one row.
struct EpiBiasAct {                  // out bf16 [M][n_total] = act(acc + bias)
    const float* bias; __nv_bfloat16* out; uint32_t n_total; int relu;
    __device__ __forceinline__ void store8(uint32_t row, uint32_t n, const uint32_t (&v)[8]) const {
        float f[8];
        #pragma unroll
        for (int i = 0; i < 8; ++i) { f[i] = __uint_as_float(v[i]) + bias[n + i]; if (relu) f[i] = fmaxf(f[i], 0.0f); }
        *reinterpret_cast<uint4*>(out + (size_t)row * n_total + n) =
            make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
    }
};
struct EpiF32 {                      // out f32 [gridDim.z][m_total][n_total]: the raw accumulators, one slice per K split
    float* out; uint32_t m_total, n_total;
    __device__ __forceinline__ void store8(uint32_t row, uint32_t n, const uint32_t (&v)[8]) const {
        float4* o = reinterpret_cast<float4*>(out + ((size_t)blockIdx.z * m_total + row) * n_total + n);
        o[0] = make_float4(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]), __uint_as_float(v[3]));
        o[1] = make_float4(__uint_as_float(v[4]), __uint_as_float(v[5]), __uint_as_float(v[6]), __uint_as_float(v[7]));
    }
};

// Split K: blockIdx.z selects a K slice. W holds the slices back to back ([gridDim.z][N_TOTAL][k_total]); the loader offsets
// its own K by blockIdx.z (the data-gradient GEMMs run with gridDim.z = 1).
template <int NT, class Loader, class Epi>
__global__ void __launch_bounds__(128) gemm_tc_kernel(Loader ld, const __nv_bfloat16* __restrict__ w, Epi epi, uint32_t m_total, uint32_t k_total,
                                                     uint32_t n_total, unsigned int* err_flag) {
    static_assert(NT % 16 == 0 && NT >= 32 && NT <= 256, "NT");
    constexpr uint32_t A_BYTES = TILE_M * KC * 2;              // 16 KB per stage
    constexpr uint32_t B_BYTES = (uint32_t)NT * KC * 2;
    constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
    constexpr uint32_t LBO = CORE_BYTES;                       // K-adjacent core matrices are contiguous
    constexpr uint32_t SBO = (KC / 8) * CORE_BYTES;            // 8-row groups are 1 KB apart
    constexpr uint32_t TMEM_COLS = NT <= 32 ? 32 : (NT <= 64 ? 64 : (NT <= 128 ? 128 : 256));
    constexpr int BV = (NT * (KC / 8) + 127) / 128;            // W chunks (16 B) per thread and stage
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar[2];
    __shared__ uint32_t tmem_slot;
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    const uint32_t n0 = blockIdx.y * NT;

    if (tid == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc(&tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    const uint32_t n_chunks = k_total / KC;
    const uint32_t n_mtiles = (m_total + TILE_M - 1) / TILE_M;
    const __nv_bfloat16* wrow = w + ((size_t)blockIdx.z * n_total + n0) * k_total;

    uint4 av[KC / 8], bv[BV];
    auto gather = [&](const typename Loader::Row& r, bool row_ok, uint32_t c) {
        #pragma unroll
        for (int j = 0; j < KC / 8; ++j) av[j] = row_ok ? ld.load8(r, c * (KC / 8) + j) : make_uint4(0u, 0u, 0u, 0u);
        #pragma unroll
        for (int i = 0; i < BV; ++i) {
            const uint32_t idx = tid + i * 128u, n = idx / (KC / 8), j = idx % (KC / 8);
            bv[i] = (n < (uint32_t)NT) ? __ldg(reinterpret_cast<const uint4*>(wrow + (size_t)n * k_total + (size_t)c * KC + j * 8)) : make_uint4(0u, 0u, 0u, 0u);
        }
    };

    uint32_t g = 0;                                            // chunks issued so far by this CTA (stage = g & 1)
    uint32_t tile = blockIdx.x;
    if (tile >= n_mtiles) { tc_fence_before(); __syncthreads(); if (warp == 0) tmem_dealloc(tmem_base, TMEM_COLS); return; }
    uint32_t my_row = tile * TILE_M + tid;
    bool row_ok = my_row < m_total;
    typename Loader::Row rprep = ld.prepare(row_ok ? my_row : 0u);
    gather(rprep, row_ok, 0);
    bool alive = true;
    while (alive) {
        for (uint32_t c = 0; c < n_chunks; ++c, ++g) {
            const uint32_t st = g & 1u;
            uint8_t* sa = smem + st * STAGE_BYTES;
            uint8_t* sb = sa + A_BYTES;
            // stage `st` was last read by the MMAs of chunk g-2
            if (g >= 2u && !mbar_wait_bounded(&bar[st], ((g - 2u) >> 1) & 1u)) { if (tid == 0 && err_flag) atomicExch(err_flag, 1u); }
            #pragma unroll
            for (int j = 0; j < KC / 8; ++j) *reinterpret_cast<uint4*>(sa + (tid >> 3) * SBO + j * LBO + (tid & 7u) * 16u) = av[j];
            #pragma unroll
            for (int i = 0; i < BV; ++i) {
                const uint32_t idx = tid + i * 128u, n = idx / (KC / 8), j = idx % (KC / 8);
                if (n < (uint32_t)NT) *reinterpret_cast<uint4*>(sb + (n >> 3) * SBO + j * LBO + (n & 7u) * 16u) = bv[i];
            }
            // next chunk's operands go in flight now (next K chunk of this tile, or chunk 0 of the CTA's next tile)
            uint32_t next_tile = tile, next_c = c + 1;
            if (next_c == n_chunks) { next_tile = tile + gridDim.x; next_c = 0; }
            typename Loader::Row nprep = rprep; bool nrow_ok = row_ok; uint32_t nrow = my_row;
            if (next_tile != tile) {
                nrow = next_tile * TILE_M + tid; nrow_ok = next_tile < n_mtiles && nrow < m_total;
                nprep = ld.prepare(nrow_ok ? nrow : 0u);
            }
            if (next_tile < n_mtiles) gather(nprep, nrow_ok, next_c);
            fence_proxy_async_smem();                          // generic-proxy writes -> visible to the tensor core (async proxy)
            __syncthreads();
            if (tid == 0) {
                tc_fence_after();
                #pragma unroll
                for (int kk = 0; kk < KC / 16; ++kk) {
                    const uint64_t da = smem_desc(smem_u32(sa) + kk * 2 * LBO, LBO, SBO);
                    const uint64_t db = smem_desc(smem_u32(sb) + kk * 2 * LBO, LBO, SBO);
                    tc_mma_bf16(tmem_base, da, db, instr_desc_bf16(TILE_M, NT), (c > 0 || kk > 0) ? 1u : 0u);
                }
                tc_commit(&bar[st]);
            }
            if (c + 1 == n_chunks) {
                // epilogue of this tile: wait for its last MMAs, thread = row (TMEM lane), 8 columns per tcgen05.ld
                if (!mbar_wait_bounded(&bar[st], (g >> 1) & 1u)) { if (tid == 0 && err_flag) atomicExch(err_flag, 1u); }
                tc_fence_after();
                #pragma unroll 1
                for (int col = 0; col < NT; col += 8) {
                    uint32_t v[8];
                    tmem_ld8(tmem_base + ((warp * 32u) << 16) + (uint32_t)col, v);
                    if (row_ok) epi.store8(my_row, n0 + (uint32_t)col, v);
                }
                tc_fence_before();                             // the next tile's first MMA overwrites the accumulator
                __syncthreads();
                tile = next_tile; my_row = nrow; row_ok = nrow_ok; rprep = nprep;
                alive = tile < n_mtiles;
            }
        }
    }
    if (warp == 0) tmem_dealloc(tmem_base, TMEM_COLS);
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) out[i] = __float2bfloat16_rn(in[i]);
}
__global__ void bf16_to_f32_kernel(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) out[i] = __bfloat162float(in[i]);
}

}  // namespace qnet
}  // namespace qlc
