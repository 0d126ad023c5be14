// qnet_conv.cuh — the three convolutions of the Q-network as "shifted-window" implicit GEMMs on tcgen05, without im2col.
//
// Idea: a stride-s convolution becomes a stride-1 convolution with few taps after a space-to-depth by s
// (conv1: 8x8/4 over 84x84x4 -> 2x2 over 21x21x64; conv2: 4x4/2 over 20x20x32 -> 2x2 over 10x10x128; conv3 is 3x3/1 over
// 9x9x64 already). With the activation stored as a matrix [row = pixel (y*W + x)][channel], tap (dy, dx) of a stride-1
// convolution is THE SAME matrix shifted by dy*W + dx rows. The tensor core reads its A operand through a shared-memory
// descriptor, so a shift is just another start address — if the layout allows arbitrary row offsets. The K-major
// no-swizzle canonical layout does when its 8-row groups are packed back to back (stride-byte-offset = 128): then row r of
// the 16-byte K chunk j lives at  j * PLANE + r * 16  ("planes" of 8 channels, rows linear), and a window shifted by S rows
// starts S * 16 bytes further. Each activation byte is staged ONCE (vs 3.6x / 4x / 9x for im2col) and no thread touches
// the operands of conv2 / conv3 at all: their planes arrive by cp.async.bulk exactly as the previous layer's epilogue
// wrote them. Output rows whose window crosses the right / bottom edge (or an item boundary) are junk and never stored.
//
// One persistent CTA per SM, warp-specialised:
//   warps 0-3  epilogue: tcgen05.ld of their TMEM lane quadrant, bias + ReLU, bf16, store in the NEXT layer's plane layout
//   warp  4    issues every tcgen05.mma of a batch (tiles x taps x K steps) and commits to mbarriers; the whole warp runs the loop
//              (elect.sync per instruction, votes on the waits) so that the descriptors stay in uniform registers
//   warp  5    one thread issues the bulk copies (conv1: the four u8 ring frames of an item, raw; conv2/3: a whole stage)
//   warps 6..  conv1 only: convert the raw u8 frames to bf16 planes (space-to-depth by 4) in shared memory
// Input stages and TMEM accumulator sets are double-buffered, so copies, conversion, MMAs and epilogue of neighbouring
// batches overlap. What bounds the kernels is the shared-memory operand fetch of the tensor core: an M = 128, K = 16 MMA with
// both operands in shared memory takes max(N/2, 32 + N/4) cycles (tools/microbench/mma_rate.cu), i.e. 40 / 48 cycles at the
// model's N = 32 / 64 instead of the tensor pipe's 16 / 32. Architecture: /root/reference/src/ql-with-tensorflow/python_model/create_ql_model_breakout_84x84x4_3_32.py:17-33.
#pragma once
#include "qnet.cuh"

namespace qlc {
namespace qnet {

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, "
        "%22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
          "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
          "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// warp-wide variants: all 32 lanes execute them with identical operands, one elected lane issues
__device__ __forceinline__ void tc_mma_bf16_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// same with the descriptors given as their low words (start address >> 4 | leading-dimension offset << 16); the high word
// is the constant stride-byte-offset 128 + descriptor version 1
__device__ __forceinline__ void tc_mma_bf16_elect_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, 0x4008};\n\t"
        "mov.b64 db, {%2, 0x4008};\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}

// Programmatic dependent launch: a kernel launched with programmaticStreamSerializationAllowed may start while its
// predecessor in the stream is still draining; everything before pdl_wait() (barrier init, TMEM allocation, the weight copy)
// overlaps that tail, pdl_wait() returns once the predecessor has completed and its writes are visible.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- layer geometry ---------------------------------------------------------------------------------------
// ROWS = pixels of one item's (space-to-depth) input, WIN its width; PL = 16-byte channel planes per tap (channels / 8);
// TY x TX taps; OH x OW valid outputs; N output channels; B items per batch (their rows are concatenated in a plane).
template <int ROWS_, int WIN_, int PL_, int TY_, int TX_, int OH_, int OW_, int N_, int B_, int NSTAGE_, bool FROM_RING_, int NCONV_>
struct ConvGeom {
    static constexpr int ROWS = ROWS_, WIN = WIN_, PL = PL_, TY = TY_, TX = TX_, OH = OH_, OW = OW_, N = N_, B = B_, NSTAGE = NSTAGE_;
    static constexpr bool FROM_RING = FROM_RING_;
    static constexpr int NCONV = FROM_RING_ ? NCONV_ : 0;                  // converter warps
    static constexpr int NRAW = 3;                                         // raw u8 item stages (conv1)
    static constexpr int TAPS = TY * TX, KSTEPS = PL / 2;                  // K = 16 per MMA = two planes
    static constexpr int M_NEEDED = (B - 1) * ROWS + (OH - 1) * WIN + OW;  // last valid output row + 1
    static constexpr int NTILES = (M_NEEDED + TILE_M - 1) / TILE_M;
    static constexpr int PLANE_BYTES = B * ROWS * 16;
    static constexpr int STAGE_BYTES = PL * PLANE_BYTES;
    static constexpr int W_BYTES = TAPS * PL * N * 16;
    static constexpr int RAW_BYTES = 4 * FRAME_BYTES;
    static constexpr int TMEM_COLS = 2 * NTILES * N <= 32 ? 32 : (2 * NTILES * N <= 64 ? 64 : (2 * NTILES * N <= 128 ? 128 : (2 * NTILES * N <= 256 ? 256 : 512)));
    static constexpr int THREADS = 32 * (6 + NCONV);
    static constexpr int NBAR = 1 + 2 * NSTAGE + 2 * NTILES + 2 + 2 * NRAW;
    static constexpr size_t SMEM_BYTES = (size_t)W_BYTES + (size_t)NSTAGE * STAGE_BYTES + (FROM_RING ? (size_t)NRAW * RAW_BYTES : 0) + 64 * 4 + NBAR * 8 + 16 + NRAW * 16;
    static_assert(M_NEEDED >= TILE_M, "a batch must fill at least one M tile");
    static_assert(2 * NTILES * N <= 512, "accumulators exceed TMEM");
    static_assert(N == 32 || N == 64, "N");
    __host__ __device__ static constexpr int row0(int t) { return t < NTILES - 1 ? t * TILE_M : M_NEEDED - TILE_M; }   // the last tile overlaps its predecessor
    __host__ __device__ static constexpr int first_new_row(int t) { return t * TILE_M; }                                  // rows below were stored by the previous tile
};
//                         ROWS WIN PL TY TX OH  OW  N  B  NSTAGE ring  NCONV
using Conv1Geom = ConvGeom<441, 21, 8, 2, 2, 20, 20, 32, 1, 2, true, 8>;
using Conv2Geom = ConvGeom<100, 10, 16, 2, 2, 9, 9, 64, 2, 2, false, 0>;
using Conv3Geom = ConvGeom<81, 9, 8, 3, 3, 7, 7, 64, 3, 2, false, 0>;

// element offset of (item, plane, row) in a global plane buffer grouped in batches of B items: [batch][plane][item in batch][row][8]
template <class G>
__host__ __device__ __forceinline__ size_t plane_elem_offset(uint32_t item, uint32_t plane, uint32_t row) {
    return ((((size_t)(item / G::B) * G::PL + plane) * G::B + item % G::B) * G::ROWS + row) * 8;
}

// ---- epilogue targets: where the bf16 outputs of pixel (ox, oy) of an item go ---------------------------------
struct OutConv2Planes {              // conv1 -> conv2 input: space-to-depth by 2, channel = (oy&1, ox&1, c), row = (oy/2)*10 + ox/2
    __nv_bfloat16* out;
    __device__ __forceinline__ void store8(uint32_t item, uint32_t ox, uint32_t oy, uint32_t c0, uint4 v) const {
        const uint32_t plane = (((oy & 1u) * 2u + (ox & 1u)) * 32u + c0) >> 3, row = (oy >> 1) * 10u + (ox >> 1);
        *reinterpret_cast<uint4*>(out + plane_elem_offset<Conv2Geom>(item, plane, row)) = v;
    }
};
struct OutConv3Planes {              // conv2 -> conv3 input: row = oy*9 + ox
    __nv_bfloat16* out;
    __device__ __forceinline__ void store8(uint32_t item, uint32_t ox, uint32_t oy, uint32_t c0, uint4 v) const {
        *reinterpret_cast<uint4*>(out + plane_elem_offset<Conv3Geom>(item, c0 >> 3, oy * 9u + ox)) = v;
    }
};

struct ConvArgs {
    const uint8_t* w;                // prepared weights: bf16 [K/8 planes][N][8], K = tap * (8 PL) + channel
    const float* bias;               // [N]
    const uint8_t* in;               // FROM_RING: the u8 frame ring; else the plane buffer written by the previous layer
    GatherParams g;                  // FROM_RING: where the items are (current observations, or replay transitions by logical index)
    uint32_t which;                  // FROM_RING: 0 = the state of the item, 1 = its state_next
    uint32_t n_items;
    unsigned int* err;
    unsigned long long* prof;        // optional (QLC_QNET_PROF): CTA 0 writes per-role cycle counters [4 roles][8]
};

// four u8 pixels -> four bf16 (exact): byte k goes into the mantissa of 2^23, minus 2^23
__device__ __forceinline__ uint2 u8x4_to_bf16x4(uint32_t w) {
    const float f0 = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540)) - 8388608.0f;
    const float f1 = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7541)) - 8388608.0f;
    const float f2 = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7542)) - 8388608.0f;
    const float f3 = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7543)) - 8388608.0f;
    return make_uint2(pack_bf16(f0, f1), pack_bf16(f2, f3));
}

template <class G, class Out>
__global__ void __launch_bounds__(G::THREADS, 1) conv_sw_kernel(ConvArgs args, Out out) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* const s_w = smem;
    uint8_t* const s_in = s_w + G::W_BYTES;
    uint8_t* const s_raw = s_in + (size_t)G::NSTAGE * G::STAGE_BYTES;
    float* const s_bias = reinterpret_cast<float*>(s_raw + (G::FROM_RING ? (size_t)G::NRAW * G::RAW_BYTES : 0));
    uint32_t* const s_slot = reinterpret_cast<uint32_t*>(s_bias + 64);      // [NRAW][4] ring frame of each slot of the item in raw stage r (16-byte aligned)
    uint64_t* const bars = reinterpret_cast<uint64_t*>(s_slot + G::NRAW * 4);
    uint64_t* const w_full = bars;                       // [1]
    uint64_t* const in_full = w_full + 1;                // [NSTAGE]
    uint64_t* const in_empty = in_full + G::NSTAGE;      // [NSTAGE]
    uint64_t* const acc_full = in_empty + G::NSTAGE;     // [2 * NTILES]
    uint64_t* const acc_empty = acc_full + 2 * G::NTILES; // [2]
    uint64_t* const raw_full = acc_empty + 2;            // [NRAW]
    uint64_t* const raw_empty = raw_full + G::NRAW;      // [NRAW]
    uint32_t* const s_misc = reinterpret_cast<uint32_t*>(bars + G::NBAR);   // [0] TMEM base, [1] abort flag

    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
    const uint32_t n_batches = (args.n_items + G::B - 1) / G::B;

    if (tid == 0) {
        mbar_init(w_full, 1);
        for (int i = 0; i < G::NSTAGE; ++i) { mbar_init(&in_full[i], G::FROM_RING ? G::NCONV : 1); mbar_init(&in_empty[i], 1); }
        for (int i = 0; i < 2 * G::NTILES; ++i) mbar_init(&acc_full[i], 1);
        for (int i = 0; i < 2; ++i) mbar_init(&acc_empty[i], 4);
        for (int i = 0; i < G::NRAW; ++i) { mbar_init(&raw_full[i], 1); mbar_init(&raw_empty[i], G::FROM_RING ? G::NCONV : 1); }
        s_misc[1] = 0u;
        fence_mbar_init();
    }
    if (tid < (uint32_t)G::N) s_bias[tid] = args.bias[tid];
    if (warp == 4) tmem_alloc(&s_misc[0], G::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = s_misc[0];
    volatile uint32_t* const abort_flag = &s_misc[1];
    if (warp == 5 && lane == 0) {                        // weights are not produced by the previous kernel: fetch them during its tail
        mbar_expect_tx(w_full, G::W_BYTES);
        for (int off = 0; off < G::W_BYTES; off += 16384) bulk_load(s_w + off, args.w + off, (uint32_t)(G::W_BYTES - off < 16384 ? G::W_BYTES - off : 16384), w_full);
    }
    pdl_wait();
    // a wait that never hangs the GPU: on time-out raise the error flag and make every role leave its loop
    const bool prof_on = args.prof != nullptr && blockIdx.x == 0 && lane == 0;
    unsigned long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const long long t_begin = clock64();
    auto wait = [&](uint64_t* bar, uint32_t parity, int slot = 7) -> bool {
        const long long t0 = prof_on ? clock64() : 0;
        const bool done = mbar_wait_bounded(bar, parity);
        if (prof_on) pc[slot] += (unsigned long long)(clock64() - t0);
        if (done) return true;
        *abort_flag = 1u;
        if (args.err) atomicExch(args.err, 2u);
        return false;
    };

    if (warp < 4) {
        // ================= epilogue =================
        for (uint32_t it = 0, bi = blockIdx.x; bi < n_batches && !*abort_flag; ++it, bi += gridDim.x) {
            const uint32_t a = it & 1u, ph = (it >> 1) & 1u;
            #pragma unroll 1
            for (int t = 0; t < G::NTILES; ++t) {
                if (!wait(&acc_full[a * G::NTILES + t], ph, 1)) break;
                tc_fence_after();
                const uint32_t m = (uint32_t)G::row0(t) + warp * 32u + lane;
                const uint32_t ib = m / (uint32_t)G::ROWS, r = m - ib * (uint32_t)G::ROWS;
                const uint32_t oy = r / (uint32_t)G::WIN, ox = r - oy * (uint32_t)G::WIN;
                const uint32_t item = bi * G::B + ib;
                const bool ok = m >= (uint32_t)G::first_new_row(t) && ib < (uint32_t)G::B && ox < (uint32_t)G::OW && oy < (uint32_t)G::OH && item < args.n_items;
                #pragma unroll
                for (int half = 0; half < G::N / 32; ++half) {
                    uint32_t v[32];
                    tmem_ld32(tmem_base + ((warp * 32u) << 16) + (uint32_t)((a * G::NTILES + t) * G::N + half * 32), v);
                    if (ok) {
                        #pragma unroll
                        for (int c = 0; c < 32; c += 8) {
                            float f[8];
                            #pragma unroll
                            for (int i = 0; i < 8; ++i) f[i] = fmaxf(__uint_as_float(v[c + i]) + s_bias[half * 32 + c + i], 0.0f);
                            out.store8(item, ox, oy, (uint32_t)(half * 32 + c),
                                       make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7])));
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[a]);
        }
    } else if (warp == 4) {
        // ================= MMA issue =================
        // The whole warp runs the loop so that every operand of tcgen05.mma stays warp-uniform (uniform registers, no
        // per-instruction broadcast loop in SASS); one elected lane issues.
        // Loop control is kept provably warp-uniform too (votes on the wait results; the TMEM base through a warp reduction,
        // which lands in a uniform register).
        constexpr uint32_t IDESC = instr_desc_bf16(TILE_M, G::N);
        const uint32_t tmem_u = __reduce_max_sync(0xFFFFFFFFu, tmem_base);
        const bool live = __all_sync(0xFFFFFFFFu, wait(w_full, 0));
        for (uint32_t it = 0, bi = blockIdx.x; live && bi < n_batches; ++it, bi += gridDim.x) {
            const uint32_t s = it % G::NSTAGE, ph_in = (it / G::NSTAGE) & 1u, a = it & 1u, ph_acc = (it >> 1) & 1u;
            const bool ok = wait(&in_full[s], ph_in, 1) && wait(&acc_empty[a], ph_acc ^ 1u, 2);
            if (!__all_sync(0xFFFFFFFFu, ok)) break;
            tc_fence_after();
            // descriptor low words: start address >> 4 (shared-memory addresses are < 2^18, all offsets multiples of 16) | LBO << 16
            const uint32_t b_lo0 = (smem_u32(s_w) >> 4) | ((uint32_t)(G::N * 16 >> 4) << 16);
            const uint32_t a_lo0 = ((smem_u32(s_in) + s * (uint32_t)G::STAGE_BYTES) >> 4) | ((uint32_t)(G::PLANE_BYTES >> 4) << 16);
            #pragma unroll 1
            for (int t = 0; t < G::NTILES; ++t) {
                const uint32_t d_tmem = tmem_u + (uint32_t)((a * G::NTILES + t) * G::N);
                const uint32_t a_lo = a_lo0 + (uint32_t)G::row0(t);                       // one row = 16 bytes = 1 address unit
                #pragma unroll
                for (int tap = 0; tap < G::TAPS; ++tap) {
                    const uint32_t shift = (uint32_t)((tap / G::TX) * G::WIN + (tap % G::TX));
                    #pragma unroll
                    for (int kk = 0; kk < G::KSTEPS; ++kk)
                        tc_mma_bf16_elect_lo(d_tmem, a_lo + shift + (uint32_t)(2 * kk) * (G::PLANE_BYTES >> 4), b_lo0 + (uint32_t)((tap * G::PL + 2 * kk) * G::N),
                                             IDESC, (tap > 0 || kk > 0) ? 1u : 0u);
                }
                tc_commit_elect(&acc_full[a * G::NTILES + t]);
            }
            tc_commit_elect(&in_empty[s]);
        }
    } else if (warp == 5) {
        // ================= bulk-copy issue =================
        if (lane == 0) {
            // which frame of the ring holds ring slot h of an item's stack (~0u: not written yet in this episode, all zero) - the
            // rules of the gather kernels (locate(), kernels.cuh); one or two global loads per item, issued ahead of the wait below
            auto slot_table = [&](uint32_t item) -> uint4 { return slot_frames(args.g, item, args.which); };
            uint4 cur = make_uint4(0u, 0u, 0u, 0u);
            if constexpr (G::FROM_RING) { if (blockIdx.x < n_batches) cur = slot_table(blockIdx.x); }
            for (uint32_t it = 0, bi = blockIdx.x; bi < n_batches && !*abort_flag; ++it, bi += gridDim.x) {
                if constexpr (G::FROM_RING) {
                    const uint32_t r = it % G::NRAW, ph = (it / G::NRAW) & 1u;
                    uint4 nxt = make_uint4(0u, 0u, 0u, 0u);                  // the next item's slot table is worked out before the wait
                    if (bi + gridDim.x < n_batches) nxt = slot_table(bi + gridDim.x);
                    if (!wait(&raw_empty[r], ph ^ 1u, 1)) break;
                    const uint32_t fi[4] = {cur.x, cur.y, cur.z, cur.w};
                    *reinterpret_cast<uint4*>(s_slot + r * 4) = cur;         // published to the converters by the arrive below (release)
                    uint32_t nv = 0;
                    #pragma unroll
                    for (int h = 0; h < 4; ++h) nv += fi[h] != 0xFFFFFFFFu;
                    if (nv) {
                        mbar_expect_tx(&raw_full[r], nv * FRAME_BYTES);
                        #pragma unroll
                        for (int h = 0; h < 4; ++h)
                            if (fi[h] != 0xFFFFFFFFu) bulk_load(s_raw + (size_t)r * G::RAW_BYTES + h * FRAME_BYTES, args.in + (size_t)fi[h] * FRAME_BYTES, FRAME_BYTES, &raw_full[r]);
                    } else {
                        mbar_arrive(&raw_full[r]);
                    }
                    cur = nxt;
                } else {
                    const uint32_t s = it % G::NSTAGE, ph = (it / G::NSTAGE) & 1u;
                    if (!wait(&in_empty[s], ph ^ 1u, 1)) break;
                    mbar_expect_tx(&in_full[s], G::STAGE_BYTES);
                    const uint8_t* src = args.in + (size_t)bi * G::STAGE_BYTES;
                    uint8_t* dst = s_in + (size_t)s * G::STAGE_BYTES;
                    constexpr int CH = (G::STAGE_BYTES / 4 + 15) & ~15;
                    for (int off = 0; off < G::STAGE_BYTES; off += CH) bulk_load(dst + off, src + off, (uint32_t)(G::STAGE_BYTES - off < CH ? G::STAGE_BYTES - off : CH), &in_full[s]);
                }
            }
            pdl_launch_dependents();                     // this CTA's last input is on its way: the next kernel may start its prologue
        }
    } else {
        // ================= conv1: u8 ring frames -> bf16 planes, space-to-depth by 4 =================
        if constexpr (G::FROM_RING) {
            const uint32_t ct = (warp - 6u) * 32u + lane;
            constexpr uint32_t CT = G::NCONV * 32;
            for (uint32_t it = 0, bi = blockIdx.x; bi < n_batches && !*abort_flag; ++it, bi += gridDim.x) {
                const uint32_t r = it % G::NRAW, ph_r = (it / G::NRAW) & 1u, s = it % G::NSTAGE, ph_s = (it / G::NSTAGE) & 1u;
                if (!wait(&raw_full[r], ph_r, 1) || !wait(&in_empty[s], ph_s ^ 1u, 2)) break;
                const uint8_t* raw = s_raw + (size_t)r * G::RAW_BYTES;
                uint8_t* dst = s_in + (size_t)s * G::STAGE_BYTES;
                uint32_t present = 0;
                #pragma unroll
                for (uint32_t h = 0; h < 4; ++h) present |= (uint32_t)(s_slot[r * 4 + h] != 0xFFFFFFFFu) << h;
                // work item = (slot h, row pair q = y/2, X = x/4): 8 pixels = channels (y&1, x&3) of plane 2h + (q&1), row (q/2)*21 + X
                #pragma unroll 7
                for (uint32_t idx = ct; idx < 4u * 882u; idx += CT) {
                    const uint32_t h = idx / 882u, rem = idx - h * 882u, q = rem / 21u, X = rem - q * 21u;
                    uint32_t lo = 0u, hi = 0u;
                    if ((present >> h) & 1u) {
                        const uint8_t* p = raw + h * FRAME_BYTES + q * (2u * FRAME_W) + X * 4u;
                        lo = *reinterpret_cast<const uint32_t*>(p);
                        hi = *reinterpret_cast<const uint32_t*>(p + FRAME_W);
                    }
                    const uint2 a = u8x4_to_bf16x4(lo), b = u8x4_to_bf16x4(hi);
                    *reinterpret_cast<uint4*>(dst + (size_t)(2u * h + (q & 1u)) * G::PLANE_BYTES + ((q >> 1) * 21u + X) * 16u) = make_uint4(a.x, a.y, b.x, b.y);
                }
                fence_proxy_async_smem();          // generic-proxy writes -> visible to the tensor core (async proxy)
                __syncwarp();
                if (lane == 0) { mbar_arrive(&in_full[s]); mbar_arrive(&raw_empty[r]); }
            }
        }
    }
    if (prof_on && (warp == 0 || warp == 4 || warp == 5 || warp == 6)) {
        const int role = warp == 0 ? 0 : (int)warp - 3;               // 0 epilogue, 1 MMA, 2 loader, 3 converter
        pc[0] = (unsigned long long)(clock64() - t_begin);
        for (int i = 0; i < 8; ++i) args.prof[role * 8 + i] = pc[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) tmem_dealloc(tmem_base, G::TMEM_COLS);
}

// ---- weight preparation: Keras [kx][ky][cin][cout] f32 -> bf16 planes [K/8][N][8] in each layer's K order ---------------
// conv1: k = tap*64 + h*16 + iy*4 + ix, tap = dy*2 + dx, kernel index (kx = 4dx + ix, ky = 4dy + iy, h)
__global__ void prep_conv1_planes_kernel(const float* __restrict__ kernel /*[8][8][4][32]*/, __nv_bfloat16* __restrict__ w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 256 * 32) return;
    const int e = i & 7, n = (i >> 3) % 32, k = (i / 256) * 8 + e;
    const int tap = k / 64, c = k % 64, dy = tap / 2, dx = tap % 2, h = c / 16, iy = (c / 4) % 4, ix = c % 4;
    w[i] = __float2bfloat16_rn(kernel[(((4 * dx + ix) * 8 + (4 * dy + iy)) * 4 + h) * 32 + n]);
}
// conv2: k = tap*128 + (iy*2 + ix)*32 + ci, tap = dy*2 + dx, kernel index (kx = 2dx + ix, ky = 2dy + iy, ci)
__global__ void prep_conv2_planes_kernel(const float* __restrict__ kernel /*[4][4][32][64]*/, __nv_bfloat16* __restrict__ w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 512 * 64) return;
    const int e = i & 7, n = (i >> 3) % 64, k = (i / 512) * 8 + e;
    const int tap = k / 128, c = k % 128, dy = tap / 2, dx = tap % 2, iy = c / 64, ix = (c / 32) % 2, ci = c % 32;
    w[i] = __float2bfloat16_rn(kernel[(((2 * dx + ix) * 4 + (2 * dy + iy)) * 32 + ci) * 64 + n]);
}
// conv3: k = tap*64 + ci, tap = dy*3 + dx, kernel index (kx = dx, ky = dy, ci)
__global__ void prep_conv3_planes_kernel(const float* __restrict__ kernel /*[3][3][64][64]*/, __nv_bfloat16* __restrict__ w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 576 * 64) return;
    const int e = i & 7, n = (i >> 3) % 64, k = (i / 512) * 8 + e;
    const int tap = k / 64, ci = k % 64, dy = tap / 3, dx = tap % 3;
    w[i] = __float2bfloat16_rn(kernel[((dx * 3 + dy) * 64 + ci) * 64 + n]);
}


// =========================================================================================================
// Dense 3136 -> 512 (+ ReLU) as a bulk-copy fed tcgen05 GEMM. A (conv3's output, Keras Flatten order) and W live in global
// memory already in the shared-memory operand layout, so one stage = one contiguous bulk copy per operand:
//   A: [M tile = item / 128][K chunk j = k / 8 (392)][item % 128][8]      (written by conv3's epilogue, OutDensePlanes)
//   W: [N tile (4)][j (392)][n % 128][8]                                  (prep_dense_planes_kernel)
// One CTA = one (M tile, N tile of NT): 128 items x NT outputs, K = 3136 in 49 stages of 64 through a 6- / 4-deep ring. The
// layer is bound by what one SM can pull from L2 (~53 B/clk measured): with NT = 256 only 64 CTAs exist at 4,096 items and
// each has to ingest 2.35 MB (24 us); NT = 128 gives 128 CTAs x 1.57 MB (18 us) but re-reads A twice as often, so it is
// used while (M tiles x 2) CTAs would not fill the SMs and NT = 256 beyond. The MMAs (64 / 128 cycles per K = 16 at
// N = 128 / 256, the tensor-pipe rate) are hidden behind the copies.
// =========================================================================================================
template <int NT_>
struct DenseGeomT {
    static constexpr int K = 3136, N = 512, NT = NT_, KSTAGE = 64, NSTAGE = NT_ == 128 ? 6 : 4;
    static constexpr int PLANES = K / 8, STAGES_K = K / KSTAGE;             // 392 planes, 49 stages
    static constexpr int A_STAGE = (KSTAGE / 8) * TILE_M * 16;               // 16 KB
    static constexpr int B_STAGE = (KSTAGE / 8) * NT * 16;                   // 16 / 32 KB
    static constexpr int A_TILE_BYTES = PLANES * TILE_M * 16;                // one M tile of A
    static constexpr int THREADS = 192;
    static constexpr size_t SMEM_BYTES = (size_t)NSTAGE * (A_STAGE + B_STAGE) + NT * 4 + 3 * NT * 4 + (2 * NSTAGE + 1) * 8 + 16;
};
struct HeadArgs {                    // Dense 512 -> 3 (+ argmax / max) fused into the dense layer's epilogue
    const float* w;                  // [3][512] f32 (prep_head_kernel)
    const float* bias;               // [3]
    float4* partial;                 // [N tiles][rows_padded]: per-N-tile partial dot products of every row
    uint32_t* row_count;             // [rows_padded], zero between forwards: how many N tiles have delivered a row
    uint32_t rows_padded;
    float* q; uint8_t* action; float* max_q;   // outputs (any may be NULL)
};
using DenseGeom = DenseGeomT<128>;   // A-side constants (PLANES, A_TILE_BYTES) do not depend on NT
struct OutDensePlanes {              // conv3 -> dense A operand, k = (ox*7 + oy)*64 + c
    __nv_bfloat16* out;
    __device__ __forceinline__ void store8(uint32_t item, uint32_t ox, uint32_t oy, uint32_t c0, uint4 v) const {
        const uint32_t j = ((ox * 7u + oy) * 64u + c0) >> 3;
        *reinterpret_cast<uint4*>(out + (((size_t)(item >> 7) * DenseGeom::PLANES + j) * TILE_M + (item & 127u)) * 8) = v;
    }
};

template <int NT>
__global__ void __launch_bounds__(DenseGeomT<NT>::THREADS, 1) dense_tc_kernel(const uint8_t* __restrict__ a_planes, const uint8_t* __restrict__ w_planes,
                                                                         const float* __restrict__ bias, __nv_bfloat16* __restrict__ out /*[items][512] or NULL*/,
                                                                         uint32_t n_items, unsigned int* err, HeadArgs head) {
    using G = DenseGeomT<NT>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* const s_a = smem;
    uint8_t* const s_b = s_a + (size_t)G::NSTAGE * G::A_STAGE;
    float* const s_bias = reinterpret_cast<float*>(s_b + (size_t)G::NSTAGE * G::B_STAGE);
    float* const s_w5 = s_bias + G::NT;                  // [3][NT]: this N tile's slice of the head weights
    uint64_t* const full = reinterpret_cast<uint64_t*>(s_w5 + 3 * G::NT);
    uint64_t* const empty = full + G::NSTAGE;
    uint64_t* const acc_full = empty + G::NSTAGE;
    uint32_t* const s_misc = reinterpret_cast<uint32_t*>(acc_full + 1);
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
    const uint32_t mtile = blockIdx.x, nhalf = blockIdx.y;       // nhalf: index of the N tile

    if (tid == 0) {
        for (int i = 0; i < G::NSTAGE; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(acc_full, 1);
        fence_mbar_init();
    }
    for (uint32_t i = tid; i < (uint32_t)G::NT; i += G::THREADS) s_bias[i] = bias[nhalf * G::NT + i];
    for (uint32_t i = tid; i < 3u * G::NT; i += G::THREADS) s_w5[i] = head.w[(i / G::NT) * G::N + nhalf * G::NT + i % G::NT];
    if (warp == 4) tmem_alloc(&s_misc[0], G::NT);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = s_misc[0];
    pdl_launch_dependents();
    pdl_wait();
    auto wait = [&](uint64_t* bar, uint32_t parity) -> bool {
        if (mbar_wait_bounded(bar, parity)) return true;
        if (err) atomicExch(err, 3u);
        return false;
    };

    if (warp < 4) {
        // epilogue: row = item, NT columns in pieces of 32: bias + ReLU, bf16; the head (Dense 512 -> 3) is applied to the rounded
        // activations on the fly. Each N tile leaves a partial dot product per row; the tile that delivers a row last (per-row
        // ticket) adds the partials in tile order - deterministic - and writes Q, the greedy action and max Q.
        if (wait(acc_full, 0)) {
            tc_fence_after();
            const uint32_t item = mtile * TILE_M + warp * 32u + lane;
            float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
            #pragma unroll 1
            for (int piece = 0; piece < G::NT / 32; ++piece) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((warp * 32u) << 16) + (uint32_t)(piece * 32), v);
                if (item < n_items) {
                    #pragma unroll
                    for (int c = 0; c < 32; c += 8) {
                        uint32_t pk[4];
                        #pragma unroll
                        for (int i = 0; i < 8; i += 2) {
                            const int col = piece * 32 + c + i;
                            const uint32_t p2 = pack_bf16(fmaxf(__uint_as_float(v[c + i]) + s_bias[col], 0.0f), fmaxf(__uint_as_float(v[c + i + 1]) + s_bias[col + 1], 0.0f));
                            pk[i >> 1] = p2;
                            const float h0 = __uint_as_float(p2 << 16), h1 = __uint_as_float(p2 & 0xFFFF0000u);      // the bf16-rounded activations
                            s0 += h0 * s_w5[col] + h1 * s_w5[col + 1];
                            s1 += h0 * s_w5[G::NT + col] + h1 * s_w5[G::NT + col + 1];
                            s2 += h0 * s_w5[2 * G::NT + col] + h1 * s_w5[2 * G::NT + col + 1];
                        }
                        if (out) *reinterpret_cast<uint4*>(out + (size_t)item * G::N + nhalf * G::NT + piece * 32 + c) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                }
            }
            if (item < n_items) {
                constexpr uint32_t NTILES = G::N / G::NT;
                head.partial[(size_t)nhalf * head.rows_padded + item] = make_float4(s0, s1, s2, 0.0f);
                __threadfence();
                if (atomicAdd(&head.row_count[item], 1u) == NTILES - 1u) {
                    __threadfence();
                    float q0 = 0.0f, q1 = 0.0f, q2 = 0.0f;
                    #pragma unroll
                    for (uint32_t t = 0; t < NTILES; ++t) {
                        const float4 p = __ldcg(&head.partial[(size_t)t * head.rows_padded + item]);
                        q0 += p.x; q1 += p.y; q2 += p.z;
                    }
                    q0 += head.bias[0]; q1 += head.bias[1]; q2 += head.bias[2];
                    if (head.q) { head.q[(size_t)item * 3] = q0; head.q[(size_t)item * 3 + 1] = q1; head.q[(size_t)item * 3 + 2] = q2; }
                    if (head.action) head.action[item] = (uint8_t)(q1 > q0 ? (q2 > q1 ? 2 : 1) : (q2 > q0 ? 2 : 0));     // first maximum, like tf.argmax
                    if (head.max_q) head.max_q[item] = fmaxf(q0, fmaxf(q1, q2));                                          // tf.reduce_max
                    head.row_count[item] = 0u;                         // ready for the next forward pass
                }
            }
        }
    } else if (warp == 4) {
        constexpr uint32_t IDESC = instr_desc_bf16(TILE_M, G::NT);
        const uint32_t tmem_u = __reduce_max_sync(0xFFFFFFFFu, tmem_base);
        for (uint32_t st = 0; st < (uint32_t)G::STAGES_K; ++st) {
            const uint32_t s = st % G::NSTAGE, ph = (st / G::NSTAGE) & 1u;
            if (!__all_sync(0xFFFFFFFFu, wait(&full[s], ph))) break;
            tc_fence_after();
            const uint32_t a_lo0 = ((smem_u32(s_a) + s * (uint32_t)G::A_STAGE) >> 4) | ((uint32_t)(TILE_M * 16 >> 4) << 16);
            const uint32_t b_lo0 = ((smem_u32(s_b) + s * (uint32_t)G::B_STAGE) >> 4) | ((uint32_t)(G::NT * 16 >> 4) << 16);
            #pragma unroll
            for (int kk = 0; kk < G::KSTAGE / 16; ++kk)
                tc_mma_bf16_elect_lo(tmem_u, a_lo0 + (uint32_t)(2 * kk) * (TILE_M * 16 >> 4), b_lo0 + (uint32_t)(2 * kk) * (G::NT * 16 >> 4), IDESC, (st > 0 || kk > 0) ? 1u : 0u);
            tc_commit_elect(&empty[s]);
        }
        tc_commit_elect(acc_full);
    } else if (lane == 0) {
        const uint8_t* a_src = a_planes + (size_t)mtile * G::A_TILE_BYTES;
        const uint8_t* b_src = w_planes + (size_t)nhalf * G::PLANES * G::NT * 16;
        for (uint32_t st = 0; st < (uint32_t)G::STAGES_K; ++st) {
            const uint32_t s = st % G::NSTAGE, ph = (st / G::NSTAGE) & 1u;
            if (!wait(&empty[s], ph ^ 1u)) break;
            mbar_expect_tx(&full[s], G::A_STAGE + G::B_STAGE);
            bulk_load(s_a + (size_t)s * G::A_STAGE, a_src + (size_t)st * G::A_STAGE, G::A_STAGE, &full[s]);
            bulk_load(s_b + (size_t)s * G::B_STAGE, b_src + (size_t)st * G::B_STAGE, G::B_STAGE / 2, &full[s]);
            bulk_load(s_b + (size_t)s * G::B_STAGE + G::B_STAGE / 2, b_src + (size_t)st * G::B_STAGE + G::B_STAGE / 2, G::B_STAGE / 2, &full[s]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) tmem_dealloc(tmem_base, G::NT);
}

// Keras dense kernel [3136][512] f32 -> bf16 [N tile][j][n % NT][8]
template <int NT>
__global__ void prep_dense_planes_kernel(const float* __restrict__ kernel, __nv_bfloat16* __restrict__ w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 3136 * 512) return;
    const int e = i & 7, nt = (i >> 3) % NT, j = (i / (8 * NT)) % 392, tile = i / (392 * 8 * NT);
    w[i] = __float2bfloat16_rn(kernel[(size_t)(j * 8 + e) * 512 + tile * NT + nt]);
}

// Dense 512 -> 3 + argmax over bf16 activations [M][512], one warp per row with 16-byte loads
__global__ void __launch_bounds__(256) head_vec_kernel(const __nv_bfloat16* __restrict__ act, const float* __restrict__ w /*[3][512]*/, const float* __restrict__ bias,
                                                       float* __restrict__ q, uint8_t* __restrict__ action, float* __restrict__ max_q, uint32_t m_total) {
    __shared__ float sw[3 * 512];
    for (uint32_t i = threadIdx.x; i < 3u * 512u; i += blockDim.x) sw[i] = w[i];
    __syncthreads();
    pdl_launch_dependents();
    pdl_wait();
    const uint32_t lane = threadIdx.x & 31u, wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nw = gridDim.x * (blockDim.x >> 5);
    for (uint32_t row = wid; row < m_total; row += nw) {
        float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
        #pragma unroll
        for (int part = 0; part < 2; ++part) {
            const uint32_t k0 = (uint32_t)part * 256u + lane * 8u;
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(act + (size_t)row * 512 + k0));
            const uint32_t u[4] = {v.x, v.y, v.z, v.w};
            #pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float a0 = __uint_as_float(u[i] << 16), a1 = __uint_as_float(u[i] & 0xFFFF0000u);
                const uint32_t k = k0 + 2 * i;
                s0 += a0 * sw[k] + a1 * sw[k + 1]; s1 += a0 * sw[512 + k] + a1 * sw[512 + k + 1]; s2 += a0 * sw[1024 + k] + a1 * sw[1024 + k + 1];
            }
        }
        for (int o = 16; o; o >>= 1) { s0 += __shfl_down_sync(~0u, s0, o); s1 += __shfl_down_sync(~0u, s1, o); s2 += __shfl_down_sync(~0u, s2, o); }
        if (lane == 0) {
            s0 += bias[0]; s1 += bias[1]; s2 += bias[2];
            if (q) { q[(size_t)row * 3] = s0; q[(size_t)row * 3 + 1] = s1; q[(size_t)row * 3 + 2] = s2; }
            if (action) action[row] = (uint8_t)(s1 > s0 ? (s2 > s1 ? 2 : 1) : (s2 > s0 ? 2 : 0));     // first maximum, like tf.argmax
            if (max_q) max_q[row] = fmaxf(s0, fmaxf(s1, s2));                                          // tf.reduce_max
        }
    }
}

}  // namespace qnet
}  // namespace qlc
