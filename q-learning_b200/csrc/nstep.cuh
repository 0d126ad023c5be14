// nstep.cuh — n-step returns and double-DQN targets read straight from the record ring (DESIGN §14).
//
// Logical index i names time T = t_oldest + i / N and env e = i mod N (locate()); its n-step successor is i + N, so a return is a
// strided walk over the u32 records [time_slots][N]. The walk over R_j = record (T + j, e) stops at the first j where R_j is done
// (terminal), R_j is truncated, j = n_step - 1, T + j is the newest time in the replay, or R_{j+1} starts an episode
// (min(k,4) = 0: a reset by the caller). Then m = j + 1, G = sum_j gamma^j r_j, disc = gamma^m (0 where terminal) and the
// bootstrap state is state_next of boot = i + (m - 1) N. The kernel is elementwise and uses no atomics: deterministic. The
// targets y are formed by qnet::target_kernel (qnet_train.cuh).
#pragma once
#include "kernels.cuh"
#include "qnet_conv.cuh"     // pdl_wait / pdl_launch_dependents

namespace qlc {
namespace nstep {

using qnet::pdl_launch_dependents;
using qnet::pdl_wait;

constexpr uint32_t CHUNK = 8;     // records loaded ahead of the stop test (independent loads, one round trip per chunk)

// G [n], disc [n], boot [n] of the items g.indices [g.n_items] (any output may be NULL). An index >= len: 0, 0, idx.
// -fmad=false: pw * r rounds before the add, pw * gamma is its own rounding.
__global__ void nstep_kernel(GatherParams g, uint32_t n_step, float gamma, float* __restrict__ ret, float* __restrict__ disc, uint32_t* __restrict__ boot) {
    pdl_launch_dependents(); pdl_wait();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n_items) return;
    const uint32_t idx = g.indices[i];
    uint64_t T; uint32_t e, k, cur;
    float G = 0.0f, d = 0.0f;
    uint32_t m = 1;
    if (locate(g, i, idx, T, e, k, cur)) {
        const uint64_t last = g.t_now - 1 - T;                        // j of the newest time in the replay
        const uint32_t j_max = (uint32_t)(last < n_step - 1u ? last : n_step - 1u);
        uint32_t slot = (uint32_t)(T % g.time_slots);
        float pw = 1.0f;
        bool terminal = false;
        for (uint32_t j0 = 0;; j0 += CHUNK) {
            uint32_t nxt[CHUNK];                                      // R_{j0+1 .. j0+CHUNK}; 0 beyond j_max (the walk stops first)
            uint32_t s = slot;
            #pragma unroll
            for (uint32_t c = 0; c < CHUNK; ++c) {
                s = s + 1u == g.time_slots ? 0u : s + 1u;
                nxt[c] = j0 + c + 1u <= j_max ? __ldg(g.records + (size_t)s * g.n_envs + e) : 0u;
            }
            bool stop = false;
            #pragma unroll
            for (uint32_t c = 0; c < CHUNK; ++c) {
                if (stop) continue;
                const uint32_t j = j0 + c;
                G = G + pw * (float)((cur >> 8) & 0xFFu);
                pw = pw * gamma;
                terminal = (cur >> 2) & 1u;
                stop = terminal || (cur & 0x10000u) || j == j_max || ((nxt[c] >> 5) & 7u) == 0u;
                if (stop) m = j + 1u;
                cur = nxt[c];
            }
            if (stop) break;
            slot = s;
        }
        d = terminal ? 0.0f : pw;
    }
    if (ret) ret[i] = G;
    if (disc) disc[i] = d;
    if (boot) boot[i] = idx + (m - 1u) * g.n_envs;
}

}  // namespace nstep
}  // namespace qlc
