// qlc_api.cu — C ABI (include/ql_cuda.h) over the sm_100a kernels. No CPU fallback: every entry point that
// computes needs a CUDA device and fails with QLC_ERR_NO_DEVICE / QLC_ERR_CUDA otherwise.
#include "../../include/ql_cuda.h"
#include "kernels.cuh"
#include "qnet.cuh"
#include "qnet_conv.cuh"
#include "qnet_train.cuh"
#include "per.cuh"
#include "nstep.cuh"
#include "host_pool.h"
#include "comm.h"

#include <nvtx3/nvToolsExt.h>   // header-only; ranges cost a few ns unless a tool (ncu --nvtx, nsys) is attached

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <string>
#include <vector>

using namespace qlc;

#ifndef QLC_SRC_HASH
#define QLC_SRC_HASH "unknown"
#endif
#ifdef QLC_PROFILING
#define QLC_PROFILING_STR "1"
#else
#define QLC_PROFILING_STR "0"
#endif
// build.py reads this marker out of the file to tell a stale library from a current one without loading it
extern "C" const char qlc_build_info_string[] = "QLC_BUILD_INFO:src_hash=" QLC_SRC_HASH ";profiling=" QLC_PROFILING_STR ";";

static thread_local std::string g_last_error;

static int32_t fail(int32_t code, const std::string& msg) { g_last_error = msg; return code; }
#define CUDA_TRY(expr)                                                                                       \
    do {                                                                                                     \
        cudaError_t _e = (expr);                                                                             \
        if (_e != cudaSuccess)                                                                               \
            return fail(QLC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));                   \
    } while (0)

// one NVTX range per public entry point that launches work ("qlc_env_step", "qlc_replay_gather", ...): lets ncu / nsys filter by call
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
#define QLC_RANGE(name) NvtxRange _qlc_nvtx_range(name)

struct qlc_env {
    qlc_config cfg;
    EnvArrays st{};
    uint8_t* frames = nullptr;
    uint32_t* records = nullptr;
    DeviceStats* stats = nullptr;
    unsigned long long* scratch = nullptr;     // 8 x u64 device scratch (histogram, err OR)
    RasterTables* tables = nullptr;            // raster tables, built once on the device
    unsigned int* work_counter = nullptr;      // dynamic work hand-out of the step kernel
    uint32_t work_base = 0;
    unsigned long long* progress = nullptr;    // per env batch: launch serial << 32 | steps done (time-chunk hand-over flag)
    unsigned int* spin_error = nullptr;
    uint32_t launch_serial = 0;
    int chunk_override = -1;                   // QLC_CHUNK: force the chunk length (0 = off)
    uint64_t submit_seq = 0;                   // qlc_env_step_host_submit calls so far
    cudaEvent_t submit_done[8] = {};           // completion of submit k in slot k % 8 (created on first use)
    cudaStream_t copy_stream = nullptr;        // pipelined submits: the H2D of step k+1 runs beside the kernel of step k
    cudaEvent_t h2d_done[2] = {};
    cudaEvent_t piece_ev[16] = {};             // host gathers: "piece i of the stacks has arrived" while the next ones are still in flight
    int zero_copy = 1;                         // QLC_ZERO_COPY=0: always stage page-locked outputs through a D2H copy
    uint32_t time_slots = 0;                   // frame/record ring length in time steps (= t_cap + 4)
    uint32_t t_cap = 0;                        // replay capacity in time steps
    uint64_t t = 0;                            // env-steps taken per env (global time)
    cudaStream_t own_stream = nullptr;         // used by the *_host entry points
    cudaEvent_t caller_done = nullptr;         // recorded after the launches of every asynchronous call; own_stream waits for it
    bool submits_pending = false;              // submitted host steps may still be running on own_stream
    // pinned staging for the host-buffer entry points
    void* pin = nullptr; size_t pin_bytes = 0;
    std::vector<qlc_host::StreamPiece> stream_pieces;
    uint32_t flag_serial = 0;                  // streamed host gathers: value the kernel raises its arrival flags to (never 0)
    void* dev_stage = nullptr; size_t dev_stage_bytes = 0;
    // episode reward window (replay_buffer.rs:100-124) — host side, fed by the caller like the reference
    std::deque<float> window;
    int advance_cfg = 0;                       // QLC_ADVANCE_CFG: force a CTA shape (0 = auto)
    int epc_override = 0;                      // QLC_EPC: force envs per CTA (0 = auto)
    int sm_count = 148;
    int debug_skip = 0;                        // QLC_DEBUG_SKIP (profiling aid)
    unsigned long long* timeline = nullptr;    // profiling builds with QLC_TIMELINE_FILE: clock stamps of the last step launch, dumped at destroy
    int persistent = 1;                        // QLC_PERSISTENT=0: one CTA per env batch
    std::vector<void*> allocs;
    std::vector<struct qlc_qnet*> qnets;       // Q-networks created on this env: invalidated (not dangling) when the env goes first
    std::vector<struct qlc_per*> pers;         // prioritized-replay trees over this env's ring: the same
    uint64_t generation = 0;                   // raised by qlc_env_load: the ring's contents were replaced (the trees rebuild)
    // episode-statistics reduction over the env shards (qlc_comm_init / qlc_stats_allreduce): NCCL on a side stream, off the step path
    struct Comm {
        qlc_comm::Comm nccl = nullptr; int rank = 0, world = 1;
        cudaStream_t stream = nullptr;
        DeviceStats* snap = nullptr;           // 4 snapshot slots, written by the last CTA of launch k into slot k % 4
        unsigned int* exit_counter = nullptr; uint32_t exit_base = 0;
        cudaEvent_t step_done = nullptr;       // recorded on the caller's step stream by qlc_stats_allreduce
        cudaEvent_t slot_read[4] = {};         // the reduction that read slot i has finished with it
        bool slot_busy[4] = {};
        double *mine = nullptr, *gathered = nullptr, *reduced = nullptr;   // device: [5], [world][5], [5]
        double* host = nullptr;                // page-locked mirror of `reduced`
        uint64_t reductions = 0;
        bool armed = false;                    // a reduction followed the previous launch: this one takes a snapshot too
        uint32_t last_serial = 0; bool have_snap = false;
    }* comm = nullptr;
};
static void qnet_release_device(struct qlc_qnet* q);
static void per_release_device(struct qlc_per* p);

static int32_t ensure_pin(qlc_env* env, size_t bytes) {
    if (bytes <= env->pin_bytes) return QLC_OK;
    if (env->pin) cudaFreeHost(env->pin);
    env->pin = nullptr; env->pin_bytes = 0;
    CUDA_TRY(cudaMallocHost(&env->pin, bytes));
    memset(env->pin, 0, bytes);                // streamed gathers keep arrival flags in here: a fresh block must not hold a serial by accident
    env->pin_bytes = bytes;
    return QLC_OK;
}
// launch with programmatic stream serialization: the kernel's prologue may overlap the tail of its predecessor in the stream
// (every kernel launched this way calls griddepcontrol.wait before it touches anything the predecessor wrote)
template <class... KArgs, class... Args>
static cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
    static const bool enabled = getenv("QLC_PDL") ? atoi(getenv("QLC_PDL")) != 0 : true;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = enabled ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

static int32_t ensure_dev_stage(qlc_env* env, size_t bytes) {
    if (bytes <= env->dev_stage_bytes) return QLC_OK;
    if (env->dev_stage) cudaFree(env->dev_stage);
    env->dev_stage = nullptr; env->dev_stage_bytes = 0;
    CUDA_TRY(cudaMalloc(&env->dev_stage, bytes));
    env->dev_stage_bytes = bytes;
    return QLC_OK;
}

template <typename T>
static int32_t dev_alloc(qlc_env* env, T** p, size_t count, bool zero) {
    void* q = nullptr;
    CUDA_TRY(cudaMalloc(&q, count * sizeof(T)));
    env->allocs.push_back(q);
    if (zero) CUDA_TRY(cudaMemset(q, 0, count * sizeof(T)));
    *p = reinterpret_cast<T*>(q);
    return QLC_OK;
}

extern "C" {

int32_t qlc_version(void) { return QLC_VERSION; }
const char* qlc_build_info(void) { return qlc_build_info_string + sizeof("QLC_BUILD_INFO:") - 1; }
const char* qlc_last_error_string(void) { return g_last_error.c_str(); }

int32_t qlc_device_count(int32_t* count) {
    if (!count) return fail(QLC_ERR_INVALID_ARG, "count is null");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *count = 0; return fail(QLC_ERR_NO_DEVICE, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e)); }
    *count = n;
    return QLC_OK;
}

float qlc_env_goal_mean(void) { return 59.0f; }   // (bricks.len() - 1) as f32, breakout_environment.rs:203-206

static int32_t set_device(const qlc_env* env) { CUDA_TRY(cudaSetDevice(env->cfg.device)); return QLC_OK; }

// Stream order (ql_cuda.h): the caller's stream and own_stream are not ordered by CUDA (own_stream is non-blocking), and the
// device-pointer calls resolve times and indices against env->t when they are queued. So an asynchronous call first waits for
// the newest submitted host step still in flight and ends with a record of caller_done on the caller's stream; a host-buffer
// call first makes own_stream wait for caller_done. An event stays valid after the caller destroys its stream; a remembered
// stream handle would not.
}  // extern "C"
template <class F>
static int32_t on_caller_stream(qlc_env* env, void* stream, F&& launches) {
    const cudaStream_t s = (cudaStream_t)stream;
    int32_t rc = set_device(env); if (rc) return rc;
    if (env->submits_pending) CUDA_TRY(cudaStreamWaitEvent(s, env->submit_done[(env->submit_seq - 1) % 8], 0));   // in order: older ones are done too
    rc = launches(); if (rc) return rc;
    CUDA_TRY(cudaEventRecord(env->caller_done, s));
    return QLC_OK;
}
extern "C" {
static int32_t after_caller_stream(qlc_env* env) {
    CUDA_TRY(cudaStreamWaitEvent(env->own_stream, env->caller_done, 0));
    return QLC_OK;
}

static int32_t launch_reset(qlc_env* env, const uint8_t* mask_dev, const float* dir_dev, int first_time, cudaStream_t s) {
    const uint32_t n = env->cfg.n_envs;
    env_reset_kernel<<<(n + 255) / 256, 256, 0, s>>>(env->st, n, env->cfg.env_id_base, env->cfg.seed, mask_dev, dir_dev, first_time);
    CUDA_TRY(cudaGetLastError());
    return QLC_OK;
}

int32_t qlc_env_create(const qlc_config* cfg, qlc_env** out) {
    if (!cfg || !out) return fail(QLC_ERR_INVALID_ARG, "cfg/out is null");
    *out = nullptr;
    if (cfg->struct_size != sizeof(qlc_config)) return fail(QLC_ERR_INVALID_ARG, "qlc_config.struct_size mismatch");
    if (cfg->n_envs == 0) return fail(QLC_ERR_INVALID_ARG, "n_envs must be > 0");
    if (cfg->frame_w != QLC_FRAME_W || cfg->frame_h != QLC_FRAME_H) return fail(QLC_ERR_INVALID_ARG, "only 84x84 frames are supported");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(QLC_ERR_NO_DEVICE, "no CUDA device: ql_cuda has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(QLC_ERR_INVALID_ARG, "device ordinal out of range");
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) return fail(QLC_ERR_NO_DEVICE, "ql_cuda is built for sm_100a (B200) only");

    qlc_env* env = new qlc_env();
    env->cfg = *cfg;
    if (env->cfg.episode_window == 0) env->cfg.episode_window = 100;
    int32_t rc = set_device(env);
    if (rc) { delete env; return rc; }
    const uint32_t n = cfg->n_envs;
    uint64_t t_cap = cfg->replay_capacity / n;
    if (t_cap == 0) t_cap = 1;
    if (t_cap > 0x7FFFFFF0ull) { delete env; return fail(QLC_ERR_INVALID_ARG, "replay_capacity too large"); }
    env->t_cap = (uint32_t)t_cap;
    env->time_slots = env->t_cap + 4;
    if (const char* c = getenv("QLC_ADVANCE_CFG")) env->advance_cfg = atoi(c);
    if (const char* c = getenv("QLC_EPC")) env->epc_override = atoi(c);
#ifdef QLC_PROFILING
    if (const char* c = getenv("QLC_DEBUG_SKIP")) env->debug_skip = atoi(c);      // ablation builds only; a release build ignores the variable
#endif
    if (const char* c = getenv("QLC_PERSISTENT")) env->persistent = atoi(c);
    if (const char* c = getenv("QLC_CHUNK")) env->chunk_override = atoi(c);
    if (const char* c = getenv("QLC_ZERO_COPY")) env->zero_copy = atoi(c);
    env->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;

#define TRY_ALLOC(x) do { rc = (x); if (rc) { qlc_env_destroy(env); return rc; } } while (0)
    TRY_ALLOC(dev_alloc(env, &env->st.ball_cx, n, false));
    TRY_ALLOC(dev_alloc(env, &env->st.ball_cy, n, false));
    TRY_ALLOC(dev_alloc(env, &env->st.ball_dx, n, false));
    TRY_ALLOC(dev_alloc(env, &env->st.ball_dy, n, false));
    TRY_ALLOC(dev_alloc(env, &env->st.pad_min_x, n, false));
    TRY_ALLOC(dev_alloc(env, &env->st.pad_max_x, n, false));
    TRY_ALLOC(dev_alloc(env, &env->st.pad_speed, n, false));
    TRY_ALLOC(dev_alloc(env, &env->st.bricks, n, false));
    TRY_ALLOC(dev_alloc(env, &env->st.score, n, true));
    TRY_ALLOC(dev_alloc(env, &env->st.episode_step, n, true));
    TRY_ALLOC(dev_alloc(env, &env->st.episode, n, true));
    TRY_ALLOC(dev_alloc(env, &env->st.err, n, true));
    TRY_ALLOC(dev_alloc(env, &env->st.finished, n, true));
    TRY_ALLOC(dev_alloc(env, &env->frames, (size_t)env->time_slots * n * FRAME_BYTES, false));
    TRY_ALLOC(dev_alloc(env, &env->records, (size_t)env->time_slots * n, true));
    TRY_ALLOC(dev_alloc(env, &env->stats, 1, false));
    TRY_ALLOC(dev_alloc(env, &env->scratch, 8, true));
    TRY_ALLOC(dev_alloc(env, &env->work_counter, 1, true));
    TRY_ALLOC(dev_alloc(env, &env->tables, 1, false));
    TRY_ALLOC(dev_alloc(env, &env->progress, n, true));
    TRY_ALLOC(dev_alloc(env, &env->spin_error, 1, true));
#undef TRY_ALLOC
    cudaError_t ce = cudaStreamCreateWithFlags(&env->own_stream, cudaStreamNonBlocking);
    if (ce != cudaSuccess) { qlc_env_destroy(env); return fail(QLC_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(ce)); }
    ce = cudaEventCreateWithFlags(&env->caller_done, cudaEventDisableTiming);
    if (ce != cudaSuccess) { qlc_env_destroy(env); return fail(QLC_ERR_CUDA, std::string("cudaEventCreate: ") + cudaGetErrorString(ce)); }
    DeviceStats init{0ull, 0ull, 0xFFFFFFFFu, 0u};
    ce = cudaMemcpy(env->stats, &init, sizeof init, cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) { qlc_env_destroy(env); return fail(QLC_ERR_CUDA, std::string("stats init: ") + cudaGetErrorString(ce)); }
#ifdef QLC_PROFILING
    if (getenv("QLC_TIMELINE_FILE")) { rc = dev_alloc(env, &env->timeline, 1024 * 16, true); if (rc) { qlc_env_destroy(env); return rc; } }
#endif
    raster_tables_kernel<<<1, 128>>>(env->tables);
    rc = launch_reset(env, nullptr, nullptr, 1, nullptr);
    if (rc) { qlc_env_destroy(env); return rc; }
    ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) { qlc_env_destroy(env); return fail(QLC_ERR_CUDA, std::string("create sync: ") + cudaGetErrorString(ce)); }
    *out = env;
    return QLC_OK;
}

int32_t qlc_env_destroy(qlc_env* env) {
    if (!env) return QLC_OK;
    cudaSetDevice(env->cfg.device);
    cudaDeviceSynchronize();
#ifdef QLC_PROFILING
    if (env->timeline)
        if (const char* path = getenv("QLC_TIMELINE_FILE")) {
            std::vector<unsigned long long> h(1024 * 16);
            if (cudaMemcpy(h.data(), env->timeline, h.size() * 8, cudaMemcpyDeviceToHost) == cudaSuccess)
                if (FILE* f = fopen(path, "wb")) { fwrite(h.data(), 8, h.size(), f); fclose(f); }
        }
#endif
    qlc_comm_destroy(env);
    for (struct qlc_qnet* q : env->qnets) qnet_release_device(q);      // their handles stay valid for qlc_qnet_destroy, every other call fails
    for (struct qlc_per* p : env->pers) per_release_device(p);         // likewise for qlc_per_destroy
    for (void* p : env->allocs) cudaFree(p);
    if (env->pin) cudaFreeHost(env->pin);
    if (env->dev_stage) cudaFree(env->dev_stage);
    for (cudaEvent_t ev : env->submit_done) if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : env->h2d_done) if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : env->piece_ev) if (ev) cudaEventDestroy(ev);
    if (env->caller_done) cudaEventDestroy(env->caller_done);
    if (env->copy_stream) cudaStreamDestroy(env->copy_stream);
    if (env->own_stream) cudaStreamDestroy(env->own_stream);
    delete env;
    return QLC_OK;
}

int32_t qlc_sync(qlc_env* env, void* stream) {
    if (!env) return fail(QLC_ERR_INVALID_ARG, "env is null");
    int32_t rc = set_device(env); if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return QLC_OK;
}

int32_t qlc_env_reset(qlc_env* env, const uint8_t* mask_host, const float* dir_x_host) {
    QLC_RANGE("qlc_env_reset");
    if (!env) return fail(QLC_ERR_INVALID_ARG, "env is null");
    int32_t rc = set_device(env); if (rc) return rc;
    const uint32_t n = env->cfg.n_envs;
    CUDA_TRY(cudaDeviceSynchronize());
    rc = ensure_dev_stage(env, (size_t)n * 8); if (rc) return rc;
    uint8_t* mask_dev = nullptr; float* dir_dev = nullptr;
    if (mask_host) { mask_dev = (uint8_t*)env->dev_stage + (size_t)n * 4; CUDA_TRY(cudaMemcpy(mask_dev, mask_host, n, cudaMemcpyHostToDevice)); }
    if (dir_x_host) { dir_dev = (float*)env->dev_stage; CUDA_TRY(cudaMemcpy(dir_dev, dir_x_host, (size_t)n * 4, cudaMemcpyHostToDevice)); }
    rc = launch_reset(env, mask_dev, dir_dev, 0, nullptr); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    return QLC_OK;
}

}  // extern "C"

// Grid shaping (measured on B200, profiles/r01_notes.md): up to one wave of 32-env CTAs the fastest split is full
// 32-env CTAs (1 per SM, 32 resident frames); shards too small to give every SM 16 envs are spread evenly instead;
// larger shards use 8-env CTAs, several resident per SM, so that prologues/tails of different CTAs overlap.
static uint32_t pick_epc(uint32_t n_envs, uint32_t sms, uint32_t max_epc) {
    if (n_envs >= sms * (max_epc / 2)) return max_epc;
    uint32_t epc = (n_envs + sms - 1) / sms;
    return epc < 1 ? 1 : epc;
}

template <int R, int NE, int D, int MINB>
static int32_t launch_advance(qlc_env* env, StepParams& p, cudaStream_t s, uint32_t chunk_request) {
    static bool configured[64] = {};
    const size_t dyn = (size_t)R * NE * FRAME_BYTES;
    auto kern = env_advance_kernel<R, NE, D, MINB>;
    if (!configured[env->cfg.device & 63]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        configured[env->cfg.device & 63] = true;
    }
    p.epc = env->epc_override ? (uint32_t)env->epc_override : pick_epc(p.n_envs, (uint32_t)env->sm_count, R * NE);
    if (p.epc > (uint32_t)(R * NE)) p.epc = R * NE;
    const uint32_t n_batches = (p.n_envs + p.epc - 1) / p.epc;
    static int occ[64] = {};
    int& o = occ[env->cfg.device & 63];
    if (o == 0) CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, 32 * (R + 1), dyn));
    const uint32_t resident = (uint32_t)(o > 0 ? o : 1) * (uint32_t)env->sm_count;
    uint32_t chunk = env->persistent ? chunk_request : 0u;
    if (env->chunk_override >= 0) chunk = env->persistent ? (uint32_t)env->chunk_override : 0u;
    if (chunk >= p.n_steps) chunk = 0;
    const uint32_t n_chunks = chunk ? (p.n_steps + chunk - 1) / chunk : 1u;
    uint32_t grid = n_batches;
    if (env->persistent) {       // CTAs take (chunk, batch) items; frames, raster tables and barriers are set up once per CTA
        grid = n_batches * n_chunks;
        if (grid > resident) grid = resident;
        // While the caller reduces the statistics after every launch, the collective's kernels (side stream) hold a few SM slots when
        // the next step launch arrives; a cooperative grid that needs EVERY slot would wait for them. Leave room: the work is handed
        // out dynamically, a few CTAs fewer cost nothing measurable on an HBM-bound launch.
        static const int reserve_sms = getenv("QLC_COMM_RESERVE_SMS") ? atoi(getenv("QLC_COMM_RESERVE_SMS")) : 4;
        if (p.snap && reserve_sms > 0 && grid == resident && env->sm_count > 2 * reserve_sms) grid = (uint32_t)(o > 0 ? o : 1) * (uint32_t)(env->sm_count - reserve_sms);
    }
    p.tables = env->tables; p.work_counter = env->work_counter; p.work_base = env->work_base;
    p.chunk_len = chunk; p.launch_serial = ++env->launch_serial; p.progress = env->progress; p.spin_error = env->spin_error;
    if (chunk) {
        // CTAs wait on one another (chunk c of a batch on chunk c-1): a cooperative launch guarantees co-residency
        void* args[] = {(void*)&env->st, (void*)&p};
        CUDA_TRY(cudaLaunchCooperativeKernel((const void*)kern, dim3(grid), dim3(32 * (R + 1)), args, dyn, s));
    } else {
        // programmatic stream serialization: the prologue (barriers, zeroed resident frames, raster tables) may run while the
        // previous kernel in the stream drains; the kernel waits (griddepcontrol.wait) before it reads anything that kernel wrote
        static const bool pdl = getenv("QLC_STEP_PDL") ? atoi(getenv("QLC_STEP_PDL")) != 0 : true;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(32 * (R + 1)); cfg.dynamicSmemBytes = dyn; cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
        CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, env->st, p));
    }
    CUDA_TRY(cudaGetLastError());
    if (n_batches * n_chunks > grid) env->work_base += n_batches * n_chunks;      // (n_items - grid) hand-outs + one failed grab per CTA
    if (env->comm) {
        if (p.snap) { env->comm->exit_base += grid; env->comm->last_serial = env->launch_serial; }
        env->comm->have_snap = p.snap != nullptr;      // a launch without a snapshot makes the older ones stale
        env->comm->armed = false;
    }
    return QLC_OK;
}

// one launch of at most time_slots steps (a longer one would wrap the frame ring inside the launch: with time chunking two CTAs
// could then have bulk stores to the same slot in flight, ordered by nothing)
static int32_t step_launch(qlc_env* env, const uint8_t* actions_dev, uint8_t* actions_out_dev, uint32_t n_steps, float* reward_dev, uint8_t* done_dev, void* stream) {
    int32_t rc = QLC_OK;
    StepParams p{};
    p.n_envs = env->cfg.n_envs; p.env_id_base = env->cfg.env_id_base; p.time_slots = env->time_slots;
    p.max_episode_steps = env->cfg.max_episode_steps; p.auto_reset = env->cfg.auto_reset; p.n_steps = n_steps;
    p.t0 = env->t; p.slot0 = (uint32_t)(env->t % env->time_slots); p.seed = env->cfg.seed; p.frames = env->frames; p.records = env->records; p.stats = env->stats;
    p.actions = actions_dev; p.actions_out = actions_out_dev; p.reward = reward_dev; p.done = done_dev;
    p.debug_skip = (uint32_t)env->debug_skip;
    p.timeline = env->timeline;
    cudaStream_t s = (cudaStream_t)stream;
    if (qlc_env::Comm* c = env->comm; c && c->armed) {           // snapshots only while the caller keeps reducing (an atomic per CTA otherwise saved)
        const uint32_t slot = (env->launch_serial + 1u) & 3u;     // launch_advance pre-increments the serial
        if (c->slot_busy[slot]) { CUDA_TRY(cudaStreamWaitEvent(s, c->slot_read[slot], 0)); c->slot_busy[slot] = false; }   // 4 launches back: long done
        p.snap = c->snap + slot; p.exit_counter = c->exit_counter; p.exit_base = c->exit_base;
    }
    // Shape selection (measured, profiles/r01_notes.md). Launches that are only a few waves of work are cut into
    // (time chunk, 8-env batch) items handed out dynamically, so that every SM / GPC keeps pulling work at its own pace —
    // this removes a 10-15 % GPU-to-GPU spread seen with one static 32-env batch per SM. Big shards are balanced by their
    // many batches alone; short launches (< 8 steps) have nothing to chunk.
    int cfg = env->advance_cfg;
    uint32_t chunk = 0;
    const uint32_t sms = (uint32_t)env->sm_count;
    if (cfg == 0) {
        if (n_steps >= 8u && p.n_envs >= sms * 16u && p.n_envs <= sms * 96u) { cfg = 5; chunk = n_steps / 4u; chunk = chunk < 4u ? 4u : (chunk > 16u ? 16u : chunk); }
        else if (n_steps < 4u) cfg = p.n_envs <= sms * 20u ? 5 : 2;    // learner-driven launches (latency bound; tools/step_latency_ab.py): 8-env batches
                                                                        // while they fit one resident wave, else 16-env batches, 2 CTAs per SM
        else cfg = p.n_envs <= sms * 32u ? 1 : 5;
    }
    switch (cfg) {
        case 1: rc = launch_advance<8, 4, 4, 1>(env, p, s, chunk); break;    // <= 32 envs / batch, 1 CTA / SM
        case 2: rc = launch_advance<8, 2, 2, 2>(env, p, s, chunk); break;    // <= 16 envs / batch, 2 CTAs / SM
        case 3: rc = launch_advance<4, 4, 4, 2>(env, p, s, chunk); break;    // <= 16 envs / batch, fewer warps
        case 4: rc = launch_advance<4, 2, 4, 3>(env, p, s, chunk); break;    // <=  8 envs / batch
        case 5: rc = launch_advance<8, 1, 4, 3>(env, p, s, chunk); break;    // <=  8 envs / batch, 3 CTAs / SM
        case 6: rc = launch_advance<16, 2, 4, 1>(env, p, s, chunk); break;   // <= 32 envs / batch, 16 render warps
        default: return fail(QLC_ERR_INVALID_ARG, "unknown QLC_ADVANCE_CFG");
    }
    if (rc) return rc;
    env->t += n_steps;
    return QLC_OK;
}

extern "C" {

static int32_t step_split(qlc_env* env, const uint8_t* actions_dev, uint8_t* actions_out_dev, uint32_t n_steps, float* reward_dev, uint8_t* done_dev, void* stream) {
    if (n_steps == 0) return QLC_OK;
    int32_t rc = set_device(env); if (rc) return rc;
    const size_t n = env->cfg.n_envs;
    for (uint32_t at = 0; at < n_steps;) {               // launches of at most one ring length each (see step_launch)
        const uint32_t part = n_steps - at < env->time_slots ? n_steps - at : env->time_slots;
        rc = step_launch(env, actions_dev ? actions_dev + (size_t)at * n : nullptr, actions_out_dev ? actions_out_dev + (size_t)at * n : nullptr, part,
                         reward_dev ? reward_dev + (size_t)at * n : nullptr, done_dev ? done_dev + (size_t)at * n : nullptr, stream);
        if (rc) return rc;
        at += part;
    }
    return QLC_OK;
}

int32_t qlc_env_step(qlc_env* env, const uint8_t* actions_dev, uint32_t n_steps, float* reward_dev, uint8_t* done_dev, void* stream) {
    QLC_RANGE("qlc_env_step");
    if (!env || !actions_dev) return fail(QLC_ERR_INVALID_ARG, "env/actions is null");
    return on_caller_stream(env, stream, [&] { return step_split(env, actions_dev, nullptr, n_steps, reward_dev, done_dev, stream); });
}

// the learner's pure-random phase: the uniform action of every env and step is drawn inside the step kernel
int32_t qlc_env_step_random(qlc_env* env, uint32_t n_steps, uint8_t* actions_out_dev, float* reward_dev, uint8_t* done_dev, void* stream) {
    QLC_RANGE("qlc_env_step_random");
    if (!env) return fail(QLC_ERR_INVALID_ARG, "env is null");
    return on_caller_stream(env, stream, [&] { return step_split(env, nullptr, actions_out_dev, n_steps, reward_dev, done_dev, stream); });
}

static bool is_pinned(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

static int32_t step_host_impl(qlc_env* env, const uint8_t* actions_host, uint32_t n_steps, float* reward_host, uint8_t* done_host, bool wait) {
    QLC_RANGE(wait ? "qlc_env_step_host" : "qlc_env_step_host_submit");
    if (!env || !actions_host) return fail(QLC_ERR_INVALID_ARG, "env/actions is null");
    if (n_steps == 0) return QLC_OK;
    int32_t rc = set_device(env); if (rc) return rc;
    const size_t n = (size_t)env->cfg.n_envs * n_steps;
    // page-locked caller buffers (qlc_host_alloc / cudaHostRegister) are used in place; pageable ones are staged
    const bool pin_a = is_pinned(actions_host), pin_r = !reward_host || is_pinned(reward_host), pin_d = !done_host || is_pinned(done_host);
    if (!wait && !(pin_a && pin_r && pin_d)) return fail(QLC_ERR_INVALID_ARG, "qlc_env_step_host_submit needs page-locked buffers (qlc_host_alloc)");
    rc = after_caller_stream(env); if (rc) return rc;
    // the asynchronous form keeps several steps in flight: each gets its own slice of the device staging ring
    const size_t off_r = (n + 15) & ~(size_t)15, off_d = off_r + n * 4, total = (off_d + n + 255) & ~(size_t)255;
    const uint32_t slot = wait ? 0u : (uint32_t)(env->submit_seq % 2u);
    if (!wait && env->submit_seq >= 8) CUDA_TRY(cudaEventSynchronize(env->submit_done[env->submit_seq % 8]));   // at most 8 steps in flight
    rc = ensure_dev_stage(env, 2 * total); if (rc) return rc;
    uint8_t* dev = (uint8_t*)env->dev_stage + slot * total;
    cudaStream_t s = env->own_stream;
    uint8_t* pin = nullptr;
    if (!(pin_a && pin_r && pin_d)) { rc = ensure_pin(env, total); if (rc) return rc; pin = (uint8_t*)env->pin; }
    const uint8_t* actions_dev = dev;
    if (pin_a && env->zero_copy >= 2) {
        actions_dev = actions_host;             // the physics lanes read (and prefetch) the action bytes straight from host memory
    } else if (pin_a && !wait) {
        // pipelined: copy on a second stream so that it overlaps the previous step's kernel; the staging slice was last read by
        // the kernel of submit seq-2
        if (!env->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&env->copy_stream, cudaStreamNonBlocking));
        cudaEvent_t& hd = env->h2d_done[slot];
        if (!hd) CUDA_TRY(cudaEventCreateWithFlags(&hd, cudaEventDisableTiming));
        if (env->submit_seq >= 2) CUDA_TRY(cudaStreamWaitEvent(env->copy_stream, env->submit_done[(env->submit_seq - 2) % 8], 0));
        CUDA_TRY(cudaMemcpyAsync(dev, actions_host, n, cudaMemcpyHostToDevice, env->copy_stream));
        CUDA_TRY(cudaEventRecord(hd, env->copy_stream));
        CUDA_TRY(cudaStreamWaitEvent(s, hd, 0));
    } else if (pin_a) {
        CUDA_TRY(cudaMemcpyAsync(dev, actions_host, n, cudaMemcpyHostToDevice, s));
    } else {
        memcpy(pin, actions_host, n);
        CUDA_TRY(cudaMemcpyAsync(dev, pin, n, cudaMemcpyHostToDevice, s));
    }
    // validate while the copy is in flight; nothing has been launched yet, so a bad action leaves the env untouched
    uint8_t bad = 0;
    for (size_t i = 0; i < n; ++i) bad |= (uint8_t)(actions_host[i] >= QLC_ACTION_SPACE);
    if (bad) {
        cudaStreamSynchronize(s);                                                   // the staging copy must not outlive the caller's buffer
        if (env->copy_stream) cudaStreamSynchronize(env->copy_stream);
        return fail(QLC_ERR_OUT_OF_RANGE, "value out of range");                    // QlError, breakout_environment.rs:117
    }
    // page-locked outputs are written by the kernel itself (zero-copy stores over PCIe while it runs, UVA pointers);
    // pageable ones go through device staging + a device->host copy
    const bool zc_r = reward_host && pin_r && env->zero_copy, zc_d = done_host && pin_d && env->zero_copy;
    rc = step_split(env, actions_dev, nullptr, n_steps, zc_r ? reward_host : (float*)(dev + off_r), zc_d ? done_host : dev + off_d, s); if (rc) return rc;
    if (reward_host && !zc_r) CUDA_TRY(cudaMemcpyAsync(pin_r ? (void*)reward_host : (void*)(pin + off_r), dev + off_r, n * 4, cudaMemcpyDeviceToHost, s));
    if (done_host && !zc_d) CUDA_TRY(cudaMemcpyAsync(pin_d ? (void*)done_host : (void*)(pin + off_d), dev + off_d, n, cudaMemcpyDeviceToHost, s));
    if (!wait) {
        cudaEvent_t& ev = env->submit_done[env->submit_seq % 8];
        if (!ev) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        CUDA_TRY(cudaEventRecord(ev, s));
        ++env->submit_seq;
        env->submits_pending = true;
        return QLC_OK;
    }
    CUDA_TRY(cudaStreamSynchronize(s));
    env->submits_pending = false;                    // own_stream is idle: every submitted step has finished
    if (reward_host && !pin_r) memcpy(reward_host, pin + off_r, n * 4);
    if (done_host && !pin_d) memcpy(done_host, pin + off_d, n);
    return QLC_OK;
}

int32_t qlc_env_step_host(qlc_env* env, const uint8_t* actions_host, uint32_t n_steps, float* reward_host, uint8_t* done_host) {
    return step_host_impl(env, actions_host, n_steps, reward_host, done_host, true);
}
int32_t qlc_env_step_host_submit(qlc_env* env, const uint8_t* actions_host, uint32_t n_steps, float* reward_host, uint8_t* done_host) {
    return step_host_impl(env, actions_host, n_steps, reward_host, done_host, false);
}
int32_t qlc_env_step_host_wait(qlc_env* env, uint32_t max_pending) {
    if (!env) return fail(QLC_ERR_INVALID_ARG, "env is null");
    if (max_pending >= 8) return fail(QLC_ERR_INVALID_ARG, "max_pending must be < 8");
    int32_t rc = set_device(env); if (rc) return rc;
    if (env->submit_seq <= max_pending) return QLC_OK;
    CUDA_TRY(cudaEventSynchronize(env->submit_done[(env->submit_seq - 1 - max_pending) % 8]));   // in-order stream: older submits are done too
    if (max_pending == 0) env->submits_pending = false;
    return QLC_OK;
}

int32_t qlc_host_alloc(size_t bytes, void** out) {
    if (!out || bytes == 0) return fail(QLC_ERR_INVALID_ARG, "out is null or bytes == 0");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(QLC_ERR_NO_DEVICE, "no CUDA device: ql_cuda has no CPU fallback");
    CUDA_TRY(cudaMallocHost(out, bytes));
    return QLC_OK;
}
int32_t qlc_host_free(void* p) {
    if (p) CUDA_TRY(cudaFreeHost(p));
    return QLC_OK;
}

static void fill_gather(const qlc_env* env, GatherParams& g) {
    g.frames = env->frames; g.records = env->records; g.episode_step = env->st.episode_step;
    g.n_envs = env->cfg.n_envs; g.time_slots = env->time_slots;
    g.t_now = env->t; g.t_oldest = env->t > env->t_cap ? env->t - env->t_cap : 0;
    g.mode = GATHER_INDICES;
}

static bool known_layout(int32_t layout) { return layout == QLC_LAYOUT_U8_BHYX || layout == QLC_LAYOUT_F32_BXYH || layout == QLC_LAYOUT_U8_BXYH; }

// Dynamic shared memory request that caps the resident CTAs per SM at `cap` (228 KB per SM, 1 KB reserved per CTA). Small grids
// launched with programmatic stream serialization start while their predecessor still holds most SMs; without a cap the block
// scheduler packs them 5-8 deep onto the few SMs that are free, and a minibatch gather then runs on a tenth of the machine.
static size_t smem_for_cap(size_t needed, uint32_t cap) {
    if (cap == 0 || cap >= 8) return needed;
    const size_t want = (size_t)228 * 1024 / (cap + 1) + 16;     // cap + 1 CTAs of this size do not fit
    const size_t most = (size_t)226 * 1024;            // the opt-in limit set below (227 KB minus the kernels' static shared memory)
    return needed > want ? needed : (want > most ? most : want);
}

static int32_t launch_gather(qlc_env* env, const GatherParams& g_in, int32_t layout, cudaStream_t s) {
    if (g_in.n_items == 0) return QLC_OK;
    GatherParams g = g_in;
    static bool configured[64] = {};
    if (!configured[env->cfg.device & 63]) {     // opt in to large dynamic shared memory (6 frames; occupancy caps)
        CUDA_TRY(cudaFuncSetAttribute(gather_u8_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
        CUDA_TRY(cudaFuncSetAttribute(gather_u8_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
        CUDA_TRY(cudaFuncSetAttribute(gather_xyh_kernel<float4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
        CUDA_TRY(cudaFuncSetAttribute(gather_xyh_kernel<uchar4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
        configured[env->cfg.device & 63] = true;
    }
    static const int slices_force = getenv("QLC_GATHER_SLICES") ? atoi(getenv("QLC_GATHER_SLICES")) : 0;
    static const int cap_force = getenv("QLC_GATHER_CAP") ? atoi(getenv("QLC_GATHER_CAP")) : -1;
    const uint32_t sms = (uint32_t)env->sm_count;
    g.slices = 1;
    // scalars only (get_many without tensorisation): the one-warp kernel has the path for it, whatever the layout
    if (layout == QLC_LAYOUT_U8_BHYX || (!g.out_state && !g.out_next)) {
        if (!known_layout(layout)) return fail(QLC_ERR_INVALID_ARG, "unknown layout");
        uint32_t cap = (g.n_items + sms - 1) / sms;                  // spread a small grid over the SMs
        if (cap_force >= 0) cap = (uint32_t)cap_force;
        // a sampled minibatch of >= 129: 7 helper warps per CTA join the index draw (one pass over the Philox stream instead of five rounds)
        if (g.mode == GATHER_SAMPLE && g.sample_batch >= SAMPLE_BLOCK_MIN_BATCH)
            CUDA_TRY(launch_pdl(gather_u8_kernel<8>, dim3(g.n_items), dim3(256), smem_for_cap(6 * FRAME_BYTES, cap), s, g));
        else
            CUDA_TRY(launch_pdl(gather_u8_kernel<1>, dim3(g.n_items), dim3(32), smem_for_cap(6 * FRAME_BYTES, cap), s, g));
    } else if (layout == QLC_LAYOUT_F32_BXYH || layout == QLC_LAYOUT_U8_BXYH) {
        // slices: enough CTAs to put a single small minibatch on every SM (each CTA stages the 4 frames again, from L2)
        const uint32_t units = g.n_items * 2u;
        g.slices = units * 4u <= 2u * sms ? 4u : (units * 2u <= 2u * sms ? 2u : 1u);
        if (slices_force == 1 || slices_force == 2 || slices_force == 4) g.slices = (uint32_t)slices_force;
        const uint32_t ctas = units * g.slices;
        size_t smem = 4 * FRAME_BYTES;           // 4 slot frames; the in-kernel sampler's table (batch > 384: 32 KB) borrows the same bytes
        if (g.mode == GATHER_SAMPLE && 8u * (size_t)sample_table_size(g.sample_batch) > smem) smem = 8u * (size_t)sample_table_size(g.sample_batch);
        uint32_t cap = (ctas + sms - 1) / sms;
        if (cap_force >= 0) cap = (uint32_t)cap_force;
        smem = smem_for_cap(smem, cap);
        if (layout == QLC_LAYOUT_F32_BXYH) CUDA_TRY(launch_pdl(gather_xyh_kernel<float4>, dim3(ctas), dim3(GATHER_XYH_THREADS), smem, s, g));
        else CUDA_TRY(launch_pdl(gather_xyh_kernel<uchar4>, dim3(ctas), dim3(GATHER_XYH_THREADS), smem, s, g));
    } else {
        return fail(QLC_ERR_INVALID_ARG, "unknown layout");
    }
    CUDA_TRY(cudaGetLastError());
    return QLC_OK;
}

static size_t item_bytes(int32_t layout) { return layout == QLC_LAYOUT_F32_BXYH ? (size_t)FRAME_BYTES * 4 * sizeof(float) : (size_t)FRAME_BYTES * 4; }

int32_t qlc_env_obs(qlc_env* env, int32_t layout, void* out_dev, void* stream) {
    QLC_RANGE("qlc_env_obs");
    if (!env || !out_dev) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    if (((uintptr_t)out_dev & 15) != 0) return fail(QLC_ERR_INVALID_ARG, "output must be 16-byte aligned");
    int32_t rc = set_device(env); if (rc) return rc;
    GatherParams g{}; fill_gather(env, g);
    g.mode = GATHER_CURRENT; g.n_items = env->cfg.n_envs; g.out_state = out_dev;
    return on_caller_stream(env, stream, [&] { return launch_gather(env, g, layout, (cudaStream_t)stream); });
}

// ---- state handles: what a cloned BreakoutState is on the host (state_as_rc / step_as_rc, prelude.rs:36,52-58) ----
int32_t qlc_obs_gather(qlc_env* env, const qlc_obs_handle* handles_dev, uint32_t n, int32_t layout, void* out_dev, void* stream) {
    QLC_RANGE("qlc_obs_gather");
    if (!env || !handles_dev || !out_dev) return fail(QLC_ERR_INVALID_ARG, "env/handles/out is null");
    if (((uintptr_t)out_dev & 15) != 0) return fail(QLC_ERR_INVALID_ARG, "output must be 16-byte aligned");
    int32_t rc = set_device(env); if (rc) return rc;
    static_assert(sizeof(qlc_obs_handle) == sizeof(ObsHandle), "handle layout");
    GatherParams g{}; fill_gather(env, g);
    g.mode = GATHER_HANDLES; g.handles = reinterpret_cast<const ObsHandle*>(handles_dev); g.n_items = n; g.out_state = out_dev;
    return on_caller_stream(env, stream, [&] { return launch_gather(env, g, layout, (cudaStream_t)stream); });
}

// a handle is usable while the frames it names are still in the ring (and it is not from the future)
static bool handle_alive(const qlc_env* env, const qlc_obs_handle& h) {
    const uint64_t need = h.k < 4u ? h.k : 4u;
    return h.env < env->cfg.n_envs && h.time <= env->t && h.time >= need && h.time - need + env->time_slots >= env->t;
}

int32_t qlc_env_state_view(qlc_env* env, qlc_state_view* out) {
    if (!env || !out) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    out->ball_cx = env->st.ball_cx; out->ball_cy = env->st.ball_cy; out->ball_dx = env->st.ball_dx; out->ball_dy = env->st.ball_dy;
    out->pad_min_x = env->st.pad_min_x; out->pad_max_x = env->st.pad_max_x; out->pad_speed = env->st.pad_speed;
    out->bricks = env->st.bricks; out->score = env->st.score; out->episode_step = env->st.episode_step; out->episode = env->st.episode;
    out->err = env->st.err; out->finished = env->st.finished; out->frames = env->frames; out->records = env->records;
    out->n_envs = env->cfg.n_envs; out->time_slots = env->time_slots; out->time = env->t;
    return QLC_OK;
}

int32_t qlc_env_read_state(qlc_env* env, const qlc_state_host* o) {
    if (!env || !o) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    int32_t rc = set_device(env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    const size_t n = env->cfg.n_envs;
#define RD(dst, src, T) do { if (o->dst) CUDA_TRY(cudaMemcpy(o->dst, env->st.src, n * sizeof(T), cudaMemcpyDeviceToHost)); } while (0)
    RD(ball_cx, ball_cx, float); RD(ball_cy, ball_cy, float); RD(ball_dx, ball_dx, float); RD(ball_dy, ball_dy, float);
    RD(pad_min_x, pad_min_x, float); RD(pad_max_x, pad_max_x, float); RD(pad_speed, pad_speed, float);
    RD(bricks, bricks, uint64_t); RD(score, score, uint32_t); RD(episode_step, episode_step, uint32_t);
    RD(episode, episode, uint32_t); RD(err, err, uint32_t); RD(finished, finished, uint8_t);
#undef RD
    return QLC_OK;
}

// "lives" of the reference game: the episode ends the first time the ball passes the paddle (mechanics.rs:131-135), so an env
// has exactly one life while it is not finished
int32_t qlc_env_lives_host(qlc_env* env, uint8_t* lives_host) {
    if (!env || !lives_host) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    int32_t rc = set_device(env); if (rc) return rc;
    const uint32_t n = env->cfg.n_envs;
    CUDA_TRY(cudaDeviceSynchronize());
    rc = ensure_dev_stage(env, n); if (rc) return rc;
    lives_kernel<<<(n + 255) / 256, 256>>>(env->st.finished, (uint8_t*)env->dev_stage, n);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(lives_host, env->dev_stage, n, cudaMemcpyDeviceToHost));
    return QLC_OK;
}

int32_t qlc_env_time(qlc_env* env, uint64_t* t) {
    if (!env || !t) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    *t = env->t; return QLC_OK;
}

int32_t qlc_env_error_flags(qlc_env* env, uint32_t* out) {
    if (!env || !out) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    int32_t rc = set_device(env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemset(env->scratch, 0, 8));
    err_or_kernel<<<64, 256>>>(env->st.err, env->cfg.n_envs, (uint32_t*)env->scratch);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(out, env->scratch, 4, cudaMemcpyDeviceToHost));
    unsigned int spin = 0;
    CUDA_TRY(cudaMemcpy(&spin, env->spin_error, 4, cudaMemcpyDeviceToHost));
    if (spin) *out |= QLC_ENVERR_HANDOVER;
    return QLC_OK;
}

// ---------------- replay ----------------
static uint64_t replay_len(const qlc_env* env) {
    const uint64_t steps = env->t < env->t_cap ? env->t : env->t_cap;
    return env->cfg.replay_capacity == 0 ? 0 : steps * env->cfg.n_envs;
}

int32_t qlc_replay_len(qlc_env* env, uint64_t* len) {
    if (!env || !len) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    *len = replay_len(env); return QLC_OK;
}
int32_t qlc_replay_capacity(qlc_env* env, uint64_t* cap) {
    if (!env || !cap) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    *cap = env->cfg.replay_capacity == 0 ? 0 : (uint64_t)env->t_cap * env->cfg.n_envs; return QLC_OK;
}

static int32_t check_sample_args(qlc_env* env, uint32_t batch, uint64_t* len_out) {
    if (batch == 0 || batch > SAMPLE_MAX_BATCH) return fail(QLC_ERR_INVALID_ARG, "batch must be in 1..1024");
    const uint64_t len = replay_len(env);
    if (len < batch) return fail(QLC_ERR_NOT_ENOUGH, "replay holds fewer transitions than the batch size");
    if (len >= 0xFFFFFFFFull) return fail(QLC_ERR_INVALID_ARG, "replay longer than 2^32-2 transitions");
    *len_out = len;
    return QLC_OK;
}

static int32_t launch_sample(qlc_env* env, uint32_t batch, uint32_t n_batches, uint64_t len, uint64_t call_index, uint32_t* idx_dev, cudaStream_t s) {
    if (batch >= SAMPLE_BLOCK_MIN_BATCH) replay_sample_kernel<8><<<n_batches, 256, 0, s>>>(idx_dev, batch, (uint32_t)len, env->cfg.seed, call_index);
    else replay_sample_kernel<1><<<n_batches, 32, 0, s>>>(idx_dev, batch, (uint32_t)len, env->cfg.seed, call_index);
    CUDA_TRY(cudaGetLastError());
    return QLC_OK;
}

int32_t qlc_replay_sample(qlc_env* env, uint32_t batch, uint32_t n_batches, uint64_t call_index, uint32_t* idx_dev, void* stream) {
    QLC_RANGE("qlc_replay_sample");
    if (!env || !idx_dev) return fail(QLC_ERR_INVALID_ARG, "env/idx is null");
    uint64_t len = 0;
    int32_t rc = check_sample_args(env, batch, &len); if (rc) return rc;
    if (n_batches == 0) return QLC_OK;
    return on_caller_stream(env, stream, [&] { return launch_sample(env, batch, n_batches, len, call_index, idx_dev, (cudaStream_t)stream); });
}

int32_t qlc_replay_gather(qlc_env* env, const uint32_t* idx_dev, uint32_t n, int32_t layout, void* state_dev, void* next_dev,
                          float* reward_dev, uint8_t* action_dev, uint8_t* done_dev, void* stream) {
    QLC_RANGE("qlc_replay_gather");
    if (!env || !idx_dev) return fail(QLC_ERR_INVALID_ARG, "env/idx is null");
    if ((((uintptr_t)state_dev) | ((uintptr_t)next_dev)) & 15) return fail(QLC_ERR_INVALID_ARG, "outputs must be 16-byte aligned");
    int32_t rc = set_device(env); if (rc) return rc;
    GatherParams g{}; fill_gather(env, g);
    g.indices = idx_dev; g.n_items = n; g.out_state = state_dev; g.out_next = next_dev;
    g.reward = reward_dev; g.action = action_dev; g.done = done_dev;
    return on_caller_stream(env, stream, [&] { return launch_gather(env, g, layout, (cudaStream_t)stream); });
}

// sample + gather in ONE launch: every CTA of the gather kernel derives the index of its own item from the Philox stream
int32_t qlc_replay_sample_gather(qlc_env* env, uint32_t batch, uint32_t n_batches, uint64_t call_index, int32_t layout, uint32_t* idx_out_dev,
                                 void* state_dev, void* next_dev, float* reward_dev, uint8_t* action_dev, uint8_t* done_dev, void* stream) {
    QLC_RANGE("qlc_replay_sample_gather");
    if (!env) return fail(QLC_ERR_INVALID_ARG, "env is null");
    if ((((uintptr_t)state_dev) | ((uintptr_t)next_dev)) & 15) return fail(QLC_ERR_INVALID_ARG, "outputs must be 16-byte aligned");
    uint64_t len = 0;
    int32_t rc = check_sample_args(env, batch, &len); if (rc) return rc;
    if (n_batches == 0) return QLC_OK;
    if ((uint64_t)batch * n_batches > 0x3FFFFFFFull) return fail(QLC_ERR_INVALID_ARG, "too many items for one call");
    rc = set_device(env); if (rc) return rc;
    GatherParams g{}; fill_gather(env, g);
    g.mode = GATHER_SAMPLE; g.sample_batch = batch; g.sample_len = (uint32_t)len; g.seed = env->cfg.seed; g.call0 = call_index; g.idx_out = idx_out_dev;
    g.n_items = batch * n_batches; g.out_state = state_dev; g.out_next = next_dev;
    g.reward = reward_dev; g.action = action_dev; g.done = done_dev;
    return on_caller_stream(env, stream, [&] { return launch_gather(env, g, layout, (cudaStream_t)stream); });
}

int32_t qlc_replay_sample_host(qlc_env* env, uint32_t batch, uint64_t call_index, uint32_t* idx_host) {
    QLC_RANGE("qlc_replay_sample_host");
    if (!env || !idx_host) return fail(QLC_ERR_INVALID_ARG, "env/idx is null");
    uint64_t len = 0;
    int32_t rc = check_sample_args(env, batch, &len); if (rc) return rc;
    rc = set_device(env); if (rc) return rc;
    rc = after_caller_stream(env); if (rc) return rc;
    rc = ensure_dev_stage(env, (size_t)batch * 4); if (rc) return rc;
    rc = launch_sample(env, batch, 1, len, call_index, (uint32_t*)env->dev_stage, env->own_stream); if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(idx_host, env->dev_stage, (size_t)batch * 4, cudaMemcpyDeviceToHost, env->own_stream));
    CUDA_TRY(cudaStreamSynchronize(env->own_stream));
    return QLC_OK;
}

// Host-buffer gathers. An f32 [b][x][y][slot] request is gathered as u8 in the same order on the device, crosses PCIe as u8 (1/4
// of the bytes) and is widened into the caller's buffer by the host pool (value = u8 as f32: bit-identical to widening on the
// device). QLC_HOST_WIDEN=0 keeps the f32 tensors on the device side of the copy (A/B measurements).
struct HostGather {
    GatherParams g; int32_t layout; uint32_t n;
    const void* h2d_src; size_t h2d_bytes;                 // indices or handles
    void* state_host; void* next_host; float* reward_host; uint8_t* action_host; uint8_t* done_host; uint32_t* idx_out_host;
};

static int32_t run_host_gather(qlc_env* env, HostGather& hg) {
    static const bool widen_on_host = getenv("QLC_HOST_WIDEN") ? atoi(getenv("QLC_HOST_WIDEN")) != 0 : true;
    int32_t rc = after_caller_stream(env); if (rc) return rc;
    const uint32_t n = hg.n;
    const bool widen = hg.layout == QLC_LAYOUT_F32_BXYH && widen_on_host;
    const int32_t dev_layout = widen ? QLC_LAYOUT_U8_BXYH : hg.layout;
    const size_t ib = item_bytes(dev_layout);
    // page-locked staging (device-visible: the kernel reads the indices / handles from it and writes the scalars into it — a few
    // hundred bytes over PCIe instead of two more copy launches): in | reward | action | done | idx_out | state | next
    const size_t o_in = 0, o_r = (hg.h2d_bytes + 255) & ~(size_t)255, o_a = o_r + (size_t)n * 4, o_d = o_a + n, o_i = (o_d + n + 15) & ~(size_t)15;
    const size_t o_s = (o_i + (size_t)n * 4 + 255) & ~(size_t)255, o_n = o_s + ib * n, total = o_n + ib * n;
    // f32 requests, streamed (QLC_HOST_STREAM=0: the piecewise copies below): the kernel stores the u8 stacks straight into the
    // page-locked staging while it runs and raises one arrival flag per CTA; the host pool widens slice i into the caller's
    // tensor as soon as its flag is up, while the slices behind it are still crossing PCIe. One launch, no copy calls, no events.
    static const int stream_mode = getenv("QLC_HOST_STREAM") ? atoi(getenv("QLC_HOST_STREAM")) : 1;
    if (widen && stream_mode == 1 && (hg.state_host || hg.next_host)) {      // (scalars only: the one-warp kernel below)
        static const bool timing = getenv("QLC_HOST_TIMING") != nullptr;
        const auto t0 = std::chrono::steady_clock::now();
        const size_t o_f = (total + 255) & ~(size_t)255, total_f = o_f + (size_t)n * 2 * 4 * sizeof(uint32_t);   // <= 4 CTAs per (item, s | s')
        rc = ensure_pin(env, total_f); if (rc) return rc;
        uint8_t* pin = (uint8_t*)env->pin;
        cudaStream_t s = env->own_stream;
        if (hg.h2d_bytes) memcpy(pin + o_in, hg.h2d_src, hg.h2d_bytes);
        GatherParams& g = hg.g;
        if (g.mode == GATHER_INDICES) g.indices = (const uint32_t*)(pin + o_in);
        if (g.mode == GATHER_HANDLES) g.handles = (const ObsHandle*)(pin + o_in);
        if (g.mode == GATHER_SAMPLE) g.idx_out = hg.idx_out_host ? (uint32_t*)(pin + o_i) : nullptr;
        g.n_items = n;
        g.out_state = hg.state_host ? pin + o_s : nullptr; g.out_next = hg.next_host ? pin + o_n : nullptr;
        const bool scalars = g.mode == GATHER_INDICES || g.mode == GATHER_SAMPLE;
        g.reward = scalars ? (float*)(pin + o_r) : nullptr; g.action = scalars ? pin + o_a : nullptr; g.done = scalars ? pin + o_d : nullptr;
        if (++env->flag_serial == 0) env->flag_serial = 1;
        g.cta_flags = (uint32_t*)(pin + o_f); g.flag_value = env->flag_serial;
        const bool sampled = g.mode == GATHER_SAMPLE;
        if (g.mode == GATHER_SAMPLE) {        // the persistent kernel takes given indices: draw them first (into the staging, the caller wants them anyway)
            uint32_t* idx = (uint32_t*)(pin + o_i);
            if (g.sample_batch >= SAMPLE_BLOCK_MIN_BATCH) replay_sample_kernel<8><<<1, 256, 0, s>>>(idx, g.sample_batch, g.sample_len, g.seed, g.call0);
            else replay_sample_kernel<1><<<1, 32, 0, s>>>(idx, g.sample_batch, g.sample_len, g.seed, g.call0);
            CUDA_TRY(cudaGetLastError());
            g.mode = GATHER_INDICES; g.indices = idx; g.idx_out = nullptr;
        }
        static const int slices_env = getenv("QLC_STREAM_SLICES") ? atoi(getenv("QLC_STREAM_SLICES")) : 0;
        static const int ctas_env = getenv("QLC_STREAM_CTAS") ? atoi(getenv("QLC_STREAM_CTAS")) : 0;
        // pieces of 14 KB for minibatch-sized requests (finer overlap of transfer and widening), whole 28 KB stacks beyond; enough CTAs
        // in flight to keep PCIe busy (each spends most of a piece's time loading and transposing), few enough that pieces land in order
        uint32_t slices = (slices_env == 1 || slices_env == 2 || slices_env == 4) ? (uint32_t)slices_env : (n <= 64 ? 2u : 1u);
        g.slices = slices;
        const bool both = hg.state_host && hg.next_host;
        const uint32_t n_ctas_all = n * (both ? 2u : 1u) * slices;

        uint32_t grid = ctas_env > 0 ? (uint32_t)ctas_env : 48u;
        if (grid > n_ctas_all) grid = n_ctas_all;
        size_t smem = 4 * (size_t)FRAME_BYTES + 2 * (4 * (size_t)FRAME_BYTES / slices);      // 4 slot frames + two staging buffers
        const size_t pre_bytes = g.mode == GATHER_INDICES ? (size_t)n * 4 : (g.mode == GATHER_HANDLES ? (size_t)n * sizeof(ObsHandle) : 0);
        g.preload = pre_bytes > 0 && pre_bytes <= 64 * 1024 ? 1u : 0u;                        // + the indices / handles, fetched over PCIe once per CTA
        if (g.preload) smem += pre_bytes;
        static bool configured[64] = {};
        if (!configured[env->cfg.device & 63]) {
            CUDA_TRY(cudaFuncSetAttribute(gather_xyh_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 12 * FRAME_BYTES + 64 * 1024));
            configured[env->cfg.device & 63] = true;
        }
        gather_xyh_stream_kernel<<<grid, GATHER_XYH_THREADS, smem, s>>>(g);
        CUDA_TRY(cudaGetLastError());
        const auto t1 = std::chrono::steady_clock::now();
        const uint32_t per = (uint32_t)(ib / slices);                 // elements per CTA: its share of the 7,056 pixels x 4 slots
        std::vector<qlc_host::StreamPiece>& pieces = env->stream_pieces;
        pieces.resize((size_t)n_ctas_all);
        for (size_t c = 0; c < pieces.size(); ++c) {
            const size_t unit = c / slices, slice = c % slices, b = both ? unit >> 1 : unit, which = both ? (unit & 1) : (hg.next_host ? 1 : 0);
            float* host = (float*)(which ? hg.next_host : hg.state_host);
            const size_t off = b * ib + slice * per;
            pieces[c] = qlc_host::StreamPiece{pin + (which ? o_n : o_s) + off, host ? host + off : nullptr, per};
        }
        const size_t missed = qlc_host::widen_stream(pieces.data(), pieces.size(), slices, (const volatile uint32_t*)(pin + o_f), g.flag_value,
                                                     [](void* st) { return cudaStreamQuery((cudaStream_t)st) == cudaErrorNotReady; }, (void*)s);
        const auto t2 = std::chrono::steady_clock::now();
        // every flag is up: all pieces and (written earlier by the same threads, before their system-scope fences) all scalars have
        // landed; the kernel is only exiting, and whatever comes next on this stream is ordered behind it. A missing piece means the
        // stream ended without it: synchronize to surface the error.
        if (missed || sampled) CUDA_TRY(cudaStreamSynchronize(s));      // (sampled: the index kernel's own stores carry no flag)
        if (timing) {
            const auto t3 = std::chrono::steady_clock::now();
            auto us = [](auto a, auto b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
            fprintf(stderr, "[qlc host gather] n=%u slices=%u: setup+launch %.1f us, widen_stream %.1f us, sync %.1f us\n", n, slices, us(t0, t1), us(t1, t2), us(t2, t3));
        }
        if (missed) return fail(QLC_ERR_CUDA, "streamed gather: the kernel finished without delivering every slice");
        if (hg.reward_host) memcpy(hg.reward_host, pin + o_r, (size_t)n * 4);
        if (hg.action_host) memcpy(hg.action_host, pin + o_a, n);
        if (hg.done_host) memcpy(hg.done_host, pin + o_d, n);
        if (hg.idx_out_host) memcpy(hg.idx_out_host, pin + o_i, (size_t)n * 4);
        return QLC_OK;
    }
    rc = ensure_dev_stage(env, 2 * ib * n); if (rc) return rc;
    rc = ensure_pin(env, total); if (rc) return rc;
    uint8_t* dev = (uint8_t*)env->dev_stage; uint8_t* pin = (uint8_t*)env->pin;
    uint8_t* dev_s = dev; uint8_t* dev_n = dev + ib * n;
    cudaStream_t s = env->own_stream;
    if (hg.h2d_bytes) memcpy(pin + o_in, hg.h2d_src, hg.h2d_bytes);
    GatherParams& g = hg.g;
    if (g.mode == GATHER_INDICES) g.indices = (const uint32_t*)(pin + o_in);
    if (g.mode == GATHER_HANDLES) g.handles = (const ObsHandle*)(pin + o_in);
    if (g.mode == GATHER_SAMPLE) g.idx_out = hg.idx_out_host ? (uint32_t*)(pin + o_i) : nullptr;
    g.n_items = n;
    g.out_state = hg.state_host ? dev_s : nullptr; g.out_next = hg.next_host ? dev_n : nullptr;
    const bool scalars = g.mode == GATHER_INDICES || g.mode == GATHER_SAMPLE;
    g.reward = scalars ? (float*)(pin + o_r) : nullptr; g.action = scalars ? pin + o_a : nullptr; g.done = scalars ? pin + o_d : nullptr;
    rc = launch_gather(env, g, dev_layout, s); if (rc) return rc;
    // The stacks cross PCIe in pieces: piece i is widened (f32 requests) or copied (pageable u8 targets) on the host while piece
    // i+1 is still in flight. u8 stacks for page-locked caller buffers (qlc_host_alloc) are copied straight into them.
    struct Piece { uint8_t* src; uint8_t* dst; size_t off, bytes; };
    Piece pieces[2 * 8]; int n_pieces = 0;
    for (int w = 0; w < 2; ++w) {
        uint8_t* host = (uint8_t*)(w ? hg.next_host : hg.state_host);
        if (!host) continue;
        const size_t stack = ib * n;
        uint8_t* devp = w ? dev_n : dev_s;
        if (!widen && is_pinned(host)) { CUDA_TRY(cudaMemcpyAsync(host, devp, stack, cudaMemcpyDeviceToHost, s)); continue; }
        size_t parts = stack / ((size_t)384 << 10);           // pieces of >= 384 KB: a 32-minibatch stack (882 KB) goes in two
        parts = parts < 1 ? 1 : (parts > 8 ? 8 : parts);
        const size_t step = ((stack / parts) + 4095) & ~(size_t)4095;
        for (size_t off = 0; off < stack; off += step) {
            const size_t m = stack - off < step ? stack - off : step;
            cudaEvent_t& ev = env->piece_ev[n_pieces];
            if (!ev) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            uint8_t* stage = pin + (w ? o_n : o_s) + off;
            CUDA_TRY(cudaMemcpyAsync(stage, devp + off, m, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaEventRecord(ev, s));
            pieces[n_pieces++] = Piece{stage, host, off, m};
        }
    }
    for (int i = 0; i < n_pieces; ++i) {
        CUDA_TRY(cudaEventSynchronize(env->piece_ev[i]));
        const Piece& p = pieces[i];
        if (widen) qlc_host::widen_u8_f32(p.src, (float*)p.dst + p.off, p.bytes);
        else memcpy(p.dst + p.off, p.src, p.bytes);
    }
    CUDA_TRY(cudaStreamSynchronize(s));
    if (hg.reward_host) memcpy(hg.reward_host, pin + o_r, (size_t)n * 4);
    if (hg.action_host) memcpy(hg.action_host, pin + o_a, n);
    if (hg.done_host) memcpy(hg.done_host, pin + o_d, n);
    if (hg.idx_out_host) memcpy(hg.idx_out_host, pin + o_i, (size_t)n * 4);
    return QLC_OK;
}

int32_t qlc_replay_gather_host(qlc_env* env, const uint32_t* idx_host, uint32_t n, int32_t layout, void* state_host, void* next_host,
                               float* reward_host, uint8_t* action_host, uint8_t* done_host) {
    QLC_RANGE("qlc_replay_gather_host");
    if (!env || !idx_host) return fail(QLC_ERR_INVALID_ARG, "env/idx is null");
    if (!known_layout(layout)) return fail(QLC_ERR_INVALID_ARG, "unknown layout");
    if (n == 0) return QLC_OK;
    const uint64_t len = replay_len(env);
    for (uint32_t i = 0; i < n; ++i) if (idx_host[i] >= len) return fail(QLC_ERR_OUT_OF_RANGE, "replay index out of range");
    int32_t rc = set_device(env); if (rc) return rc;
    HostGather hg{}; fill_gather(env, hg.g);
    hg.layout = layout; hg.n = n; hg.h2d_src = idx_host; hg.h2d_bytes = (size_t)n * 4;
    hg.state_host = state_host; hg.next_host = next_host; hg.reward_host = reward_host; hg.action_host = action_host; hg.done_host = done_host;
    return run_host_gather(env, hg);
}

int32_t qlc_replay_sample_gather_host(qlc_env* env, uint32_t batch, uint64_t call_index, int32_t layout, uint32_t* idx_out_host,
                                      void* state_host, void* next_host, float* reward_host, uint8_t* action_host, uint8_t* done_host) {
    QLC_RANGE("qlc_replay_sample_gather_host");
    if (!env) return fail(QLC_ERR_INVALID_ARG, "env is null");
    if (!known_layout(layout)) return fail(QLC_ERR_INVALID_ARG, "unknown layout");
    uint64_t len = 0;
    int32_t rc = check_sample_args(env, batch, &len); if (rc) return rc;
    rc = set_device(env); if (rc) return rc;
    HostGather hg{}; fill_gather(env, hg.g);
    hg.g.mode = GATHER_SAMPLE; hg.g.sample_batch = batch; hg.g.sample_len = (uint32_t)len; hg.g.seed = env->cfg.seed; hg.g.call0 = call_index;
    hg.layout = layout; hg.n = batch; hg.idx_out_host = idx_out_host;
    hg.state_host = state_host; hg.next_host = next_host; hg.reward_host = reward_host; hg.action_host = action_host; hg.done_host = done_host;
    return run_host_gather(env, hg);
}

int32_t qlc_env_obs_host(qlc_env* env, int32_t layout, void* out_host) {
    QLC_RANGE("qlc_env_obs_host");
    if (!env || !out_host) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    if (!known_layout(layout)) return fail(QLC_ERR_INVALID_ARG, "unknown layout");
    int32_t rc = set_device(env); if (rc) return rc;
    HostGather hg{}; fill_gather(env, hg.g);
    hg.g.mode = GATHER_CURRENT;
    hg.layout = layout; hg.n = env->cfg.n_envs; hg.state_host = out_host;
    return run_host_gather(env, hg);
}

// batch_to_multi_dim_array for host-side state handles (breakout_environment.rs:56-77): n stacks into out_host
int32_t qlc_obs_gather_host(qlc_env* env, const qlc_obs_handle* handles_host, uint32_t n, int32_t layout, void* out_host) {
    QLC_RANGE("qlc_obs_gather_host");
    if (!env || !handles_host || !out_host) return fail(QLC_ERR_INVALID_ARG, "env/handles/out is null");
    if (!known_layout(layout)) return fail(QLC_ERR_INVALID_ARG, "unknown layout");
    if (n == 0) return QLC_OK;
    for (uint32_t i = 0; i < n; ++i)
        if (!handle_alive(env, handles_host[i])) return fail(QLC_ERR_OUT_OF_RANGE, "stale state handle: its frames have left the frame ring (or it belongs to another env)");
    int32_t rc = set_device(env); if (rc) return rc;
    HostGather hg{}; fill_gather(env, hg.g);
    hg.g.mode = GATHER_HANDLES;
    hg.layout = layout; hg.n = n; hg.h2d_src = handles_host; hg.h2d_bytes = (size_t)n * sizeof(qlc_obs_handle);
    hg.state_host = out_host;
    return run_host_gather(env, hg);
}

int32_t qlc_replay_action_counts(qlc_env* env, uint64_t counts[3]) {
    if (!env || !counts) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    int32_t rc = set_device(env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemset(env->scratch, 0, 3 * sizeof(unsigned long long)));
    counts[0] = counts[1] = counts[2] = 0;
    if (replay_len(env) == 0) return QLC_OK;
    const uint64_t t_old = env->t > env->t_cap ? env->t - env->t_cap : 0;
    action_histogram_kernel<<<296, 256>>>(env->records, env->cfg.n_envs, env->time_slots, t_old, env->t, env->scratch);
    CUDA_TRY(cudaGetLastError());
    unsigned long long h[3];
    CUDA_TRY(cudaMemcpy(h, env->scratch, sizeof h, cudaMemcpyDeviceToHost));
    counts[0] = h[0]; counts[1] = h[1]; counts[2] = h[2];
    return QLC_OK;
}

// ---------------- episode statistics ----------------
int32_t qlc_stats_read(qlc_env* env, qlc_episode_stats* out) {
    if (!env || !out) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    int32_t rc = set_device(env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    DeviceStats d;
    CUDA_TRY(cudaMemcpy(&d, env->stats, sizeof d, cudaMemcpyDeviceToHost));
    out->sum_return = d.sum_return; out->episodes = d.episodes; out->steps = env->t * env->cfg.n_envs;
    out->min_return = d.min_return; out->max_return = d.max_return;
    return QLC_OK;
}
int32_t qlc_stats_export(qlc_env* env, double* out_dev, void* stream) {
    if (!env || !out_dev) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    return on_caller_stream(env, stream, [&] {
        stats_export_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(env->stats, env->t * env->cfg.n_envs, out_dev);
        CUDA_TRY(cudaGetLastError());
        return QLC_OK;
    });
}
// ---------------- statistics reduction over the env shards: NCCL behind the C ABI, on a side stream ----------------
int32_t qlc_comm_unique_id(uint8_t* id128) {
    if (!id128) return fail(QLC_ERR_INVALID_ARG, "id is null");
    std::string why;
    const qlc_comm::Api* nccl = qlc_comm::api(&why);
    if (!nccl) return fail(QLC_ERR_COMM, why);
    qlc_comm::UniqueId id;
    const int r = nccl->GetUniqueId(&id);
    if (r != 0) return fail(QLC_ERR_COMM, std::string("ncclGetUniqueId: ") + nccl->GetErrorString(r));
    memcpy(id128, id.internal, QLC_COMM_ID_BYTES);
    return QLC_OK;
}

int32_t qlc_comm_destroy(qlc_env* env) {
    if (!env || !env->comm) return QLC_OK;
    qlc_env::Comm* c = env->comm;
    cudaSetDevice(env->cfg.device);
    cudaDeviceSynchronize();
    if (c->nccl) { std::string why; if (const qlc_comm::Api* nccl = qlc_comm::api(&why)) nccl->CommDestroy(c->nccl); }
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->step_done) cudaEventDestroy(c->step_done);
    for (cudaEvent_t ev : c->slot_read) if (ev) cudaEventDestroy(ev);
    cudaFree(c->snap); cudaFree(c->exit_counter); cudaFree(c->mine); cudaFree(c->gathered); cudaFree(c->reduced);
    if (c->host) cudaFreeHost(c->host);
    delete c;
    env->comm = nullptr;
    return QLC_OK;
}

int32_t qlc_comm_init(qlc_env* env, int32_t rank, int32_t world, const uint8_t* id128) {
    QLC_RANGE("qlc_comm_init");
    if (!env) return fail(QLC_ERR_INVALID_ARG, "env is null");
    if (world < 1 || rank < 0 || rank >= world) return fail(QLC_ERR_INVALID_ARG, "need 0 <= rank < world");
    if (world > 1 && !id128) return fail(QLC_ERR_INVALID_ARG, "a communicator of more than one rank needs the id from qlc_comm_unique_id on rank 0");
    if (env->comm) return fail(QLC_ERR_INVALID_ARG, "this env already has a communicator");
    int32_t rc = set_device(env); if (rc) return rc;
    qlc_env::Comm* c = new qlc_env::Comm();
    c->rank = rank; c->world = world;
    env->comm = c;
    auto bail = [&](int32_t code, const std::string& msg) { qlc_comm_destroy(env); return fail(code, msg); };
    if (id128) {        // world == 1 without an id: no NCCL at all (the reduction is the identity)
        std::string why;
        const qlc_comm::Api* nccl = qlc_comm::api(&why);
        if (!nccl) return bail(QLC_ERR_COMM, why);
        qlc_comm::UniqueId id; memcpy(id.internal, id128, QLC_COMM_ID_BYTES);
        // one CTA for the collective (QLC_COMM_CTAS=0: NCCL's own choice); a library without ncclCommInitRankConfig, or one that
        // refuses the config, gets the plain call
        static const bool one_cta = getenv("QLC_COMM_CTAS") ? atoi(getenv("QLC_COMM_CTAS")) == 1 : true;
        int r = -1;
        if (one_cta && nccl->CommInitRankConfig) {
            qlc_comm::Config cfg = qlc_comm::one_cta_config();
            r = nccl->CommInitRankConfig(&c->nccl, world, id, rank, &cfg);
            if (r != 0) c->nccl = nullptr;
        }
        if (r != 0) r = nccl->CommInitRank(&c->nccl, world, id, rank);
        if (r != 0) { c->nccl = nullptr; return bail(QLC_ERR_COMM, std::string("ncclCommInitRank: ") + nccl->GetErrorString(r)); }
    }
    cudaError_t e = cudaSuccess;
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);                    // lowest priority: step CTAs are scheduled first
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, lo);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->step_done, cudaEventDisableTiming);
    for (cudaEvent_t& ev : c->slot_read) if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(&c->snap, 4 * sizeof(DeviceStats));
    if (e == cudaSuccess) e = cudaMalloc(&c->exit_counter, 4);
    if (e == cudaSuccess) e = cudaMemset(c->exit_counter, 0, 4);
    if (e == cudaSuccess) e = cudaMalloc(&c->mine, 5 * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&c->gathered, (size_t)world * 5 * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&c->reduced, 5 * sizeof(double));
    if (e == cudaSuccess) e = cudaMallocHost(&c->host, 5 * sizeof(double));
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return bail(QLC_ERR_CUDA, std::string("qlc_comm_init: ") + cudaGetErrorString(e));
    for (int i = 0; i < 5; ++i) c->host[i] = i < 3 ? 0.0 : -1.0e300;
    return QLC_OK;
}

int32_t qlc_comm_info(qlc_env* env, int32_t* rank, int32_t* world, int32_t* nccl_version, int32_t* nccl_ranks) {
    if (!env || !env->comm) return fail(QLC_ERR_INVALID_ARG, "no communicator (qlc_comm_init)");
    if (rank) *rank = env->comm->rank;
    if (world) *world = env->comm->world;
    if (nccl_version) *nccl_version = 0;
    if (nccl_ranks) *nccl_ranks = 0;
    if (env->comm->nccl) {
        std::string why;
        const qlc_comm::Api* nccl = qlc_comm::api(&why);
        int v = 0, n = 0;
        if (nccl && nccl->GetVersion(&v) == 0 && nccl_version) *nccl_version = v;
        if (nccl && nccl->CommCount(env->comm->nccl, &n) == 0 && nccl_ranks) *nccl_ranks = n;
    }
    return QLC_OK;
}

// Enqueues one reduction of {sum_return, episodes, steps, min, max} over all ranks. Nothing but an event record lands on
// `stream` (the caller's step stream): the export, ONE ncclAllGather of 5 doubles, the combine and the copy to the host mirror
// run on the communicator's own low-priority stream, behind the work `stream` holds now, next to whatever it is given later.
int32_t qlc_stats_allreduce(qlc_env* env, void* stream) {
    QLC_RANGE("qlc_stats_allreduce");
    if (!env || !env->comm) return fail(QLC_ERR_INVALID_ARG, "no communicator (qlc_comm_init)");
    int32_t rc = set_device(env); if (rc) return rc;
    qlc_env::Comm* c = env->comm;
    CUDA_TRY(cudaEventRecord(c->step_done, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamWaitEvent(c->stream, c->step_done, 0));
    const uint64_t steps = env->t * env->cfg.n_envs;
    const uint32_t slot = c->last_serial & 3u;
    // the snapshot the last launch left (launches after it may already be running); before the first launch: the accumulators
    stats_export_kernel<<<1, 1, 0, c->stream>>>(c->have_snap ? c->snap + slot : env->stats, steps, c->mine);
    CUDA_TRY(cudaGetLastError());
    if (c->have_snap) { CUDA_TRY(cudaEventRecord(c->slot_read[slot], c->stream)); c->slot_busy[slot] = true; }
    const double* result = c->mine;
    if (c->nccl) {
        std::string why;
        const qlc_comm::Api* nccl = qlc_comm::api(&why);
        if (!nccl) return fail(QLC_ERR_COMM, why);
        const int r = nccl->AllGather(c->mine, c->gathered, 5, qlc_comm::kFloat64, c->nccl, (void*)c->stream);
        if (r != 0) return fail(QLC_ERR_COMM, std::string("ncclAllGather: ") + nccl->GetErrorString(r));
        stats_combine_kernel<<<1, 1, 0, c->stream>>>(c->gathered, c->world, c->reduced);
        CUDA_TRY(cudaGetLastError());
        result = c->reduced;
    }
    CUDA_TRY(cudaMemcpyAsync(c->host, result, 5 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    c->reductions += 1;
    c->armed = true;
    return QLC_OK;
}

// The job-wide statistics of the last reduction that has completed (wait != 0: of the last one enqueued).
int32_t qlc_stats_global(qlc_env* env, qlc_episode_stats* out, int32_t wait) {
    if (!env || !out) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    if (!env->comm) return fail(QLC_ERR_INVALID_ARG, "no communicator (qlc_comm_init)");
    int32_t rc = set_device(env); if (rc) return rc;
    if (wait) CUDA_TRY(cudaStreamSynchronize(env->comm->stream));
    const volatile double* h = env->comm->host;
    out->sum_return = (uint64_t)h[0]; out->episodes = (uint64_t)h[1]; out->steps = (uint64_t)h[2];
    const bool any = out->episodes != 0;
    out->min_return = any ? (uint32_t)(-h[3]) : 0xFFFFFFFFu; out->max_return = any ? (uint32_t)h[4] : 0u;
    return QLC_OK;
}

int32_t qlc_stats_push(qlc_env* env, float r) {                      // Buffer::add (replay_buffer.rs:21-29)
    if (!env) return fail(QLC_ERR_INVALID_ARG, "env is null");
    if (env->window.size() >= env->cfg.episode_window) env->window.pop_front();
    env->window.push_back(r);
    return QLC_OK;
}
int32_t qlc_stats_mean(qlc_env* env, float* out) {                   // avg_episode_reward :107-111
    if (!env || !out) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    if (env->window.empty()) return fail(QLC_ERR_NOT_ENOUGH, "episode reward history is empty");
    float sum = 0.0f;
    for (float v : env->window) sum = sum + v;
    *out = sum / (float)env->window.size();
    return QLC_OK;
}
int32_t qlc_stats_min(qlc_env* env, float* out) {                    // min_episode_reward :113-120
    if (!env || !out) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    if (env->window.empty()) return fail(QLC_ERR_NOT_ENOUGH, "episode reward history is empty");
    float mn = env->window.front();
    for (float v : env->window) if (v < mn) mn = v;
    *out = mn;
    return QLC_OK;
}
int32_t qlc_stats_window(qlc_env* env, float* out, uint32_t cap, uint32_t* n) {   // episode_rewards :124
    if (!env || !n) return fail(QLC_ERR_INVALID_ARG, "env/n is null");
    uint32_t i = 0;
    for (float v : env->window) { if (out && i < cap) out[i] = v; ++i; }
    *n = i;
    return QLC_OK;
}

// ---------------- checkpoint / resume (SURVEY.md 8f-4; the reference checkpoints only the model) ----------------
namespace {
struct CkptHeader {
    char magic[8];                 // "QLCCKPT1"
    uint32_t version, header_bytes;
    qlc_config cfg;
    uint32_t time_slots, t_cap;
    uint64_t t;
    DeviceStats stats;
    uint32_t window_len, reserved;
};
struct CkptArray { void* ptr; size_t bytes; };

static std::vector<CkptArray> ckpt_arrays(qlc_env* env) {
    const size_t n = env->cfg.n_envs;
    return {
        {env->st.ball_cx, n * 4}, {env->st.ball_cy, n * 4}, {env->st.ball_dx, n * 4}, {env->st.ball_dy, n * 4},
        {env->st.pad_min_x, n * 4}, {env->st.pad_max_x, n * 4}, {env->st.pad_speed, n * 4}, {env->st.bricks, n * 8},
        {env->st.score, n * 4}, {env->st.episode_step, n * 4}, {env->st.episode, n * 4}, {env->st.err, n * 4}, {env->st.finished, n},
        {env->records, (size_t)env->time_slots * n * 4}, {env->frames, (size_t)env->time_slots * n * FRAME_BYTES},
    };
}
}  // namespace

int32_t qlc_env_save(qlc_env* env, const char* path) {
    QLC_RANGE("qlc_env_save");
    if (!env || !path) return fail(QLC_ERR_INVALID_ARG, "env/path is null");
    int32_t rc = set_device(env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    FILE* f = fopen(path, "wb");
    if (!f) return fail(QLC_ERR_INVALID_ARG, std::string("cannot open ") + path);
    CkptHeader h{};
    memcpy(h.magic, "QLCCKPT1", 8); h.version = 1; h.header_bytes = sizeof h; h.cfg = env->cfg;
    h.time_slots = env->time_slots; h.t_cap = env->t_cap; h.t = env->t; h.window_len = (uint32_t)env->window.size();
    cudaError_t e = cudaMemcpy(&h.stats, env->stats, sizeof h.stats, cudaMemcpyDeviceToHost);
    bool ok = e == cudaSuccess && fwrite(&h, sizeof h, 1, f) == 1;
    for (float v : env->window) ok = ok && fwrite(&v, 4, 1, f) == 1;
    const size_t CH = (size_t)64 << 20;
    if (ok && ensure_pin(env, CH) != QLC_OK) ok = false;
    for (const CkptArray& a : ckpt_arrays(env)) {
        for (size_t off = 0; ok && off < a.bytes; off += CH) {
            const size_t m = a.bytes - off < CH ? a.bytes - off : CH;
            ok = cudaMemcpy(env->pin, (const char*)a.ptr + off, m, cudaMemcpyDeviceToHost) == cudaSuccess && fwrite(env->pin, 1, m, f) == m;
        }
    }
    ok = (fclose(f) == 0) && ok;
    if (!ok) return fail(QLC_ERR_CUDA, std::string("writing checkpoint failed: ") + path);
    return QLC_OK;
}

int32_t qlc_env_load(qlc_env* env, const char* path) {
    QLC_RANGE("qlc_env_load");
    if (!env || !path) return fail(QLC_ERR_INVALID_ARG, "env/path is null");
    int32_t rc = set_device(env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    FILE* f = fopen(path, "rb");
    if (!f) return fail(QLC_ERR_INVALID_ARG, std::string("cannot open ") + path);
    CkptHeader h{};
    if (fread(&h, sizeof h, 1, f) != 1 || memcmp(h.magic, "QLCCKPT1", 8) != 0 || h.version != 1 || h.header_bytes != sizeof h) {
        fclose(f); return fail(QLC_ERR_INVALID_ARG, "not a ql_cuda checkpoint (or another version)");
    }
    const qlc_config& a = h.cfg; const qlc_config& b = env->cfg;
    if (a.n_envs != b.n_envs || a.env_id_base != b.env_id_base || a.seed != b.seed || h.time_slots != env->time_slots || h.t_cap != env->t_cap ||
        a.max_episode_steps != b.max_episode_steps || a.auto_reset != b.auto_reset) {
        fclose(f); return fail(QLC_ERR_INVALID_ARG, "checkpoint was taken with a different configuration (n_envs / env_id_base / seed / replay_capacity / episode limits)");
    }
    bool ok = true;
    std::deque<float> window;
    for (uint32_t i = 0; ok && i < h.window_len; ++i) { float v; ok = fread(&v, 4, 1, f) == 1; window.push_back(v); }
    const size_t CH = (size_t)64 << 20;
    if (ok && ensure_pin(env, CH) != QLC_OK) ok = false;
    for (const CkptArray& arr : ckpt_arrays(env)) {
        for (size_t off = 0; ok && off < arr.bytes; off += CH) {
            const size_t m = arr.bytes - off < CH ? arr.bytes - off : CH;
            ok = fread(env->pin, 1, m, f) == m && cudaMemcpy((char*)arr.ptr + off, env->pin, m, cudaMemcpyHostToDevice) == cudaSuccess;
        }
    }
    fclose(f);
    ++env->generation;                               // the ring may have been (partly) overwritten, whether or not the load succeeds
    if (ok) ok = cudaMemcpy(env->stats, &h.stats, sizeof h.stats, cudaMemcpyHostToDevice) == cudaSuccess;
    // a pageable host-to-device copy may return before its DMA lands: done before a step or an export on a non-blocking stream
    if (ok) ok = cudaDeviceSynchronize() == cudaSuccess;
    if (!ok) return fail(QLC_ERR_CUDA, std::string("reading checkpoint failed (the env state is now undefined): ") + path);
    env->t = h.t; env->window = window;
    if (env->comm) env->comm->have_snap = false;     // the snapshots belong to the run that was replaced
    return QLC_OK;
}

// ---------------- debug / known-answer ----------------
static int32_t run_debug(int which, float cx, float cy, float r, float mvx, float mvy, float minx, float miny, float maxx, float maxy,
                         int32_t* some, float* way, float* approx, float* nx, float* ny, uint32_t* err) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(QLC_ERR_NO_DEVICE, "no CUDA device: ql_cuda has no CPU fallback");
    float* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, 8 * sizeof(float)));
    debug_collision_kernel<<<1, 1>>>(which, cx, cy, r, mvx, mvy, minx, miny, maxx, maxy, d, (uint32_t*)(d + 6));
    cudaError_t e = cudaGetLastError();
    float h[8];
    if (e == cudaSuccess) e = cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(QLC_ERR_CUDA, std::string("debug kernel: ") + cudaGetErrorString(e));
    if (some) *some = h[0] != 0.0f;
    if (way) *way = h[1];
    if (approx) *approx = h[2];
    if (nx) *nx = h[3];
    if (ny) *ny = h[4];
    if (err) memcpy(err, &h[6], 4);
    return QLC_OK;
}
int32_t qlc_debug_collision_rect_batch(const float* in_host, float* out_host, uint32_t n) {
    if (!in_host || !out_host) return fail(QLC_ERR_INVALID_ARG, "in/out is null");
    if (n == 0) return QLC_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(QLC_ERR_NO_DEVICE, "no CUDA device: ql_cuda has no CPU fallback");
    float *din = nullptr, *dout = nullptr;
    CUDA_TRY(cudaMalloc(&din, (size_t)n * 9 * sizeof(float)));
    cudaError_t e = cudaMalloc(&dout, (size_t)n * 6 * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(din, in_host, (size_t)n * 9 * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) { debug_collision_batch_kernel<<<(n + 127) / 128, 128>>>(din, dout, n); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaMemcpy(out_host, dout, (size_t)n * 6 * sizeof(float), cudaMemcpyDeviceToHost);
    cudaFree(din); cudaFree(dout);
    if (e != cudaSuccess) return fail(QLC_ERR_CUDA, std::string("debug batch: ") + cudaGetErrorString(e));
    return QLC_OK;
}
}  // extern "C"

// gemm_tc_kernel over n_splits K slices (gridDim.z); persistent CTAs along M, as many as fit beside the other N tiles
template <int NT, class Loader, class Epi>
static cudaError_t launch_gemm(const Loader& ld, const __nv_bfloat16* w, const Epi& epi, uint32_t m, uint32_t k, uint32_t n_total, uint32_t n_splits,
                               unsigned int* err, cudaStream_t s) {
    const size_t dyn = 2 * ((size_t)qnet::TILE_M * qnet::KC * 2 + (size_t)NT * qnet::KC * 2);
    auto kern = qnet::gemm_tc_kernel<NT, Loader, Epi>;
    static int occ_dev[64] = {}, sms_dev[64] = {};
    int cur_dev = 0; cudaGetDevice(&cur_dev);
    int &occ = occ_dev[cur_dev & 63], &sms = sms_dev[cur_dev & 63];
    cudaError_t e = cudaSuccess;
    if (occ == 0) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
        if (e != cudaSuccess) return e;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 128, dyn);
        if (e != cudaSuccess) return e;
        int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const int tmem_limit = 512 / (NT <= 32 ? 32 : (NT <= 64 ? 64 : (NT <= 128 ? 128 : 256)));   // TMEM columns per SM
        if (occ > tmem_limit) occ = tmem_limit;
        if (occ < 1) occ = 1;
    }
    const uint32_t n_mtiles = (m + qnet::TILE_M - 1) / qnet::TILE_M, n_ntiles = n_total / NT;
    uint32_t gx = (uint32_t)(occ * sms) / (n_ntiles * n_splits);
    if (gx < 1) gx = 1;
    if (gx > n_mtiles) gx = n_mtiles;
    kern<<<dim3(gx, n_ntiles, n_splits), 128, dyn, s>>>(ld, w, epi, m, k, n_total, err);
    return cudaGetLastError();
}

template <class G, class Out>
static cudaError_t launch_conv_sw(const qnet::ConvArgs& a, const Out& o, cudaStream_t s) {
    auto kern = qnet::conv_sw_kernel<G, Out>;
    static int sms[64] = {};                             // per device: function attributes are per context
    int dev = 0; cudaGetDevice(&dev);
    int& n_sm = sms[dev & 63];
    if (n_sm == 0) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    }
    const uint32_t n_batches = (a.n_items + G::B - 1) / G::B;
    return launch_pdl(kern, dim3(n_batches < (uint32_t)n_sm ? n_batches : (uint32_t)n_sm), dim3(G::THREADS), G::SMEM_BYTES, s, a, o);      // persistent: one CTA per SM
}

extern "C" {

// ---------------- Q-network forward on the tensor cores (SURVEY.md 8f-3) ----------------
struct qlc_qnet {
    qlc_env* env = nullptr;                                                 // NULL once the env has been destroyed: every call but destroy fails
    int device = 0;
    float* w5 = nullptr;
    float *b1 = nullptr, *b2 = nullptr, *b3 = nullptr, *b4 = nullptr, *b5 = nullptr;
    __nv_bfloat16 *w1p = nullptr, *w2p = nullptr, *w3p = nullptr, *w4p = nullptr, *w4p256 = nullptr;   // operand-layout weights (dense: N tiles of 128 and of 256): planes [K/8][N][8]
    __nv_bfloat16* a4 = nullptr; uint32_t* slot_frame = nullptr; unsigned int* err = nullptr;
    float4* head_partial = nullptr; uint32_t* head_count = nullptr;       // dense epilogue -> fused head (per-N-tile partials, per-row tickets)
    __nv_bfloat16 *a1p = nullptr, *a2p = nullptr, *a3p = nullptr;         // conv outputs in the next layer's operand (plane) layout
    unsigned long long* prof = nullptr;                                    // QLC_QNET_PROF: per-role cycle counters of CTA 0, printed after each forward
    uint32_t cap_items = 0;
    // training (qlc_qnet_train): f32 masters of the 10 Keras variables back to back (b1..b5 point into it), their gradients,
    // Adam moments; bf16 weight copies in the data-gradient GEMMs' operand layouts; scratch sized for train_cap items
    float *master = nullptr, *grad = nullptr, *adam_m = nullptr, *adam_v = nullptr, *norm_partial = nullptr;
    __nv_bfloat16 *w4k = nullptr, *w3r = nullptr, *w2r = nullptr;
    qlc_adam_config adam{2.5e-4f, 0.9f, 0.999f, 1e-7f, 1.0f};
    uint64_t adam_t = 0;                                                   // updates since set_weights / set_adam
    uint32_t train_cap = 0, y_cap = 0;
    float *t_q = nullptr, *t_dq = nullptr, *t_loss = nullptr, *t_dh = nullptr, *t_d3 = nullptr, *t_d2 = nullptr, *t_d1 = nullptr, *t_split = nullptr, *t_colsum = nullptr;
    __nv_bfloat16 *t_dh_bf = nullptr, *t_d3_bf = nullptr, *t_d2_bf = nullptr, *t_pack = nullptr;
    // targets of one call, sized for y_cap items: y, target-network max-Q; for n-step / double DQN also returns, discounts,
    // bootstrap indices, target-network q [n][3], online greedy actions. All seven grow together, so a one-step call also holds
    // the n-step arrays (25 bytes per item: 0.8 MB at 32,768 items) in exchange for one allocation rule.
    float *t_y = nullptr, *t_maxq = nullptr, *t_ret = nullptr, *t_disc = nullptr, *t_tq = nullptr; uint32_t* t_boot = nullptr; uint8_t* t_act = nullptr;
    size_t split_floats = 0, pack_elems = 0;
};

// per-minibatch scratch of the backward (sized for train_cap items)
static void qnet_free_scratch(qlc_qnet* q) {
    void* p[] = {q->t_q, q->t_dq, q->t_loss, q->t_dh, q->t_d3, q->t_d2, q->t_d1, q->t_split, q->t_colsum, q->t_dh_bf, q->t_d3_bf, q->t_d2_bf, q->t_pack};
    for (void* x : p) cudaFree(x);
    q->t_q = q->t_dq = q->t_loss = q->t_dh = q->t_d3 = q->t_d2 = q->t_d1 = q->t_split = q->t_colsum = nullptr;
    q->t_dh_bf = q->t_d3_bf = q->t_d2_bf = q->t_pack = nullptr; q->train_cap = 0; q->split_floats = 0; q->pack_elems = 0;
}
// targets of one call (sized for y_cap items)
static void qnet_free_targets(qlc_qnet* q) {
    cudaFree(q->t_y); cudaFree(q->t_maxq); cudaFree(q->t_ret); cudaFree(q->t_disc); cudaFree(q->t_tq); cudaFree(q->t_boot); cudaFree(q->t_act);
    q->t_y = q->t_maxq = q->t_ret = q->t_disc = q->t_tq = nullptr; q->t_boot = nullptr; q->t_act = nullptr; q->y_cap = 0;
}
static void qnet_free_train(qlc_qnet* q) { qnet_free_scratch(q); qnet_free_targets(q); }

static void qnet_free_acts(qlc_qnet* q) {
    cudaFree(q->a4); cudaFree(q->slot_frame); cudaFree(q->a1p); cudaFree(q->a2p); cudaFree(q->a3p); cudaFree(q->head_partial); cudaFree(q->head_count);
    q->a4 = q->a1p = q->a2p = q->a3p = nullptr; q->head_partial = nullptr; q->head_count = nullptr; q->slot_frame = nullptr; q->cap_items = 0;
}

}  // extern "C"

// frees everything the network holds on the device and cuts its tie to the env (called by qlc_qnet_destroy, and by
// qlc_env_destroy for networks that outlive their env: their handle stays valid, but only for qlc_qnet_destroy)
static void qnet_release_device(qlc_qnet* q) {
    if (!q->env) return;
    cudaSetDevice(q->device);
    cudaDeviceSynchronize();
    qnet_free_acts(q);
    qnet_free_train(q);
    cudaFree(q->w5); cudaFree(q->w1p); cudaFree(q->w2p); cudaFree(q->w3p); cudaFree(q->w4p); cudaFree(q->w4p256);
    cudaFree(q->master); cudaFree(q->grad); cudaFree(q->adam_m); cudaFree(q->adam_v); cudaFree(q->norm_partial); cudaFree(q->w4k); cudaFree(q->w3r); cudaFree(q->w2r);
    cudaFree(q->err); cudaFree(q->prof);
    q->w1p = q->w2p = q->w3p = q->w4p = q->w4p256 = nullptr; q->w5 = nullptr;
    q->master = q->grad = q->adam_m = q->adam_v = q->norm_partial = nullptr; q->w4k = q->w3r = q->w2r = nullptr;
    q->b1 = q->b2 = q->b3 = q->b4 = q->b5 = nullptr; q->err = nullptr; q->prof = nullptr;
    q->env = nullptr;
}

extern "C" {

int32_t qlc_qnet_destroy(qlc_qnet* q) {
    if (!q) return QLC_OK;
    if (qlc_env* env = q->env) {
        for (size_t i = 0; i < env->qnets.size(); ++i)
            if (env->qnets[i] == q) { env->qnets.erase(env->qnets.begin() + i); break; }
        qnet_release_device(q);
    }
    delete q;
    return QLC_OK;
}

// MMA completion time-out flag of the device-path forward (qlc_qnet_forward never synchronises): read and clear
int32_t qlc_qnet_error(qlc_qnet* q, uint32_t* flag) {
    if (!q || !flag) return fail(QLC_ERR_INVALID_ARG, "qnet/out is null");
    if (!q->env) return fail(QLC_ERR_INVALID_ARG, "the environment of this Q-network has been destroyed");
    int32_t rc = set_device(q->env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    unsigned int herr = 0;
    CUDA_TRY(cudaMemcpy(&herr, q->err, 4, cudaMemcpyDeviceToHost));
    *flag = herr;
    if (herr) {
        // a pass that gave up may have left per-row tickets of the fused head behind: start the next one clean
        if (q->head_count) CUDA_TRY(cudaMemset(q->head_count, 0, (size_t)((q->cap_items + 127u) / 128u) * 128u * 4));
        CUDA_TRY(cudaMemset(q->err, 0, 4));
        CUDA_TRY(cudaDeviceSynchronize());              // legacy-stream memsets: done before work on a non-blocking stream
    }
    return QLC_OK;
}

static const float* const* weight_ptrs(const qlc_qnet_weights* w, const float* (&out)[qnet::NVARS]) {
    const float* p[qnet::NVARS] = {w->conv1_kernel, w->conv1_bias, w->conv2_kernel, w->conv2_bias, w->conv3_kernel, w->conv3_bias, w->dense1_kernel, w->dense1_bias, w->dense2_kernel, w->dense2_bias};
    for (int i = 0; i < qnet::NVARS; ++i) out[i] = p[i];
    return out;
}

// operand-layout bf16 copies of the f32 masters (the forward's, and the backward's data-gradient weights), on `s`
static cudaError_t qnet_prep_weights(qlc_qnet* q, cudaStream_t s) {
    const float* m = q->master;
    auto V = [&](int v) { return m + qnet::var_offset(v); };
    qnet::prep_conv1_planes_kernel<<<(32 * 256 + 255) / 256, 256, 0, s>>>(V(0), q->w1p);
    qnet::prep_conv2_planes_kernel<<<(512 * 64 + 255) / 256, 256, 0, s>>>(V(2), q->w2p);
    qnet::prep_conv3_planes_kernel<<<(576 * 64 + 255) / 256, 256, 0, s>>>(V(4), q->w3p);
    qnet::prep_dense_planes_kernel<128><<<(3136 * 512 + 255) / 256, 256, 0, s>>>(V(6), q->w4p);
    qnet::prep_dense_planes_kernel<256><<<(3136 * 512 + 255) / 256, 256, 0, s>>>(V(6), q->w4p256);
    qnet::prep_head_kernel<<<(3 * 512 + 255) / 256, 256, 0, s>>>(V(8), q->w5);
    qnet::prep_dgrad_weights_kernel<16, 32, 64><<<(16 * 32 * 64 + 255) / 256, 256, 0, s>>>(V(2), q->w2r);
    qnet::prep_dgrad_weights_kernel<9, 64, 64><<<(9 * 64 * 64 + 255) / 256, 256, 0, s>>>(V(4), q->w3r);
    qnet::f32_to_bf16_kernel<<<1024, 256, 0, s>>>(V(6), q->w4k, (size_t)3136 * 512);
    return cudaGetLastError();
}

static int32_t qnet_reset_adam(qlc_qnet* q) {
    CUDA_TRY(cudaMemset(q->adam_m, 0, (size_t)qnet::N_PARAMS * 4));
    CUDA_TRY(cudaMemset(q->adam_v, 0, (size_t)qnet::N_PARAMS * 4));
    CUDA_TRY(cudaDeviceSynchronize());                  // legacy-stream memsets: done before an update on a non-blocking stream
    q->adam_t = 0;
    return QLC_OK;
}

int32_t qlc_qnet_set_weights(qlc_qnet* q, const qlc_qnet_weights* w) {
    if (!q || !w) return fail(QLC_ERR_INVALID_ARG, "qnet/weights is null");
    if (!q->env) return fail(QLC_ERR_INVALID_ARG, "the environment of this Q-network has been destroyed");
    const float* srcs[qnet::NVARS];
    weight_ptrs(w, srcs);
    for (int i = 0; i < qnet::NVARS; ++i) if (!srcs[i]) return fail(QLC_ERR_INVALID_ARG, "a weight pointer is null");
    int32_t rc = set_device(q->env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    for (int v = 0; v < qnet::NVARS; ++v) CUDA_TRY(cudaMemcpy(q->master + qnet::var_offset(v), srcs[v], (size_t)qnet::var_size(v) * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(qnet_prep_weights(q, nullptr));
    CUDA_TRY(cudaDeviceSynchronize());
    return qnet_reset_adam(q);
}

int32_t qlc_qnet_get_weights(qlc_qnet* q, const qlc_qnet_weights* w) {
    if (!q || !w) return fail(QLC_ERR_INVALID_ARG, "qnet/weights is null");
    if (!q->env) return fail(QLC_ERR_INVALID_ARG, "the environment of this Q-network has been destroyed");
    const float* dst[qnet::NVARS];
    weight_ptrs(w, dst);
    for (int i = 0; i < qnet::NVARS; ++i) if (!dst[i]) return fail(QLC_ERR_INVALID_ARG, "a weight pointer is null");
    int32_t rc = set_device(q->env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    for (int v = 0; v < qnet::NVARS; ++v) CUDA_TRY(cudaMemcpy(const_cast<float*>(dst[v]), q->master + qnet::var_offset(v), (size_t)qnet::var_size(v) * 4, cudaMemcpyDeviceToHost));
    return QLC_OK;
}

int32_t qlc_qnet_set_adam(qlc_qnet* q, const qlc_adam_config* cfg) {
    if (!q || !cfg) return fail(QLC_ERR_INVALID_ARG, "qnet/cfg is null");
    if (!q->env) return fail(QLC_ERR_INVALID_ARG, "the environment of this Q-network has been destroyed");
    if (!(cfg->lr >= 0.0f) || !(cfg->beta1 >= 0.0f && cfg->beta1 < 1.0f) || !(cfg->beta2 >= 0.0f && cfg->beta2 < 1.0f) || !(cfg->epsilon >= 0.0f) || cfg->clipnorm != cfg->clipnorm)
        return fail(QLC_ERR_INVALID_ARG, "adam config out of range");
    int32_t rc = set_device(q->env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    q->adam = *cfg;
    return qnet_reset_adam(q);
}

int32_t qlc_qnet_create(qlc_env* env, const qlc_qnet_weights* w, qlc_qnet** out) {
    if (!env || !w || !out) return fail(QLC_ERR_INVALID_ARG, "env/weights/out is null");
    *out = nullptr;
    int32_t rc = set_device(env); if (rc) return rc;
    qlc_qnet* q = new qlc_qnet();
    q->env = env; q->device = env->cfg.device;
    env->qnets.push_back(q);
    cudaError_t e = cudaSuccess;
    auto A = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
    A((void**)&q->w5, 3 * 512 * 4);
    A((void**)&q->w1p, 32 * 256 * 2); A((void**)&q->w2p, 64 * 512 * 2); A((void**)&q->w3p, 64 * 576 * 2); A((void**)&q->w4p, (size_t)512 * 3136 * 2); A((void**)&q->w4p256, (size_t)512 * 3136 * 2);
    if (getenv("QLC_QNET_PROF")) A((void**)&q->prof, 3 * 32 * 8);
    A((void**)&q->master, (size_t)qnet::N_PARAMS * 4); A((void**)&q->grad, (size_t)qnet::N_PARAMS * 4);
    A((void**)&q->adam_m, (size_t)qnet::N_PARAMS * 4); A((void**)&q->adam_v, (size_t)qnet::N_PARAMS * 4); A((void**)&q->norm_partial, qnet::NVARS * qnet::NORM_CHUNKS * 4);
    A((void**)&q->w4k, (size_t)3136 * 512 * 2); A((void**)&q->w3r, 64 * 576 * 2); A((void**)&q->w2r, 32 * 1024 * 2); A((void**)&q->err, 4);
    if (e == cudaSuccess) {
        q->b1 = q->master + qnet::var_offset(1); q->b2 = q->master + qnet::var_offset(3); q->b3 = q->master + qnet::var_offset(5);
        q->b4 = q->master + qnet::var_offset(7); q->b5 = q->master + qnet::var_offset(9);
        e = cudaMemset(q->err, 0, 4);
    }
    if (e != cudaSuccess) { qlc_qnet_destroy(q); return fail(QLC_ERR_CUDA, std::string("qnet alloc: ") + cudaGetErrorString(e)); }
    rc = qlc_qnet_set_weights(q, w);
    if (rc) { qlc_qnet_destroy(q); return rc; }
    *out = q;
    return QLC_OK;
}

}  // extern "C"

// the forward chain; hidden (training): keep the bf16 dense-1 activations in q->a4
static int32_t qnet_forward(qlc_qnet* q, const uint32_t* idx_dev, uint32_t n, int32_t which, float* q_dev, uint8_t* action_dev, float* max_q_dev, bool hidden_out,
                            void* stream) {
    if (!q) return fail(QLC_ERR_INVALID_ARG, "qnet is null");
    qlc_env* env = q->env;
    if (!env) return fail(QLC_ERR_INVALID_ARG, "the environment of this Q-network has been destroyed");
    int32_t rc = set_device(env); if (rc) return rc;
    if (!idx_dev) { n = env->cfg.n_envs; which = 0; }
    if (n == 0) return QLC_OK;
    if ((uint64_t)n * 400ull >= 0xFFFFFFFFull) return fail(QLC_ERR_INVALID_ARG, "too many items for one forward pass");
    cudaStream_t s = (cudaStream_t)stream;
    if (n > q->cap_items) {
        // the new buffers are cleared on `s`: a plain cudaMemset runs on the legacy stream, which a non-blocking stream (the
        // env's own) does not wait for, and could then zero conv outputs and head tickets under this pass's kernels
        CUDA_TRY(cudaDeviceSynchronize());
        qnet_free_acts(q);
        CUDA_TRY(cudaMalloc(&q->a4, (size_t)n * 512 * 2)); CUDA_TRY(cudaMalloc(&q->slot_frame, (size_t)n * 16));
        const size_t a1p_bytes = (size_t)((n + qnet::Conv2Geom::B - 1) / qnet::Conv2Geom::B) * qnet::Conv2Geom::STAGE_BYTES;
        const size_t a2p_bytes = (size_t)((n + qnet::Conv3Geom::B - 1) / qnet::Conv3Geom::B) * qnet::Conv3Geom::STAGE_BYTES;
        CUDA_TRY(cudaMalloc(&q->a1p, a1p_bytes)); CUDA_TRY(cudaMalloc(&q->a2p, a2p_bytes));
        const size_t a3p_bytes = (size_t)((n + 127) / 128) * qnet::DenseGeom::A_TILE_BYTES;
        CUDA_TRY(cudaMalloc(&q->a3p, a3p_bytes)); CUDA_TRY(cudaMemsetAsync(q->a3p, 0, a3p_bytes, s));
        const size_t rows_padded = (size_t)((n + 127) / 128) * 128;
        CUDA_TRY(cudaMalloc(&q->head_partial, 4 * rows_padded * sizeof(float4))); CUDA_TRY(cudaMalloc(&q->head_count, rows_padded * 4));
        CUDA_TRY(cudaMemsetAsync(q->head_count, 0, rows_padded * 4, s));
        CUDA_TRY(cudaMemsetAsync(q->a1p, 0, a1p_bytes, s)); CUDA_TRY(cudaMemsetAsync(q->a2p, 0, a2p_bytes, s));     // rows of a partial last batch are read (never used)
        q->cap_items = n;
    }
    GatherParams g{}; fill_gather(env, g);
    g.indices = idx_dev; g.n_items = n; g.mode = idx_dev ? GATHER_INDICES : GATHER_CURRENT;
    // conv1's loader works out where each item's four frames are (the gather kernels' locate()) - no separate kernel
    const qnet::ConvArgs c1{(const uint8_t*)q->w1p, q->b1, env->frames, g, which ? 1u : 0u, n, q->err, q->prof};
    cudaError_t e = launch_conv_sw<qnet::Conv1Geom>(c1, qnet::OutConv2Planes{q->a1p}, s);
    if (e != cudaSuccess) return fail(QLC_ERR_CUDA, std::string("conv1: ") + cudaGetErrorString(e));
    const qnet::ConvArgs c2{(const uint8_t*)q->w2p, q->b2, (const uint8_t*)q->a1p, GatherParams{}, 0u, n, q->err, q->prof ? q->prof + 32 : nullptr};
    e = launch_conv_sw<qnet::Conv2Geom>(c2, qnet::OutConv3Planes{q->a2p}, s);
    if (e != cudaSuccess) return fail(QLC_ERR_CUDA, std::string("conv2: ") + cudaGetErrorString(e));
    const qnet::ConvArgs c3{(const uint8_t*)q->w3p, q->b3, (const uint8_t*)q->a2p, GatherParams{}, 0u, n, q->err, q->prof ? q->prof + 64 : nullptr};
    e = launch_conv_sw<qnet::Conv3Geom>(c3, qnet::OutDensePlanes{q->a3p}, s);
    if (e != cudaSuccess) return fail(QLC_ERR_CUDA, std::string("conv3: ") + cudaGetErrorString(e));
    static bool attr_set[64] = {};
    if (!attr_set[env->cfg.device & 63]) {
        CUDA_TRY(cudaFuncSetAttribute(qnet::dense_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qnet::DenseGeomT<128>::SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(qnet::dense_tc_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qnet::DenseGeomT<256>::SMEM_BYTES));
        attr_set[env->cfg.device & 63] = true;
    }
    // N tiles of 128 while (M tiles x 2) CTAs would leave SMs idle (the layer is bound by per-SM L2 ingest), 256 beyond
    const uint32_t m_tiles = (n + 127) / 128;
    const bool narrow = m_tiles * 2u < (uint32_t)env->sm_count;
    // the head (Dense 512 -> 3, argmax, max) runs in the dense epilogue; rows_padded is that of the allocation (cap_items)
    const qnet::HeadArgs head{q->w5, q->b5, q->head_partial, q->head_count, ((q->cap_items + 127u) / 128u) * 128u, q_dev, action_dev, max_q_dev};
    __nv_bfloat16* hidden = hidden_out ? q->a4 : nullptr;                 // the 512 hidden activations are only needed by training
    if (narrow)
        CUDA_TRY(launch_pdl(qnet::dense_tc_kernel<128>, dim3(m_tiles, 4), dim3(qnet::DenseGeomT<128>::THREADS), qnet::DenseGeomT<128>::SMEM_BYTES, s, (const uint8_t*)q->a3p,
                            (const uint8_t*)q->w4p, (const float*)q->b4, hidden, n, q->err, head));
    else
        CUDA_TRY(launch_pdl(qnet::dense_tc_kernel<256>, dim3(m_tiles, 2), dim3(qnet::DenseGeomT<256>::THREADS), qnet::DenseGeomT<256>::SMEM_BYTES, s, (const uint8_t*)q->a3p,
                            (const uint8_t*)q->w4p256, (const float*)q->b4, hidden, n, q->err, head));
    CUDA_TRY(cudaGetLastError());
    if (q->prof) {
        unsigned long long h[96];
        CUDA_TRY(cudaStreamSynchronize(s));
        CUDA_TRY(cudaMemcpy(h, q->prof, sizeof(h), cudaMemcpyDeviceToHost));
        static const char* roles[4] = {"epilogue", "mma", "loader", "converter"};
        for (int l = 0; l < 3; ++l) for (int r = 0; r < 4; ++r)
            fprintf(stderr, "qnet prof conv%d %-9s total %8llu wait1 %8llu wait2 %8llu other-wait %8llu\n", l + 1, roles[r], h[l * 32 + r * 8], h[l * 32 + r * 8 + 1], h[l * 32 + r * 8 + 2], h[l * 32 + r * 8 + 7]);
    }
    return QLC_OK;
}

extern "C" int32_t qlc_qnet_forward(qlc_qnet* q, const uint32_t* idx_dev, uint32_t n, int32_t which, float* q_dev, uint8_t* action_dev, float* max_q_dev, void* stream) {
    QLC_RANGE("qlc_qnet_forward");
    if (!q) return fail(QLC_ERR_INVALID_ARG, "qnet is null");
    if (!q->env) return fail(QLC_ERR_INVALID_ARG, "the environment of this Q-network has been destroyed");
    return on_caller_stream(q->env, stream, [&] { return qnet_forward(q, idx_dev, n, which, q_dev, action_dev, max_q_dev, false, stream); });
}

extern "C" {

int32_t qlc_qnet_forward_host(qlc_qnet* q, const uint32_t* idx_host, uint32_t n, int32_t which, float* q_host, uint8_t* action_host, float* max_q_host) {
    QLC_RANGE("qlc_qnet_forward_host");
    if (!q) return fail(QLC_ERR_INVALID_ARG, "qnet is null");
    qlc_env* env = q->env;
    if (!env) return fail(QLC_ERR_INVALID_ARG, "the environment of this Q-network has been destroyed");
    int32_t rc = set_device(env); if (rc) return rc;
    if (!idx_host) n = env->cfg.n_envs;
    if (n == 0) return QLC_OK;
    if (idx_host) { const uint64_t len = replay_len(env); for (uint32_t i = 0; i < n; ++i) if (idx_host[i] >= len) return fail(QLC_ERR_OUT_OF_RANGE, "replay index out of range"); }
    rc = after_caller_stream(env); if (rc) return rc;
    const size_t o_idx = 0, o_q = ((size_t)n * 4 + 255) & ~(size_t)255, o_m = o_q + (size_t)n * 12, o_a = o_m + (size_t)n * 4, total = o_a + n;
    rc = ensure_dev_stage(env, total); if (rc) return rc;
    uint8_t* dev = (uint8_t*)env->dev_stage;
    cudaStream_t s = env->own_stream;
    if (idx_host) CUDA_TRY(cudaMemcpyAsync(dev + o_idx, idx_host, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    rc = qnet_forward(q, idx_host ? (const uint32_t*)(dev + o_idx) : nullptr, n, which, (float*)(dev + o_q), dev + o_a, (float*)(dev + o_m), false, s); if (rc) return rc;
    if (q_host) CUDA_TRY(cudaMemcpyAsync(q_host, dev + o_q, (size_t)n * 12, cudaMemcpyDeviceToHost, s));
    if (max_q_host) CUDA_TRY(cudaMemcpyAsync(max_q_host, dev + o_m, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    if (action_host) CUDA_TRY(cudaMemcpyAsync(action_host, dev + o_a, n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    uint32_t herr = 0;
    rc = qlc_qnet_error(q, &herr); if (rc) return rc;
    if (herr) return fail(QLC_ERR_CUDA, "qnet: an MMA completion barrier timed out");
    return QLC_OK;
}

}  // extern "C"

// ---------------- Q-network training (qnet_train.cuh, DESIGN §11) ----------------
// K slices of a weight-gradient GEMM: enough CTAs for the machine (about two per SM), at least two 64-wide K chunks per slice
struct SplitK { uint32_t splits, kc; };
static SplitK pick_splits(uint32_t k_valid, uint32_t mn_tiles) {
    const uint32_t chunks = (k_valid + qnet::KC - 1) / qnet::KC;
    uint32_t sp = (296u + mn_tiles - 1u) / mn_tiles;
    if (sp > 64u) sp = 64u;
    if (sp > (chunks + 1u) / 2u) sp = (chunks + 1u) / 2u;
    if (sp < 1u) sp = 1u;
    const uint32_t per = (chunks + sp - 1u) / sp;
    return SplitK{(chunks + per - 1u) / per, per * (uint32_t)qnet::KC};
}
// the four weight-gradient GEMMs of a minibatch of b items: {K valid, M x N tiles, N, M}
struct WGradShape { uint32_t k_valid, mn_tiles, n, m; };
static void wgrad_shapes(uint32_t b, WGradShape (&w)[4]) {
    w[0] = {b, 25u * 2u, 512u, 3136u};          // dense 1 (N tiles of 256)
    w[1] = {b * 49u, 5u, 64u, 576u};            // conv3
    w[2] = {b * 81u, 4u, 64u, 512u};            // conv2
    w[3] = {b * 400u, 2u, 32u, 256u};           // conv1
}
static uint32_t colsum_rows_per_split(uint32_t rows) { const uint32_t r = (rows + 63u) / 64u; return r < 256u ? 256u : r; }
constexpr uint32_t COLSUM_MAX_SPLITS = 64, COLSUM_MAX_COLS = 1536;

static int32_t qnet_train_alloc(qlc_qnet* q, uint32_t b) {
    if (b <= q->train_cap) return QLC_OK;
    CUDA_TRY(cudaDeviceSynchronize());
    qnet_free_scratch(q);                   // a failed allocation below leaves train_cap = 0 and no stale pointers
    WGradShape ws[4]; wgrad_shapes(b, ws);
    size_t split_floats = 0, pack_elems = 0;
    for (const WGradShape& w : ws) {
        const SplitK sk = pick_splits(w.k_valid, w.mn_tiles);
        split_floats = std::max(split_floats, (size_t)sk.splits * w.m * w.n);
        pack_elems = std::max(pack_elems, (size_t)sk.splits * w.n * sk.kc);
    }
    const size_t n = b;
    cudaError_t e = cudaSuccess;
    auto A = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
    A((void**)&q->t_q, n * 3 * 4); A((void**)&q->t_dq, n * 3 * 4); A((void**)&q->t_loss, n * 4);
    A((void**)&q->t_dh, n * 512 * 4); A((void**)&q->t_dh_bf, n * 512 * 2);
    A((void**)&q->t_d3, n * 3136 * 4); A((void**)&q->t_d3_bf, n * 3136 * 2);
    A((void**)&q->t_d2, n * 5184 * 4); A((void**)&q->t_d2_bf, n * 5184 * 2);
    A((void**)&q->t_d1, n * 12800 * 4);
    A((void**)&q->t_split, split_floats * 4); A((void**)&q->t_pack, pack_elems * 2);
    A((void**)&q->t_colsum, (size_t)COLSUM_MAX_SPLITS * COLSUM_MAX_COLS * 4);
    if (e != cudaSuccess) { cudaGetLastError(); qnet_free_scratch(q); return fail(QLC_ERR_CUDA, std::string("qnet training scratch: ") + cudaGetErrorString(e)); }
    q->split_floats = split_floats; q->pack_elems = pack_elems; q->train_cap = b;
    return QLC_OK;
}

// out[c] = sum over rows of x [rows][c] (fixed order) / div
static cudaError_t launch_colsum(qlc_qnet* q, const float* x, uint32_t rows, uint32_t c, float div, float* out, cudaStream_t s) {
    const uint32_t rps = colsum_rows_per_split(rows), splits = (rows + rps - 1) / rps;
    cudaError_t e = launch_pdl(qnet::colsum_partial_kernel, dim3((c + 31) / 32, splits), dim3(32, 8), 0, s, x, rows, c, rps, q->t_colsum);
    if (e != cudaSuccess) return e;
    return launch_pdl(qnet::colsum_final_kernel, dim3((c + 255) / 256), dim3(256), 0, s, (const float*)q->t_colsum, splits, c, div, out);
}
// dW [m][n] (Keras layout, into the gradient block) = A^T(loader) * dZ [k_valid rows][n] over K slices
template <int NT, class Loader>
static cudaError_t launch_wgrad(qlc_qnet* q, const WGradShape& w, Loader ld, const float* dz, float* out, cudaStream_t s) {
    const SplitK sk = pick_splits(w.k_valid, w.mn_tiles);
    ld.k_valid = w.k_valid; ld.kc = sk.kc;
    const size_t pack = (size_t)sk.splits * w.n * sk.kc;
    cudaError_t e = launch_pdl(qnet::pack_splits_kernel, dim3((uint32_t)std::min<size_t>((pack + 255) / 256, 4096)), dim3(256), 0, s, dz, w.k_valid, w.n, sk.kc, sk.splits, q->t_pack);
    if (e != cudaSuccess) return e;
    e = launch_gemm<NT>(ld, (const __nv_bfloat16*)q->t_pack, qnet::EpiF32{q->t_split, w.m, w.n}, w.m, sk.kc, w.n, sk.splits, q->err, s);
    if (e != cudaSuccess) return e;
    const uint32_t mn = w.m * w.n;
    return launch_pdl(qnet::reduce_splits_kernel, dim3(std::min<uint32_t>((mn + 255) / 256, 2048)), dim3(256), 0, s, (const float*)q->t_split, sk.splits, mn, out);
}

// forward + backward of one minibatch (idx_dev [b], targets y_dev [b], loss weights w_dev [b] or NULL = 1) into q->grad; loss_dev
// (optional) gets the mean weighted Huber loss, td_dev (optional) Q(s)[a] - y; apply: clip + Adam + operand copies of the new weights
static int32_t qnet_train_step(qlc_qnet* q, const uint32_t* idx_dev, uint32_t b, const float* y_dev, const float* w_dev, float* loss_dev, float* td_dev,
                               bool apply, cudaStream_t s) {
    using namespace qnet;
    qlc_env* env = q->env;
    int32_t rc = qnet_train_alloc(q, b); if (rc) return rc;
    rc = qnet_forward(q, idx_dev, b, 0, q->t_q, nullptr, nullptr, true, s); if (rc) return rc;
    float* const g = q->grad;
    auto G = [&](int v) { return g + var_offset(v); };
    GatherParams gp{}; fill_gather(env, gp);
    gp.indices = idx_dev; gp.n_items = b; gp.mode = GATHER_INDICES;
    WGradShape ws[4]; wgrad_shapes(b, ws);
    const uint32_t ew_blocks = 4096;
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t x) { if (e == cudaSuccess) e = x; return e == cudaSuccess; };
    // head: dQ, loss, dH (masked), dW5, db5, db4
    ok(launch_pdl(head_backward_kernel, dim3((b + 7) / 8), dim3(256), 0, s, gp, (const float*)q->t_q, y_dev, w_dev, (const __nv_bfloat16*)q->a4,
                  (const float*)(q->master + var_offset(8)), q->t_dq, q->t_loss, q->t_dh, q->t_dh_bf, td_dev));
    {
        const uint32_t rps = colsum_rows_per_split(b), splits = (b + rps - 1) / rps;
        ok(launch_pdl(head_wgrad_partial_kernel, dim3(16, splits), dim3(32, 8), 0, s, (const __nv_bfloat16*)q->a4, (const float*)q->t_dq, b, rps, q->t_colsum));
        ok(launch_pdl(colsum_final_kernel, dim3(6), dim3(256), 0, s, (const float*)q->t_colsum, splits, 1536u, 1.0f, G(8)));
    }
    ok(launch_colsum(q, q->t_dq, b, 3, 1.0f, G(9), s));
    if (loss_dev) ok(launch_colsum(q, q->t_loss, b, 1, (float)b, loss_dev, s));
    ok(launch_colsum(q, q->t_dh, b, 512, 1.0f, G(7), s));
    // dense 1: dW4 = a3^T dH (K = items), dA3 = dH W4^T, masked by conv3's ReLU
    ok(launch_wgrad<256>(q, ws[0], LoadA3T{q->a3p, 0, 0}, q->t_dh, G(6), s));
    if (e == cudaSuccess) ok(launch_gemm<64>(LoadRowMajorBf16{q->t_dh_bf, 512u}, (const __nv_bfloat16*)q->w4k, EpiF32{q->t_d3, b, 3136u}, b, 512u, 3136u, 1u, q->err, s));
    ok(launch_pdl(mask_conv3_kernel, dim3(ew_blocks), dim3(256), 0, s, q->t_d3, (const __nv_bfloat16*)q->a3p, q->t_d3_bf, b));
    ok(launch_colsum(q, q->t_d3, b * 49u, 64, 1.0f, G(5), s));
    // conv3: dW3, dA2 (full correlation), masked by conv2's ReLU
    ok(launch_wgrad<64>(q, ws[1], LoadIm2colT3{q->a2p, 0, 0}, q->t_d3, G(4), s));
    if (e == cudaSuccess) ok(launch_gemm<64>(LoadDz3Taps{q->t_d3_bf}, (const __nv_bfloat16*)q->w3r, EpiF32{q->t_d2, b * 81u, 64u}, b * 81u, 576u, 64u, 1u, q->err, s));
    ok(launch_pdl(mask_conv2_kernel, dim3(ew_blocks), dim3(256), 0, s, q->t_d2, (const __nv_bfloat16*)q->a2p, q->t_d2_bf, b));
    ok(launch_colsum(q, q->t_d2, b * 81u, 64, 1.0f, G(3), s));
    // conv2: dW2, dA1 (stride-2 transposed convolution), masked by conv1's ReLU
    ok(launch_wgrad<64>(q, ws[2], LoadIm2colT2{q->a1p, 0, 0}, q->t_d2, G(2), s));
    if (e == cudaSuccess) ok(launch_gemm<32>(LoadDz2Taps{q->t_d2_bf}, (const __nv_bfloat16*)q->w2r, EpiF32{q->t_d1, b * 400u, 32u}, b * 400u, 1024u, 32u, 1u, q->err, s));
    ok(launch_pdl(mask_conv1_kernel, dim3(ew_blocks), dim3(256), 0, s, q->t_d1, (const __nv_bfloat16*)q->a1p, b));
    ok(launch_colsum(q, q->t_d1, b * 400u, 32, 1.0f, G(1), s));
    // conv1: dW1 from the u8 ring frames (no data gradient)
    ok(launch_pdl(qnet_locate_kernel, dim3((b + 127) / 128), dim3(128), 0, s, gp, 0u, q->slot_frame));
    ok(launch_wgrad<32>(q, ws[3], LoadIm2colT1{env->frames, q->slot_frame, 0, 0}, q->t_d1, G(0), s));
    if (e != cudaSuccess) return fail(QLC_ERR_CUDA, std::string("qnet backward: ") + cudaGetErrorString(e));
    if (!apply) return QLC_OK;
    // per-variable clipnorm + Adam, then the operand copies of the new weights
    const uint64_t t = ++q->adam_t;
    const qlc_adam_config& c = q->adam;
    const double alpha = (double)c.lr * std::sqrt(1.0 - std::pow((double)c.beta2, (double)t)) / (1.0 - std::pow((double)c.beta1, (double)t));
    ok(launch_pdl(sumsq_partial_kernel, dim3(NVARS, NORM_CHUNKS), dim3(256), 0, s, (const float*)g, q->norm_partial));
    ok(launch_pdl(adam_kernel, dim3((N_PARAMS + 1023) / 1024), dim3(256), 0, s, q->master, q->adam_m, q->adam_v, (const float*)g, (const float*)q->norm_partial,
                  AdamStep{(float)alpha, (float)(1.0 - (double)c.beta1), (float)(1.0 - (double)c.beta2), c.epsilon, c.clipnorm}));
    ok(qnet_prep_weights(q, s));
    if (e != cudaSuccess) return fail(QLC_ERR_CUDA, std::string("qnet update: ") + cudaGetErrorString(e));
    return QLC_OK;
}

extern "C" {

static int32_t check_train_args(qlc_qnet* q, const void* idx, uint32_t batch, uint32_t n_batches, const float* target, qlc_qnet* target_net) {
    if (!q || !idx) return fail(QLC_ERR_INVALID_ARG, "qnet/indices is null");
    if (!q->env) return fail(QLC_ERR_INVALID_ARG, "the environment of this Q-network has been destroyed");
    if (batch == 0) return fail(QLC_ERR_INVALID_ARG, "batch must be > 0");
    if ((uint64_t)batch * n_batches * 400ull >= 0xFFFFFFFFull) return fail(QLC_ERR_INVALID_ARG, "too many items for one call");
    if (!target) {
        if (!target_net) return fail(QLC_ERR_INVALID_ARG, "give either targets or a target network");
        if (!target_net->env) return fail(QLC_ERR_INVALID_ARG, "the environment of the target network has been destroyed");
        if (target_net->env != q->env) return fail(QLC_ERR_INVALID_ARG, "the target network belongs to another environment");
    }
    return QLC_OK;
}

// where the targets of a training call come from: given (y [n]), or from target_net (same env) as the one-step TD target of
// the items' records (n_step = 0) or through the n-step walk (n_step >= 1; nstep.cuh, DESIGN §14), optionally double DQN
struct TargetSource {
    const float* y;
    qlc_qnet* target_net;
    float gamma;
    uint32_t n_step;
    bool double_dqn;
};

// grows the targets of one call to n items: synchronise, free, allocate (a failed allocation leaves y_cap = 0 and no stale pointers)
static int32_t qnet_targets_alloc(qlc_qnet* q, uint32_t n) {
    if (n <= q->y_cap) return QLC_OK;
    CUDA_TRY(cudaDeviceSynchronize());
    qnet_free_targets(q);
    const size_t m = n;
    cudaError_t e = cudaSuccess;
    auto A = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
    A((void**)&q->t_y, m * 4); A((void**)&q->t_maxq, m * 4); A((void**)&q->t_ret, m * 4); A((void**)&q->t_disc, m * 4);
    A((void**)&q->t_boot, m * 4); A((void**)&q->t_tq, m * 12); A((void**)&q->t_act, m);
    if (e != cudaSuccess) { cudaGetLastError(); qnet_free_targets(q); return fail(QLC_ERR_CUDA, std::string("qnet TD targets: ") + cudaGetErrorString(e)); }
    q->y_cap = n;
    return QLC_OK;
}

static cudaError_t launch_nstep(qlc_env* env, const uint32_t* idx_dev, uint32_t n, uint32_t n_step, float gamma, float* ret, float* disc, uint32_t* boot,
                                cudaStream_t s) {
    GatherParams g{}; fill_gather(env, g);
    g.indices = idx_dev; g.n_items = n;
    return launch_pdl(nstep::nstep_kernel, dim3((n + 127) / 128), dim3(128), 0, s, g, n_step, gamma, ret, disc, boot);
}

// the updates of one training call on `s` (arguments checked, n_batches > 0). Computed targets are written to y_out [n] if it
// is given, else to the network's scratch. The target network runs once per call; with double DQN the online network's
// greedy action for minibatch j comes from the weights after updates 0 .. j-1, so n_batches = k is k calls.
static int32_t qnet_train_calls(qlc_qnet* q, const uint32_t* idx_dev, const float* weight_dev, uint32_t batch, uint32_t n_batches, const TargetSource& t,
                                float* loss_dev, float* td_dev, float* y_out, cudaStream_t s) {
    int32_t rc = QLC_OK;
    const uint32_t n = batch * n_batches;
    GatherParams gp{}; fill_gather(q->env, gp);
    // y [m] = target_kernel over gp.indices [m]: G = ret or r of the record, d = disc or gamma, Q_boot = max_q or tq at t_act
    auto target = [&](uint32_t m, const float* ret, const float* disc, const float* max_q, const float* tq, float* y) {
        gp.n_items = m;
        return launch_pdl(qnet::target_kernel, dim3((m + 255) / 256), dim3(256), 0, s, gp, ret, disc, t.gamma, max_q, tq,
                          (const uint8_t*)(tq ? q->t_act : nullptr), y);
    };
    float* y = nullptr;
    if (!t.y) {
        rc = qnet_targets_alloc(q, n); if (rc) return rc;
        y = y_out ? y_out : q->t_y;
        if (t.n_step == 0) {
            rc = qnet_forward(t.target_net, idx_dev, n, 1, nullptr, nullptr, q->t_maxq, false, s); if (rc) return rc;
            gp.indices = idx_dev;
            CUDA_TRY(target(n, nullptr, nullptr, q->t_maxq, nullptr, y));
        } else {
            // G, disc, boot of the whole call; then the target network on the bootstrap states
            CUDA_TRY(launch_nstep(q->env, idx_dev, n, t.n_step, t.gamma, q->t_ret, q->t_disc, q->t_boot, s));
            rc = qnet_forward(t.target_net, q->t_boot, n, 1, t.double_dqn ? q->t_tq : nullptr, nullptr, t.double_dqn ? nullptr : q->t_maxq, false, s);
            if (rc) return rc;
            gp.indices = q->t_boot;
            if (!t.double_dqn) CUDA_TRY(target(n, q->t_ret, q->t_disc, q->t_maxq, nullptr, y));
        }
    }
    const float* const y_in = t.y ? t.y : y;
    for (uint32_t j = 0; j < n_batches; ++j) {
        const size_t o = (size_t)j * batch;
        if (t.double_dqn) {
            rc = qnet_forward(q, q->t_boot + o, batch, 1, nullptr, q->t_act, nullptr, false, s); if (rc) return rc;
            gp.indices = q->t_boot + o;
            CUDA_TRY(target(batch, q->t_ret + o, q->t_disc + o, nullptr, q->t_tq + o * 3, y + o));
        }
        rc = qnet_train_step(q, idx_dev + o, batch, y_in + o, weight_dev ? weight_dev + o : nullptr, loss_dev ? loss_dev + j : nullptr,
                             td_dev ? td_dev + o : nullptr, true, s);
        if (rc) return rc;
    }
    return QLC_OK;
}

int32_t qlc_qnet_train_weighted(qlc_qnet* q, const uint32_t* idx_dev, const float* weight_dev, uint32_t batch, uint32_t n_batches, const float* target_dev,
                                qlc_qnet* target_net, float gamma, float* loss_dev, float* td_dev, void* stream) {
    QLC_RANGE("qlc_qnet_train_weighted");
    int32_t rc = check_train_args(q, idx_dev, batch, n_batches, target_dev, target_net); if (rc) return rc;
    if (n_batches == 0) return QLC_OK;
    return on_caller_stream(q->env, stream, [&] {
        return qnet_train_calls(q, idx_dev, weight_dev, batch, n_batches, TargetSource{target_dev, target_net, gamma, 0, false}, loss_dev, td_dev, nullptr,
                                (cudaStream_t)stream);
    });
}

int32_t qlc_qnet_train(qlc_qnet* q, const uint32_t* idx_dev, uint32_t batch, uint32_t n_batches, const float* target_dev, qlc_qnet* target_net,
                       float gamma, float* loss_dev, void* stream) {
    return qlc_qnet_train_weighted(q, idx_dev, nullptr, batch, n_batches, target_dev, target_net, gamma, loss_dev, nullptr, stream);
}

// stages host indices / targets / loss weights (may be NULL) in the env's device staging buffer, with room for n_loss losses and
// n TD errors; checks the indices against the replay length
static int32_t stage_train_inputs(qlc_qnet* q, const uint32_t* idx_host, uint32_t n, const float* target_host, const float* weight_host, uint32_t n_loss,
                                  uint32_t** idx_dev, float** y_dev, float** w_dev, float** loss_dev, float** td_dev) {
    qlc_env* env = q->env;
    const uint64_t len = replay_len(env);
    for (uint32_t i = 0; i < n; ++i) if (idx_host[i] >= len) return fail(QLC_ERR_INVALID_ARG, "replay index out of range");
    const size_t arr = ((size_t)n * 4 + 255) & ~(size_t)255;
    const size_t o_y = arr, o_w = 2 * arr, o_td = 3 * arr, o_l = 4 * arr, total = o_l + (size_t)n_loss * 4 + 16;
    int32_t rc = ensure_dev_stage(env, total); if (rc) return rc;
    uint8_t* dev = (uint8_t*)env->dev_stage;
    CUDA_TRY(cudaMemcpyAsync(dev, idx_host, (size_t)n * 4, cudaMemcpyHostToDevice, env->own_stream));
    if (target_host) CUDA_TRY(cudaMemcpyAsync(dev + o_y, target_host, (size_t)n * 4, cudaMemcpyHostToDevice, env->own_stream));
    if (weight_host) CUDA_TRY(cudaMemcpyAsync(dev + o_w, weight_host, (size_t)n * 4, cudaMemcpyHostToDevice, env->own_stream));
    *idx_dev = (uint32_t*)dev; *y_dev = target_host ? (float*)(dev + o_y) : nullptr; *w_dev = weight_host ? (float*)(dev + o_w) : nullptr;
    *loss_dev = (float*)(dev + o_l); *td_dev = (float*)(dev + o_td);
    return QLC_OK;
}

int32_t qlc_qnet_train_host(qlc_qnet* q, const uint32_t* idx_host, uint32_t batch, uint32_t n_batches, const float* target_host, qlc_qnet* target_net,
                            float gamma, float* loss_host) {
    QLC_RANGE("qlc_qnet_train_host");
    int32_t rc = check_train_args(q, idx_host, batch, n_batches, target_host, target_net); if (rc) return rc;
    if (n_batches == 0) return QLC_OK;
    rc = set_device(q->env); if (rc) return rc;
    rc = after_caller_stream(q->env); if (rc) return rc;
    uint32_t* idx_dev; float *y_dev, *w_dev, *loss_dev, *td_dev;
    rc = stage_train_inputs(q, idx_host, batch * n_batches, target_host, nullptr, n_batches, &idx_dev, &y_dev, &w_dev, &loss_dev, &td_dev); if (rc) return rc;
    cudaStream_t s = q->env->own_stream;
    rc = qnet_train_calls(q, idx_dev, nullptr, batch, n_batches, TargetSource{y_dev, target_net, gamma, 0, false}, loss_host ? loss_dev : nullptr, nullptr,
                          nullptr, s);
    if (rc) return rc;
    if (loss_host) CUDA_TRY(cudaMemcpyAsync(loss_host, loss_dev, (size_t)n_batches * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    uint32_t herr = 0;
    rc = qlc_qnet_error(q, &herr); if (rc) return rc;
    if (herr) return fail(QLC_ERR_CUDA, "qnet: an MMA completion barrier timed out");
    return QLC_OK;
}

int32_t qlc_qnet_debug_grads_weighted(qlc_qnet* q, const uint32_t* idx_host, uint32_t n, const float* target_host, const float* weight_host,
                                      const qlc_qnet_weights* grads_out, float* td_out_host) {
    int32_t rc = check_train_args(q, idx_host, n, 1, target_host, nullptr); if (rc) return rc;
    if (!grads_out) return fail(QLC_ERR_INVALID_ARG, "grads_out is null");
    const float* dst[qnet::NVARS];
    weight_ptrs(grads_out, dst);
    for (int i = 0; i < qnet::NVARS; ++i) if (!dst[i]) return fail(QLC_ERR_INVALID_ARG, "a gradient pointer is null");
    rc = set_device(q->env); if (rc) return rc;
    rc = after_caller_stream(q->env); if (rc) return rc;
    uint32_t* idx_dev; float *y_dev, *w_dev, *loss_dev, *td_dev;
    rc = stage_train_inputs(q, idx_host, n, target_host, weight_host, 1, &idx_dev, &y_dev, &w_dev, &loss_dev, &td_dev); if (rc) return rc;
    cudaStream_t s = q->env->own_stream;
    rc = qnet_train_step(q, idx_dev, n, y_dev, w_dev, nullptr, td_out_host ? td_dev : nullptr, false, s); if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(s));
    uint32_t herr = 0;
    rc = qlc_qnet_error(q, &herr); if (rc) return rc;
    if (herr) return fail(QLC_ERR_CUDA, "qnet: an MMA completion barrier timed out");
    for (int v = 0; v < qnet::NVARS; ++v) CUDA_TRY(cudaMemcpy(const_cast<float*>(dst[v]), q->grad + qnet::var_offset(v), (size_t)qnet::var_size(v) * 4, cudaMemcpyDeviceToHost));
    if (td_out_host) CUDA_TRY(cudaMemcpy(td_out_host, td_dev, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return QLC_OK;
}

int32_t qlc_qnet_debug_grads(qlc_qnet* q, const uint32_t* idx_host, uint32_t n, const float* target_host, const qlc_qnet_weights* grads_out) {
    return qlc_qnet_debug_grads_weighted(q, idx_host, n, target_host, nullptr, grads_out, nullptr);
}

// ---------------- n-step returns and double-DQN targets (nstep.cuh, DESIGN §14) ----------------
static int32_t check_nstep_args(uint32_t n_step, float gamma) {
    if (n_step < 1 || n_step > QLC_NSTEP_MAX) return fail(QLC_ERR_INVALID_ARG, "n_step must be in [1, QLC_NSTEP_MAX]");
    if (!(gamma >= 0.0f && gamma <= 1.0f)) return fail(QLC_ERR_INVALID_ARG, "gamma must be finite and in [0, 1]");
    return QLC_OK;
}
// before anything reads a handle's env: a call that passes validation on a machine without a device fails here
static int32_t check_device_present() {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(QLC_ERR_NO_DEVICE, "no CUDA device: ql_cuda has no CPU fallback");
    return QLC_OK;
}

int32_t qlc_replay_nstep(qlc_env* env, const uint32_t* idx_dev, uint32_t n, uint32_t n_step, float gamma, float* return_dev, float* discount_dev,
                         uint32_t* boot_idx_dev, void* stream) {
    QLC_RANGE("qlc_replay_nstep");
    int32_t rc = check_nstep_args(n_step, gamma); if (rc) return rc;
    if (!env || !idx_dev) return fail(QLC_ERR_INVALID_ARG, "env/idx is null");
    rc = check_device_present(); if (rc) return rc;
    if (n == 0) return QLC_OK;
    return on_caller_stream(env, stream, [&] {
        CUDA_TRY(launch_nstep(env, idx_dev, n, n_step, gamma, return_dev, discount_dev, boot_idx_dev, (cudaStream_t)stream));
        return QLC_OK;
    });
}

int32_t qlc_qnet_train_nstep(qlc_qnet* q, const uint32_t* idx_dev, const float* weight_dev, uint32_t batch, uint32_t n_batches, qlc_qnet* target_net,
                             float gamma, uint32_t n_step, int32_t double_dqn, float* loss_dev, float* td_dev, float* y_dev, void* stream) {
    QLC_RANGE("qlc_qnet_train_nstep");
    int32_t rc = check_nstep_args(n_step, gamma); if (rc) return rc;
    if (double_dqn != 0 && double_dqn != 1) return fail(QLC_ERR_INVALID_ARG, "double_dqn must be 0 or 1");
    if (!target_net) return fail(QLC_ERR_INVALID_ARG, "target_net is null");
    rc = check_train_args(q, idx_dev, batch, n_batches, nullptr, target_net); if (rc) return rc;
    rc = check_device_present(); if (rc) return rc;
    if (n_batches == 0) return QLC_OK;
    return on_caller_stream(q->env, stream, [&] {
        return qnet_train_calls(q, idx_dev, weight_dev, batch, n_batches, TargetSource{nullptr, target_net, gamma, n_step, double_dqn != 0}, loss_dev, td_dev,
                                y_dev, (cudaStream_t)stream);
    });
}

// test hook: out[M][N] = act(bf16(a)[M][K] * bf16(w)[N][K]^T + bias) through the tcgen05 GEMM kernel (host f32 in / out)

int32_t qlc_debug_gemm_bf16(const float* a_host, const float* w_host, const float* bias_host, int32_t relu, float* out_host, uint32_t m, uint32_t n, uint32_t k) {
    if (!a_host || !w_host || !bias_host || !out_host) return fail(QLC_ERR_INVALID_ARG, "null pointer");
    if (k % qnet::KC != 0 || !(n == 32 || n == 64 || n == 128 || n == 256 || n == 512) || m == 0) return fail(QLC_ERR_INVALID_ARG, "need K % 64 == 0 and N in {32, 64, 128, 256, 512}");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(QLC_ERR_NO_DEVICE, "no CUDA device: ql_cuda has no CPU fallback");
    float *da = nullptr, *dw = nullptr, *db = nullptr, *dof = nullptr; __nv_bfloat16 *ba = nullptr, *bw = nullptr, *bo = nullptr; unsigned int* derr = nullptr;
    cudaError_t e = cudaSuccess;
    auto A = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
    A((void**)&da, (size_t)m * k * 4); A((void**)&dw, (size_t)n * k * 4); A((void**)&db, (size_t)n * 4); A((void**)&dof, (size_t)m * n * 4);
    A((void**)&ba, (size_t)m * k * 2); A((void**)&bw, (size_t)n * k * 2); A((void**)&bo, (size_t)m * n * 2); A((void**)&derr, 4);
    if (e == cudaSuccess) e = cudaMemset(derr, 0, 4);
    if (e == cudaSuccess) e = cudaMemcpy(da, a_host, (size_t)m * k * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dw, w_host, (size_t)n * k * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, bias_host, (size_t)n * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        qnet::f32_to_bf16_kernel<<<256, 256>>>(da, ba, (size_t)m * k);
        qnet::f32_to_bf16_kernel<<<256, 256>>>(dw, bw, (size_t)n * k);
        const qnet::LoadRowMajorBf16 ld{ba, k};
        const qnet::EpiBiasAct epi{db, bo, n, relu};
        switch (n) {
            case 32: e = launch_gemm<32>(ld, bw, epi, m, k, n, 1u, derr, nullptr); break;
            case 64: e = launch_gemm<64>(ld, bw, epi, m, k, n, 1u, derr, nullptr); break;
            case 128: e = launch_gemm<128>(ld, bw, epi, m, k, n, 1u, derr, nullptr); break;
            case 256: e = launch_gemm<256>(ld, bw, epi, m, k, n, 1u, derr, nullptr); break;
            default: e = launch_gemm<128>(ld, bw, epi, m, k, n, 1u, derr, nullptr); break;      // 512 = 4 N tiles of 128
        }
    }
    unsigned int herr = 0;
    if (e == cudaSuccess) { qnet::bf16_to_f32_kernel<<<256, 256>>>(bo, dof, (size_t)m * n); e = cudaMemcpy(out_host, dof, (size_t)m * n * 4, cudaMemcpyDeviceToHost); }
    if (e == cudaSuccess) e = cudaMemcpy(&herr, derr, 4, cudaMemcpyDeviceToHost);
    cudaFree(da); cudaFree(dw); cudaFree(db); cudaFree(dof); cudaFree(ba); cudaFree(bw); cudaFree(bo); cudaFree(derr);
    if (e != cudaSuccess) return fail(QLC_ERR_CUDA, std::string("tensor-core GEMM: ") + cudaGetErrorString(e));
    if (herr) return fail(QLC_ERR_CUDA, "tensor-core GEMM: the MMA completion barrier timed out");
    return QLC_OK;
}

int32_t qlc_debug_collision_wall(int32_t which, float cx, float cy, float radius, float mvx, float mvy, int32_t* some, float* way,
                                 float* approximation, float* nx, float* ny, uint32_t* err) {
    if (which < 0 || which > 2) return fail(QLC_ERR_INVALID_ARG, "which must be 0..2");
    return run_debug(which, cx, cy, radius, mvx, mvy, 0, 0, 0, 0, some, way, approximation, nx, ny, err);
}
int32_t qlc_debug_collision_rect(float cx, float cy, float radius, float mvx, float mvy, float min_x, float min_y, float max_x, float max_y,
                                 int32_t* some, float* way, float* approximation, float* nx, float* ny, uint32_t* err) {
    return run_debug(3, cx, cy, radius, mvx, mvy, min_x, min_y, max_x, max_y, some, way, approximation, nx, ny, err);
}

}  // extern "C"

// ---------------- prioritized replay: a sum tree over the replay ring (per.cuh, DESIGN.md §13) ----------------
struct qlc_per {
    qlc_env* env = nullptr;                    // NULL once the env has been destroyed: every call but destroy fails
    int device = 0;
    float alpha = 0.6f, epsilon = 1e-6f;
    per::Tree tree{};
    void* block = nullptr;                     // one allocation: leaves, node levels, running max
    bool synced = false;                       // the leaves describe the ring at (synced_t, synced_gen)
    uint64_t synced_t = 0, synced_gen = 0;
};

static void per_release_device(qlc_per* p) {
    if (!p->env) return;
    cudaSetDevice(p->device);
    cudaDeviceSynchronize();
    cudaFree(p->block);
    p->block = nullptr; p->tree = per::Tree{}; p->env = nullptr;
}

static uint32_t per_grid(const qlc_env* env, uint64_t items, uint32_t threads) {
    const uint64_t want = (items + threads - 1) / threads, most = (uint64_t)env->sm_count * 8u;
    return (uint32_t)(want < 1 ? 1 : (want > most ? most : want));
}

// Brings the leaves up to the env's time: rows whose time entered the replay get the running max, rows whose time left it 0;
// then their ancestors are re-summed. A load (new generation) or a jump of time_slots steps or more rewrites every row.
static int32_t per_sync(qlc_per* p, cudaStream_t s) {
    qlc_env* env = p->env;
    const uint64_t t = env->t, oldest = t > env->t_cap ? t - env->t_cap : 0;
    if (p->synced && p->synced_gen == env->generation && p->synced_t == t) return QLC_OK;
    const uint32_t ts = env->time_slots, n_envs = env->cfg.n_envs;
    per::Intervals slots{};
    auto add_times = [&](uint64_t a, uint64_t b) {       // times [a, b), b - a < time_slots, as ring-slot intervals
        if (b <= a) return;
        const uint64_t s0 = a % ts, n = b - a;
        if (s0 + n <= ts) { slots.lo[slots.n] = s0; slots.hi[slots.n++] = s0 + n; }
        else { slots.lo[slots.n] = s0; slots.hi[slots.n++] = ts; slots.lo[slots.n] = 0; slots.hi[slots.n++] = s0 + n - ts; }
    };
    if (!p->synced || p->synced_gen != env->generation || t < p->synced_t || t - p->synced_t >= ts) {
        slots.n = 1; slots.lo[0] = 0; slots.hi[0] = ts;
    } else {
        const uint64_t t0 = p->synced_t, oldest0 = t0 > env->t_cap ? t0 - env->t_cap : 0;
        add_times(oldest0, oldest);                        // left the replay
        add_times(t0, t);                                  // written since the last sync
    }
    per::Intervals iv = slots;
    uint64_t total = 0;
    for (uint32_t k = 0; k < iv.n; ++k) { iv.lo[k] *= n_envs; iv.hi[k] *= n_envs; total += iv.hi[k] - iv.lo[k]; }
    CUDA_TRY(launch_pdl(per::per_sync_leaves_kernel, dim3(per_grid(env, total, 256)), dim3(256), 0, s, p->tree, iv, total, t, oldest));
    for (uint32_t level = 1; level <= p->tree.depth; ++level) {
        per::Intervals nv = iv;
        total = 0;
        for (uint32_t k = 0; k < nv.n; ++k) {
            nv.lo[k] = iv.lo[k] >> (per::LOG_FAN * level); nv.hi[k] = ((iv.hi[k] - 1) >> (per::LOG_FAN * level)) + 1;
            total += nv.hi[k] - nv.lo[k];
        }
        CUDA_TRY(launch_pdl(per::per_resum_intervals_kernel, dim3(per_grid(env, total, 256)), dim3(256), 0, s, p->tree, level, nv, total));
    }
    p->synced = true; p->synced_t = t; p->synced_gen = env->generation;
    return QLC_OK;
}

extern "C" {

int32_t qlc_per_create(qlc_env* env, float alpha, float epsilon, qlc_per** out) {
    if (!(alpha >= 0.0f && alpha <= 1.0f)) return fail(QLC_ERR_INVALID_ARG, "alpha must be in [0, 1]");
    if (!(epsilon > 0.0f) || !std::isfinite(epsilon)) return fail(QLC_ERR_INVALID_ARG, "epsilon must be finite and > 0");
    if (!env || !out) return fail(QLC_ERR_INVALID_ARG, "env/out is null");
    *out = nullptr;
    int ndev = 0;                                      // before anything reads the env

    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(QLC_ERR_NO_DEVICE, "no CUDA device: ql_cuda has no CPU fallback");
    if (env->cfg.replay_capacity == 0) return fail(QLC_ERR_INVALID_ARG, "the env keeps no replay (replay_capacity == 0)");
    int32_t rc = set_device(env); if (rc) return rc;
    qlc_per* p = new qlc_per();
    p->device = env->cfg.device; p->alpha = alpha; p->epsilon = epsilon;
    per::Tree& t = p->tree;
    t.n_envs = env->cfg.n_envs; t.time_slots = env->time_slots;
    uint64_t cnt = (uint64_t)env->time_slots * env->cfg.n_envs;
    t.count[0] = cnt;
    while (cnt > 1 || t.depth == 0) { cnt = (cnt + per::FAN - 1) / per::FAN; t.count[++t.depth] = cnt; }
    auto padded = [](uint64_t n, size_t elem) { return ((((n + per::FAN - 1) / per::FAN) * per::FAN * elem) + 255) & ~(size_t)255; };
    size_t bytes = padded(t.count[0], 4);
    for (uint32_t k = 1; k <= t.depth; ++k) bytes += padded(t.count[k], 8);
    bytes += 256;
    cudaError_t e = cudaMalloc(&p->block, bytes);
    if (e == cudaSuccess) e = cudaMemset(p->block, 0, bytes);
    if (e == cudaSuccess) {
        uint8_t* b = (uint8_t*)p->block;
        t.leaves = (float*)b; b += padded(t.count[0], 4);
        for (uint32_t k = 1; k <= t.depth; ++k) { t.node[k] = (double*)b; b += padded(t.count[k], 8); }
        t.max_bits = (unsigned int*)b;
        const float one = 1.0f;
        e = cudaMemcpy(t.max_bits, &one, 4, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();   // legacy-stream init: done before a sync or sample on a non-blocking stream
    if (e != cudaSuccess) { cudaGetLastError(); cudaFree(p->block); delete p; return fail(QLC_ERR_CUDA, std::string("prioritized replay alloc: ") + cudaGetErrorString(e)); }
    p->env = env;
    env->pers.push_back(p);
    *out = p;
    return QLC_OK;
}

int32_t qlc_per_destroy(qlc_per* p) {
    if (!p) return QLC_OK;
    if (qlc_env* env = p->env) {
        for (size_t i = 0; i < env->pers.size(); ++i)
            if (env->pers[i] == p) { env->pers.erase(env->pers.begin() + i); break; }
        per_release_device(p);
    }
    delete p;
    return QLC_OK;
}

static int32_t check_per(qlc_per* p) {
    if (!p) return fail(QLC_ERR_INVALID_ARG, "per is null");
    if (!p->env) return fail(QLC_ERR_INVALID_ARG, "the environment of this prioritized replay has been destroyed");
    return QLC_OK;
}

int32_t qlc_per_sample(qlc_per* p, uint32_t batch, uint32_t n_batches, uint64_t call_index, float beta, uint32_t* idx_dev, float* weight_dev, void* stream) {
    QLC_RANGE("qlc_per_sample");
    if (batch == 0) return fail(QLC_ERR_INVALID_ARG, "batch must be > 0");
    if (!(beta >= 0.0f && beta <= 1.0f)) return fail(QLC_ERR_INVALID_ARG, "beta must be in [0, 1]");
    if ((uint64_t)batch * n_batches > 0x3FFFFFFFull) return fail(QLC_ERR_INVALID_ARG, "too many items for one call");
    int32_t rc = check_per(p); if (rc) return rc;
    if (!idx_dev) return fail(QLC_ERR_INVALID_ARG, "idx is null");
    qlc_env* env = p->env;
    const uint64_t len = replay_len(env);
    if (len == 0) return fail(QLC_ERR_NOT_ENOUGH, "the replay is empty");
    if (len >= 0xFFFFFFFFull) return fail(QLC_ERR_INVALID_ARG, "replay longer than 2^32-2 transitions");
    if (n_batches == 0) return QLC_OK;
    return on_caller_stream(env, stream, [&] {
        cudaStream_t s = (cudaStream_t)stream;
        int32_t rc = per_sync(p, s); if (rc) return rc;
        const uint32_t n = batch * n_batches;
        const uint64_t oldest = env->t > env->t_cap ? env->t - env->t_cap : 0;
        CUDA_TRY(launch_pdl(per::per_sample_kernel, dim3((n + 127) / 128), dim3(128), 0, s, p->tree, batch, n, call_index, env->cfg.seed, env->t, oldest,
                            idx_dev, weight_dev));
        if (weight_dev) CUDA_TRY(launch_pdl(per::per_weight_kernel, dim3(n_batches), dim3(256), 0, s, weight_dev, batch, beta));
        return QLC_OK;
    });
}

int32_t qlc_per_update(qlc_per* p, const uint32_t* idx_dev, const float* td_dev, uint32_t n, void* stream) {
    QLC_RANGE("qlc_per_update");
    int32_t rc = check_per(p); if (rc) return rc;
    if (!idx_dev || !td_dev) return fail(QLC_ERR_INVALID_ARG, "idx/td is null");
    qlc_env* env = p->env;
    const uint64_t len = replay_len(env);
    if (len >= 0xFFFFFFFFull) return fail(QLC_ERR_INVALID_ARG, "replay longer than 2^32-2 transitions");
    return on_caller_stream(env, stream, [&] {
        cudaStream_t s = (cudaStream_t)stream;
        int32_t rc = per_sync(p, s); if (rc) return rc;
        if (n == 0) return QLC_OK;
        const uint64_t oldest = env->t > env->t_cap ? env->t - env->t_cap : 0;
        const dim3 grid((n + 255) / 256);
        CUDA_TRY(launch_pdl(per::per_update_clear_kernel, grid, dim3(256), 0, s, p->tree, idx_dev, td_dev, n, (uint32_t)len, oldest, p->alpha, p->epsilon));
        CUDA_TRY(launch_pdl(per::per_update_set_kernel, grid, dim3(256), 0, s, p->tree, idx_dev, td_dev, n, (uint32_t)len, oldest, p->alpha, p->epsilon));
        for (uint32_t level = 1; level <= p->tree.depth; ++level)
            CUDA_TRY(launch_pdl(per::per_resum_items_kernel, grid, dim3(256), 0, s, p->tree, level, idx_dev, n, (uint32_t)len, oldest));
        return QLC_OK;
    });
}

int32_t qlc_per_read_host(qlc_per* p, float* leaves_host, double* total_host, float* max_priority_host) {
    int32_t rc = check_per(p); if (rc) return rc;
    qlc_env* env = p->env;
    rc = set_device(env); if (rc) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    rc = per_sync(p, env->own_stream); if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(env->own_stream));
    if (leaves_host) {
        // logical order = rows of times t_oldest .. t - 1, contiguous in the ring up to one wrap
        const uint64_t n_envs = env->cfg.n_envs, rows = replay_len(env) / n_envs, ts = env->time_slots;
        const uint64_t s0 = (env->t > env->t_cap ? env->t - env->t_cap : 0) % ts, first = std::min(rows, ts - s0);
        CUDA_TRY(cudaMemcpy(leaves_host, p->tree.leaves + s0 * n_envs, first * n_envs * 4, cudaMemcpyDeviceToHost));
        if (rows > first) CUDA_TRY(cudaMemcpy(leaves_host + first * n_envs, p->tree.leaves, (rows - first) * n_envs * 4, cudaMemcpyDeviceToHost));
    }
    if (total_host) CUDA_TRY(cudaMemcpy(total_host, p->tree.node[p->tree.depth], 8, cudaMemcpyDeviceToHost));
    if (max_priority_host) CUDA_TRY(cudaMemcpy(max_priority_host, p->tree.max_bits, 4, cudaMemcpyDeviceToHost));
    return QLC_OK;
}

}  // extern "C"
