/* ql_cuda.h — C ABI of the B200-native Breakout env + DQN replay hot path.
 *
 * This is the drop-in boundary: exactly what a Rust `ql-cuda` crate (or any FFI host) binds to stand in for
 * the reference's CPU implementation of the path. Plain C types only; the library owns all device memory;
 * every call returns an int32 status (QLC_OK = 0), the text of the last failure is qlc_last_error_string().
 * A handle is NOT thread-safe: one host thread and one CUDA stream per handle / per GPU
 * (the reference learner is single-threaded behind Arc<RwLock<E>>: self_driving_tf_q_learner.rs:74,171).
 * Stream order: every call is ordered after all work that earlier calls on the same handle (or on its env, for Q-network and
 * prioritized-replay handles) queued, whether on the caller's stream or on the library's own stream (the *_host calls, submitted
 * host steps). So a host-buffer call after qlc_env_step on the caller's stream sees the step, and a device-pointer call after
 * qlc_env_step_host_submit sees the submitted steps. This holds for one caller stream per handle: work on a second caller
 * stream is not ordered by the library.
 *
 * Reference interfaces replaced (paths relative to /root/reference/src):
 *   Environment trait ................. ql/src/prelude.rs:21-63
 *   Action trait (BreakoutAction) ..... ql/src/prelude.rs:12-18, _breakout-ml/src/breakout_environment.rs:94-120
 *   BreakoutEnvironment ............... _breakout-ml/src/breakout_environment.rs:131-207
 *   BreakoutMechanics::time_step ...... breakout-game/src/mechanics.rs:119-129
 *   FrameRingBuffer ................... _breakout-ml/src/util/frame_ring_buffer.rs:17-63
 *   ToMultiDimArray ................... ql-with-tensorflow/src/ml_model/model.rs:12-26,
 *                                       _breakout-ml/src/breakout_environment.rs:39-78
 *   ReplayBuffer ...................... ql-with-tensorflow/src/learn/replay_buffer.rs:53-146
 *   generate_distinct_random_ids ...... ql-with-tensorflow/src/learn/self_driving_tf_q_learner.rs:276-296
 * The reference-side binding a maintainer would add is shown in INTEGRATION.md.
 */
#ifndef QL_CUDA_H
#define QL_CUDA_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QLC_VERSION 200

/* status codes */
#define QLC_OK                0
#define QLC_ERR_INVALID_ARG   1   /* null pointer, zero size, unsupported frame size ... */
#define QLC_ERR_CUDA          2   /* a CUDA runtime call failed; see qlc_last_error_string() */
#define QLC_ERR_OUT_OF_RANGE  3   /* QlError("value out of range"): action >= 3, index >= len (breakout_environment.rs:112-119) */
#define QLC_ERR_NO_DEVICE     4   /* no CUDA device / not an sm_100 part: there is NO CPU fallback */
#define QLC_ERR_NOT_ENOUGH    5   /* replay shorter than the batch (assert at self_driving_tf_q_learner.rs:282) */
#define QLC_ERR_COMM          6   /* NCCL could not be loaded (dlopen) or an NCCL call failed */

/* BreakoutAction::numeric (breakout_environment.rs:104-110) */
#define QLC_ACTION_NONE  0
#define QLC_ACTION_LEFT  1
#define QLC_ACTION_RIGHT 2
#define QLC_ACTION_SPACE 3

#define QLC_FRAME_W 84
#define QLC_FRAME_H 84
#define QLC_FRAME_BYTES (QLC_FRAME_W * QLC_FRAME_H)
#define QLC_NUM_FRAMES 4             /* WORLD_STATE_NUM_FRAMES, breakout_environment.rs:15 */

/* per-env sticky error flags (the reference panics on these; mechanics.rs:145,265,284,303,511) */
#define QLC_ENVERR_WALL_DISTANCE 1u
#define QLC_ENVERR_APPROX_RANGE  2u
#define QLC_ENVERR_RECURSION     4u
#define QLC_ENVERR_BISECTION     8u
#define QLC_ENVERR_DEGENERATE   16u  /* informational: parry2d degenerate-contact branch taken */
#define QLC_ENVERR_ACTION       32u  /* action byte >= 3 seen on the device path (treated as None) */
#define QLC_ENVERR_HANDOVER     64u  /* (shard-wide) a time-chunk hand-over between CTAs timed out inside the step kernel */

/* output layouts of the state gather (ToMultiDimArray) */
#define QLC_LAYOUT_U8_BHYX   0  /* [b][slot h][y][x] u8  — fast path, frame-major                     */
#define QLC_LAYOUT_F32_BXYH  1  /* [b][x][y][slot h] f32 — BreakoutState::batch_to_multi_dim_array, value = u8 as f32 */
#define QLC_LAYOUT_U8_BXYH   2  /* [b][x][y][slot h] u8  — the same element order at 1/4 of the bytes (the *_host calls move
                                   this over PCIe and widen to f32 on the host; a GPU consumer can widen it itself) */

typedef struct qlc_env qlc_env;      /* opaque: N envs + their frame ring + replay shard on one GPU */

/* A state handle: what `Clone` of a BreakoutState is on the host (state_as_rc / step_as_rc, prelude.rs:36,52-58) - two
 * integers naming frames in the HBM frame ring instead of 4 x 7,056 copied pixels. It names the observation of env `env`
 * after `time` env-steps, `k` of them in the current episode (k = 0 right after reset: an all-zero stack,
 * breakout_environment.rs:177-180): frames F_{time-d}, d = 1..min(k,4), in ring slot (k-d) mod 4 (frame_ring_buffer.rs:53-63).
 * A handle stays usable while those frames are in the ring, i.e. for replay_capacity / n_envs further steps - exactly as
 * long as the reference's ReplayBuffer keeps the Rc it wraps when step_buffer_len <= replay_capacity. */
typedef struct qlc_obs_handle {
    uint64_t time;
    uint32_t k;
    uint32_t env;
} qlc_obs_handle;

typedef struct qlc_config {
    uint32_t struct_size;            /* = sizeof(qlc_config) */
    int32_t  device;                 /* CUDA device ordinal */
    uint32_t n_envs;                 /* independent Breakout instances on this GPU */
    uint32_t env_id_base;            /* global id of local env 0 (sharding: ids seed the per-env random streams) */
    uint32_t frame_w, frame_h;       /* BreakoutEnvironment::new(frame_size_x, frame_size_y); only 84 x 84 */
    uint64_t seed;                   /* Philox key for reset directions and index sampling */
    uint64_t replay_capacity;        /* ReplayBuffer::new(step_buffer_len, ..): transitions, rounded down to a
                                        multiple of n_envs (>= n_envs); 0 = keep only the current observation */
    uint32_t max_episode_steps;      /* Parameter::max_steps_per_episode; 0 = unlimited */
    uint32_t episode_window;         /* Parameter::episode_reward_history_buffer_len (default 100) */
    uint32_t auto_reset;             /* 1: finished/truncated envs restart on device inside the step kernel;
                                        0: reference behaviour, the caller resets (learn_episode :142) */
    uint32_t reserved;
} qlc_config;

/* device pointers to the structure-of-arrays env state (valid until qlc_env_destroy) */
typedef struct qlc_state_view {
    const float* ball_cx; const float* ball_cy; const float* ball_dx; const float* ball_dy;
    const float* pad_min_x; const float* pad_max_x; const float* pad_speed;
    const uint64_t* bricks;          /* bit 20*row + k = brick alive (mechanics.rs:67-95 order) */
    const uint32_t* score;
    const uint32_t* episode_step;    /* frames written in the current episode */
    const uint32_t* episode;         /* episode index (selects the reset direction draw) */
    const uint32_t* err;             /* QLC_ENVERR_* */
    const uint8_t*  finished;
    const uint8_t*  frames;          /* frame ring [time_slots][n_envs][84*84] u8 */
    const uint32_t* records;         /* transition records [time_slots][n_envs] (packing: DESIGN.md) */
    uint32_t n_envs; uint32_t time_slots; uint64_t time;
} qlc_state_view;

/* host-side copy of the SoA state (all pointers caller-allocated, n_envs elements each, any may be NULL) */
typedef struct qlc_state_host {
    float* ball_cx; float* ball_cy; float* ball_dx; float* ball_dy;
    float* pad_min_x; float* pad_max_x; float* pad_speed;
    uint64_t* bricks; uint32_t* score; uint32_t* episode_step; uint32_t* episode; uint32_t* err; uint8_t* finished;
} qlc_state_host;

/* shard episode statistics (order-independent accumulators; reduced across GPUs by the caller with NCCL) */
typedef struct qlc_episode_stats {
    uint64_t sum_return;             /* sum of finished episodes' returns (returns are integral: 1 per brick) */
    uint64_t episodes;
    uint64_t steps;                  /* env-steps executed */
    uint32_t min_return, max_return; /* min = UINT32_MAX, max = 0 while episodes == 0 */
} qlc_episode_stats;

/* ---- lifecycle ---- */
int32_t qlc_version(void);
/* "src_hash=<sha256 of the sources the library was built from>;profiling=<0|1>;" - profiling=1 marks an ablation build
 * (-DQLC_PROFILING) in which QLC_DEBUG_SKIP can remove work from the step kernel; release builds ignore that variable. */
const char* qlc_build_info(void);
const char* qlc_last_error_string(void);
int32_t qlc_device_count(int32_t* count);
int32_t qlc_env_create(const qlc_config* cfg, qlc_env** out);         /* BreakoutEnvironment::new + ReplayBuffer::new */
int32_t qlc_env_destroy(qlc_env* env);
int32_t qlc_sync(qlc_env* env, void* stream);
/* page-locked host memory for the *_host entry points: buffers from here (or cudaHostRegister'ed ones) are copied
 * to / from the device in place, without the library's internal staging copy. */
int32_t qlc_host_alloc(size_t bytes, void** out);
int32_t qlc_host_free(void* p);

/* ---- Environment (prelude.rs:21-63) ---- */
/* reset(): mask_host NULL = all envs, else n_envs bytes (non-zero = reset). dir_x_host NULL = draw the initial
 * ball direction from the env's Philox stream (mechanics.rs:103), else n_envs explicit values. Synchronous. */
int32_t qlc_env_reset(qlc_env* env, const uint8_t* mask_host, const float* dir_x_host);
/* step() x n_steps for all envs in ONE launch (launches of more steps than the frame ring has time slots,
 * replay_capacity / n_envs + 4, are split at that length). actions_dev [n_steps][n_envs] u8 (device);
 * reward_dev [n_steps][n_envs] f32 and done_dev [n_steps][n_envs] u8 (device, either may be NULL).
 * Each step also renders the 84x84 u8 frame into the frame ring and writes the replay transition record
 * (ReplayBuffer::add). Asynchronous on `stream` (a cudaStream_t, NULL = default stream). */
int32_t qlc_env_step(qlc_env* env, const uint8_t* actions_dev, uint32_t n_steps, float* reward_dev, uint8_t* done_dev, void* stream);
/* The learner's pure-random phase (self_driving_tf_q_learner.rs:153-157: rng.gen_range(0..ACTION_SPACE) while step_count <
 * epsilon_pure_random_steps) without an action buffer: the step kernel draws the uniform action of env e at time t itself
 * (word 0 of philox({env_id_base + e, t, 0, 'ACTI'}, seed) * 3 >> 32) and writes it to actions_out_dev [n_steps][n_envs] if
 * that is not NULL (the replay record keeps it either way). */
int32_t qlc_env_step_random(qlc_env* env, uint32_t n_steps, uint8_t* actions_out_dev, float* reward_dev, uint8_t* done_dev, void* stream);
/* same with HOST buffers: validates actions (QLC_ERR_OUT_OF_RANGE), H2D, step, D2H, synchronises. */
int32_t qlc_env_step_host(qlc_env* env, const uint8_t* actions_host, uint32_t n_steps, float* reward_host, uint8_t* done_host);
/* Pipelined form for action streams that do not depend on the previous result (the learner's random-policy phase
 * self_driving_tf_q_learner.rs:153-160, replayed traces): submit validates, queues the copies and the launch and returns
 * (it blocks only while 8 steps are already in flight); qlc_env_step_host_wait blocks until at most `max_pending` (0..7) of the
 * submitted steps are still running - the reward / done of all earlier ones are then in the caller's buffers. All three
 * buffers must be page-locked (qlc_host_alloc, else QLC_ERR_INVALID_ARG) and stay untouched until their step has been waited
 * for; steps execute in submission order. */
int32_t qlc_env_step_host_submit(qlc_env* env, const uint8_t* actions_host, uint32_t n_steps, float* reward_host, uint8_t* done_host);
int32_t qlc_env_step_host_wait(qlc_env* env, uint32_t max_pending);
/* state(): current observation stacks of all envs, [n_envs] x layout, into a device / host buffer */
int32_t qlc_env_obs(qlc_env* env, int32_t layout, void* out_dev, void* stream);
int32_t qlc_env_obs_host(qlc_env* env, int32_t layout, void* out_host);
int32_t qlc_env_state_view(qlc_env* env, qlc_state_view* out);
int32_t qlc_env_read_state(qlc_env* env, const qlc_state_host* out);
float   qlc_env_goal_mean(void);                                      /* episode_reward_goal_mean() = 59 */
int32_t qlc_env_time(qlc_env* env, uint64_t* steps_taken);
/* lives[n_envs]: the reference game has no lives counter - the episode ends the first time the ball passes the paddle
 * (mechanics.rs:131-135) - so this is 1 while an env is not finished and 0 once it is. Synchronous. */
int32_t qlc_env_lives_host(qlc_env* env, uint8_t* lives_host);
/* batch_to_multi_dim_array for state handles (breakout_environment.rs:56-77): the stacks of n handles, [n] x layout, into a
 * device / host buffer. The host form checks every handle (QLC_ERR_OUT_OF_RANGE: "stale state handle"); on the device path
 * a dead handle gives an all-zero stack. */
int32_t qlc_obs_gather(qlc_env* env, const qlc_obs_handle* handles_dev, uint32_t n, int32_t layout, void* out_dev, void* stream);
int32_t qlc_obs_gather_host(qlc_env* env, const qlc_obs_handle* handles_host, uint32_t n, int32_t layout, void* out_host);
int32_t qlc_env_error_flags(qlc_env* env, uint32_t* or_of_all);

/* ---- ReplayBuffer (replay_buffer.rs:53-146) ---- */
int32_t qlc_replay_len(qlc_env* env, uint64_t* len);                  /* ReplayBuffer::len */
int32_t qlc_replay_capacity(qlc_env* env, uint64_t* capacity);
/* generate_distinct_random_ids: n_batches x batch DISTINCT (per batch) uniform indices in [0, len) into
 * idx_dev [n_batches][batch] u32; minibatch i uses Philox stream (seed, call_index + i). batch <= 1024. */
int32_t qlc_replay_sample(qlc_env* env, uint32_t batch, uint32_t n_batches, uint64_t call_index, uint32_t* idx_dev, void* stream);
/* get_many + batch_to_multi_dim_array: gather n transitions by logical index (0 = oldest). state_dev / next_dev
 * [n] x layout (either may be NULL), reward_dev [n] f32, action_dev [n] u8, done_dev [n] u8 (any may be NULL).
 * Indices are not range-checked on the device path: an index >= len gives all-zero stacks and zero scalars. */
int32_t qlc_replay_gather(qlc_env* env, const uint32_t* idx_dev, uint32_t n, int32_t layout,
                          void* state_dev, void* next_dev, float* reward_dev, uint8_t* action_dev, uint8_t* done_dev, void* stream);
/* generate_distinct_random_ids + get_many + batch_to_multi_dim_array in ONE kernel launch (self_driving_tf_q_learner.rs:181-185):
 * every CTA of the gather kernel derives the index of its own item from the Philox stream (seed, call_index + minibatch) -
 * the same indices qlc_replay_sample gives. Items = n_batches x batch; idx_out_dev [n_batches][batch] u32 may be NULL. */
int32_t qlc_replay_sample_gather(qlc_env* env, uint32_t batch, uint32_t n_batches, uint64_t call_index, int32_t layout, uint32_t* idx_out_dev,
                                 void* state_dev, void* next_dev, float* reward_dev, uint8_t* action_dev, uint8_t* done_dev, void* stream);
/* host-buffer forms (range-check indices: QLC_ERR_OUT_OF_RANGE; copies inside; synchronous). QLC_LAYOUT_F32_BXYH stacks cross
 * PCIe as u8 and are widened into the caller's buffer by a small host thread pool (QLC_HOST_THREADS; bit-identical). */
int32_t qlc_replay_sample_host(qlc_env* env, uint32_t batch, uint64_t call_index, uint32_t* idx_host);
int32_t qlc_replay_gather_host(qlc_env* env, const uint32_t* idx_host, uint32_t n, int32_t layout,
                               void* state_host, void* next_host, float* reward_host, uint8_t* action_host, uint8_t* done_host);
int32_t qlc_replay_sample_gather_host(qlc_env* env, uint32_t batch, uint64_t call_index, int32_t layout, uint32_t* idx_out_host,
                                      void* state_host, void* next_host, float* reward_host, uint8_t* action_host, uint8_t* done_host);
int32_t qlc_replay_action_counts(qlc_env* env, uint64_t counts[3]);   /* actions() histogram (learner log :242-245) */

/* ---- episode statistics (replay_buffer.rs:100-124, self_driving_tf_q_learner.rs:134-139,220-223) ---- */
int32_t qlc_stats_read(qlc_env* env, qlc_episode_stats* out);         /* synchronous */
/* device vector of 5 doubles {sum_return, episodes, steps, -min_return, max_return} refreshed on `stream`;
 * sum the first three and max-reduce the last two across ranks (ncclAllReduce / torch.distributed). */
int32_t qlc_stats_export(qlc_env* env, double* out_dev, void* stream);
/* ---- the same reduction behind the C ABI (a host without torch.distributed, e.g. the Rust `ql-cuda` crate): NCCL is bound at
 * run time (dlopen "libnccl.so.2", QLC_NCCL_LIB overrides), one process per GPU, one communicator per env handle. Rank 0 calls
 * qlc_comm_unique_id and hands the 128 bytes to the other ranks by whatever channel the host has (file, socket, env var);
 * every rank then calls qlc_comm_init (collective, blocking). world == 1 with id == NULL needs no NCCL at all.
 * qlc_stats_allreduce enqueues one reduction: nothing but an event record lands on `stream` (the caller's step stream) - the
 * export of the shard's statistics as of the end of the last step launch (a snapshot the step kernel's last CTA takes, so later
 * launches may already be running), ONE ncclAllGather of 5 doubles, the combine and the copy into a host mirror run on the
 * communicator's own low-priority stream: it can be called after every step without being on the step path.
 * qlc_stats_global returns the job-wide statistics of the last completed reduction (wait != 0: waits for the last enqueued). ---- */
#define QLC_COMM_ID_BYTES 128
int32_t qlc_comm_unique_id(uint8_t* id128);
int32_t qlc_comm_init(qlc_env* env, int32_t rank, int32_t world, const uint8_t* id128);
int32_t qlc_comm_destroy(qlc_env* env);                              /* also done by qlc_env_destroy */
int32_t qlc_comm_info(qlc_env* env, int32_t* rank, int32_t* world, int32_t* nccl_version, int32_t* nccl_ranks);
int32_t qlc_stats_allreduce(qlc_env* env, void* stream);
int32_t qlc_stats_global(qlc_env* env, qlc_episode_stats* out, int32_t wait);

int32_t qlc_stats_push(qlc_env* env, float episode_reward);           /* add_episode_reward */
int32_t qlc_stats_mean(qlc_env* env, float* out);                     /* avg_episode_reward */
int32_t qlc_stats_min(qlc_env* env, float* out);                      /* min_episode_reward */
int32_t qlc_stats_window(qlc_env* env, float* out, uint32_t cap, uint32_t* n);  /* episode_rewards() */

/* ---- Q-network forward on the tensor cores (tcgen05, bf16 operands, f32 accumulation) — SURVEY.md 8f-3. Architecture of
 * python_model/create_ql_model_breakout_84x84x4_3_32.py:17-33; the first convolution reads the u8 frames straight from
 * the frame ring. Replaces QLearningTensorflowModel::predict_action / batch_predict_max_future_reward
 * (ql-with-tensorflow/src/ml_model/tensorflow_python/q_learning_model.rs:107-152) for inference. ---- */
typedef struct qlc_qnet qlc_qnet;
typedef struct qlc_qnet_weights {          /* host f32 arrays in the Keras layouts */
    const float* conv1_kernel; const float* conv1_bias;    /* [8][8][4][32], [32]  (axes: x offset, y offset, ring slot, out) */
    const float* conv2_kernel; const float* conv2_bias;    /* [4][4][32][64], [64] */
    const float* conv3_kernel; const float* conv3_bias;    /* [3][3][64][64], [64] */
    const float* dense1_kernel; const float* dense1_bias;  /* [3136][512], [512]   (input order of Flatten([7][7][64])) */
    const float* dense2_kernel; const float* dense2_bias;  /* [512][3], [3] */
} qlc_qnet_weights;
int32_t qlc_qnet_create(qlc_env* env, const qlc_qnet_weights* weights_host, qlc_qnet** out);
int32_t qlc_qnet_set_weights(qlc_qnet* qnet, const qlc_qnet_weights* weights_host);
int32_t qlc_qnet_destroy(qlc_qnet* qnet);   /* valid before or after qlc_env_destroy of its env; after it, every other qnet call fails */
/* qlc_qnet_forward is asynchronous and cannot report a failed pass; this synchronises the device, returns the sticky flag
 * (non-zero: an MMA completion barrier timed out, the outputs of that pass are undefined) and clears it. */
int32_t qlc_qnet_error(qlc_qnet* qnet, uint32_t* flag);
/* idx_dev NULL: the current observation of all n_envs envs (predict_action for every env); else n replay transitions by
 * logical index, which = 0 their state / 1 their state_next. Outputs (device, any may be NULL): q [n][3] f32, action [n] u8
 * (first maximum, tf.argmax), max_q [n] f32 (tf.reduce_max). Asynchronous on `stream`. */
int32_t qlc_qnet_forward(qlc_qnet* qnet, const uint32_t* idx_dev, uint32_t n, int32_t which, float* q_dev, uint8_t* action_dev, float* max_q_dev, void* stream);
int32_t qlc_qnet_forward_host(qlc_qnet* qnet, const uint32_t* idx_host, uint32_t n, int32_t which, float* q_host, uint8_t* action_host, float* max_q_host);

/* ---- Q-network training on the device: the reference's DeepQLearningModel::train (ml_model/model.rs:59-71) for the Keras
 * model (Huber(delta 1) loss on Q(s)[a] averaged over the minibatch, clipnorm per variable, Adam). Master weights, Adam
 * moments and gradients are f32; GEMM operands bf16 with f32 accumulation. Deterministic: the same inputs give the same
 * weight bits. Adam moments are not part of qlc_env_save checkpoints; a resumed run restarts them. ---- */
typedef struct qlc_adam_config { float lr, beta1, beta2, epsilon, clipnorm; } qlc_adam_config;   /* default 2.5e-4, 0.9, 0.999, 1e-7, 1.0; clipnorm <= 0: off */
int32_t qlc_qnet_set_adam(qlc_qnet* qnet, const qlc_adam_config* cfg);           /* also resets m, v and the step count t (as qlc_qnet_set_weights does) */
int32_t qlc_qnet_get_weights(qlc_qnet* qnet, const qlc_qnet_weights* out_host);  /* the f32 masters in the Keras layouts (writes through the pointers) */
/* n_batches successive updates on the minibatches idx_dev[j * batch .. (j + 1) * batch) of replay transitions (state =
 * which 0 of qlc_qnet_forward, action = record bits 0-1). Targets: target_dev [n_batches][batch] f32, or, when it is NULL,
 * y = r + max_a Q_target(state_next) * gamma (y = r where done) from target_net (same env), evaluated once for the whole
 * call. loss_dev (optional): [n_batches] Huber losses, before each update. Asynchronous on `stream`; MMA time-outs raise
 * the sticky flag of qlc_qnet_error. */
int32_t qlc_qnet_train(qlc_qnet* qnet, const uint32_t* idx_dev, uint32_t batch, uint32_t n_batches, const float* target_dev, qlc_qnet* target_net,
                       float gamma, float* loss_dev, void* stream);
int32_t qlc_qnet_train_host(qlc_qnet* qnet, const uint32_t* idx_host, uint32_t batch, uint32_t n_batches, const float* target_host, qlc_qnet* target_net,
                            float gamma, float* loss_host);
/* forward + backward only, for tests: the unclipped f32 gradients of the loss over n transitions with targets target_host [n] */
int32_t qlc_qnet_debug_grads(qlc_qnet* qnet, const uint32_t* idx_host, uint32_t n, const float* target_host, const qlc_qnet_weights* grads_out_host);
/* qlc_qnet_train with per-item loss weights: minibatch loss = mean of w * Huber(Q(s)[a] - y). weight_dev [n_batches][batch] (NULL = 1:
 * exactly qlc_qnet_train's arithmetic); td_dev [n_batches][batch] out (NULL = not written) gets Q(s)[a] - y from the forward that
 * precedes each item's own update - what qlc_per_update takes. */
int32_t qlc_qnet_train_weighted(qlc_qnet* qnet, const uint32_t* idx_dev, const float* weight_dev, uint32_t batch, uint32_t n_batches,
                                const float* target_dev, qlc_qnet* target_net, float gamma, float* loss_dev, float* td_dev, void* stream);
/* test hook, like qlc_qnet_debug_grads: unclipped gradients of the weighted loss (weight_host NULL = 1), and the TD errors
 * td_out_host [n] (may be NULL) */
int32_t qlc_qnet_debug_grads_weighted(qlc_qnet* qnet, const uint32_t* idx_host, uint32_t n, const float* target_host,
                                      const float* weight_host, const qlc_qnet_weights* grads_out_host, float* td_out_host);

/* ---- n-step returns and double-DQN targets read straight from the replay ring (DESIGN.md §14). Transition i (logical index)
 * is followed in its env by i + n_envs. The walk from i takes records j = 0, 1, ... and stops at the first j where the record is
 * done (terminal) or truncated, j = n_step - 1, j is the newest time in the replay, or the next record starts an episode (a
 * reset by the caller). With m = j + 1 records: G = sum gamma^j r_j (f32, in order), disc = gamma^m (0 where terminal), and the
 * bootstrap state is state_next of boot = i + (m - 1) n_envs. The target is y = G where terminal, else G + Q_boot * disc, with
 * Q_boot = max_a Q_target(boot), or with double DQN Q_target(boot)[argmax_a Q_online(boot)]. Deterministic. ---- */
#define QLC_NSTEP_MAX 64
/* n-step returns of replay transitions idx_dev [n] (logical indices): return_dev [n] f32 = G, discount_dev [n] f32 = disc
 * (0 where terminal), boot_idx_dev [n] u32 = the logical index whose state_next bootstraps (any output may be NULL).
 * 1 <= n_step <= QLC_NSTEP_MAX, 0 <= gamma <= 1. An index >= len gives 0, 0 and the index itself. Asynchronous on `stream`. */
int32_t qlc_replay_nstep(qlc_env* env, const uint32_t* idx_dev, uint32_t n, uint32_t n_step, float gamma,
                         float* return_dev, float* discount_dev, uint32_t* boot_idx_dev, void* stream);
/* qlc_qnet_train_weighted with n-step / double-DQN targets from target_net (required, same env); y_dev [n_batches][batch]
 * (may be NULL) receives the target each item was trained on. n_step = 1, double_dqn = 0 is qlc_qnet_train_weighted's
 * arithmetic bit for bit. The target network is evaluated once per call; with double_dqn = 1 the online network's greedy
 * action for minibatch j comes from the weights after updates 0 .. j-1, so n_batches = k calls give the bits of k calls. */
int32_t qlc_qnet_train_nstep(qlc_qnet* qnet, const uint32_t* idx_dev, const float* weight_dev, uint32_t batch, uint32_t n_batches,
                             qlc_qnet* target_net, float gamma, uint32_t n_step, int32_t double_dqn,
                             float* loss_dev, float* td_dev, float* y_dev, void* stream);

/* ---- proportional prioritized replay (Schaul et al., ICLR 2016) on the device: a sum tree over the replay ring (DESIGN.md §13).
 * Priorities p = (|delta| + epsilon)^alpha, one per transition; a transition enters the replay at the running maximum priority
 * (which starts at 1.0 and never decreases). The tree follows the ring lazily: every call first catches up with the steps taken
 * since the previous one, so qlc_env_step is unchanged and nothing is read back to the host. Sample, train and update must see
 * the same env time: a step in between shifts the logical indices (as it does between qlc_replay_sample and qlc_qnet_train).
 * Priorities are not part of qlc_env_save checkpoints; after qlc_env_load every transition restarts at the running maximum.
 * Deterministic: the same calls give the same indices, weights and tree bits. ---- */
typedef struct qlc_per qlc_per;
/* 0 <= alpha <= 1, epsilon > 0 (finite); the env's replay_capacity > 0 */
int32_t qlc_per_create(qlc_env* env, float alpha, float epsilon, qlc_per** out);
/* valid before or after qlc_env_destroy; afterwards every other call fails */
int32_t qlc_per_destroy(qlc_per* per);
/* n_batches stratified minibatches drawn with replacement, P(i) = p_i / total: idx_dev [n_batches][batch] u32 logical indices
 * (0 = oldest), weight_dev [n_batches][batch] f32 importance weights (p_min / p_i)^beta, p_min the smallest priority in the item's
 * minibatch (may be NULL); 0 <= beta <= 1. Minibatch m uses the Philox stream (seed, call_index + m, 'PRIO'). Asynchronous. */
int32_t qlc_per_sample(qlc_per* per, uint32_t batch, uint32_t n_batches, uint64_t call_index, float beta,
                       uint32_t* idx_dev, float* weight_dev, void* stream);
/* priorities of n transitions from their TD errors td_dev [n]: an index given twice keeps its largest priority, indices >= len
 * are ignored, a non-finite delta gives the running maximum. Asynchronous. */
int32_t qlc_per_update(qlc_per* per, const uint32_t* idx_dev, const float* td_dev, uint32_t n, void* stream);
/* synchronous; leaves_host [len] in logical order (may be NULL), total = root, max = running max priority (either may be NULL) */
int32_t qlc_per_read_host(qlc_per* per, float* leaves_host, double* total_host, float* max_priority_host);

/* ---- checkpoint / resume of the env shard + replay ring (the reference checkpoints only the model:
 * q_learning_model.rs:191-202). qlc_env_load needs an env created with the same n_envs / env_id_base / seed /
 * replay_capacity / episode limits; a resumed run continues bit-identically. Synchronous. ---- */
int32_t qlc_env_save(qlc_env* env, const char* path);
int32_t qlc_env_load(qlc_env* env, const char* path);

/* ---- debug / known-answer entry points: run the DEVICE collision routines on the GPU for one input
 * (used to replay the reference's rstest vectors mechanics.rs:659-752 through the product code) ---- */
int32_t qlc_debug_collision_wall(int32_t which /*0 left,1 right,2 top*/, float cx, float cy, float radius, float mvx, float mvy,
                                 int32_t* some, float* way, float* approximation, float* nx, float* ny, uint32_t* err);
int32_t qlc_debug_collision_rect(float cx, float cy, float radius, float mvx, float mvy,
                                 float min_x, float min_y, float max_x, float max_y,
                                 int32_t* some, float* way, float* approximation, float* nx, float* ny, uint32_t* err);

/* batched rectangle sweep: in_host [n][9] = cx, cy, radius, mvx, mvy, min_x, min_y, max_x, max_y;
 * out_host [n][6] = some (0/1), way, approximation, nx, ny, err (u32 bits in a float slot) */
int32_t qlc_debug_collision_rect_batch(const float* in_host, float* out_host, uint32_t n);

/* test hook of the tcgen05 GEMM the Q-network layers are built from: out[m][n] = act(bf16(a)[m][k] * bf16(w)[n][k]^T + bias),
 * host f32 buffers in and out; k % 64 == 0, n in {32, 64, 128, 256, 512} */
int32_t qlc_debug_gemm_bf16(const float* a_host, const float* w_host, const float* bias_host, int32_t relu, float* out_host,
                            uint32_t m, uint32_t n, uint32_t k);

#ifdef __cplusplus
}
#endif
#endif /* QL_CUDA_H */
