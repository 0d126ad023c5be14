//! Raw bindings, 1:1 with include/ql_cuda.h.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

pub const QLC_OK: i32 = 0;
pub const QLC_ERR_OUT_OF_RANGE: i32 = 3;
pub const QLC_LAYOUT_U8_BHYX: i32 = 0;
pub const QLC_LAYOUT_F32_BXYH: i32 = 1;
pub const QLC_LAYOUT_U8_BXYH: i32 = 2;
pub const QLC_COMM_ID_BYTES: usize = 128;
pub const QLC_FRAME_W: usize = 84;
pub const QLC_FRAME_H: usize = 84;
pub const QLC_NUM_FRAMES: usize = 4;
pub const QLC_NSTEP_MAX: u32 = 64;

#[repr(C)]
pub struct qlc_env {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct qlc_config {
    pub struct_size: u32,
    pub device: i32,
    pub n_envs: u32,
    pub env_id_base: u32,
    pub frame_w: u32,
    pub frame_h: u32,
    pub seed: u64,
    pub replay_capacity: u64,
    pub max_episode_steps: u32,
    pub episode_window: u32,
    pub auto_reset: u32,
    pub reserved: u32,
}

/// A state handle: the observation of env `env` after `time` env-steps, `k` of them in the current episode.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct qlc_obs_handle {
    pub time: u64,
    pub k: u32,
    pub env: u32,
}

#[repr(C)]
pub struct qlc_state_host {
    pub ball_cx: *mut f32,
    pub ball_cy: *mut f32,
    pub ball_dx: *mut f32,
    pub ball_dy: *mut f32,
    pub pad_min_x: *mut f32,
    pub pad_max_x: *mut f32,
    pub pad_speed: *mut f32,
    pub bricks: *mut u64,
    pub score: *mut u32,
    pub episode_step: *mut u32,
    pub episode: *mut u32,
    pub err: *mut u32,
    pub finished: *mut u8,
}

/// device pointers to the structure-of-arrays env state (valid until qlc_env_destroy)
#[repr(C)]
pub struct qlc_state_view {
    pub ball_cx: *const f32,
    pub ball_cy: *const f32,
    pub ball_dx: *const f32,
    pub ball_dy: *const f32,
    pub pad_min_x: *const f32,
    pub pad_max_x: *const f32,
    pub pad_speed: *const f32,
    pub bricks: *const u64,
    pub score: *const u32,
    pub episode_step: *const u32,
    pub episode: *const u32,
    pub err: *const u32,
    pub finished: *const u8,
    pub frames: *const u8,
    pub records: *const u32,
    pub n_envs: u32,
    pub time_slots: u32,
    pub time: u64,
}

#[repr(C)]
pub struct qlc_qnet {
    _private: [u8; 0],
}

/// proportional prioritized replay: a sum tree over an env's replay ring
#[repr(C)]
pub struct qlc_per {
    _private: [u8; 0],
}

/// host f32 arrays in the Keras layouts
#[repr(C)]
pub struct qlc_qnet_weights {
    pub conv1_kernel: *const f32,
    pub conv1_bias: *const f32,
    pub conv2_kernel: *const f32,
    pub conv2_bias: *const f32,
    pub conv3_kernel: *const f32,
    pub conv3_bias: *const f32,
    pub dense1_kernel: *const f32,
    pub dense1_bias: *const f32,
    pub dense2_kernel: *const f32,
    pub dense2_bias: *const f32,
}

/// Adam + clipnorm settings of qlc_qnet_train (default: the Keras model's 2.5e-4, 0.9, 0.999, 1e-7, clipnorm 1.0).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct qlc_adam_config {
    pub lr: f32,
    pub beta1: f32,
    pub beta2: f32,
    pub epsilon: f32,
    pub clipnorm: f32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct qlc_episode_stats {
    pub sum_return: u64,
    pub episodes: u64,
    pub steps: u64,
    pub min_return: u32,
    pub max_return: u32,
}

extern "C" {
    pub fn qlc_version() -> i32;
    pub fn qlc_build_info() -> *const c_char;
    pub fn qlc_last_error_string() -> *const c_char;
    pub fn qlc_device_count(count: *mut i32) -> i32;
    pub fn qlc_env_create(cfg: *const qlc_config, out: *mut *mut qlc_env) -> i32;
    pub fn qlc_env_destroy(env: *mut qlc_env) -> i32;
    pub fn qlc_sync(env: *mut qlc_env, stream: *mut c_void) -> i32;
    pub fn qlc_host_alloc(bytes: usize, out: *mut *mut c_void) -> i32;
    pub fn qlc_host_free(p: *mut c_void) -> i32;
    pub fn qlc_env_reset(env: *mut qlc_env, mask_host: *const u8, dir_x_host: *const f32) -> i32;
    pub fn qlc_env_step(env: *mut qlc_env, actions_dev: *const u8, n_steps: u32, reward_dev: *mut f32, done_dev: *mut u8, stream: *mut c_void) -> i32;
    pub fn qlc_env_step_random(env: *mut qlc_env, n_steps: u32, actions_out_dev: *mut u8, reward_dev: *mut f32, done_dev: *mut u8, stream: *mut c_void) -> i32;
    pub fn qlc_env_step_host(env: *mut qlc_env, actions_host: *const u8, n_steps: u32, reward_host: *mut f32, done_host: *mut u8) -> i32;
    pub fn qlc_env_step_host_submit(env: *mut qlc_env, actions_host: *const u8, n_steps: u32, reward_host: *mut f32, done_host: *mut u8) -> i32;
    pub fn qlc_env_step_host_wait(env: *mut qlc_env, max_pending: u32) -> i32;
    pub fn qlc_env_obs(env: *mut qlc_env, layout: i32, out_dev: *mut c_void, stream: *mut c_void) -> i32;
    pub fn qlc_env_obs_host(env: *mut qlc_env, layout: i32, out_host: *mut c_void) -> i32;
    pub fn qlc_env_state_view(env: *mut qlc_env, out: *mut qlc_state_view) -> i32;
    pub fn qlc_env_read_state(env: *mut qlc_env, out: *const qlc_state_host) -> i32;
    pub fn qlc_env_goal_mean() -> f32;
    pub fn qlc_env_time(env: *mut qlc_env, steps_taken: *mut u64) -> i32;
    pub fn qlc_env_lives_host(env: *mut qlc_env, lives_host: *mut u8) -> i32;
    pub fn qlc_obs_gather(env: *mut qlc_env, handles_dev: *const qlc_obs_handle, n: u32, layout: i32, out_dev: *mut c_void, stream: *mut c_void) -> i32;
    pub fn qlc_obs_gather_host(env: *mut qlc_env, handles_host: *const qlc_obs_handle, n: u32, layout: i32, out_host: *mut c_void) -> i32;
    pub fn qlc_env_error_flags(env: *mut qlc_env, or_of_all: *mut u32) -> i32;
    pub fn qlc_replay_len(env: *mut qlc_env, len: *mut u64) -> i32;
    pub fn qlc_replay_capacity(env: *mut qlc_env, capacity: *mut u64) -> i32;
    pub fn qlc_replay_sample(env: *mut qlc_env, batch: u32, n_batches: u32, call_index: u64, idx_dev: *mut u32, stream: *mut c_void) -> i32;
    pub fn qlc_replay_gather(env: *mut qlc_env, idx_dev: *const u32, n: u32, layout: i32, state_dev: *mut c_void, next_dev: *mut c_void,
                             reward_dev: *mut f32, action_dev: *mut u8, done_dev: *mut u8, stream: *mut c_void) -> i32;
    pub fn qlc_replay_sample_gather(env: *mut qlc_env, batch: u32, n_batches: u32, call_index: u64, layout: i32, idx_out_dev: *mut u32,
                                    state_dev: *mut c_void, next_dev: *mut c_void, reward_dev: *mut f32, action_dev: *mut u8, done_dev: *mut u8,
                                    stream: *mut c_void) -> i32;
    pub fn qlc_replay_sample_host(env: *mut qlc_env, batch: u32, call_index: u64, idx_host: *mut u32) -> i32;
    pub fn qlc_replay_sample_gather_host(env: *mut qlc_env, batch: u32, call_index: u64, layout: i32, idx_out_host: *mut u32, state_host: *mut c_void,
                                         next_host: *mut c_void, reward_host: *mut f32, action_host: *mut u8, done_host: *mut u8) -> i32;
    pub fn qlc_replay_gather_host(env: *mut qlc_env, idx_host: *const u32, n: u32, layout: i32, state_host: *mut c_void, next_host: *mut c_void,
                                  reward_host: *mut f32, action_host: *mut u8, done_host: *mut u8) -> i32;
    pub fn qlc_replay_action_counts(env: *mut qlc_env, counts: *mut u64) -> i32;
    pub fn qlc_env_save(env: *mut qlc_env, path: *const c_char) -> i32;
    pub fn qlc_env_load(env: *mut qlc_env, path: *const c_char) -> i32;
    pub fn qlc_stats_read(env: *mut qlc_env, out: *mut qlc_episode_stats) -> i32;
    pub fn qlc_stats_export(env: *mut qlc_env, out_dev: *mut f64, stream: *mut c_void) -> i32;
    pub fn qlc_comm_unique_id(id128: *mut u8) -> i32;
    pub fn qlc_comm_init(env: *mut qlc_env, rank: i32, world: i32, id128: *const u8) -> i32;
    pub fn qlc_comm_destroy(env: *mut qlc_env) -> i32;
    pub fn qlc_comm_info(env: *mut qlc_env, rank: *mut i32, world: *mut i32, nccl_version: *mut i32, nccl_ranks: *mut i32) -> i32;
    pub fn qlc_stats_allreduce(env: *mut qlc_env, stream: *mut c_void) -> i32;
    pub fn qlc_stats_global(env: *mut qlc_env, out: *mut qlc_episode_stats, wait: i32) -> i32;
    pub fn qlc_stats_push(env: *mut qlc_env, episode_reward: f32) -> i32;
    pub fn qlc_stats_mean(env: *mut qlc_env, out: *mut f32) -> i32;
    pub fn qlc_stats_min(env: *mut qlc_env, out: *mut f32) -> i32;
    pub fn qlc_stats_window(env: *mut qlc_env, out: *mut f32, cap: u32, n: *mut u32) -> i32;
    pub fn qlc_debug_collision_wall(which: i32, cx: f32, cy: f32, radius: f32, mvx: f32, mvy: f32, some: *mut i32, way: *mut f32,
                                    approximation: *mut f32, nx: *mut f32, ny: *mut f32, err: *mut u32) -> i32;
    pub fn qlc_debug_collision_rect(cx: f32, cy: f32, radius: f32, mvx: f32, mvy: f32, min_x: f32, min_y: f32, max_x: f32, max_y: f32,
                                    some: *mut i32, way: *mut f32, approximation: *mut f32, nx: *mut f32, ny: *mut f32, err: *mut u32) -> i32;
    pub fn qlc_debug_collision_rect_batch(in_host: *const f32, out_host: *mut f32, n: u32) -> i32;
    pub fn qlc_qnet_create(env: *mut qlc_env, weights_host: *const qlc_qnet_weights, out: *mut *mut qlc_qnet) -> i32;
    pub fn qlc_qnet_set_weights(qnet: *mut qlc_qnet, weights_host: *const qlc_qnet_weights) -> i32;
    pub fn qlc_qnet_destroy(qnet: *mut qlc_qnet) -> i32;
    pub fn qlc_qnet_error(qnet: *mut qlc_qnet, flag: *mut u32) -> i32;
    pub fn qlc_qnet_forward(qnet: *mut qlc_qnet, idx_dev: *const u32, n: u32, which: i32, q_dev: *mut f32, action_dev: *mut u8, max_q_dev: *mut f32, stream: *mut c_void) -> i32;
    pub fn qlc_qnet_forward_host(qnet: *mut qlc_qnet, idx_host: *const u32, n: u32, which: i32, q_host: *mut f32, action_host: *mut u8, max_q_host: *mut f32) -> i32;
    pub fn qlc_qnet_set_adam(qnet: *mut qlc_qnet, cfg: *const qlc_adam_config) -> i32;
    pub fn qlc_qnet_get_weights(qnet: *mut qlc_qnet, out_host: *const qlc_qnet_weights) -> i32;
    pub fn qlc_qnet_train(qnet: *mut qlc_qnet, idx_dev: *const u32, batch: u32, n_batches: u32, target_dev: *const f32, target_net: *mut qlc_qnet,
                          gamma: f32, loss_dev: *mut f32, stream: *mut c_void) -> i32;
    pub fn qlc_qnet_train_host(qnet: *mut qlc_qnet, idx_host: *const u32, batch: u32, n_batches: u32, target_host: *const f32, target_net: *mut qlc_qnet,
                               gamma: f32, loss_host: *mut f32) -> i32;
    pub fn qlc_qnet_debug_grads(qnet: *mut qlc_qnet, idx_host: *const u32, n: u32, target_host: *const f32, grads_out_host: *const qlc_qnet_weights) -> i32;
    pub fn qlc_qnet_train_weighted(qnet: *mut qlc_qnet, idx_dev: *const u32, weight_dev: *const f32, batch: u32, n_batches: u32, target_dev: *const f32,
                                   target_net: *mut qlc_qnet, gamma: f32, loss_dev: *mut f32, td_dev: *mut f32, stream: *mut c_void) -> i32;
    pub fn qlc_qnet_debug_grads_weighted(qnet: *mut qlc_qnet, idx_host: *const u32, n: u32, target_host: *const f32, weight_host: *const f32,
                                         grads_out_host: *const qlc_qnet_weights, td_out_host: *mut f32) -> i32;
    pub fn qlc_replay_nstep(env: *mut qlc_env, idx_dev: *const u32, n: u32, n_step: u32, gamma: f32, return_dev: *mut f32, discount_dev: *mut f32,
                            boot_idx_dev: *mut u32, stream: *mut c_void) -> i32;
    pub fn qlc_qnet_train_nstep(qnet: *mut qlc_qnet, idx_dev: *const u32, weight_dev: *const f32, batch: u32, n_batches: u32, target_net: *mut qlc_qnet,
                                gamma: f32, n_step: u32, double_dqn: i32, loss_dev: *mut f32, td_dev: *mut f32, y_dev: *mut f32, stream: *mut c_void) -> i32;
    pub fn qlc_per_create(env: *mut qlc_env, alpha: f32, epsilon: f32, out: *mut *mut qlc_per) -> i32;
    pub fn qlc_per_destroy(per: *mut qlc_per) -> i32;
    pub fn qlc_per_sample(per: *mut qlc_per, batch: u32, n_batches: u32, call_index: u64, beta: f32, idx_dev: *mut u32, weight_dev: *mut f32,
                          stream: *mut c_void) -> i32;
    pub fn qlc_per_update(per: *mut qlc_per, idx_dev: *const u32, td_dev: *const f32, n: u32, stream: *mut c_void) -> i32;
    pub fn qlc_per_read_host(per: *mut qlc_per, leaves_host: *mut f32, total_host: *mut f64, max_priority_host: *mut f32) -> i32;
    pub fn qlc_debug_gemm_bf16(a_host: *const f32, w_host: *const f32, bias_host: *const f32, relu: i32, out_host: *mut f32, m: u32, n: u32, k: u32) -> i32;
}
