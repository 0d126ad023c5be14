//! Raw bindings, 1:1 with include/ql_cuda_nstep.h: n-step returns and double-DQN targets on the device.
#![allow(non_camel_case_types)]
use std::os::raw::c_void;

use crate::ffi::{qlc_env, qlc_qnet};

pub const QLC_NSTEP_MAX: u32 = 64;

extern "C" {
    pub fn qlc_replay_nstep(env: *mut qlc_env, idx_dev: *const u32, n: u32, n_step: u32, gamma: f32, return_dev: *mut f32, discount_dev: *mut f32,
                            boot_idx_dev: *mut u32, stream: *mut c_void) -> i32;
    pub fn qlc_qnet_train_nstep(qnet: *mut qlc_qnet, idx_dev: *const u32, weight_dev: *const f32, batch: u32, n_batches: u32, target_net: *mut qlc_qnet,
                                gamma: f32, n_step: u32, double_dqn: i32, loss_dev: *mut f32, td_dev: *mut f32, y_dev: *mut f32, stream: *mut c_void) -> i32;
}
