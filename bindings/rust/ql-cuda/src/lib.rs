//! ql-cuda: B200-native drop-in for the Breakout environment and its state in bitmagier/q-learning.
//!
//! * [`CudaBreakoutEnvironment`]`: ql::prelude::Environment` — `reset` / `state` / `step` drive the fused CUDA kernel
//!   (physics + rasteriser + grayscale + frame-ring append) through the C ABI.
//! * [`CudaBreakoutState`] is a *handle* (env, time, frames-in-episode): `Clone` and `Rc::new(state.clone())`
//!   (`state_as_rc` / `step_as_rc`, ql/src/prelude.rs:36,52-58) copy two integers, the pixels stay in the HBM frame ring.
//! * The learner's replay memory is **the reference's own, unchanged** `ReplayBuffer<Rc<E::S>, E::A>`
//!   (ql-with-tensorflow/src/learn/replay_buffer.rs:53-146, held at self_driving_tf_q_learner.rs:81): it is generic over `S`,
//!   so with `S = CudaBreakoutState` its five deques hold handles and scalars, and the pixels of a minibatch move exactly
//!   once — on the GPU — when the model calls `S::batch_to_multi_dim_array(batch)` (q_learning_model.rs:137,171;
//!   `src/tensor.rs` here): ONE gather kernel + one u8 copy over PCIe instead of `N * 28,224` `Tensor::set` calls.
//!   `self_driving_tf_q_learner.rs` is not touched at all — not even its `use` lines.
//! * [`TensorCoreQModel`]: optional inference half of `DeepQLearningModel` on the library's tcgen05 Q-network.
pub mod ffi;

mod env;
mod model;
#[cfg(feature = "tensorflow")]
mod tensor;

pub use env::{BreakoutAction, CudaBreakoutEnvironment, CudaBreakoutState, EpisodeStats};
pub use model::{QNetWeights, TensorCoreQModel};

use ql::prelude::QlError;
use std::ffi::CStr;

pub(crate) fn check(rc: i32) -> anyhow::Result<()> {
    if rc == ffi::QLC_OK {
        return Ok(());
    }
    let msg = unsafe { CStr::from_ptr(ffi::qlc_last_error_string()) }.to_string_lossy().into_owned();
    Err(QlError(msg).into())
}
