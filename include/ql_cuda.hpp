// ql_cuda.hpp — C++ host-side mirror of the reference's Rust interfaces for the hot path, over the C ABI (ql_cuda.h).
//
// The reference is compiled Rust and this image has no cargo/rustc, so the host layer above the C ABI is written in
// C++ with the SAME names, argument meaning and error behaviour as the reference, so that the learner loop
// (self_driving_tf_q_learner.rs:141-233) reads the same against it:
//
//   ql::prelude::Action / BreakoutAction ....... prelude.rs:12-18, breakout_environment.rs:94-120  -> ql::BreakoutAction
//   ql::prelude::Environment ................... prelude.rs:21-63                                  -> ql::BreakoutEnvironment
//   BreakoutState + ToMultiDimArray ............ breakout_environment.rs:24-78, model.rs:12-26      -> ql::BreakoutState (a handle)
//   Buffer<T>, ReplayBuffer<S, A>, BufferSample  replay_buffer.rs:5-146                             -> ql::Buffer / ql::ReplayBuffer / ql::BufferSample,
//                                                                                                      generic with the same signatures
//   generate_distinct_random_ids(rng, range) ... self_driving_tf_q_learner.rs:276-296               -> ql::generate_distinct_random_ids (host, the learner's own)
//
// A Rust `ql-cuda` crate with the same shape is in bindings/rust/ql-cuda (source only; see INTEGRATION.md).
// Header-only; link with libqlcuda.so. No CPU fallback: every call fails with QlError when CUDA is unavailable.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <deque>
#include <memory>
#include <random>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "ql_cuda.h"

namespace ql {

using ModelActionType = uint8_t;                                   // prelude.rs:10

struct QlError : std::runtime_error {                              // prelude.rs:70-86
    int32_t code;
    QlError(const std::string& msg, int32_t c = QLC_ERR_INVALID_ARG) : std::runtime_error(msg), code(c) {}
};

inline void check(int32_t rc) {
    if (rc != QLC_OK) throw QlError(qlc_last_error_string(), rc);
}

// ---- Action (breakout_environment.rs:94-120) ----
enum class BreakoutAction : ModelActionType { None = 0, Left = 1, Right = 2 };
struct BreakoutActionTrait {
    static constexpr ModelActionType ACTION_SPACE = 3;
    static ModelActionType numeric(BreakoutAction a) { return static_cast<ModelActionType>(a); }
    static BreakoutAction try_from_numeric(ModelActionType v) {
        if (v >= ACTION_SPACE) throw QlError("value out of range", QLC_ERR_OUT_OF_RANGE);
        return static_cast<BreakoutAction>(v);
    }
};

// ---- Tensor<f32> stand-in: dims + row-major data (what ToMultiDimArray<Tensor<f32>> produces) ----
struct Tensor {
    std::vector<uint64_t> dims;
    std::vector<float> data;
};

class EnvHandle {   // owns the qlc_env; shared by the environment and every state handle
public:
    explicit EnvHandle(const qlc_config& cfg) { check(qlc_env_create(&cfg, &h_)); n_envs_ = cfg.n_envs; }
    ~EnvHandle() { qlc_env_destroy(h_); }
    EnvHandle(const EnvHandle&) = delete;
    EnvHandle& operator=(const EnvHandle&) = delete;
    qlc_env* get() const { return h_; }
    uint32_t n_envs() const { return n_envs_; }
    uint64_t time() const { uint64_t t = 0; check(qlc_env_time(h_, &t)); return t; }
private:
    qlc_env* h_ = nullptr;
    uint32_t n_envs_ = 0;
};

// ---- BreakoutState (breakout_environment.rs:24-28) as a HANDLE: the observation of the env after `time` steps, `k` of them in
// the current episode. Copying it (Clone, Rc::new(state.clone()): prelude.rs:36,57) copies two integers; the four frames it names
// stay in the HBM frame ring and remain readable for replay_capacity further steps. ----
class BreakoutState {
public:
    BreakoutState(std::shared_ptr<EnvHandle> env, uint64_t time, uint32_t k) : env_(std::move(env)), time_(time), k_(k) {}

    std::array<uint64_t, 3> dims() const { return {QLC_FRAME_W, QLC_FRAME_H, QLC_NUM_FRAMES}; }   // model_dims :148

    // ToMultiDimArray::to_multi_dim_array (:42-54): [x][y][slot] f32, value = u8 as f32
    Tensor to_multi_dim_array() const {
        const std::shared_ptr<BreakoutState> self = std::make_shared<BreakoutState>(*this);
        Tensor t = batch_to_multi_dim_array<1>({&self});
        t.dims.erase(t.dims.begin());
        return t;
    }

    // ToMultiDimArray::batch_to_multi_dim_array (:56-77), `batch: &[&Rc<Self>; N]`: [b][x][y][slot] f32 — ONE gather kernel for
    // the batch; the stacks cross PCIe as u8 and are widened into the tensor by the library's host pool
    template <size_t N>
    static Tensor batch_to_multi_dim_array(const std::array<const std::shared_ptr<BreakoutState>*, N>& batch) {
        static_assert(N > 0, "empty batch");
        const BreakoutState& first = **batch[0];
        const size_t per = (size_t)QLC_FRAME_W * QLC_FRAME_H * QLC_NUM_FRAMES;
        Tensor t;
        t.dims = {N, QLC_FRAME_W, QLC_FRAME_H, QLC_NUM_FRAMES};
        t.data.resize(N * per);
        std::array<qlc_obs_handle, N> h;
        for (size_t b = 0; b < N; ++b) {
            const BreakoutState& s = **batch[b];
            if (s.env_ != first.env_) throw QlError("states of different environments in one batch");
            h[b] = s.raw();
        }
        check(qlc_obs_gather_host(first.env_->get(), h.data(), (uint32_t)N, QLC_LAYOUT_F32_BXYH, t.data.data()));
        return t;
    }

    std::string one_line_info() const {                            // DebugVisualizer :81-89 (the env's current mechanics)
        float cx = 0, cy = 0, pmin = 0, pmax = 0; uint64_t bricks = 0;
        qlc_state_host sh{};
        sh.ball_cx = &cx; sh.ball_cy = &cy; sh.pad_min_x = &pmin; sh.pad_max_x = &pmax; sh.bricks = &bricks;
        check(qlc_env_read_state(env_->get(), &sh));
        return "Breakout [" + std::to_string(__builtin_popcountll(bricks)) + " bricks, ball_pos: [" + std::to_string(cx) + " " +
               std::to_string(cy) + "], panel_pos: [" + std::to_string((pmin + pmax) / 2.0f) + " 570]]";
    }
    uint64_t time() const { return time_; }
    uint32_t k() const { return k_; }
    qlc_obs_handle raw() const { return qlc_obs_handle{time_, k_, 0u}; }
    const std::shared_ptr<EnvHandle>& env() const { return env_; }

private:
    std::shared_ptr<EnvHandle> env_;
    uint64_t time_;
    uint32_t k_;
};

// ---- Environment (prelude.rs:21-63) for ONE Breakout env: the drop-in the unchanged learner drives ----
class BreakoutEnvironment {
public:
    using S = BreakoutState;
    using A = BreakoutAction;

    // BreakoutEnvironment::new(frame_size_x, frame_size_y) (:139-153). history_buffer_len = Parameter::history_buffer_len of the
    // learner that will hold the handles (default: Parameter::default(), self_driving_tf_q_learner.rs:59).
    BreakoutEnvironment(uint32_t frame_size_x, uint32_t frame_size_y, uint64_t history_buffer_len = 1000000, uint64_t seed = 0, int32_t device = 0) {
        qlc_config cfg{};
        cfg.struct_size = sizeof cfg; cfg.device = device; cfg.n_envs = 1; cfg.env_id_base = 0;
        cfg.frame_w = frame_size_x; cfg.frame_h = frame_size_y; cfg.seed = seed; cfg.replay_capacity = history_buffer_len;
        cfg.max_episode_steps = 0; cfg.episode_window = 100; cfg.auto_reset = 0;     // the learner resets (learn_episode :142)
        env_ = std::make_shared<EnvHandle>(cfg);
        state_ = std::make_unique<BreakoutState>(env_, 0, 0);
    }

    void reset() {                                                  // :177-180
        check(qlc_env_reset(env_->get(), nullptr, nullptr));
        state_ = std::make_unique<BreakoutState>(env_, env_->time(), 0);
    }
    const S& state() const { return *state_; }                      // :182
    std::shared_ptr<S> state_as_rc() const { return std::make_shared<S>(*state_); }   // prelude.rs:36

    std::tuple<const S&, float, bool> step(A action) {              // :184-201
        const uint8_t a = BreakoutActionTrait::numeric(action);
        float reward = 0.0f; uint8_t done = 0;
        check(qlc_env_step_host(env_->get(), &a, 1, &reward, &done));
        state_ = std::make_unique<BreakoutState>(env_, state_->time() + 1, state_->k() + 1);
        return {*state_, reward, done != 0};
    }
    std::tuple<std::shared_ptr<S>, float, bool> step_as_rc(A action) {   // prelude.rs:52-58
        auto [s, r, d] = step(action);
        return {std::make_shared<S>(s), r, d};
    }
    float episode_reward_goal_mean() const { return qlc_env_goal_mean(); }   // :203-206
    // 1 while the episode runs, 0 once it is over: the reference game ends with the first miss (mechanics.rs:131-135)
    uint8_t lives() const { uint8_t l = 0; check(qlc_env_lives_host(env_->get(), &l)); return l; }

    const std::shared_ptr<EnvHandle>& handle() const { return env_; }

private:
    std::shared_ptr<EnvHandle> env_;
    std::unique_ptr<BreakoutState> state_;
};

// ---- Buffer<T>, ReplayBuffer<S, A>, BufferSample (replay_buffer.rs:5-146): generic over the state type exactly like the
// reference. With S = std::shared_ptr<BreakoutState> (the learner's Rc<E::S>, self_driving_tf_q_learner.rs:81) the buffers hold
// handles and scalars; no pixel ever lives here. ----
template <class T>
struct Buffer {
    size_t max_buffer_len;
    std::deque<T> buffer;

    explicit Buffer(size_t max_len) : max_buffer_len(max_len) { if (max_len == 0) throw QlError("max_buffer_len must be > 0"); }
    size_t len() const { return buffer.size(); }
    void add(T element) {
        if (buffer.size() >= max_buffer_len) buffer.pop_front();
        buffer.push_back(std::move(element));
    }
    template <size_t N>
    std::array<const T*, N> get_many(const std::array<size_t, N>& indices) const {        // [&T; N]
        std::array<const T*, N> out;
        for (size_t i = 0; i < N; ++i) out[i] = &buffer.at(indices[i]);
        return out;
    }
    template <size_t N>
    std::array<T, N> get_many_as_val(const std::array<size_t, N>& indices) const {        // [T; N], T: Copy
        std::array<T, N> out;
        for (size_t i = 0; i < N; ++i) out[i] = buffer.at(indices[i]);
        return out;
    }
};

template <size_t N, class S, class A>
struct BufferSample {
    std::array<const S*, N> state;
    std::array<const S*, N> state_next;
    std::array<float, N> reward;
    std::array<A, N> action;
    std::array<bool, N> done;
};

template <class S, class A>
class ReplayBuffer {
public:
    ReplayBuffer(size_t step_buffer_len, size_t episode_reward_buffer_len)                       // :69-81
        : action_history(step_buffer_len), state_history(step_buffer_len), state_next_history(step_buffer_len), reward_history(step_buffer_len),
          done_history(step_buffer_len), episode_reward_history(episode_reward_buffer_len) {}
    size_t len() const { return done_history.len(); }                                             // :83
    void add(A action, S state, S state_next, float reward, bool done) {                          // :85-98
        action_history.add(action); state_history.add(std::move(state)); state_next_history.add(std::move(state_next));
        reward_history.add(reward); done_history.add(done);
    }
    void add_episode_reward(float r) { episode_reward_history.add(r); }                           // :100-105
    float avg_episode_reward() const {                                                            // :107-111
        if (episode_reward_history.len() == 0) throw QlError("episode reward history is empty", QLC_ERR_NOT_ENOUGH);
        float sum = 0.0f;
        for (float v : episode_reward_history.buffer) sum = sum + v;
        return sum / (float)episode_reward_history.len();
    }
    float min_episode_reward() const {                                                            // :113-120
        if (episode_reward_history.len() == 0) throw QlError("episode reward history is empty", QLC_ERR_NOT_ENOUGH);
        float mn = episode_reward_history.buffer.front();
        for (float v : episode_reward_history.buffer) if (v < mn) mn = v;
        return mn;
    }
    const Buffer<A>& actions() const { return action_history; }                                   // :122
    std::vector<float> episode_rewards() const { return {episode_reward_history.buffer.begin(), episode_reward_history.buffer.end()}; }   // :124
    template <size_t N>
    BufferSample<N, S, A> get_many(const std::array<size_t, N>& indices) const {                  // :126-137
        return {state_history.template get_many<N>(indices), state_next_history.template get_many<N>(indices),
                reward_history.template get_many_as_val<N>(indices), action_history.template get_many_as_val<N>(indices),
                done_history.template get_many_as_val<N>(indices)};
    }

private:
    Buffer<A> action_history;
    Buffer<S> state_history, state_next_history;
    Buffer<float> reward_history;
    Buffer<bool> done_history;
    Buffer<float> episode_reward_history;
};

// generate_distinct_random_ids (self_driving_tf_q_learner.rs:276-296): the learner's own private function — BATCH_SIZE distinct
// uniform ids in [range_start, range_end) by rejection, on the host. It stays with the learner; only the pixel gather behind
// batch_to_multi_dim_array goes to the device. (The device-side equivalent for vectorised callers is qlc_replay_sample /
// qlc_replay_sample_gather.)
template <size_t BATCH_SIZE, class Rng>
std::array<size_t, BATCH_SIZE> generate_distinct_random_ids(Rng& rng, size_t range_start, size_t range_end) {
    if (range_end - range_start < BATCH_SIZE) throw QlError("range smaller than the batch", QLC_ERR_NOT_ENOUGH);
    std::array<size_t, BATCH_SIZE> result{};
    std::uniform_int_distribution<size_t> distribution(range_start, range_end - 1);
    for (size_t i = 0; i < BATCH_SIZE; ++i) {
        for (;;) {
            const size_t x = distribution(rng);
            bool seen = false;
            for (size_t j = 0; j < i; ++j) seen = seen || result[j] == x;
            if (!seen) { result[i] = x; break; }
        }
    }
    return result;
}

// ---- the inference half of DeepQLearningModel (ml_model/model.rs:29-77) on the library's tensor-core Q-network ----
// predict_action (:40-46) and batch_predict_max_future_reward (:48-57) for BreakoutState handles: the network reads the u8
// frames in the frame ring directly, no tensor is materialised. train() (:59-71) stays with the caller, who hands updated
// weights over with set_weights (ten f32 arrays in the Keras layouts, see qlc_qnet_weights).
class TensorCoreQModel {
public:
    TensorCoreQModel(const BreakoutEnvironment& env, const qlc_qnet_weights& weights) : env_(env.handle()) { check(qlc_qnet_create(env_->get(), &weights, &q_)); }
    ~TensorCoreQModel() { qlc_qnet_destroy(q_); }
    TensorCoreQModel(const TensorCoreQModel&) = delete;
    TensorCoreQModel& operator=(const TensorCoreQModel&) = delete;
    void set_weights(const qlc_qnet_weights& weights) { check(qlc_qnet_set_weights(q_, &weights)); }

    // The ten Keras arrays (f32 masters, layouts of qlc_qnet_weights) owned by the caller.
    struct Weights {
        std::vector<float> conv1_kernel = std::vector<float>(8 * 8 * 4 * 32), conv1_bias = std::vector<float>(32);
        std::vector<float> conv2_kernel = std::vector<float>(4 * 4 * 32 * 64), conv2_bias = std::vector<float>(64);
        std::vector<float> conv3_kernel = std::vector<float>(3 * 3 * 64 * 64), conv3_bias = std::vector<float>(64);
        std::vector<float> dense1_kernel = std::vector<float>((size_t)3136 * 512), dense1_bias = std::vector<float>(512);
        std::vector<float> dense2_kernel = std::vector<float>(512 * 3), dense2_bias = std::vector<float>(3);
        qlc_qnet_weights view() const {
            return {conv1_kernel.data(), conv1_bias.data(), conv2_kernel.data(), conv2_bias.data(), conv3_kernel.data(), conv3_bias.data(),
                    dense1_kernel.data(), dense1_bias.data(), dense2_kernel.data(), dense2_bias.data()};
        }
    };
    Weights weights() const {                                       // checkpoint / target sync (set_weights(w.view()))
        Weights w;
        const qlc_qnet_weights v = w.view();
        check(qlc_qnet_get_weights(q_, &v));
        return w;
    }
    // DeepQLearningModel::train (model.rs:59-71) on replay transitions by logical index (state and action read from the ring),
    // one Keras-Adam update with the given TD targets; returns the Huber loss before the update.
    float train_replay(const std::vector<uint32_t>& idx, const std::vector<float>& targets) {
        if (idx.size() != targets.size() || idx.empty()) throw QlError("train_replay: one target per index, at least one index");
        float loss = 0.0f;
        check(qlc_qnet_train_host(q_, idx.data(), (uint32_t)idx.size(), 1, targets.data(), nullptr, 0.0f, &loss));
        return loss;
    }

    BreakoutAction predict_action(const BreakoutState& state) const {
        uint8_t a = 0;
        q_values(state, &a);
        return BreakoutActionTrait::try_from_numeric(a);
    }
    std::array<float, 3> q_values(const BreakoutState& state, uint8_t* action = nullptr) const {
        std::array<float, 3> qv{};
        uint8_t a = 0;
        uint32_t idx = 0; int32_t which = 0;
        if (locate(state, &idx, &which)) check(qlc_qnet_forward_host(q_, &idx, 1, which, qv.data(), &a, nullptr));
        else check(qlc_qnet_forward_host(q_, nullptr, 1, 0, qv.data(), &a, nullptr));
        if (action) *action = a;
        return qv;
    }
    template <size_t N>
    std::array<float, N> batch_predict_max_future_reward(const std::array<const std::shared_ptr<BreakoutState>*, N>& batch) const {
        std::array<float, N> out{};
        for (int32_t which = 1; which >= 0; --which) {          // state_next rows (the usual case), then rows taken right after a reset
            std::vector<uint32_t> idx; std::vector<size_t> pos;
            for (size_t b = 0; b < N; ++b) {
                uint32_t i = 0; int32_t w = 0;
                if (locate(**batch[b], &i, &w)) { if (w == which) { idx.push_back(i); pos.push_back(b); } }
                else if (which == 1) { const auto q = q_values(**batch[b]); out[b] = std::max(q[0], std::max(q[1], q[2])); }
            }
            if (idx.empty()) continue;
            std::vector<float> mq(idx.size());
            check(qlc_qnet_forward_host(q_, idx.data(), (uint32_t)idx.size(), which, nullptr, nullptr, mq.data()));
            for (size_t j = 0; j < pos.size(); ++j) out[pos[j]] = mq[j];
        }
        return out;
    }

private:
    // A handle names the observation after `time` steps: `state_next` of the transition taken at time - 1 (k >= 1) or `state` of
    // the one taken at `time` (k = 0). false = the live observation right after a reset (no transition after it yet).
    bool locate(const BreakoutState& s, uint32_t* idx, int32_t* which) const {
        if (s.env() != env_) throw QlError("state of another environment");
        const uint64_t now = env_->time();
        if (s.time() == now && s.k() == 0) return false;
        uint64_t cap = 0, len = 0;
        check(qlc_replay_capacity(env_->get(), &cap)); check(qlc_replay_len(env_->get(), &len));
        const uint64_t oldest = now > cap ? now - cap : 0;
        const uint64_t t = s.k() >= 1 ? s.time() - 1 : s.time();
        *which = s.k() >= 1 ? 1 : 0;
        if (t < oldest || t - oldest >= len) throw QlError("stale state handle: its frames have left the frame ring", QLC_ERR_OUT_OF_RANGE);
        *idx = (uint32_t)(t - oldest);
        return true;
    }
    std::shared_ptr<EnvHandle> env_;
    qlc_qnet* q_ = nullptr;
};

}  // namespace ql
