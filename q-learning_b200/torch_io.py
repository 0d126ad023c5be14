"""Zero-copy hand-off of the hot path's outputs to a torch consumer (SURVEY.md §8f-2): the gather kernels write straight
into CUDA tensors that the model reads — no host round trip. torch is plumbing here (device memory + streams); every byte
is produced by the kernels in csrc/."""
import torch

from . import FRAME_H, FRAME_W, LAYOUT_F32_BXYH, LAYOUT_U8_BHYX, NUM_FRAMES, QlError


def _stream():
    return torch.cuda.current_stream().cuda_stream


class DeviceSampler:
    """Reusable device buffers for `n_batches` minibatches of `batch` transitions; `sample()` = ONE kernel launch
    (`qlc_replay_sample_gather`: the gather kernel draws the distinct indices itself) on torch's current stream, returns views
    on the buffers."""

    def __init__(self, replay, batch, n_batches=1, layout=LAYOUT_F32_BXYH, device=None):
        self.replay, self.batch, self.n_batches, self.layout = replay, batch, n_batches, layout
        dev = torch.device("cuda", replay._env.device if device is None else device)
        n = batch * n_batches
        if layout == LAYOUT_F32_BXYH:
            shape, dt = (n_batches, batch, FRAME_W, FRAME_H, NUM_FRAMES), torch.float32
        elif layout == LAYOUT_U8_BHYX:
            shape, dt = (n_batches, batch, NUM_FRAMES, FRAME_H, FRAME_W), torch.uint8
        else:
            raise QlError("unknown layout")
        self.indices = torch.empty((n_batches, batch), dtype=torch.int32, device=dev)
        self.state = torch.empty(shape, dtype=dt, device=dev)
        self.state_next = torch.empty(shape, dtype=dt, device=dev)
        self.reward = torch.empty((n_batches, batch), dtype=torch.float32, device=dev)
        self.action = torch.empty((n_batches, batch), dtype=torch.uint8, device=dev)
        self.done = torch.empty((n_batches, batch), dtype=torch.uint8, device=dev)

    def sample(self, call_index):
        self.replay.sample_gather_device(self.batch, self.n_batches, call_index, self.layout, self.indices.data_ptr(), self.state.data_ptr(),
                                         self.state_next.data_ptr(), self.reward.data_ptr(), self.action.data_ptr(), self.done.data_ptr(), _stream())
        return self


def observe(env, layout=LAYOUT_F32_BXYH, out=None):
    """Current observation stacks of all envs as a CUDA tensor (Environment::state + ToMultiDimArray, no host copy)."""
    dev = torch.device("cuda", env.device)
    if layout == LAYOUT_F32_BXYH:
        shape, dt = (env.n_envs, FRAME_W, FRAME_H, NUM_FRAMES), torch.float32
    else:
        shape, dt = (env.n_envs, NUM_FRAMES, FRAME_H, FRAME_W), torch.uint8
    if out is None:
        out = torch.empty(shape, dtype=dt, device=dev)
    env.obs_device(layout, out.data_ptr(), _stream())
    return out


def step(env, actions, reward=None, done=None):
    """One launch advancing all envs by actions.shape[0] steps; actions / reward / done are CUDA tensors [K][N]."""
    if actions.dtype != torch.uint8 or actions.dim() != 2 or actions.shape[1] != env.n_envs or not actions.is_contiguous():
        raise QlError("actions must be a contiguous u8 CUDA tensor [n_steps][n_envs]")
    k = actions.shape[0]
    if reward is None:
        reward = torch.empty((k, env.n_envs), dtype=torch.float32, device=actions.device)
    if done is None:
        done = torch.empty((k, env.n_envs), dtype=torch.uint8, device=actions.device)
    env.step_device(actions.data_ptr(), k, reward.data_ptr(), done.data_ptr(), _stream())
    return reward, done


def keras_weights_from_torch(net):
    """Weights of a torch network with the reference architecture (create_ql_model_breakout_84x84x4_3_32.py:17-33; convs in
    NCHW with H = x, W = y as in examples/dqn_breakout_torch.py) in the Keras layouts `QNetwork` takes (QNET_SHAPES)."""
    convs = [m for m in net.modules() if isinstance(m, torch.nn.Conv2d)]
    dense = [m for m in net.modules() if isinstance(m, torch.nn.Linear)]
    if len(convs) != 3 or len(dense) != 2:
        raise QlError("expected 3 Conv2d and 2 Linear layers")
    w = {}
    for i, c in enumerate(convs, 1):
        w["conv%d_kernel" % i] = c.weight.detach().permute(2, 3, 1, 0).contiguous().float().cpu().numpy()      # [cout][cin][kh][kw] -> [kh][kw][cin][cout]
        w["conv%d_bias" % i] = c.bias.detach().float().cpu().numpy()
    d1 = dense[0].weight.detach().float()                                                                      # [512][c*49 + x*7 + y]
    w["dense1_kernel"] = d1.view(512, 64, 7, 7).permute(2, 3, 1, 0).reshape(3136, 512).contiguous().cpu().numpy()   # Keras Flatten: (x*7 + y)*64 + c
    w["dense1_bias"] = dense[0].bias.detach().float().cpu().numpy()
    w["dense2_kernel"] = dense[1].weight.detach().float().t().contiguous().cpu().numpy()
    w["dense2_bias"] = dense[1].bias.detach().float().cpu().numpy()
    return w


class TensorCoreActor:
    """The inference half of DeepQLearningModel (ml_model/model.rs:29-77) on the library's tcgen05 Q-network, fed straight
    from the frame ring: `predict_action()` for every env without materialising the f32 observation, and
    `max_future_reward(indices)` for sampled transitions without gathering their state_next. Training stays with the
    caller's torch model; `sync(net)` copies its weights over (bf16 operands, f32 accumulation)."""

    def __init__(self, env, net):
        from . import QNetwork
        self.env = env
        self.qnet = QNetwork(env, keras_weights_from_torch(net))
        dev = torch.device("cuda", env.device)
        self.actions = torch.empty((1, env.n_envs), dtype=torch.uint8, device=dev)
        self.q = torch.empty((env.n_envs, 3), dtype=torch.float32, device=dev)

    def sync(self, net):
        self.qnet.set_weights(keras_weights_from_torch(net))

    def predict_action(self, states=None, want_q=False):
        """Greedy action of every env as a CUDA u8 tensor [1][n_envs] (the shape `step` takes); `states` is ignored — the
        network reads the frames where the step kernel wrote them."""
        self.qnet.forward_device(None, self.env.n_envs, 0, self.q.data_ptr() if want_q else None, self.actions.data_ptr(), None, _stream())
        return self.actions

    def max_future_reward(self, indices, out=None):
        """batch_predict_max_future_reward for the state_next of the replay transitions `indices` (CUDA int32 / uint32 tensor)."""
        n = indices.numel()
        if out is None:
            out = torch.empty((n,), dtype=torch.float32, device=indices.device)
        self.qnet.forward_device(indices.data_ptr(), n, 1, None, None, out.data_ptr(), _stream())
        return out

    def close(self):
        self.qnet.close()


class TensorCoreLearner:
    """The three DeepQLearningModel methods (ml_model/model.rs:29-77) on the library's tcgen05 Q-network, training included,
    with an online and a target (stabilized) network on the replay ring of `env`: `predict_action()` for every env,
    `train_indices(idx)` — `n_batches` Keras-Adam updates on replay transitions by index, the TD target
    y = r + max Q_target(s') * gamma (y = r where done) computed on the device — and `sync_target()`. No state tensor is
    materialised anywhere: the kernels read the u8 frames where the step kernel wrote them. `weights`: Keras-layout f32 arrays
    (QNET_SHAPES) for both networks. `per_alpha` (not None): prioritized replay over the same ring (PrioritizedReplay), used by
    `train_prioritized()`. `n_step` > 1 and `double_dqn`: both training calls bootstrap from n-step returns read from the ring
    (DESIGN.md §14) and, with `double_dqn`, take Q_target at the online network's greedy action instead of max Q_target."""

    def __init__(self, env, weights, gamma=0.99, lr=2.5e-4, clipnorm=1.0, per_alpha=None, per_epsilon=1e-6, n_step=1, double_dqn=False):
        from . import PrioritizedReplay, QNetwork
        self.env, self.gamma = env, float(gamma)
        self.n_step, self.double_dqn = int(n_step), bool(double_dqn)
        self.online = QNetwork(env, weights)
        self.target = QNetwork(env, weights)
        self.online.set_adam(lr=lr, clipnorm=clipnorm)
        self.per = None if per_alpha is None else PrioritizedReplay(env, per_alpha, per_epsilon)
        self._per_bufs = None
        dev = torch.device("cuda", env.device)
        self.actions = torch.empty((1, env.n_envs), dtype=torch.uint8, device=dev)
        self.losses = []

    def predict_action(self):
        """Greedy action of every env as a CUDA u8 tensor [1][n_envs] (the shape `step` takes)."""
        self.online.forward_device(None, self.env.n_envs, 0, None, self.actions.data_ptr(), None, _stream())
        return self.actions

    def train_indices(self, indices):
        """One update per row of `indices` (CUDA int32 / uint32 tensor [n_batches][batch], e.g. DeviceSampler.indices filled by
        ReplayBuffer.sample_device); returns the CUDA f32 tensor [n_batches] of losses, each before its update."""
        if indices.dim() != 2 or not indices.is_cuda or not indices.is_contiguous() or indices.dtype not in (torch.int32, torch.uint32):
            raise QlError("indices must be a contiguous int32 CUDA tensor [n_batches][batch]")
        nb, batch = indices.shape
        loss = torch.empty(nb, dtype=torch.float32, device=indices.device)
        if self._nstep_targets():
            self.online.train_nstep_device(indices.data_ptr(), None, batch, nb, self.target, self.gamma, self.n_step, self.double_dqn, loss.data_ptr(),
                                           None, None, _stream())
        else:
            self.online.train_device(indices.data_ptr(), batch, nb, None, self.target, self.gamma, loss.data_ptr(), _stream())
        self.losses.append(loss)
        return loss

    def train_prioritized(self, batch, n_batches, call_index, beta):
        """`n_batches` updates on minibatches of `batch` transitions drawn by priority, each weighted by its importance weights
        (exponent `beta`); the TD errors of the updates become the new priorities. Sample, train and update are queued on the
        current stream without a host synchronisation; returns the CUDA f32 tensor [n_batches] of weighted losses."""
        if self.per is None:
            raise QlError("this learner was created without per_alpha")
        dev = torch.device("cuda", self.env.device)
        if self._per_bufs is None or self._per_bufs[0].shape != (n_batches, batch):
            self._per_bufs = (torch.empty((n_batches, batch), dtype=torch.int32, device=dev), torch.empty((n_batches, batch), dtype=torch.float32, device=dev),
                              torch.empty((n_batches, batch), dtype=torch.float32, device=dev))
        idx, w, td = self._per_bufs
        s = _stream()
        loss = torch.empty(n_batches, dtype=torch.float32, device=dev)
        self.per.sample_device(batch, n_batches, call_index, beta, idx.data_ptr(), w.data_ptr(), s)
        if self._nstep_targets():
            self.online.train_nstep_device(idx.data_ptr(), w.data_ptr(), batch, n_batches, self.target, self.gamma, self.n_step, self.double_dqn,
                                           loss.data_ptr(), td.data_ptr(), None, s)
        else:
            self.online.train_weighted_device(idx.data_ptr(), w.data_ptr(), batch, n_batches, None, self.target, self.gamma, loss.data_ptr(), td.data_ptr(), s)
        self.per.update_device(idx.data_ptr(), td.data_ptr(), batch * n_batches, s)
        self.losses.append(loss)
        return loss

    def _nstep_targets(self):
        return self.n_step != 1 or self.double_dqn

    def sync_target(self):
        """target <- online (get + set of the f32 master weights)."""
        self.target.set_weights(self.online.get_weights())

    def get_weights(self):
        return self.online.get_weights()

    def write_checkpoint(self, path):
        """The online network's weights as an .npz of the Keras arrays (QNET_SHAPES names)."""
        import numpy as np
        np.savez(path, **self.online.get_weights())

    def error(self):
        """Sticky MMA time-out flags of both networks (0 = fine); synchronises."""
        return self.online.error() | self.target.error()

    def close(self):
        if self.per is not None:
            self.per.close()
        self.online.close()
        self.target.close()
