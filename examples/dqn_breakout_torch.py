#!/usr/bin/env python
"""End-to-end DQN on the B200 path: N Breakout envs + replay on the GPU (this repo) feeding a torch Q-network
(library code standing in for the reference's TensorFlow SavedModel — the model is OUT of this repo's scope).

Architecture and optimiser follow the reference's Keras definition
(/root/reference/src/ql-with-tensorflow/python_model/create_ql_model_breakout_84x84x4_3_32.py:10-33):
Conv(32, 8, stride 4) -> Conv(64, 4, stride 2) -> Conv(64, 3, stride 1) -> Dense 512 -> Dense 3, ReLU, Adam 2.5e-4 with
clipnorm 1, Huber loss; input [B, 84, 84, 4] f32 exactly as BreakoutState::batch_to_multi_dim_array lays it out
(x, y, ring slot; value 0..255, no scaling). The loop is q-learning_b200/learner.py (the vectorised twin of
SelfDrivingQLearner); observations and minibatches reach the model without leaving the device (torch_io.py).

    python examples/dqn_breakout_torch.py --envs 1024 --iterations 200
"""
import argparse
import importlib
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch
import torch.nn as nn

q = importlib.import_module("q-learning_b200")
L = importlib.import_module("q-learning_b200.learner")
tio = importlib.import_module("q-learning_b200.torch_io")


class QNet(nn.Module):
    def __init__(self, n_actions=3):
        super().__init__()
        self.body = nn.Sequential(
            nn.Conv2d(4, 32, 8, stride=4), nn.ReLU(), nn.Conv2d(32, 64, 4, stride=2), nn.ReLU(), nn.Conv2d(64, 64, 3, stride=1), nn.ReLU(),
            nn.Flatten(), nn.Linear(64 * 7 * 7, 512), nn.ReLU(), nn.Linear(512, n_actions))

    def forward(self, x_bxyh):                       # [B, 84, 84, 4] channels-last as the reference feeds Keras
        return self.body(x_bxyh.permute(0, 3, 1, 2))


class TorchDQNModel:
    """The three DeepQLearningModel methods (ml_model/model.rs:29-77) on CUDA tensors."""

    def __init__(self, device, lr=2.5e-4):
        self.net = QNet().to(device).to(memory_format=torch.channels_last)
        self.opt = torch.optim.Adam(self.net.parameters(), lr=lr)
        self.loss_fn = nn.HuberLoss()
        self.losses = []

    @torch.no_grad()
    def predict_action(self, states):
        return self.net(states).argmax(dim=1).to(torch.uint8)

    @torch.no_grad()
    def batch_predict_max_future_reward(self, states):
        return self.net(states).max(dim=1).values

    def train(self, state_batch, action_batch, updated_q_values):
        qv = self.net(state_batch).gather(1, action_batch.long().unsqueeze(1)).squeeze(1)
        loss = self.loss_fn(qv, updated_q_values)
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        nn.utils.clip_grad_norm_(self.net.parameters(), 1.0)          # clipnorm=1.0
        self.opt.step()
        self.losses.append(loss.detach())

    def load_from(self, other):
        self.net.load_state_dict(other.net.state_dict())


def run(n_envs=1024, iterations=200, batch=32, minibatches_per_call=None, seed=0, device=0, quiet=False, tensor_core_actor=False, actor_sync_every=10,
        env_id_base=0, skip_model=False, random_phase_steps=None, tensor_core_learner=False, target_sync_every=250, prioritized=False,
        n_step=1, double_dqn=False):
    """Device-resident variant of learner.SelfDrivingQLearner.learn_iteration: same rules, tensors never leave the GPU.
    skip_model: run the data path only (step, replay insert, sample + gather, TD-target inputs) without the network calls —
    what is left of an iteration when the learner costs nothing (bench.py uses it to attribute the iteration time).
    tensor_core_learner: the whole model on the library (torch_io.TensorCoreLearner): greedy actions and training on the
    tcgen05 Q-network; minibatches are drawn by qlc_replay_sample into an index tensor (no gather, no state tensor) and
    trained by qlc_qnet_train (one update per call on all of them, like the torch path) with the TD target from the target
    network, which follows every `target_sync_every` iterations.
    prioritized (with tensor_core_learner): proportional prioritized replay (alpha 0.6) instead of uniform minibatches — one
    stratified minibatch of the same nb * batch items per iteration, importance weights with beta annealed linearly from 0.4 to
    1.0 over the run, priorities updated from the TD errors of the update.
    n_step, double_dqn: TD targets from n-step returns read from the replay ring (qlc_replay_nstep), bootstrapped from the
    state_next of the last transition walked; double_dqn takes Q_target there at the online network's greedy action instead of
    max Q_target. The tensor-core learner computes them on the device; the torch learner gathers the bootstrap states and forms
    y = G + disc * Q_boot in torch. n_step=1 without double_dqn is the one-step target above."""
    if prioritized and not tensor_core_learner:
        raise ValueError("prioritized replay runs on the tensor-core learner (tensor_core_learner=True)")
    dev = torch.device("cuda", device)
    torch.cuda.set_device(dev)
    p = L.Parameter(history_buffer_len=n_envs * 128, epsilon_pure_random_steps=n_envs * 20 if random_phase_steps is None else random_phase_steps,
                    epsilon_greedy_steps=float(n_envs * 400), max_steps_per_episode=10_000)
    env = q.BreakoutEnvironment(n_envs=n_envs, seed=seed, env_id_base=env_id_base, replay_capacity=p.history_buffer_len,
                                max_episode_steps=p.max_steps_per_episode, device=device)
    rb = q.ReplayBuffer(env)
    model, target = TorchDQNModel(dev), TorchDQNModel(dev)
    target.load_from(model)
    learner = tio.TensorCoreLearner(env, tio.keras_weights_from_torch(model.net), gamma=p.gamma.item(), per_alpha=0.6 if prioritized else None,
                                    n_step=n_step, double_dqn=double_dqn) if tensor_core_learner else None
    # optional: action selection on the library's tcgen05 Q-network, reading the frame ring directly (no f32 observation
    # is materialised); its weights follow the torch model every `actor_sync_every` iterations
    actor = tio.TensorCoreActor(env, model.net) if tensor_core_actor else None
    due_per_iter = n_envs // p.update_after_actions               # one minibatch per 4 env-steps (self_driving_tf_q_learner.rs:181)
    nb = minibatches_per_call or due_per_iter
    if learner is None:
        sampler = tio.DeviceSampler(rb, batch, nb, q.LAYOUT_F32_BXYH)
        if n_step != 1 or double_dqn:
            n_ret, n_disc = (torch.empty(nb * batch, dtype=torch.float32, device=dev) for _ in range(2))
            n_boot = torch.empty(nb * batch, dtype=torch.int32, device=dev)
    else:
        idx = torch.empty((nb, batch), dtype=torch.int32, device=dev)
    gen = torch.Generator(device=dev); gen.manual_seed(seed)
    obs = None
    epsilon, delta = p.epsilon_max, p.epsilon_interval() / p.epsilon_greedy_steps
    step_count, calls, returns = 0, 0, torch.zeros(n_envs, device=dev)
    finished_returns = []
    t0 = time.time()
    for it in range(iterations):
        a_rand = torch.randint(0, 3, (1, n_envs), dtype=torch.uint8, device=dev, generator=gen)
        u = torch.rand(n_envs, device=dev, generator=gen)
        eps = torch.clamp(epsilon - torch.arange(n_envs, device=dev) * delta, min=p.epsilon_min)
        random_mask = (eps > u) | (step_count + 1 + torch.arange(n_envs, device=dev) < p.epsilon_pure_random_steps)
        actions = a_rand
        if not skip_model and not bool(random_mask.all()):
            if learner is not None:
                greedy = learner.predict_action()[0]
            elif actor is not None:
                if it % actor_sync_every == 0:
                    actor.sync(model.net)
                greedy = actor.predict_action()[0]
            else:
                obs = tio.observe(env, q.LAYOUT_F32_BXYH, obs)
                greedy = model.predict_action(obs)
            actions = torch.where(random_mask, a_rand[0], greedy).unsqueeze(0).contiguous()
        epsilon = max(epsilon - n_envs * delta, p.epsilon_min)
        reward, done = tio.step(env, actions)
        returns += reward[0]
        step_count += n_envs
        if rb.len() > batch:
            for _ in range(max(1, due_per_iter // nb)):
                if prioritized:
                    if not skip_model:
                        learner.train_prioritized(nb * batch, 1, calls, 0.4 + 0.6 * it / max(1, iterations - 1))
                    calls += nb
                    continue
                if learner is not None:
                    rb.sample_device(batch, nb, calls, idx.data_ptr(), tio._stream()); calls += nb
                    if not skip_model:
                        learner.train_indices(idx.view(1, -1))     # one update on the nb minibatches together, as the torch model trains them
                    continue
                s = sampler.sample(calls); calls += nb
                st, nx = s.state.view(nb * batch, 84, 84, 4), s.state_next.view(nb * batch, 84, 84, 4)
                if skip_model:
                    continue
                if n_step != 1 or double_dqn:
                    # G, disc and the bootstrap index of every sampled transition; its state_next replaces the sampled one
                    rb.nstep_device(s.indices.data_ptr(), nb * batch, n_step, p.gamma.item(), n_ret.data_ptr(), n_disc.data_ptr(), n_boot.data_ptr(), tio._stream())
                    rb.gather_device(n_boot.data_ptr(), nb * batch, q.LAYOUT_F32_BXYH, None, s.state_next.data_ptr(), stream=tio._stream())
                    with torch.no_grad():
                        if double_dqn:
                            a_star = model.predict_action(nx).long()
                            q_boot = target.net(nx).gather(1, a_star.unsqueeze(1)).squeeze(1)
                        else:
                            q_boot = target.batch_predict_max_future_reward(nx)
                    updated_q = n_ret + n_disc * q_boot
                else:
                    max_future = target.batch_predict_max_future_reward(nx)
                    rwd, dn = s.reward.view(-1), s.done.view(-1)
                    updated_q = torch.where(dn != 0, rwd, rwd + p.gamma.item() * max_future)      # TD target (:192-199)
                model.train(st, s.action.view(-1), updated_q)
        if learner is not None and (it + 1) % target_sync_every == 0:
            learner.sync_target()
        ended = done[0] != 0
        if bool(ended.any()):
            finished_returns.extend(returns[ended].tolist()); returns[ended] = 0
        if (it + 1) % 50 == 0 and not quiet:
            torch.cuda.synchronize()
            print("iter %d  env-steps %d  eps %.3f  loss %.4f  episodes %d  mean return %.2f  %.0f env-steps/s" % (
                it + 1, step_count, epsilon, float(torch.cat([x.reshape(-1) for x in (learner.losses if learner else model.losses)[-20:]]).mean())
                if (learner.losses if learner else model.losses) else float("nan"),
                len(finished_returns), float(np.mean(finished_returns[-500:])) if finished_returns else float("nan"), step_count / (time.time() - t0)), flush=True)
    torch.cuda.synchronize()
    stats = env.stats()
    losses = model.losses if learner is None else learner.losses
    out = {"env_steps": step_count, "seconds": time.time() - t0, "episodes": int(stats["episodes"]), "train_calls": len(losses), "minibatches": calls,
           "last_loss": float(losses[-1].reshape(-1)[-1]) if losses else None, "epsilon": epsilon, "error_flags": env.error_flags()}
    if learner is not None:
        out["losses_finite"] = bool(all(torch.isfinite(x).all() for x in learner.losses))
        out["qnet_error"] = learner.error()
        if learner.per is not None:
            out["per_leaves"], out["per_total"], out["per_max"] = learner.per.read()      # logical order; the ring is at env.time()
            out["env_time"] = env.time()
        learner.close()
    if actor is not None:
        actor.close()
    env.close()
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--iterations", type=int, default=200)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--tensor-core-learner", action="store_true", help="the whole model on the library: greedy actions and training (qlc_qnet_train) "
                    "on its tcgen05 Q-network, minibatches sampled as indices only")
    ap.add_argument("--tensor-core-actor", action="store_true", help="greedy actions from the library's tcgen05 Q-network (weights synced from the torch model)")
    ap.add_argument("--prioritized", action="store_true", help="with --tensor-core-learner: proportional prioritized replay (alpha 0.6, beta 0.4 -> 1.0)")
    ap.add_argument("--n-step", type=int, default=1, help="TD targets from n-step returns read from the replay ring (1 = one-step)")
    ap.add_argument("--double-dqn", action="store_true", help="double-DQN targets: Q_target at the online network's greedy action")
    args = ap.parse_args()
    if args.prioritized and not args.tensor_core_learner:
        ap.error("--prioritized needs --tensor-core-learner")
    print(run(args.envs, args.iterations, args.batch, tensor_core_actor=args.tensor_core_actor, tensor_core_learner=args.tensor_core_learner,
              prioritized=args.prioritized, n_step=args.n_step, double_dqn=args.double_dqn))
