"""Q-network training on the device (qlc_qnet_train): the reference's DeepQLearningModel::train for the Keras model —
Huber(delta 1) on Q(s)[a] averaged over the minibatch, clipnorm 1 per variable, Keras 2.12 Adam. Gradients are compared
with torch autograd on the same bf16-quantised forward; the optimizer step with float64 numpy on the library's own
gradients (an update is deterministic, so they are the bits the update used)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KERAS_ADAM = dict(lr=2.5e-4, beta1=0.9, beta2=0.999, epsilon=1e-7)


def _random_weights(qlb, seed):
    rng = np.random.default_rng(seed)
    w = {}
    for name, shape in qlb.QNET_SHAPES.items():
        if name.endswith("kernel"):
            fan_in = int(np.prod(shape[:-1])); fan_out = shape[-1]
            lim = np.sqrt(6.0 / (fan_in + fan_out))                      # Keras default glorot_uniform
            w[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)
        else:
            w[name] = rng.uniform(-0.1, 0.1, size=shape).astype(np.float32)
    return w


def _replay(qlb, n_envs=300, seed=5):
    """An env whose replay holds episode starts (zero-filled ring slots) and partially filled stacks."""
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=n_envs * 64)
    rng = np.random.default_rng(seed)
    env.step_many(rng.integers(0, 3, size=(30, n_envs), dtype=np.uint8))
    env.reset(mask=(np.arange(n_envs) % 7 == 0).astype(np.uint8))
    env.step_many(rng.integers(0, 3, size=(10, n_envs), dtype=np.uint8))
    return env, qlb.ReplayBuffer(env)


def _torch_loss(torch, w, obs_bxyh, action, target, quantise):
    """Huber loss of the Keras model on [B, 84(x), 84(y), 4(slot)] as an fp32 torch graph over leaf tensors `w` (Keras
    layouts); quantise=True rounds weights and the activations between layers to bf16 at the points of the tensor-core
    forward (the rounding passes the gradient through unchanged, as it does on the device)."""
    F = torch.nn.functional
    bf = (lambda t: t.to(torch.bfloat16).to(torch.float32)) if quantise else (lambda t: t)
    x = torch.from_numpy(obs_bxyh).permute(0, 3, 1, 2).contiguous()
    for i in (1, 2, 3):
        k = bf(w["conv%d_kernel" % i].permute(3, 2, 0, 1))
        x = bf(torch.relu(F.conv2d(x, k, w["conv%d_bias" % i], stride={1: 4, 2: 2, 3: 1}[i])))
    x = x.permute(0, 2, 3, 1).reshape(x.shape[0], -1)
    x = bf(torch.relu(x @ bf(w["dense1_kernel"]) + w["dense1_bias"]))
    q = x @ w["dense2_kernel"] + w["dense2_bias"]
    qa = q.gather(1, torch.from_numpy(action.astype(np.int64)).unsqueeze(1)).squeeze(1)
    return torch.nn.functional.huber_loss(qa, torch.from_numpy(target), delta=1.0)


def _torch_grads(torch, w_np, obs, action, target, quantise):
    w = {k: torch.from_numpy(v.copy()).requires_grad_(True) for k, v in w_np.items()}
    _torch_loss(torch, w, obs, action, target, quantise).backward()
    return {k: w[k].grad.numpy().astype(np.float64) for k in w}


def _saturating_targets(net, idx, sample, seed):
    """Targets at least 2 from the library's Q(s)[a]: the Huber gradient is then +-1/batch on both sides, so forward
    rounding differences do not reach dL/dq."""
    q, _, _ = net.forward(idx, 0)
    qa = q[np.arange(idx.size), sample.action.astype(np.int64)]
    rng = np.random.default_rng(seed)
    return (qa + rng.choice([-1.0, 1.0], size=idx.size) * (2.0 + rng.uniform(0, 1, size=idx.size))).astype(np.float32)


@pytest.mark.parametrize("batch", [1, 32, 300, 2000])
def test_gradients_match_torch_autograd(qlb, batch):
    """Per variable ||g - g_ref|| <= tol * ||g_ref||. Tolerances: against autograd on the forward quantised at the same
    points 2e-2 — the backward rounds its GEMM operands (the back-propagated gradients) to bf16, 2^-9 relative each, through
    up to four layers, plus accumulation order; against pure fp32 1.5e-1 — the bf16 forward itself moves activations and
    ReLU masks (the forward test allows 4e-2 of max|Q| on Q alone)."""
    torch = pytest.importorskip("torch")
    env, rb = _replay(qlb)
    w = _random_weights(qlb, 3)
    net = qlb.QNetwork(env, w)
    idx = np.random.default_rng(batch).choice(rb.len(), size=batch, replace=False).astype(np.uint32)
    smp = rb.get_many(idx, qlb.LAYOUT_F32_BXYH)
    y = _saturating_targets(net, idx, smp, batch)
    g = net.debug_grads(idx, y)
    ref_q = _torch_grads(torch, w, smp.state, smp.action, y, quantise=True)
    ref_f = _torch_grads(torch, w, smp.state, smp.action, y, quantise=False)
    for name in qlb.QNET_SHAPES:
        assert np.all(np.isfinite(g[name])), name
        nref = np.linalg.norm(ref_q[name])
        assert nref > 0, name
        eq = np.linalg.norm(g[name] - ref_q[name]) / nref
        ef = np.linalg.norm(g[name] - ref_f[name]) / np.linalg.norm(ref_f[name])
        assert eq <= 2e-2, (name, eq)
        assert ef <= 1.5e-1, (name, ef)
    net.close(); env.close()


def test_replay_minibatch_includes_episode_starts(qlb):
    """The replay used by the gradient tests holds states with zero-filled ring slots (episode starts)."""
    env, rb = _replay(qlb)
    idx = np.random.default_rng(2000).choice(rb.len(), size=2000, replace=False).astype(np.uint32)
    st = rb.get_many(idx, qlb.LAYOUT_F32_BXYH).state
    assert (st.reshape(2000, -1, 4).max(axis=1) == 0).any()
    env.close()


def _keras_step(w, g, m, v, t, clipnorm, lr=2.5e-4, b1=0.9, b2=0.999, eps=1e-7):
    """Keras 2.12 Adam with per-variable clipnorm in float64 (m, v updated in place)."""
    alpha = lr * np.sqrt(1 - b2 ** t) / (1 - b1 ** t)
    out = {}
    for k in w:
        gk = g[k].astype(np.float64)
        nrm = np.sqrt(np.sum(gk * gk))
        if clipnorm > 0:
            gk = gk * clipnorm / max(nrm, clipnorm)
        m[k] += (gk - m[k]) * (1 - b1)
        v[k] += (gk * gk - v[k]) * (1 - b2)
        out[k] = w[k].astype(np.float64) - alpha * m[k] / (np.sqrt(v[k]) + eps)
    return out


def test_adam_step_matches_keras(qlb):
    """Each of five updates moves every weight by Keras Adam + per-variable clipnorm computed in float64 from the
    library's gradients, within f32 rounding: 2 ulp of the weight, plus 1e-3 of the step, plus 1e-4 of alpha_t for steps
    where m nearly cancels (the per-variable norm is an f32 sum of up to 1.6M squares, ~1e-5 relative). clipnorm is set between the
    variables' gradient norms so that some variables are clipped and others are not."""
    env, rb = _replay(qlb)
    net = qlb.QNetwork(env, _random_weights(qlb, 7))
    idx = rb.generate_distinct_random_ids(32, 1)
    smp = rb.get_many(idx, qlb.LAYOUT_F32_BXYH)
    y = (smp.reward + np.float32(0.5)).astype(np.float32)
    g0 = net.debug_grads(idx, y)
    norms = sorted(float(np.linalg.norm(g0[k].astype(np.float64))) for k in g0)
    clipnorm = float(np.float32((norms[4] + norms[5]) / 2))
    net.set_adam(clipnorm=clipnorm, **KERAS_ADAM)
    m = {k: np.zeros(s, np.float64) for k, s in qlb.QNET_SHAPES.items()}
    v = {k: np.zeros(s, np.float64) for k, s in qlb.QNET_SHAPES.items()}
    clipped = set()
    for t in range(1, 6):
        w = net.get_weights()
        g = net.debug_grads(idx, y)
        clipped |= {k for k in g if np.linalg.norm(g[k].astype(np.float64)) > clipnorm}
        exp = _keras_step(w, g, m, v, t, clipnorm)
        alpha = 2.5e-4 * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)
        net.train(idx, y)
        got = net.get_weights()
        for k in got:
            tol = 2 * np.spacing(np.abs(exp[k]).astype(np.float32)).astype(np.float64) + 1e-3 * np.abs(exp[k] - w[k]) + 1e-4 * alpha
            err = np.abs(got[k] - exp[k])
            assert np.all(err <= tol), (t, k, float(err.max()))
    assert 0 < len(clipped) < 10, clipped
    net.close(); env.close()


def test_td_target_is_bit_identical_to_numpy(qlb):
    """The on-device target y = r + maxQ_target(s') * gamma (y = r where done) gives the same update bits as the numpy
    target of learner.py with maxQ from target.forward(idx, 1) and r / done from get_many."""
    env, rb = _replay(qlb)
    w0, wt = _random_weights(qlb, 1), _random_weights(qlb, 2)
    target = qlb.QNetwork(env, wt)
    a, b = qlb.QNetwork(env, w0), qlb.QNetwork(env, w0)
    idx = rb.generate_distinct_random_ids(64, 3)
    smp = rb.get_many(idx, qlb.LAYOUT_F32_BXYH)
    _, _, max_q = target.forward(idx, 1)
    gamma = np.float32(0.99)
    y = smp.reward + max_q * gamma
    y = np.where(smp.done != 0, smp.reward, y).astype(np.float32)
    la = a.train(idx, target_net=target, gamma=float(gamma))
    lb = b.train(idx, targets=y)
    assert np.array_equal(la.view(np.uint32), lb.view(np.uint32))
    wa, wb = a.get_weights(), b.get_weights()
    for k in wa:
        assert np.array_equal(wa[k].view(np.uint32), wb[k].view(np.uint32)), k
    for n in (a, b, target):
        n.close()
    env.close()


def test_sequential_minibatches_and_determinism(qlb):
    """One call with n_batches = 4 equals four calls with n_batches = 1, bit for bit, and two runs from the same seed and
    weights end in identical weight bits (no float atomics; fixed-order sums)."""
    def run(split):
        env, rb = _replay(qlb)
        tgt = qlb.QNetwork(env, _random_weights(qlb, 12))
        net = qlb.QNetwork(env, _random_weights(qlb, 11))
        idx = np.concatenate([rb.generate_distinct_random_ids(48, c) for c in range(4)])
        if split:
            loss = np.concatenate([net.train(idx[j * 48:(j + 1) * 48], target_net=tgt) for j in range(4)])
        else:
            loss = net.train(idx, target_net=tgt, n_batches=4)
        out = net.get_weights(), loss
        net.close(); tgt.close(); env.close()
        return out
    (w1, l1), (w2, l2), (w3, l3) = run(False), run(True), run(False)
    assert np.all(np.isfinite(l1))
    assert np.array_equal(l1.view(np.uint32), l2.view(np.uint32)) and np.array_equal(l1.view(np.uint32), l3.view(np.uint32))
    for k in w1:
        assert np.array_equal(w1[k].view(np.uint32), w2[k].view(np.uint32)), k
        assert np.array_equal(w1[k].view(np.uint32), w3[k].view(np.uint32)), k


def test_repeated_updates_reduce_the_loss_like_torch(qlb):
    """60 updates on one fixed minibatch with fixed targets cut the loss (mean of the last 10 steps) to below a quarter of
    its start, and a torch model with the same rules (fp32, Keras Adam form, per-variable clipnorm 1) on the same data does
    the same. lr = 5e-6: with unscaled 0..255 pixels and fresh Glorot weights the Keras model's 2.5e-4 overshoots on a
    single minibatch (both implementations). The curves, not the weights, are compared (Adam's first steps amplify the sign
    of near-zero gradients): means over windows of 10 steps agree within a factor 3."""
    torch = pytest.importorskip("torch")
    lr, steps = 5e-6, 60
    env, rb = _replay(qlb)
    w = _random_weights(qlb, 21)
    net = qlb.QNetwork(env, w)
    net.set_adam(lr=lr)
    idx = rb.generate_distinct_random_ids(32, 9)
    smp = rb.get_many(idx, qlb.LAYOUT_F32_BXYH)
    q, _, _ = net.forward(idx, 0)
    rng = np.random.default_rng(4)
    y = (q[np.arange(32), smp.action.astype(np.int64)] + rng.uniform(-3, 3, size=32)).astype(np.float32)
    lib = np.array([net.train(idx, y)[0] for _ in range(steps)], dtype=np.float64)
    tw = {k: torch.from_numpy(v.copy()).requires_grad_(True) for k, v in w.items()}
    m = {k: torch.zeros_like(v) for k, v in tw.items()}
    v2 = {k: torch.zeros_like(v) for k, v in tw.items()}
    ref = []
    for t in range(1, steps + 1):
        for p in tw.values():
            p.grad = None
        loss = _torch_loss(torch, tw, smp.state, smp.action, y, quantise=False)
        loss.backward()
        ref.append(float(loss.detach()))
        alpha = lr * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)
        with torch.no_grad():
            for k, p in tw.items():
                gk = p.grad * 1.0 / torch.clamp(p.grad.norm(), min=1.0)
                m[k] += (gk - m[k]) * (1 - 0.9)
                v2[k] += (gk * gk - v2[k]) * (1 - 0.999)
                p -= (m[k] * alpha) / (torch.sqrt(v2[k]) + 1e-7)
    ref = np.array(ref)
    assert np.all(np.isfinite(lib))
    assert abs(lib[0] - ref[0]) <= 0.05 * ref[0], (lib[0], ref[0])        # same start (bf16 forward)
    wl, wr = lib.reshape(-1, 10).mean(axis=1), ref.reshape(-1, 10).mean(axis=1)
    assert wl[-1] < lib[0] / 4 and wr[-1] < ref[0] / 4, (wl, wr)
    assert np.all((wl / wr > 1 / 3) & (wl / wr < 3)), (wl, wr)
    net.close(); env.close()


def test_weight_round_trip_and_errors(qlb):
    """set_weights -> get_weights is bit-exact; bad arguments are QLC_ERR_INVALID_ARG; training after the env is
    destroyed is an error, not a crash."""
    env, rb = _replay(qlb, n_envs=64)
    w = _random_weights(qlb, 30)
    net = qlb.QNetwork(env, w)
    got = net.get_weights()
    for k in w:
        assert np.array_equal(got[k].view(np.uint32), w[k].view(np.uint32)), k
    idx = rb.generate_distinct_random_ids(32, 0)
    y = np.zeros(32, np.float32)
    with pytest.raises(qlb.QlError) as e:
        net.train(np.array([rb.len()], np.uint32), np.zeros(1, np.float32))
    assert e.value.code == qlb.ERR_INVALID_ARG
    with pytest.raises(qlb.QlError) as e:
        net.train(idx)                                                   # neither targets nor a target network
    assert e.value.code == qlb.ERR_INVALID_ARG
    env2, _ = _replay(qlb, n_envs=64, seed=6)
    other = qlb.QNetwork(env2, w)
    with pytest.raises(qlb.QlError) as e:
        net.train(idx, target_net=other)
    assert e.value.code == qlb.ERR_INVALID_ARG
    with pytest.raises(qlb.QlError) as e:
        net.train(np.zeros(0, np.uint32), np.zeros(0, np.float32))   # batch 0
    assert e.value.code == qlb.ERR_INVALID_ARG
    net.train(idx, y)
    assert net.error() == 0
    env.close()
    with pytest.raises(qlb.QlError) as e:
        net.train(idx, y)
    assert "destroyed" in str(e.value)
    net.close(); other.close(); env2.close()


def test_huber_quadratic_and_linear_branches(qlb):
    """dL/dq_a = clip(q_a - y, -1, 1) / batch and the loss = mean Huber(q_a - y), checked exactly against float64 numpy on
    the library's own Q(s)[a] with targets that put about half the items inside |d| < 1 (quadratic branch) and half
    outside: the dense-2 bias gradient is sum over items with a = j of dL/dq_a, which depends on nothing deeper. Tolerance:
    f32 summation of 64 terms, 1e-6 relative (+1e-9)."""
    env, rb = _replay(qlb)
    net = qlb.QNetwork(env, _random_weights(qlb, 41))
    idx = rb.generate_distinct_random_ids(64, 17)
    smp = rb.get_many(idx, qlb.LAYOUT_F32_BXYH)
    q, _, _ = net.forward(idx, 0)
    a = smp.action.astype(np.int64)
    qa = q[np.arange(64), a]
    y = (qa - np.random.default_rng(3).uniform(-2.5, 2.5, size=64)).astype(np.float32)
    d = (qa - y).astype(np.float64)
    assert 10 < np.count_nonzero(np.abs(d) < 1) < 54
    g = net.debug_grads(idx, y)
    exp_db5 = np.array([np.sum(np.clip(d[a == j], -1, 1)) / 64 for j in range(3)])
    assert np.all(np.abs(g["dense2_bias"] - exp_db5) <= 1e-6 * np.abs(exp_db5) + 1e-9), (g["dense2_bias"], exp_db5)
    exp_loss = np.mean(np.where(np.abs(d) <= 1, 0.5 * d * d, np.abs(d) - 0.5))
    loss = net.train(idx, y)[0]
    assert abs(loss - exp_loss) <= 1e-6 * exp_loss, (loss, exp_loss)
    net.close(); env.close()


def test_closed_loop_example_with_tensor_core_learner(qlb):
    """examples/dqn_breakout_torch.py --tensor-core-learner at 1,024 envs for 20 iterations: greedy actions, index-only
    sampling and training all on the library; every loss is finite, no env error flag, no MMA time-out."""
    import importlib.util
    import os
    pytest.importorskip("torch")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("dqn_breakout_torch", os.path.join(root, "examples", "dqn_breakout_torch.py"))
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    out = ex.run(n_envs=1024, iterations=20, quiet=True, random_phase_steps=0, tensor_core_learner=True, target_sync_every=5)
    assert out["train_calls"] == 20 and out["minibatches"] == 20 * 256, out
    assert out["losses_finite"] and np.isfinite(out["last_loss"]), out
    assert out["error_flags"] == 0 and out["qnet_error"] == 0, out
