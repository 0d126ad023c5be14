"""Prioritized replay on the device (qlc_per_*, qlc_qnet_train_weighted). The sum tree, the stratified descent and the
importance weights are rebuilt in numpy from the leaves the library reports (a numpy Philox4x32-10 checked against the
Random123 answer oracle/selftest.c pins; the summation and descent order of DESIGN.md §13), so everything downstream of the
leaves is compared bit for bit."""
import numpy as np
import pytest

from test_qnet_train import _random_weights, _replay, _saturating_targets

pytestmark = pytest.mark.gpu

N_ENVS, T_CAP = 64, 16
TIME_SLOTS = T_CAP + 4
STREAM_PRIORITY = 0x5052494F
M32 = np.uint64(0xFFFFFFFF)


# ---------------------------------------------------------------- numpy reference
def philox4x32_10(c0, c1, c2, c3, key):
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in (c0, c1, c2, c3)]
    c = np.broadcast_arrays(*c)
    c = [x.copy() for x in c]
    k0, k1 = np.uint64(key & 0xFFFFFFFF), np.uint64(key >> 32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return [x.astype(np.uint32) for x in c]


def test_numpy_philox_matches_random123():
    r = philox4x32_10(0, 0, 0, 0, 0)
    assert [int(x) for x in r] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]


def ring_window(t):
    oldest = t - T_CAP if t > T_CAP else 0
    return oldest, (t - oldest) * N_ENVS


def physical_leaves(leaves, t, n_envs=N_ENVS, t_cap=T_CAP):
    """the leaves in the ring's layout [time_slots][n_envs] (0 outside the replay) from their logical order"""
    ts = t_cap + 4
    oldest = t - t_cap if t > t_cap else 0
    phys = np.zeros(ts * n_envs, dtype=np.float32)
    times = oldest + np.arange(leaves.size) // n_envs
    phys[(times % ts) * n_envs + np.arange(leaves.size) % n_envs] = leaves
    return phys


def tree_levels(phys):
    """levels[0] = leaves (f64), levels[k] = f64 nodes, each the sum of its 32 children added left to right from 0.0"""
    levels = [phys.astype(np.float64)]
    while levels[-1].size > 1 or len(levels) == 1:
        a = levels[-1]
        a = np.concatenate([a, np.zeros((-a.size) % 32)]).reshape(-1, 32)
        s = np.zeros(a.shape[0])
        for c in range(32):
            s = s + a[:, c]
        levels.append(s)
    return levels


def reference_sample(phys, t, batch, n_batches, call_index, seed, beta, n_envs=N_ENVS, t_cap=T_CAP):
    levels = tree_levels(phys)
    total = levels[-1][0]
    n = batch * n_batches
    item = np.arange(n, dtype=np.uint64)
    m, i = item // np.uint64(batch), item % np.uint64(batch)
    c = np.uint64(call_index) + m
    words = philox4x32_10(i >> np.uint64(2), c & M32, c >> np.uint64(32), STREAM_PRIORITY, seed)
    w32 = np.choose((i & np.uint64(3)).astype(np.int64), words)
    u = (i.astype(np.float64) + (w32.astype(np.float64) + 0.5) * 2.0 ** -32) * total / float(batch)
    node = np.zeros(n, dtype=np.int64)
    for level in range(len(levels) - 1, 0, -1):
        below = np.concatenate([levels[level - 1], np.zeros(32)])
        c0 = node * 32
        pick = np.full(n, -1, dtype=np.int64)
        last_nz = np.zeros(n, dtype=np.int64)
        for k in range(32):
            v = below[np.minimum(c0 + k, below.size - 1)]
            v = np.where(c0 + k < levels[level - 1].size, v, 0.0)
            last_nz = np.where(v > 0.0, k, last_nz)
            active = pick < 0
            take = active & (u < v)
            pick = np.where(take, k, pick)
            u = np.where(active & ~take, u - v, u)
        node = c0 + np.where(pick < 0, last_nz, pick)
    ts = t_cap + 4
    oldest = t - t_cap if t > t_cap else 0
    slot, e = node // n_envs, node % n_envs
    d = ((t - 1) % ts - slot) % ts
    T = t - 1 - d
    idx = ((T - oldest) * n_envs + e).astype(np.uint32)
    p = phys[node].reshape(n_batches, batch).astype(np.float64)
    wts = np.power(p.min(axis=1, keepdims=True) / p, np.float64(beta))
    return idx.reshape(n_batches, batch), wts, phys[node].reshape(n_batches, batch), total


def priority64(td, alpha, eps):
    return np.power(np.abs(td.astype(np.float64)) + np.float64(np.float32(eps)), np.float64(np.float32(alpha)))


# ---------------------------------------------------------------- fixtures
def _env(qlb, seed=7):
    return qlb.BreakoutEnvironment(n_envs=N_ENVS, seed=seed, replay_capacity=N_ENVS * T_CAP)


def _step(env, n, seed):
    env.step_many(np.random.default_rng(seed).integers(0, 3, size=(n, env.n_envs), dtype=np.uint8))


def _len(qlb, env):
    return qlb.ReplayBuffer(env).len()


def _check_tree(qlb, per, env, expect_len=None):
    """len(leaves) == replay len, and the root equals the numpy tree over the leaves placed in the ring's layout, exactly"""
    leaves, total, mx = per.read()
    t = env.time()
    _, n = ring_window(t)
    assert leaves.size == n == _len(qlb, env)
    if expect_len is not None:
        assert n == expect_len
    phys = physical_leaves(leaves, t)
    assert total == tree_levels(phys)[-1][0]
    return leaves, total, mx


def _update(torch, per, idx, td):
    i = torch.as_tensor(np.asarray(idx, dtype=np.int64).astype(np.int32), device="cuda")
    d = torch.as_tensor(np.asarray(td, dtype=np.float32), device="cuda")
    per.update_device(i.data_ptr(), d.data_ptr(), i.numel(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()


def _sample(torch, per, batch, n_batches, call_index, beta):
    i = torch.empty((n_batches, batch), dtype=torch.int32, device="cuda")
    w = torch.empty((n_batches, batch), dtype=torch.float32, device="cuda")
    per.sample_device(batch, n_batches, call_index, beta, i.data_ptr(), w.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return i.cpu().numpy().view(np.uint32), w.cpu().numpy()


# ---------------------------------------------------------------- 1. ring tracking
def test_tree_follows_the_ring(qlb, tmp_path):
    env = _env(qlb)
    per = qlb.PrioritizedReplay(env)
    leaves, total, mx = _check_tree(qlb, per, env, 0)
    assert total == 0.0 and mx == 1.0
    for steps, expect in ((5, 5), (11, 16), (7, 16), (1, 16), (3, 16), (30, 16)):     # not full, exactly full, wrapped, ..., > time_slots
        _step(env, steps, env.time())
        leaves, total, mx = _check_tree(qlb, per, env, expect * N_ENVS)
        assert np.all(leaves == mx) and mx == 1.0
    env.save(str(tmp_path / "ckpt"))
    torch = pytest.importorskip("torch")
    _update(torch, per, np.arange(0, 16 * N_ENVS, 3), np.linspace(0.0, 40.0, (16 * N_ENVS + 2) // 3))
    leaves, total, mx = _check_tree(qlb, per, env)
    assert mx > 1.0 and len(np.unique(leaves)) > 2
    _step(env, 2, 99)
    env.load(str(tmp_path / "ckpt"))                   # the ring goes back: every transition restarts at the running max
    leaves2, total2, mx2 = _check_tree(qlb, per, env, 16 * N_ENVS)
    assert mx2 == mx and np.all(leaves2 == mx)
    per.close(); env.close()


# ---------------------------------------------------------------- 2. exact sampling
@pytest.mark.parametrize("batch", [1, 32, 1000, 32768])
def test_sampling_matches_the_numpy_tree(qlb, batch):
    torch = pytest.importorskip("torch")
    env = _env(qlb, seed=11)
    _step(env, 27, 5)                                   # wrapped ring
    per = qlb.PrioritizedReplay(env)
    n = _len(qlb, env)
    rng = np.random.default_rng(batch)
    td = rng.exponential(1.0, size=n).astype(np.float32)
    td[rng.random(n) < 0.2] = 0.0
    td[rng.random(n) < 0.02] = 1e4
    _update(torch, per, np.arange(n), td)
    leaves, total, _ = per.read()
    phys = physical_leaves(leaves, env.time())
    for call_index in (0, 12345678901):
        idx, w = _sample(torch, per, batch, 2, call_index, 0.7)
        ref_idx, ref_w, p, ref_total = reference_sample(phys, env.time(), batch, 2, call_index, 11, 0.7)
        assert ref_total == total
        assert np.array_equal(idx, ref_idx), (batch, call_index)
        assert idx.max() < n
        assert np.all(np.abs(w.astype(np.float64) - ref_w) <= 2.0 ** -22 * ref_w)
        for mb in range(2):
            assert w[mb][np.argmin(p[mb])] == 1.0
    per.close(); env.close()


# ---------------------------------------------------------------- 3. frequencies
def test_draw_frequencies_follow_the_priorities(qlb):
    torch = pytest.importorskip("torch")
    env = _env(qlb, seed=3)
    _step(env, 20, 3)
    per = qlb.PrioritizedReplay(env, alpha=1.0, epsilon=1e-6)
    n = _len(qlb, env)
    cls = np.arange(n) % 4
    _update(torch, per, np.arange(n), np.array([0.5, 1.0, 2.0, 4.0], dtype=np.float32)[cls])
    leaves, total, _ = per.read()
    idx, _ = _sample(torch, per, 4096, 256, 77, 0.5)
    counts = np.bincount(cls[idx.ravel()], minlength=4).astype(np.float64)
    expect = idx.size * np.array([leaves[cls == k].sum(dtype=np.float64) for k in range(4)]) / total
    chi2 = float(((counts - expect) ** 2 / expect).sum())
    assert chi2 < 30.0, (counts, expect, chi2)         # 3 degrees of freedom
    per.close(); env.close()


# ---------------------------------------------------------------- 4. update semantics
def test_update_semantics(qlb):
    torch = pytest.importorskip("torch")
    env = _env(qlb, seed=5)
    _step(env, 10, 1)
    alpha, eps = 0.6, 1e-6
    per = qlb.PrioritizedReplay(env, alpha, eps)
    n = _len(qlb, env)
    rng = np.random.default_rng(0)
    td = (rng.standard_normal(n) * 3).astype(np.float32)
    td[:5] = 0.0
    _update(torch, per, np.arange(n), td)
    leaves, _, mx = _check_tree(qlb, per, env)
    ref = priority64(td, alpha, eps)
    assert np.all(np.abs(leaves - ref) <= np.spacing(ref.astype(np.float32)))        # within 1 f32 ulp of the f64 value
    assert mx == max(1.0, leaves.max())
    # duplicates keep the largest priority; indices >= len change nothing
    _update(torch, per, [5, 5, 5, n, n + 1000, 0xFFFFFFF0], [0.1, 3.0, -1.0, 100.0, 100.0, 100.0])
    l2, _, mx2 = _check_tree(qlb, per, env)
    assert l2[5] == np.float32(priority64(np.float32([3.0]), alpha, eps)[0])
    assert np.array_equal(np.delete(l2, 5), np.delete(leaves, 5)) and mx2 == mx
    # a non-finite delta takes the running max, raised by the same update's finite ones
    big = np.float32(500.0)
    _update(torch, per, [7, 8, 9], [np.nan, np.inf, big])
    l3, _, mx3 = _check_tree(qlb, per, env)
    assert mx3 == np.float32(priority64(np.float32([big]), alpha, eps)[0])
    assert l3[7] == mx3 and l3[8] == mx3 and l3[9] == mx3
    # new transitions enter at the raised running max
    _step(env, 1, 2)
    l4, _, mx4 = _check_tree(qlb, per, env)
    assert mx4 == mx3 and np.all(l4[-N_ENVS:] == mx3)
    per.close()
    # alpha = 0: every priority is 1
    per0 = qlb.PrioritizedReplay(env, alpha=0.0)
    _update(torch, per0, np.arange(n), td)
    l5, _, _ = _check_tree(qlb, per0, env)
    assert np.all(l5 == 1.0)
    per0.close(); env.close()


# ---------------------------------------------------------------- 5. no drift
def test_no_drift_over_interleaved_calls(qlb):
    torch = pytest.importorskip("torch")
    env = _env(qlb, seed=9)
    _step(env, 3, 9)
    per = qlb.PrioritizedReplay(env)
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    s = torch.cuda.current_stream().cuda_stream
    idx = torch.empty(32, dtype=torch.int32, device="cuda")
    w = torch.empty(32, dtype=torch.float32, device="cuda")
    for it in range(200):
        if it % 3 == 0:
            env.step_random_device(1 + it % 5, stream=s)
        per.sample_device(32, 1, it, 0.5, idx.data_ptr(), w.data_ptr(), s)
        td = torch.randn(32, device="cuda", generator=g) * (1.0 + it % 7)
        per.update_device(idx.data_ptr(), td.data_ptr(), 32, s)
        if it % 50 == 49:
            _check_tree(qlb, per, env)
    _check_tree(qlb, per, env)
    per.close(); env.close()


# ---------------------------------------------------------------- 6. unweighted training is unchanged
def test_weighted_training_with_unit_weights_is_bit_identical(qlb):
    torch = pytest.importorskip("torch")
    env, rb = _replay(qlb)
    w = _random_weights(qlb, 4)
    tgt = qlb.QNetwork(env, w)
    nets = [qlb.QNetwork(env, w) for _ in range(3)]
    batch, nb = 64, 3
    idx = torch.as_tensor(np.random.default_rng(1).choice(rb.len(), size=batch * nb, replace=False).astype(np.int32), device="cuda")
    ones = torch.ones(batch * nb, dtype=torch.float32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    losses = [torch.empty(nb, dtype=torch.float32, device="cuda") for _ in range(3)]
    nets[0].train_device(idx.data_ptr(), batch, nb, None, tgt, 0.99, losses[0].data_ptr(), s)
    nets[1].train_weighted_device(idx.data_ptr(), None, batch, nb, None, tgt, 0.99, losses[1].data_ptr(), None, s)
    nets[2].train_weighted_device(idx.data_ptr(), ones.data_ptr(), batch, nb, None, tgt, 0.99, losses[2].data_ptr(), None, s)
    torch.cuda.synchronize()
    assert all(n.error() == 0 for n in nets)
    l0 = losses[0].cpu().numpy()
    ws = [n.get_weights() for n in nets]
    for k in (1, 2):
        assert np.array_equal(losses[k].cpu().numpy().view(np.uint32), l0.view(np.uint32))
        for name in qlb.QNET_SHAPES:
            assert np.array_equal(ws[k][name].view(np.uint32), ws[0][name].view(np.uint32)), (k, name)
    for n in nets + [tgt]:
        n.close()
    env.close()


# ---------------------------------------------------------------- 7. weighted gradients vs torch autograd
def _torch_weighted_grads(torch, w_np, obs_bxyh, action, target, weight, quantise):
    """the graph of test_qnet_train._torch_loss with the loss mean(w * huber)"""
    F = torch.nn.functional
    w = {k: torch.from_numpy(v.copy()).requires_grad_(True) for k, v in w_np.items()}
    bf = (lambda t: t.to(torch.bfloat16).to(torch.float32)) if quantise else (lambda t: t)
    x = torch.from_numpy(obs_bxyh).permute(0, 3, 1, 2).contiguous()
    for i in (1, 2, 3):
        k = bf(w["conv%d_kernel" % i].permute(3, 2, 0, 1))
        x = bf(torch.relu(F.conv2d(x, k, w["conv%d_bias" % i], stride={1: 4, 2: 2, 3: 1}[i])))
    x = x.permute(0, 2, 3, 1).reshape(x.shape[0], -1)
    x = bf(torch.relu(x @ bf(w["dense1_kernel"]) + w["dense1_bias"]))
    q = x @ w["dense2_kernel"] + w["dense2_bias"]
    qa = q.gather(1, torch.from_numpy(action.astype(np.int64)).unsqueeze(1)).squeeze(1)
    loss = (torch.from_numpy(weight) * F.huber_loss(qa, torch.from_numpy(target), delta=1.0, reduction="none")).mean()
    loss.backward()
    return {k: w[k].grad.numpy().astype(np.float64) for k in w}


@pytest.mark.parametrize("batch", [1, 32, 300, 2000])
def test_weighted_gradients_match_torch_autograd(qlb, batch):
    """Tolerances of test_qnet_train.test_gradients_match_torch_autograd: 2e-2 against the bf16-quantised graph, 1.5e-1 against
    fp32. The TD errors are Q(s)[a] - y of the library's own forward, bit for bit."""
    torch = pytest.importorskip("torch")
    env, rb = _replay(qlb)
    w = _random_weights(qlb, 3)
    net = qlb.QNetwork(env, w)
    rng = np.random.default_rng(batch + 1)
    idx = rng.choice(rb.len(), size=batch, replace=False).astype(np.uint32)
    smp = rb.get_many(idx, qlb.LAYOUT_F32_BXYH)
    y = _saturating_targets(net, idx, smp, batch)
    wt = rng.uniform(0.0, 1.0, size=batch).astype(np.float32)
    wt = np.where(wt == 0.0, np.float32(1.0), wt)
    g, td = net.debug_grads_weighted(idx, y, wt)
    q, _, _ = net.forward(idx, 0)
    assert np.array_equal(td.view(np.uint32), (q[np.arange(batch), smp.action.astype(np.int64)] - y).view(np.uint32))
    ref_q = _torch_weighted_grads(torch, w, smp.state, smp.action, y, wt, quantise=True)
    ref_f = _torch_weighted_grads(torch, w, smp.state, smp.action, y, wt, quantise=False)
    for name in qlb.QNET_SHAPES:
        assert np.all(np.isfinite(g[name])), name
        nref = np.linalg.norm(ref_q[name])
        assert nref > 0, name
        eq = np.linalg.norm(g[name] - ref_q[name]) / nref
        ef = np.linalg.norm(g[name] - ref_f[name]) / np.linalg.norm(ref_f[name])
        assert eq <= 2e-2, (name, eq)
        assert ef <= 1.5e-1, (name, ef)
    net.close(); env.close()


# ---------------------------------------------------------------- 8. determinism
def test_prioritized_training_is_deterministic(qlb):
    torch = pytest.importorskip("torch")

    def run():
        env, rb = _replay(qlb, n_envs=128, seed=6)
        w = _random_weights(qlb, 8)
        net, tgt = qlb.QNetwork(env, w), qlb.QNetwork(env, w)
        per = qlb.PrioritizedReplay(env)
        s = torch.cuda.current_stream().cuda_stream
        batch = 32
        idx = torch.empty(batch, dtype=torch.int32, device="cuda")
        wt = torch.empty(batch, dtype=torch.float32, device="cuda")
        td = torch.empty(batch, dtype=torch.float32, device="cuda")
        seen = []
        for it in range(10):
            per.sample_device(batch, 1, it, 0.4 + 0.06 * it, idx.data_ptr(), wt.data_ptr(), s)
            net.train_weighted_device(idx.data_ptr(), wt.data_ptr(), batch, 1, None, tgt, 0.99, None, td.data_ptr(), s)
            per.update_device(idx.data_ptr(), td.data_ptr(), batch, s)
            seen.append(idx.cpu().numpy().copy())
        torch.cuda.synchronize()
        assert net.error() == 0
        out = (net.get_weights(), per.read()[0], np.concatenate(seen))
        per.close(); net.close(); tgt.close(); env.close()
        return out

    a, b = run(), run()
    for name in qlb.QNET_SHAPES:
        assert np.array_equal(a[0][name].view(np.uint32), b[0][name].view(np.uint32)), name
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    assert np.array_equal(a[2], b[2])
    assert len(np.unique(a[1])) > 2                     # the priorities did move


# ---------------------------------------------------------------- 9. lifetimes
def test_handle_outlives_its_env(qlb):
    import ctypes
    env = _env(qlb)
    _step(env, 2, 0)
    per = qlb.PrioritizedReplay(env)
    per.read()
    env.close()
    lib = qlb.load_library()
    total = ctypes.c_double(0)
    assert lib.qlc_per_read_host(per._h, None, ctypes.byref(total), None) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_update(per._h, ctypes.c_void_p(16), ctypes.c_void_p(16), 1, None) == qlb.ERR_INVALID_ARG
    with pytest.raises(qlb.QlError) as ei:
        per.sample_device(32, 1, 0, 0.5, 16, None)
    assert ei.value.code == qlb.ERR_INVALID_ARG
    per.close()
    assert per._h is None


def test_empty_replay_is_not_enough(qlb):
    env = _env(qlb)
    per = qlb.PrioritizedReplay(env)
    with pytest.raises(qlb.QlError) as ei:
        per.sample_device(32, 1, 0, 0.5, 16, None)
    assert ei.value.code == qlb.ERR_NOT_ENOUGH
    per.close(); env.close()


# ---------------------------------------------------------------- 10. closed loop
def test_closed_loop_example_with_prioritized_replay(qlb):
    import importlib.util
    import os
    pytest.importorskip("torch")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("dqn_breakout_torch", os.path.join(root, "examples", "dqn_breakout_torch.py"))
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    out = ex.run(n_envs=1024, iterations=20, quiet=True, random_phase_steps=0, tensor_core_learner=True, prioritized=True, target_sync_every=5)
    assert out["train_calls"] == 20 and out["minibatches"] == 20 * 256, out
    assert out["losses_finite"] and np.isfinite(out["last_loss"]), out
    assert out["error_flags"] == 0 and out["qnet_error"] == 0, out
    leaves, t = out["per_leaves"], out["env_time"]
    assert leaves.size == min(t, 128) * 1024 and np.all(leaves > 0)
    phys = physical_leaves(leaves, t, n_envs=1024, t_cap=128)
    assert out["per_total"] == tree_levels(phys)[-1][0]
    assert len(np.unique(leaves)) > 2                    # priorities were updated from the TD errors
