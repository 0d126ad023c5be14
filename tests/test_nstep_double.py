"""n-step returns and double-DQN targets on the device (nstep.cuh, qlc_replay_nstep, qlc_qnet_train_nstep; DESIGN.md §14)
against the numpy model of tests/test_nstep_abi.py, bit for bit:

1. qlc_replay_nstep for every logical index of wrapped rings (1, 37 and 4,096 envs), auto-reset on and off with resets by the
   caller, truncating episode limits, n_step 1 to 64, gamma 0 to 1, and indices >= len.
2. n_step = 1 without double DQN is qlc_qnet_train_weighted (weighted and unweighted) and qlc_qnet_train, except at an index
   >= len, where the one-step target bootstraps from the zero stack and the n-step target is 0.
3. The targets equal the model's y built from qlc_replay_nstep and qlc_qnet_forward on the bootstrap states.
4. Each minibatch is qlc_qnet_train_weighted on the targets y_dev reports; n_batches = 3 is 3 calls; runs repeat bit for bit.
5. The prioritized learner feeds its n-step double-DQN TD errors to the tree.
6. The example's closed loop with --n-step 3 --double-dqn on both learners."""
import importlib
import importlib.util
import os

import numpy as np
import pytest

from test_nstep_abi import nstep_model, target_model
from test_qnet_train import _random_weights

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
array_io = importlib.import_module("q-learning_b200.array_io")
torch_io = importlib.import_module("q-learning_b200.torch_io")


def _s():
    return torch.cuda.current_stream().cuda_stream


def _ring_state(env, rb):
    """(records u32 [time_slots][n_envs], t_oldest, t_now) read from the device"""
    torch.cuda.synchronize()
    v = array_io.device_views(env)
    rec = torch.as_tensor(v["records"], device="cuda").cpu().numpy()
    t = v["_time"]
    return rec, t - rb.len() // env.n_envs, t


def _dev_idx(idx):
    return torch.as_tensor(np.asarray(idx, dtype=np.uint32).view(np.int32), device="cuda")


def _nstep(rb, idx_t, n_step, gamma):
    n = idx_t.numel()
    G = torch.empty(n, dtype=torch.float32, device="cuda")
    d = torch.empty(n, dtype=torch.float32, device="cuda")
    b = torch.empty(n, dtype=torch.int32, device="cuda")
    rb.nstep_device(idx_t.data_ptr(), n, n_step, gamma, G.data_ptr(), d.data_ptr(), b.data_ptr(), _s())
    torch.cuda.synchronize()
    return G.cpu().numpy(), d.cpu().numpy(), b.cpu().numpy().view(np.uint32)


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def _check_every_index(env, rb, combos):
    rec, t_old, t_now = _ring_state(env, rb)
    n_len = rb.len()
    idx = np.concatenate([np.arange(n_len), n_len + np.array([0, 1, env.n_envs, 1 << 20]), [0xFFFFFFFF]]).astype(np.uint32)
    idx_t = _dev_idx(idx)
    for n_step, gamma in combos:
        G, d, b = _nstep(rb, idx_t, n_step, gamma)
        mG, md, mb, _ = nstep_model(rec, t_old, t_now, idx, n_step, gamma)
        for name, got, want in (("G", _bits(G), _bits(mG)), ("disc", _bits(d), _bits(md)), ("boot", b, mb)):
            bad = np.nonzero(got != want)[0]
            assert bad.size == 0, (n_step, gamma, name, bad[:4], idx[bad[:4]], got[bad[:4]], want[bad[:4]])


ALL_COMBOS = [(n, g) for n in (1, 2, 3, 5, 64) for g in (0.0, 0.5, 0.99, 1.0)]


# ---------------------------------------------------------------- 1. returns, exactly
@pytest.mark.parametrize("n_envs,t_cap,max_steps", [(1, 300, 0), (1, 40, 9), (37, 16, 0), (37, 16, 5)])
def test_returns_every_index_auto_reset(qlb, n_envs, t_cap, max_steps):
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=5, replay_capacity=n_envs * t_cap, max_episode_steps=max_steps)
    rb = qlb.ReplayBuffer(env)
    rng = np.random.default_rng(n_envs + max_steps)
    env.step_many(rng.integers(0, 3, size=(3, n_envs), dtype=np.uint8))
    _check_every_index(env, rb, [(3, 0.99), (64, 1.0)])                     # a ring that is not full yet
    env.step_many(rng.integers(0, 3, size=(t_cap + 207, n_envs), dtype=np.uint8))
    rec, t_old, t_now = _ring_state(env, rb)
    assert t_old > 0 and t_old % (t_cap + 4) != 0                        # wrapped
    if max_steps:
        assert ((rec >> 16) & 1).any()                                    # truncations
    _check_every_index(env, rb, ALL_COMBOS)
    env.close()


@pytest.mark.parametrize("n_envs,max_steps", [(1, 0), (37, 6)])
def test_returns_every_index_resets_by_the_caller(qlb, n_envs, max_steps):
    """auto_reset off: finished envs keep writing done records until the caller resets them; a reset of a running env ends
    its episode without a done record (the next record has min(k,4) = 0)."""
    t_cap = 16
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=9, replay_capacity=n_envs * t_cap, max_episode_steps=max_steps, auto_reset=False)
    rb = qlb.ReplayBuffer(env)
    rng = np.random.default_rng(1)
    for it in range(12):
        env.step_many(rng.integers(0, 3, size=(int(rng.integers(2, 6)), n_envs), dtype=np.uint8))
        env.reset(mask=(rng.random(n_envs) < 0.4).astype(np.uint8) if n_envs > 1 else np.array([it % 2 == 0], np.uint8))
    env.step_many(rng.integers(0, 3, size=(2, n_envs), dtype=np.uint8))
    rec, t_old, t_now = _ring_state(env, rb)
    assert t_old > 0
    kmin = (rec >> 5) & 7
    assert (kmin == 0).sum() > 1
    _check_every_index(env, rb, ALL_COMBOS)
    env.close()


def test_returns_every_index_4096_envs(qlb):
    n_envs, cap = 4096, 1 << 20
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=2, replay_capacity=cap, max_episode_steps=200)
    rb = qlb.ReplayBuffer(env)
    env.step_random_device(cap // n_envs + 37, stream=_s())
    rec, t_old, _ = _ring_state(env, rb)
    assert t_old > 0 and ((rec >> 2) & 1).any()
    _check_every_index(env, rb, [(1, 0.99), (3, 0.99), (5, 1.0), (64, 0.5), (2, 0.0)])
    env.close()


# ---------------------------------------------------------------- training fixtures
def _setup(qlb, seed=3, n_envs=37, t_cap=16, steps=21, max_steps=11):
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=n_envs * t_cap, max_episode_steps=max_steps)
    rb = qlb.ReplayBuffer(env)
    env.step_many(np.random.default_rng(seed).integers(0, 3, size=(steps, n_envs), dtype=np.uint8))
    return env, rb


def _nets(qlb, env, w, k):
    nets = [qlb.QNetwork(env, w) for _ in range(k)]
    for n in nets:
        n.set_adam(lr=2.5e-4, clipnorm=1.0)
    return nets


def _weights_equal(a, b):
    wa, wb = a.get_weights(), b.get_weights()
    return all(np.array_equal(wa[k].view(np.uint32), wb[k].view(np.uint32)) for k in wa)


def _bufs(n_batches, batch):
    return (torch.empty(n_batches, dtype=torch.float32, device="cuda"), torch.empty(n_batches * batch, dtype=torch.float32, device="cuda"),
            torch.empty(n_batches * batch, dtype=torch.float32, device="cuda"))


# ---------------------------------------------------------------- 2. n = 1 is the old path
def test_one_step_is_the_weighted_update(qlb):
    env, rb = _setup(qlb)
    w0, w1 = _random_weights(qlb, 11), _random_weights(qlb, 12)
    target = qlb.QNetwork(env, w1)
    batch, nb = 32, 3
    idx = _dev_idx(np.random.default_rng(0).integers(0, rb.len(), size=nb * batch))
    wts = torch.as_tensor(np.random.default_rng(1).uniform(0.1, 1.0, size=nb * batch).astype(np.float32), device="cuda")
    for wt in (wts, None):
        a, b, c = _nets(qlb, env, w0, 3)
        ra, rb_, rc = _bufs(nb, batch), _bufs(nb, batch), _bufs(nb, batch)
        wp = None if wt is None else wt.data_ptr()
        a.train_nstep_device(idx.data_ptr(), wp, batch, nb, target, 0.99, 1, False, ra[0].data_ptr(), ra[1].data_ptr(), ra[2].data_ptr(), _s())
        b.train_weighted_device(idx.data_ptr(), wp, batch, nb, None, target, 0.99, rb_[0].data_ptr(), rb_[1].data_ptr(), _s())
        if wt is None:
            c.train_device(idx.data_ptr(), batch, nb, None, target, 0.99, rc[0].data_ptr(), _s())
        torch.cuda.synchronize()
        assert a.error() == 0 and b.error() == 0 and c.error() == 0
        assert np.array_equal(_bits(ra[0].cpu()), _bits(rb_[0].cpu()))
        assert np.array_equal(_bits(ra[1].cpu()), _bits(rb_[1].cpu()))
        assert _weights_equal(a, b)
        if wt is None:
            assert np.array_equal(_bits(ra[0].cpu()), _bits(rc[0].cpu())) and _weights_equal(a, c)
        for n in (a, b, c):
            n.close()
    target.close(); env.close()


def test_one_step_target_of_an_index_beyond_len(qlb):
    """Where the one-step and the n-step targets differ: an index >= len has record 0 and the all-zero stacks. The one-step
    target is then y = 0 + maxQ_target(zero stack)·gamma with action 0, so td = Q_online(zero stack)[0] - y; the n-step walk
    gives G = 0, disc = 0, so y = 0."""
    env, rb = _setup(qlb, seed=8)
    w0, w1 = _random_weights(qlb, 51), _random_weights(qlb, 52)
    target = qlb.QNetwork(env, w1)
    batch, gamma, k = 32, 0.99, 7
    idx_np = np.random.default_rng(5).integers(0, rb.len(), size=batch).astype(np.uint32)
    idx_np[k] = rb.len() + 5
    idx = _dev_idx(idx_np)
    a, b = _nets(qlb, env, w0, 2)
    q_on, max_t = torch.empty((batch, 3), dtype=torch.float32, device="cuda"), torch.empty(batch, dtype=torch.float32, device="cuda")
    a.forward_device(idx.data_ptr(), batch, 0, q_on.data_ptr(), None, None, _s())          # the online weights before the update
    target.forward_device(idx.data_ptr(), batch, 1, None, None, max_t.data_ptr(), _s())
    loss, td, y = _bufs(1, batch)
    a.train_weighted_device(idx.data_ptr(), None, batch, 1, None, target, gamma, loss.data_ptr(), td.data_ptr(), _s())
    b.train_nstep_device(idx.data_ptr(), None, batch, 1, target, gamma, 1, False, None, None, y.data_ptr(), _s())
    torch.cuda.synchronize()
    assert a.error() == 0 and b.error() == 0
    q0, mt = q_on.cpu().numpy()[k, 0], max_t.cpu().numpy()[k]
    want = np.float32(q0 - np.float32(mt * np.float32(gamma)))
    assert _bits(td.cpu().numpy()[k]) == _bits(want), (td.cpu().numpy()[k], want)
    assert y.cpu().numpy()[k] == 0.0
    for n in (a, b, target):
        n.close()
    env.close()


# ---------------------------------------------------------------- 3. targets
def _y_of_call(qlb, env, w_online, target, idx, double, n_step=3, gamma=0.99):
    (net,) = _nets(qlb, env, w_online, 1)
    y = torch.empty(idx.numel(), dtype=torch.float32, device="cuda")
    net.train_nstep_device(idx.data_ptr(), None, idx.numel(), 1, target, gamma, n_step, double, None, None, y.data_ptr(), _s())
    torch.cuda.synchronize()
    assert net.error() == 0
    net.close()
    return y.cpu().numpy()


def test_targets_match_the_model(qlb):
    env, rb = _setup(qlb, seed=4, n_envs=256, t_cap=64, steps=400, max_steps=0)
    w0, w1 = _random_weights(qlb, 21), _random_weights(qlb, 22)
    target = qlb.QNetwork(env, w1)
    online = qlb.QNetwork(env, w0)
    n, gamma = 96, 0.99
    rec, t_old, t_now = _ring_state(env, rb)
    # half of the items end in a done record within 3 steps (terminal), the rest are drawn uniformly
    ends = np.nonzero(nstep_model(rec, t_old, t_now, np.arange(rb.len()), 3, gamma)[3])[0]
    assert ends.size
    rng = np.random.default_rng(2)
    idx_np = np.concatenate([rng.choice(ends, n // 2), rng.integers(0, rb.len(), size=n - n // 2)]).astype(np.uint32)
    idx = _dev_idx(idx_np)
    G, d, b = _nstep(rb, idx, 3, gamma)
    mG, md, mb, term = nstep_model(rec, t_old, t_now, idx_np, 3, gamma)
    assert np.array_equal(_bits(G), _bits(mG)) and np.array_equal(_bits(d), _bits(md)) and np.array_equal(b, mb)
    assert term.any() and (~term).any() and (b != idx_np).any()
    tq, _, tmax = target.forward(b, 1)
    _, a_on, _ = online.forward(b, 1)
    y_van = _y_of_call(qlb, env, w0, target, idx, False, gamma=gamma)
    y_dbl = _y_of_call(qlb, env, w0, target, idx, True, gamma=gamma)
    assert np.array_equal(_bits(y_van), _bits(target_model(G, d, term, tmax)))
    assert np.array_equal(_bits(y_dbl), _bits(target_model(G, d, term, tq[np.arange(n), a_on.astype(np.int64)])))
    assert (_bits(y_dbl) != _bits(y_van)).any()                              # different online and target weights
    # equal weights: double DQN is vanilla
    same = qlb.QNetwork(env, w0)
    assert np.array_equal(_bits(_y_of_call(qlb, env, w0, same, idx, True, gamma=gamma)), _bits(_y_of_call(qlb, env, w0, same, idx, False, gamma=gamma)))
    for x in (same, online, target):
        x.close()
    env.close()


# ---------------------------------------------------------------- 4. decomposition, k calls, repeatability
@pytest.mark.parametrize("double", [False, True])
def test_minibatches_decompose(qlb, double):
    env, rb = _setup(qlb, seed=6)
    w0, w1 = _random_weights(qlb, 31), _random_weights(qlb, 32)
    target = qlb.QNetwork(env, w1)
    batch, nb = 32, 3
    idx = _dev_idx(np.random.default_rng(3).integers(0, rb.len(), size=nb * batch))
    wts = torch.as_tensor(np.random.default_rng(4).uniform(0.1, 1.0, size=nb * batch).astype(np.float32), device="cuda")
    a, b, c, d = _nets(qlb, env, w0, 4)
    ra, rb_, rc, rd = (_bufs(nb, batch) for _ in range(4))
    ya, yc, yd = (torch.empty(nb * batch, dtype=torch.float32, device="cuda") for _ in range(3))
    a.train_nstep_device(idx.data_ptr(), wts.data_ptr(), batch, nb, target, 0.99, 3, double, ra[0].data_ptr(), ra[1].data_ptr(), ya.data_ptr(), _s())
    # the same updates from qlc_qnet_train_weighted on the targets the n-step call reports
    b.train_weighted_device(idx.data_ptr(), wts.data_ptr(), batch, nb, ya.data_ptr(), None, 0.99, rb_[0].data_ptr(), rb_[1].data_ptr(), _s())
    # three calls of one minibatch each
    for j in range(nb):
        o = j * batch
        c.train_nstep_device(idx[o:].data_ptr(), wts[o:].data_ptr(), batch, 1, target, 0.99, 3, double, rc[0][j:].data_ptr(), rc[1][o:].data_ptr(),
                             yc[o:].data_ptr(), _s())
    d.train_nstep_device(idx.data_ptr(), wts.data_ptr(), batch, nb, target, 0.99, 3, double, rd[0].data_ptr(), rd[1].data_ptr(), yd.data_ptr(), _s())
    torch.cuda.synchronize()
    for n in (a, b, c, d):
        assert n.error() == 0
    for other, y in ((rb_, None), (rc, yc), (rd, yd)):
        assert np.array_equal(_bits(ra[0].cpu()), _bits(other[0].cpu()))
        assert np.array_equal(_bits(ra[1].cpu()), _bits(other[1].cpu()))
        if y is not None:
            assert np.array_equal(_bits(ya.cpu()), _bits(y.cpu()))
    assert _weights_equal(a, b) and _weights_equal(a, c) and _weights_equal(a, d)
    for n in (a, b, c, d, target):
        n.close()
    env.close()


# ---------------------------------------------------------------- 5. prioritized
def test_prioritized_learner_feeds_nstep_double_td_errors(qlb):
    n_envs, t_cap, seed = 37, 16, 23
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=n_envs * t_cap, max_episode_steps=9)
    env.step_many(np.random.default_rng(4).integers(0, 3, size=(t_cap + 6, n_envs), dtype=np.uint8))
    w0 = _random_weights(qlb, 41)
    learner = torch_io.TensorCoreLearner(env, w0, gamma=0.99, per_alpha=0.6, n_step=3, double_dqn=True)
    online, target = _nets(qlb, env, w0, 1)[0], qlb.QNetwork(env, w0)
    twin_per = qlb.PrioritizedReplay(env, 0.6)
    batch = 32
    idx_t = torch.empty(batch, dtype=torch.int32, device="cuda")
    w_t, td_t = (torch.empty(batch, dtype=torch.float32, device="cuda") for _ in range(2))
    for it in range(3):
        if it:
            env.step_random_device(3, stream=_s())
        learner.train_prioritized(batch, 1, 100 + it, 0.5)
        twin_per.sample_device(batch, 1, 100 + it, 0.5, idx_t.data_ptr(), w_t.data_ptr(), _s())
        online.train_nstep_device(idx_t.data_ptr(), w_t.data_ptr(), batch, 1, target, 0.99, 3, True, None, td_t.data_ptr(), None, _s())
        twin_per.update_device(idx_t.data_ptr(), td_t.data_ptr(), batch, _s())
        torch.cuda.synchronize()
        assert learner.error() == 0 and online.error() == 0
        l_idx, _, l_td = (x.cpu().numpy() for x in learner._per_bufs)
        assert np.array_equal(l_idx.ravel(), idx_t.cpu().numpy())
        assert np.array_equal(_bits(l_td.ravel()), _bits(td_t.cpu().numpy())), it
        leaves = learner.per.read()[0]
        assert np.array_equal(leaves.view(np.uint32), twin_per.read()[0].view(np.uint32)), it
        # the sampled transitions carry (|td| + eps)^alpha of this update's TD errors (the largest where an index repeats)
        p = np.power(np.abs(l_td.ravel().astype(np.float64)) + np.float64(np.float32(1e-6)), np.float64(np.float32(0.6)))
        for i in np.unique(l_idx.ravel()):
            want = p[l_idx.ravel() == i].max()
            assert abs(float(leaves[i]) - want) <= 2.0 ** -23 * want, (it, i)
        assert _weights_equal(learner.online, online)
    for x in (twin_per, online, target):
        x.close()
    learner.close(); env.close()


# ---------------------------------------------------------------- 6. closed loop
@pytest.mark.parametrize("learner", ["tensor_core", "tensor_core_prioritized", "torch"])
def test_closed_loop_example_nstep_double(qlb, learner):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("dqn_breakout_torch", os.path.join(root, "examples", "dqn_breakout_torch.py"))
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    tc = learner != "torch"
    out = ex.run(n_envs=1024, iterations=12, quiet=True, random_phase_steps=0, tensor_core_learner=tc, prioritized=learner.endswith("prioritized"),
                 target_sync_every=5, n_step=3, double_dqn=True)
    assert out["train_calls"] > 0 and np.isfinite(out["last_loss"]), out
    assert out["error_flags"] == 0, out
    if tc:
        assert out["losses_finite"] and out["qnet_error"] == 0, out
