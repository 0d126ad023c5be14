"""n-step and double-DQN training (qlc_qnet_train_nstep, nstep.cuh; DESIGN.md §14) where it can go wrong. The reference for y is
the model of tests/test_nstep_abi.py applied to the library's own parts: G, disc, boot and terminal from nstep_model on the
records read back from the device, Q_boot from qlc_qnet_forward(which = 1) on boot at the item count the call itself uses (so
the same dense path), and for double DQN the target's q[boot] at the first-maximum action of an online twin brought to the
weights after updates 0 .. j-1 with qlc_qnet_train_weighted on the reported y. Composed this way y is exact: it is compared bit
for bit, +0 and -0 equal. td is compared bit for bit with Q(s)[a] - y from the forward that precedes the item's own update.

1. Every stop kind (done, truncation, reset by the caller, newest time, n_step reached) in every minibatch, with duplicate
   indices and indices >= len, on wrapped rings of 1, 37 and 300 envs, n_step 1 to 64, gamma 0 to 1, vanilla and double.
2. Both dense paths: the target network's forward (all items), the online double-DQN forward and the training forward (one
   minibatch each) on either side of the narrow / wide boundary, and 32,768 items on a 1 M-transition ring.
3. Scratch growth and reuse: n-step, plain and weighted calls of one network on a side stream at growing and shrinking sizes,
   each equal to a fresh twin that makes only that call.
4. Stream order of the two n-step calls: both are under test_stream_order.py's asynchronous rule and see submitted host steps;
   host calls of the network wait for an n-step update queued behind a sleep."""
import time
from types import SimpleNamespace

import numpy as np
import pytest

import test_stream_order as so
from test_nstep_abi import _ring, nstep_model, target_model
from test_nstep_double import _bits, _dev_idx, _ring_state, _weights_equal
from test_qnet_batch_edges import _random_weights, _size

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

DONE, TRUNCATION, RESET, NEWEST, N_STEP = range(5)
KINDS = ("done", "truncation", "reset by the caller", "newest time", "n_step reached")


# ---------------------------------------------------------------- helpers (checked on the CPU below)
def stop_kinds(records, t_oldest, t_now, idx, n_step):
    """Why nstep_model's walk of each logical index stops, as an index into KINDS; -1 for an index >= len. Where several
    reasons hold at the stop record, the first in KINDS order: a reset by the caller means the record after the stop starts
    an episode, and n_step reached means no other reason holds (then the walk has taken n_step records)."""
    ts, n_envs = records.shape
    idx = np.asarray(idx, dtype=np.uint64)
    _, _, boot, term = nstep_model(records, t_oldest, t_now, idx, n_step, 1.0)
    N = np.uint64(n_envs)
    T = np.uint64(t_oldest) + idx // N
    valid = T < np.uint64(t_now)
    e = (idx % N).astype(np.int64)
    m = np.where(valid, (boot.astype(np.uint64) - idx) // N, 0) + np.uint64(1)
    t_stop = T + m - np.uint64(1)
    rec = records[(t_stop % np.uint64(ts)).astype(np.int64), e]
    nxt = records[(np.minimum(t_stop + np.uint64(1), np.uint64(t_now - 1)) % np.uint64(ts)).astype(np.int64), e]
    newest = t_stop == np.uint64(t_now - 1)
    kind = np.select([~valid, term, (rec & 0x10000) != 0, ~newest & (((nxt >> 5) & 7) == 0), newest],
                     [-1, DONE, TRUNCATION, RESET, NEWEST], N_STEP)
    assert np.all(m[kind == N_STEP] == n_step), "a walk stopped early for no reason"
    return kind


PER_KIND = 6


def draw_minibatches(kinds, expected, n_len, n_envs, batch, n_batches, rng):
    """n_batches minibatches of batch logical indices, each holding PER_KIND items of every kind in `expected` (drawn with
    replacement), two repeated items, one index >= len and uniform indices for the rest, in random order."""
    pools = {c: np.nonzero(kinds == c)[0] for c in expected}
    for c, p in pools.items():
        assert p.size, "the ring produced no '%s' stops" % KINDS[c]
    beyond = [n_len, n_len + n_envs + 3, 0xFFFFFFFF]
    out = []
    for j in range(n_batches):
        mb = np.concatenate([rng.choice(pools[c], PER_KIND) for c in sorted(expected)])
        mb = np.concatenate([mb, mb[:2], [beyond[j % 3]], rng.integers(0, n_len, size=batch - mb.size - 3)])
        out.append(rng.permutation(mb))
    return np.concatenate(out).astype(np.uint32)


def differ(got, want):
    """positions where got and want (f32) differ bit for bit, with +0 and -0 equal"""
    g, w = (np.where(x == 0, np.float32(0), x).astype(np.float32) for x in (got, want))
    return np.nonzero(g.view(np.uint32) != w.view(np.uint32))[0]


def narrow(n, sm):
    """qnet_forward's choice of dense_tc_kernel<128> for n items"""
    return (n + 127) // 128 * 2 < sm


def last_narrow(sm):
    """the largest item count that still runs dense_tc_kernel<128> (test_qnet_batch_edges.py's last_narrow)"""
    return 128 * ((sm - 1) // 2)


def dense_shapes(ln):
    """(batch, n_batches) for the last narrow size ln: the target network's forward (all items) wide and the minibatch
    narrow, at the boundary (ln in 2 minibatches) and just past it (ln + 2 items); then every forward wide, at the first
    wide size, in 1 and in 2 minibatches."""
    w = SimpleNamespace(last_narrow=ln)
    wide = _size(w, "last_narrow+1")
    return [(_size(w, "last_narrow"), 2), (ln // 2 + 1, 2), (wide, 1), (wide, 2)]


# ---------------------------------------------------------------- CPU checks of the helpers
def test_stop_kinds_of_the_hand_worked_rings():
    """The rings of test_nstep_abi.py, whose walks are worked out by hand there."""
    # 2 envs, times 0..3: env 0 done at t1 and t2, env 1 truncated at t2; t3 is the newest time
    rows = [[dict(k=1, reward=1), dict(k=5, reward=1)],
            [dict(k=2, reward=2, done=True), dict(k=6, reward=2)],
            [dict(k=3, reward=3, done=True), dict(k=7, reward=3, truncated=True)],
            [dict(k=0, reward=4), dict(k=0, reward=4)]]
    got = stop_kinds(_ring(rows), 0, 4, np.arange(9), 3).tolist()
    assert got == [DONE, TRUNCATION, DONE, TRUNCATION, DONE, TRUNCATION, NEWEST, NEWEST, -1]
    # 1 env, times 0..4: the record at t3 starts an episode (a reset by the caller after t2)
    rows = [[dict(k=1, reward=1)], [dict(k=2, reward=1)], [dict(k=3, reward=1)], [dict(k=0, reward=2)], [dict(k=1, reward=2)]]
    rec = _ring(rows, ts=7)
    assert stop_kinds(rec, 0, 5, np.arange(6), 10).tolist() == [RESET, RESET, RESET, NEWEST, NEWEST, -1]
    # n_step 2: idx 0 takes 2 records (t0, t1) and t2 continues the episode; idx 1 stops at t2 before the reset (also its
    # n_step-th record: the reset comes first); idx 3 reaches the newest time with its n_step-th record (newest first)
    assert stop_kinds(rec, 0, 5, np.arange(6), 2).tolist() == [N_STEP, RESET, RESET, NEWEST, NEWEST, -1]
    # wrapped: 2 envs, 6 slots, times 3..8 live, no episode ends: T <= 4 takes 4 records, T >= 5 reaches t = 8
    rows = [[dict(k=t + 1, reward=t), dict(k=t + 1, reward=2 * t)] for t in range(9)]
    got = stop_kinds(_ring(rows, ts=6), 3, 9, np.arange(13), 4).tolist()
    assert got == [N_STEP] * 4 + [NEWEST] * 8 + [-1]


def test_minibatches_hold_every_kind_a_repeat_and_an_index_beyond_len():
    rng = np.random.default_rng(0)
    kinds = rng.integers(-1, 5, size=500)
    n_len = 500
    idx = draw_minibatches(kinds, {DONE, TRUNCATION, RESET, NEWEST, N_STEP}, n_len, 7, 40, 3, rng)
    assert idx.size == 120
    for j in range(3):
        mb = idx[j * 40:(j + 1) * 40]
        inside = mb[mb < n_len]
        assert set(kinds[inside]) >= set(range(5)) and np.unique(inside).size < inside.size
        assert (mb >= n_len).sum() == 1
    assert idx.max() == 0xFFFFFFFF


def test_differ_equates_signed_zeros_only():
    z = np.array([0.0, -0.0, 1.0, np.nan, 2.0], np.float32)
    assert differ(z, np.array([-0.0, 0.0, 1.0, np.nan, 2.0], np.float32)).size == 0
    assert differ(z, np.array([0.0, 0.0, np.nextafter(np.float32(1), np.float32(2)), np.nan, -2.0], np.float32)).tolist() == [2, 4]
    assert differ(z, np.array([0.0, 0.0, 1.0, 0.0, 2.0], np.float32)).tolist() == [3]


@pytest.mark.parametrize("sm", [148, 132, 160, 9])
def test_dense_shapes_straddle_the_boundary(sm):
    ln = last_narrow(sm)
    assert narrow(ln, sm) and not narrow(ln + 1, sm)
    sides = [(narrow(b * nb, sm), narrow(b, sm)) for b, nb in dense_shapes(ln)]
    assert sides == [(False, True), (False, True), (False, False), (False, False)]


# ---------------------------------------------------------------- 4a. both n-step calls are asynchronous and have a consumer test
def test_every_nstep_entry_point_has_an_ordering_rule():
    """test_stream_order.py places both calls under its asynchronous rule; each has a submitted-steps consumer case below."""
    assert {"qlc_replay_nstep", "qlc_qnet_train_nstep"} <= so.ASYNC
    assert {"qlc_replay_nstep", "qlc_qnet_train_nstep"} == set(SUBMITTED_CONSUMERS.values())


# ---------------------------------------------------------------- GPU helpers
LR = 1e-2            # large steps: the online argmax of double DQN moves between minibatches


class Ring:
    """An env's replay ring read back from the device, and the model on it."""

    def __init__(self, qlb, env):
        self.env, self.rb, self.n_envs = env, qlb.ReplayBuffer(env), env.n_envs
        self.rec, self.t_old, self.t_now = _ring_state(env, self.rb)
        self.len = self.rb.len()

    def model(self, idx, n_step, gamma):
        return nstep_model(self.rec, self.t_old, self.t_now, idx, n_step, gamma)

    def kinds(self, n_step):
        return stop_kinds(self.rec, self.t_old, self.t_now, np.arange(self.len), n_step)

    def actions(self, idx):
        """the action bits of each transition's record (0 for an index >= len, as locate() gives)"""
        idx = np.asarray(idx, np.uint64)
        T = self.t_old + idx // np.uint64(self.n_envs)
        ok = T < np.uint64(self.t_now)
        slot = (np.where(ok, T, 0) % np.uint64(self.rec.shape[0])).astype(np.int64)
        return np.where(ok, self.rec[slot, (idx % np.uint64(self.n_envs)).astype(np.int64)] & 3, 0).astype(np.int64)

    def close(self):
        self.env.close()


def forward(net, idx, which):
    """qlc_qnet_forward on the device (it takes indices >= len): (q [n][3], first-maximum action [n], max_q [n])"""
    n = idx.size
    q, a, m = (torch.empty(s, dtype=t, device="cuda") for s, t in (((n, 3), torch.float32), (n, torch.uint8), (n, torch.float32)))
    d = _dev_idx(idx)
    net.forward_device(d.data_ptr(), n, which, q.data_ptr(), a.data_ptr(), m.data_ptr())
    torch.cuda.synchronize()
    assert net.error() == 0
    return q.cpu().numpy(), a.cpu().numpy().astype(np.int64), m.cpu().numpy()


def check_nstep_call(r, net, twin, target, w0, idx, wts, batch, nb, gamma, n_step, double, lr=2.5e-4):
    """One train_nstep_device call of `net` from w0 with fresh Adam state, against the model (module docstring). `twin` (may be
    `net` itself: everything of the call is read back first) replays it minibatch by minibatch. Returns the reported y, the
    model's G, and the number of items of minibatches j >= 1 whose online action (double DQN) differs from that of w0."""
    n = batch * nb
    idx_d = _dev_idx(idx)
    wt = None if wts is None else torch.as_tensor(wts, device="cuda")
    loss_d, td_d, y_d = (torch.full((k,), float("nan"), device="cuda") for k in (nb, n, n))     # unwritten outputs stay NaN
    net.set_weights(w0)
    net.set_adam(lr=lr)
    net.train_nstep_device(idx_d.data_ptr(), None if wt is None else wt.data_ptr(), batch, nb, target, gamma, n_step, double,
                           loss_d.data_ptr(), td_d.data_ptr(), y_d.data_ptr())
    torch.cuda.synchronize()
    assert net.error() == 0
    loss, td, y = (x.cpu().numpy() for x in (loss_d, td_d, y_d))
    w_after = net.get_weights()
    what = "n_step %d gamma %g double %d batch %d x %d" % (n_step, gamma, double, batch, nb)

    G, disc, boot, term = r.model(idx, n_step, gamma)
    tq, _, tmax = forward(target, boot, 1)                   # all n items, as the call runs the target network
    a = r.actions(idx)
    twin.set_weights(w0)
    twin.set_adam(lr=lr)
    a0 = [forward(twin, boot[j * batch:(j + 1) * batch], 1)[1] for j in range(nb)] if double else None
    moved = 0
    for j in range(nb):
        s = slice(j * batch, (j + 1) * batch)
        if double:
            _, a_on, _ = forward(twin, boot[s], 1)           # the online weights after updates 0 .. j-1
            q_boot = tq[s][np.arange(batch), a_on]
            moved += int((a_on != a0[j]).sum()) if j else 0
        else:
            q_boot = tmax[s]
        y_model = target_model(G[s], disc[s], term[s], q_boot)
        bad = differ(y[s], y_model)[:4]
        assert bad.size == 0, (what, "y of minibatch", j, idx[s][bad], y[s][bad], y_model[bad])
        q, _, _ = forward(twin, idx[s], 0)                   # the forward that precedes this minibatch's update
        td_model = (q[np.arange(batch), a[s]] - y_model).astype(np.float32)
        bad = differ(td[s], td_model)[:4]
        assert bad.size == 0, (what, "td of minibatch", j, idx[s][bad], td[s][bad], td_model[bad])
        l_twin = torch.empty(1, device="cuda")
        twin.train_weighted_device(idx_d[j * batch:].data_ptr(), None if wt is None else wt[j * batch:].data_ptr(), batch, 1,
                                   y_d[j * batch:].data_ptr(), None, gamma, l_twin.data_ptr())
        torch.cuda.synchronize()
        assert twin.error() == 0
        assert np.array_equal(_bits(l_twin.cpu().numpy()), _bits(loss[j:j + 1])), (what, "loss of minibatch", j)
    so.assert_weights(w_after, twin.get_weights())
    beyond = idx >= r.len
    assert beyond.any() and np.all(y[beyond] == 0), what   # an index >= len: the kernel gives G = 0 and disc = 0, so y = 0
    return y, G, moved


# ---------------------------------------------------------------- 1. every stop kind, vanilla and double
MAX_EP = 162         # random play ends an episode after 158 to 174 steps: some episodes end in done, the others truncate
BATCH, NB = 40, 3
N_STEPS, GAMMAS = (1, 2, 5, 64), (0.0, 0.5, 0.99, 1.0)
RINGS = {   # n_envs: (time steps held, steps taken); each window holds episode ends of both kinds and 64-step stretches
    1: (1000, 1500),                  # without one
    37: (128, 400),
    300: (128, 400),
}


def build_ring(qlb, n_envs, auto_reset, seed):
    """auto_reset: random steps, episodes end in done or at MAX_EP. Otherwise the caller resets: after every chunk of 3 to 7
    steps it resets the envs that ended (done and truncated records repeat until then) and some running ones (1 in 100 per
    chunk; with one env, every 40th chunk), whose next record starts an episode without a done."""
    t_cap, steps = RINGS[n_envs]
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=n_envs * t_cap, max_episode_steps=MAX_EP,
                                  auto_reset=auto_reset)
    rng = np.random.default_rng(seed)
    if auto_reset:
        env.step_many(rng.integers(0, 3, size=(steps, n_envs), dtype=np.uint8))
    else:
        c = 0
        while env.time() < steps:
            env.step_many(rng.integers(0, 3, size=(int(rng.integers(3, 8)), n_envs), dtype=np.uint8))
            st = env.read_state()
            ended = (st["finished"] != 0) | (st["episode_step"] >= MAX_EP)
            running = rng.random(n_envs) < 0.01 if n_envs > 1 else np.array([c % 40 == 17])
            env.reset(mask=(ended | running).astype(np.uint8))
            c += 1
    r = Ring(qlb, env)
    assert r.t_old > 0 and r.t_old % (t_cap + 4) != 0                 # wrapped
    return r


@gpu
@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto_reset", "caller_resets"])
@pytest.mark.parametrize("n_envs", sorted(RINGS))
def test_every_stop_kind(qlb, n_envs, auto_reset):
    """y of every stop kind in every minibatch, n_step x gamma x (vanilla, double), 3 minibatches per call. The auto-reset
    ring has no resets by the caller; it must produce the four other kinds at every n_step, the caller-reset ring all five."""
    r = build_ring(qlb, n_envs, auto_reset, seed=11 + n_envs)
    expected = {DONE, TRUNCATION, NEWEST, N_STEP} | (set() if auto_reset else {RESET})
    w0, w1 = _random_weights(qlb, 51), _random_weights(qlb, 52)
    net, twin, target = qlb.QNetwork(r.env, w0), qlb.QNetwork(r.env, w0), qlb.QNetwork(r.env, w1)
    rng = np.random.default_rng(n_envs)
    moved, trunc_bootstraps = 0, 0
    for n_step in N_STEPS:
        kinds = r.kinds(n_step)
        occurred = set(np.unique(kinds[kinds >= 0]).tolist())
        assert occurred == expected, (n_step, [KINDS[c] for c in expected - occurred])
        idx = draw_minibatches(kinds, expected, r.len, n_envs, BATCH, NB, rng)
        wts = rng.uniform(0.1, 1.0, size=idx.size).astype(np.float32)
        trunc = np.nonzero(idx < r.len)[0]
        trunc = trunc[kinds[idx[trunc]] == TRUNCATION]
        for gamma in GAMMAS:
            for double in (False, True):
                y, G, mv = check_nstep_call(r, net, twin, target, w0, idx, wts, BATCH, NB, gamma, n_step, double, lr=LR)
                moved += mv
                trunc_bootstraps += differ(y[trunc], G[trunc]).size
    # controls: a truncated walk bootstraps (y != G), and the online action of double DQN changes between minibatches
    assert trunc_bootstraps > 0 and moved > 0, (trunc_bootstraps, moved)
    for x in (net, twin, target):
        x.close()
    r.close()


# ---------------------------------------------------------------- 2. both dense paths
def _draw_uniform(r, n, seed):
    """n indices with repeats and a few >= len, in random order"""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, r.len, size=n).astype(np.uint32)
    idx[rng.choice(n, 3, replace=False)] = [r.len, r.len + 5, 0xFFFFFFFF]
    return idx


@gpu
def test_32768_items_on_a_1m_ring(qlb):
    """4,096 envs, 2^20 transitions, wrapped, with episode ends: 32,768 items in 1 minibatch and in 2, vanilla and double. The
    network is its own twin (restored to w0): a second training network's scratch at this size would take 5 GB more."""
    n_envs, cap = 4096, 1 << 20
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=2, replay_capacity=cap, max_episode_steps=MAX_EP)
    env.step_random_device(cap // n_envs + 37)
    r = Ring(qlb, env)
    assert r.t_old > 0 and ((r.rec >> 2) & 1).any() and ((r.rec >> 16) & 1).any()
    w0 = _random_weights(qlb, 71)
    net, target = qlb.QNetwork(env, w0), qlb.QNetwork(env, _random_weights(qlb, 72))
    for nb in (1, 2):
        idx = _draw_uniform(r, 32768, nb)
        for double in (False, True):
            check_nstep_call(r, net, net, target, w0, idx, None, 32768 // nb, nb, 0.99, 5, double)
    net.close(); target.close()
    r.close()


@pytest.fixture(scope="module")
def dense_ring(qlb):
    """40,960 transitions of 1,024 envs with episode ends, a target network and two online networks"""
    env = qlb.BreakoutEnvironment(n_envs=1024, seed=8, replay_capacity=1024 * 40, max_episode_steps=25)
    env.step_many(np.random.default_rng(8).integers(0, 3, size=(70, 1024), dtype=np.uint8))
    r = Ring(qlb, env)
    w0 = _random_weights(qlb, 61)
    nets = SimpleNamespace(r=r, w0=w0, net=qlb.QNetwork(env, w0), twin=qlb.QNetwork(env, w0), target=qlb.QNetwork(env, _random_weights(qlb, 62)),
                           last_narrow=last_narrow(torch.cuda.get_device_properties(0).multi_processor_count))
    yield nets
    for x in (nets.net, nets.twin, nets.target):
        x.close()
    r.close()


@gpu
@pytest.mark.parametrize("double", [False, True])
@pytest.mark.parametrize("shape", range(4))
def test_dense_paths(qlb, dense_ring, shape, double):
    """dense_shapes on this device's SM count: the target network's forward of all items wide while the online and training
    forwards of one minibatch are narrow, and every forward wide (n_step 3, unweighted)."""
    d = dense_ring
    batch, nb = dense_shapes(d.last_narrow)[shape]
    idx = _draw_uniform(d.r, batch * nb, batch + nb)
    check_nstep_call(d.r, d.net, d.twin, d.target, d.w0, idx, None, batch, nb, 0.99, 3, double)


# ---------------------------------------------------------------- 3. scratch growth and reuse
GROWTH = [   # (call, batch, n_batches, double): n-step scratch grows, is reused when smaller, is freed by the plain call's larger
    ("nstep", 32, 1, False), ("nstep", 64, 3, True), ("nstep", 300, 2, False), ("nstep", 48, 2, True),   # y_cap and comes back
    ("plain", 512, 2, None), ("nstep", 200, 3, False), ("weighted", 100, 2, None), ("nstep", 700, 2, True),
]


@gpu
def test_scratch_growth_and_reuse_on_a_side_stream(qlb):
    """One network runs GROWTH on a torch side stream (non-blocking), with its Adam state reset before each call. After each
    call its loss, td, y and weights equal those of a fresh twin (same weights, fresh Adam state) that makes only that call on
    the legacy stream. The first call at each new size (an allocation) is the case under test."""
    env = qlb.BreakoutEnvironment(n_envs=256, seed=13, replay_capacity=256 * 16, max_episode_steps=11)
    env.step_many(np.random.default_rng(13).integers(0, 3, size=(30, 256), dtype=np.uint8))
    n_len = qlb.ReplayBuffer(env).len()
    net, target = qlb.QNetwork(env, _random_weights(qlb, 81)), qlb.QNetwork(env, _random_weights(qlb, 82))
    side = torch.cuda.Stream()
    rng = np.random.default_rng(13)

    def call(n, kind, idx, wt, batch, nb, double, stream):
        out = {k: torch.full((s,), float("nan"), device="cuda") for k, s in (("loss", nb), ("td", batch * nb), ("y", batch * nb))}
        if kind == "nstep":
            n.train_nstep_device(idx.data_ptr(), wt.data_ptr(), batch, nb, target, 0.99, 3, double, out["loss"].data_ptr(),
                                 out["td"].data_ptr(), out["y"].data_ptr(), stream)
        elif kind == "plain":
            n.train_device(idx.data_ptr(), batch, nb, None, target, 0.99, out["loss"].data_ptr(), stream)
        else:
            n.train_weighted_device(idx.data_ptr(), wt.data_ptr(), batch, nb, None, target, 0.99, out["loss"].data_ptr(),
                                    out["td"].data_ptr(), stream)
        return out

    for kind, batch, nb, double in GROWTH:
        n = batch * nb
        idx = _dev_idx(rng.integers(0, n_len, size=n))
        wt = torch.as_tensor(rng.uniform(0.1, 1.0, size=n).astype(np.float32), device="cuda")
        net.set_adam()
        twin = qlb.QNetwork(env, net.get_weights())
        twin.set_adam()
        got = call(net, kind, idx, wt, batch, nb, double, side.cuda_stream)
        side.synchronize()
        want = call(twin, kind, idx, wt, batch, nb, double, None)
        torch.cuda.synchronize()
        assert net.error() == 0 and twin.error() == 0
        for k in got:
            assert np.array_equal(_bits(got[k].cpu().numpy()), _bits(want[k].cpu().numpy())), (kind, batch, nb, k)
        assert not np.isnan(got["loss"].cpu().numpy()).any()
        assert _weights_equal(net, twin), (kind, batch, nb)
        twin.close()
    net.close(); target.close(); env.close()


# ---------------------------------------------------------------- 4b. consumers of submitted host steps
@pytest.fixture(params=["legacy", "side"])
def stream(request):
    return torch.cuda.default_stream() if request.param == "legacy" else torch.cuda.Stream()


SUBMITTED_CONSUMERS = {"replay_nstep": "qlc_replay_nstep", "train_nstep": "qlc_qnet_train_nstep"}


@gpu
@pytest.mark.parametrize("consumer", sorted(SUBMITTED_CONSUMERS))
def test_nstep_call_after_submitted_steps(qlb, stream, consumer):
    """test_stream_order.py's test_device_call_after_submitted_steps for the n-step calls: 16,384 envs x 32 steps x 6 submits
    (every slot of the ring rewritten), not waited for, then the call on the caller's stream. It must see every submitted
    step: compared with a twin env stepped synchronously (returns of 4,096 indices spread over the ring; a double-DQN update
    of 256 items, whose twin network was warmed up the same way). Without the ordering this fails likely, not certainly."""
    n = so.BIG_N
    envs = [qlb.BreakoutEnvironment(n_envs=n, seed=so.SEED, replay_capacity=n * so.BIG_T_CAP, max_episode_steps=40) for _ in range(2)]
    rng = np.random.default_rng(7)
    warm = rng.integers(0, 3, size=(so.BIG_T_CAP + 5, n), dtype=np.uint8)
    for e in envs:
        e.step_many(warm)
    k, subs = 32, 6
    acts = [qlb.PinnedArray((k, n), np.uint8) for _ in range(subs)]
    outs = [(qlb.PinnedArray((k, n), np.float32), qlb.PinnedArray((k, n), np.uint8)) for _ in range(subs)]
    for a in acts:
        a.array[:] = rng.integers(0, 3, size=(k, n), dtype=np.uint8)
    L = qlb.ReplayBuffer(envs[0]).capacity()
    m = 4096 if consumer == "replay_nstep" else 256
    idx = _dev_idx(np.concatenate([rng.integers(0, L, size=m - 64), np.arange(L - 64, L)]))
    w0, w1 = _random_weights(qlb, 91), _random_weights(qlb, 92)
    nets = [(qlb.QNetwork(e, w0), qlb.QNetwork(e, w1)) for e in envs] if consumer == "train_nstep" else None

    def run(i, s):
        if consumer == "replay_nstep":
            G, d, b = (torch.empty(m, dtype=t, device="cuda") for t in (torch.float32, torch.float32, torch.int32))
            qlb.ReplayBuffer(envs[i]).nstep_device(idx.data_ptr(), m, 5, 0.99, G.data_ptr(), d.data_ptr(), b.data_ptr(), s)
            return [G, d, b]
        out = [torch.empty(x, dtype=torch.float32, device="cuda") for x in (1, m, m)]
        nets[i][0].train_nstep_device(idx.data_ptr(), None, m, 1, nets[i][1], 0.99, 3, True, *[t.data_ptr() for t in out], s)
        return out

    for i in range(2):          # warm-up, the same on both: buffers allocated
        run(i, None)
    torch.cuda.synchronize()
    for a in acts:
        envs[1].step_many(a.array)
    want = run(1, None)
    torch.cuda.synchronize()
    for a, (r, d) in zip(acts, outs):
        envs[0].step_many_submit(a.array, r.array, d.array)
    got = run(0, stream.cuda_stream or None)
    torch.cuda.synchronize()
    envs[0].step_many_wait(0)
    for g, o in zip(got, want):
        so.assert_same(g.cpu().numpy(), o.cpu().numpy(), consumer)
    if nets:
        assert _weights_equal(nets[0][0], nets[1][0])
        for pair in nets:
            for x in pair:
                x.close()
    assert envs[0].time() == envs[1].time()
    for a in acts:
        a.free()
    for r, d in outs:
        r.free(); d.free()
    for e in envs:
        e.close()


# ---------------------------------------------------------------- 4c. host calls after an n-step update
SLEEP_S = 0.25       # the delay in front of every producer: test_stream_order.py's bound (>= 20 x the consumer) with room for
                     # a host call slowed by other work on the machine


@pytest.fixture(scope="module")
def cycles():
    """torch.cuda._sleep cycles for SLEEP_S seconds, measured with CUDA events (as in test_stream_order.py)"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20_000_000
    torch.cuda._sleep(n)
    a.record(); torch.cuda._sleep(n); b.record(); b.synchronize()
    return int(n * SLEEP_S * 1000.0 / a.elapsed_time(b))


def timed(f, twin):
    """test_stream_order.timed against SLEEP_S: a warm-up call of the consumer, then a timed one, each followed by the same
    call on the twin"""
    f()
    twin()
    t0 = time.perf_counter()
    f()
    dt = time.perf_counter() - t0
    twin()
    assert 20 * dt < SLEEP_S, "consumer takes %.1f ms: too slow for the sleep in front of the producer" % (dt * 1e3)


@gpu
@pytest.mark.parametrize("double", [False, True], ids=["vanilla", "double"])
@pytest.mark.parametrize("consumer", ["forward", "get_weights"])
def test_host_call_after_nstep_update(qlb, cycles, stream, consumer, double):
    """test_stream_order.py's test_host_call_after_device_update with train_nstep_device (n_step 3, 32 items spread over the
    ring) as the producer on stream A behind the sleep: forward() of the current stacks and get_weights() must see the
    updated weights. Checked against a twin updated with a synchronise; every buffer of both networks is warmed up first."""
    w = so.World(qlb, None, oracle=False)
    net, twin = so._nets(qlb, w)
    target = qlb.QNetwork(w.env, so.random_weights(qlb, 12))
    idx = _dev_idx(np.random.default_rng(4).integers(0, w.rb.len(), size=32))
    upd = lambda n, s: n.train_nstep_device(idx.data_ptr(), None, 32, 1, target, 0.99, 3, double, None, None, None, s)
    f = {"forward": lambda n: n.forward(), "get_weights": lambda n: n.get_weights()}[consumer]
    for n in (net, twin):
        upd(n, None); n.forward(); f(n)
    torch.cuda.synchronize()
    timed(lambda: f(net), lambda: f(twin))
    got, waited = so.host_after(torch, stream, cycles, lambda s: upd(net, s), lambda: f(net))
    upd(twin, None)
    torch.cuda.synchronize()
    want = f(twin)
    if consumer == "get_weights":
        so.assert_weights(got, want)
    else:
        for g, o in zip(got, want):
            so.assert_same(g, o)
    so.assert_waited(waited)
    net.close(); twin.close(); target.close(); w.close()
