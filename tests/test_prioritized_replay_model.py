"""Prioritized replay (per.cuh, qlc_per_*) against a numpy model of every transition's priority. The model keys priorities
by absolute time and env (T, e), not by ring slot, so it shares none of the library's slot arithmetic (leaf_of, slot_owner,
the sync intervals). After every step, update, sample and checkpoint load, the leaves the library reports in logical order,
the root and the running maximum must equal the model; the root bit for bit against a tree rebuilt from the model's own
leaves, so a wrong read order and a priority on the wrong transition both show. Sampled indices are compared exactly with
the numpy descent through the model's tree.

Shapes: one-env rings (a one-transition replay; a 300-step one), odd env counts (37 envs put sync interval ends inside
level-1 nodes; 300 envs), today's 64 x 16 ring, and the 1 M-transition benchmark ring (5 levels above the leaves). Their
step schedules reach sync catch-ups of 1, 2, 3 and 4 slot intervals, one of time_slots - 1 steps and full rewrites; a CPU
test restates per_sync's interval arithmetic to show that they do."""
import numpy as np
import pytest

from test_prioritized_replay import physical_leaves, reference_sample, tree_levels
from test_qnet_train import _random_weights

FLT_MIN = np.float32(1.17549435e-38)              # priority() floor: the smallest normal f32
FLT_MAX = np.finfo(np.float32).max
SUB_MIN = 2.0 ** -149                              # the smallest f32 subnormal
WEIGHT_RTOL = 2.0 ** -22

# (n_envs, replay_capacity): t_cap = capacity / n_envs, time_slots = t_cap + 4
SHAPES = [(1, 1), (1, 300), (37, 37 * 16), (300, 300 * 9), (64, 64 * 16)]
BENCH_SHAPE = (4096, 1 << 20)


def ring_dims(n_envs, capacity):
    t_cap = max(capacity // n_envs, 1)
    return t_cap, t_cap + 4


# ---------------------------------------------------------------- per_sync's interval arithmetic, restated
def sync_slot_intervals(synced, t0, gen0, t, gen, time_slots, t_cap):
    """The ring-slot intervals a sync at time t rewrites after a sync at (t0, gen0): ('full', [(0, time_slots)]) for a first
    sync, a load or a jump of time_slots steps or more; else ('catch-up', rows that left then rows that entered, each split
    at the wrap); None when nothing changed."""
    if synced and gen0 == gen and t0 == t:
        return None
    if not synced or gen0 != gen or t < t0 or t - t0 >= time_slots:
        return "full", [(0, time_slots)]
    slots = []

    def add_times(a, b):
        if b > a:
            s0, n = a % time_slots, b - a
            slots.extend([(s0, s0 + n)] if s0 + n <= time_slots else [(s0, time_slots), (0, s0 + n - time_slots)])

    add_times(t0 - t_cap if t0 > t_cap else 0, t - t_cap if t > t_cap else 0)
    add_times(t0, t)
    return "catch-up", slots


def schedule(time_slots, t_cap):
    """Step counts between syncs ('save' / 'load': a checkpoint of the env), run from t = 0 after a first sync there."""
    ts = time_slots
    return [1, 2, t_cap, "save", 1, 2, 3, ts - 1, 5, 6, ts // 2 + 1, ts - 2, 3, ts, 4, ts + 7, 2, "load", 3, ts - 1, 1]


def simulate_syncs(ops, time_slots, t_cap):
    """[(op, kind, slot intervals, t)] of the sync after each op of `ops`, starting with a sync at t = 0."""
    synced, t0, gen0 = True, 0, 0
    t, gen, saved, out = 0, 0, None, []
    for op in ops:
        if op == "save":
            saved = t
            continue
        if op == "load":
            t, gen = saved, gen + 1
        else:
            t += op
        r = sync_slot_intervals(synced, t0, gen0, t, gen, time_slots, t_cap)
        synced, t0, gen0 = True, t, gen
        if r is not None:
            out.append((op, r[0], r[1], t))
    return out


def tree_counts(n_envs, time_slots):
    """qlc_per_create's level sizes: leaves, then ceil(/32) until one node"""
    cnt = [time_slots * n_envs]
    while cnt[-1] > 1 or len(cnt) == 1:
        cnt.append(-(-cnt[-1] // 32))
    return cnt


@pytest.mark.parametrize("shape", SHAPES)
def test_schedules_reach_every_catch_up(shape):
    """CPU only: each shape's schedule makes per_sync catch up by 1, 2, 3 and 4 slot intervals, by exactly time_slots - 1
    steps, and rewrite everything after >= time_slots steps and after a load. At 37 envs some leaf interval starts or ends
    inside a level-1 node (off a multiple of 32), so the node intervals round inward and outward."""
    n_envs, cap = shape
    t_cap, ts = ring_dims(n_envs, cap)
    syncs = simulate_syncs(schedule(ts, t_cap), ts, t_cap)
    catch_ups = [(op, iv) for op, kind, iv, _ in syncs if kind == "catch-up"]
    assert {len(iv) for _, iv in catch_ups} == {1, 2, 3, 4}
    assert any(op == ts - 1 for op, _ in catch_ups)
    assert any(kind == "full" and op != "load" and op >= ts for op, kind, _, _ in syncs)
    assert any(kind == "full" and op == "load" for op, kind, _, _ in syncs)
    for _, iv in catch_ups:                                         # intervals stay inside the ring and cover op rows each way
        assert all(0 <= lo < hi <= ts for lo, hi in iv)
    leaf_ends = {x * n_envs for _, _, iv, _ in syncs for lo_hi in iv for x in lo_hi}
    if n_envs == 37:
        assert any(x % 32 for x in leaf_ends)


def test_tree_shapes():
    """CPU only: the levels above the leaves per shape; the 1 M-transition tree has 5, its 33-node level padded to 64."""
    levels = {s: tree_counts(s[0], ring_dims(*s)[1]) for s in SHAPES + [BENCH_SHAPE]}
    assert [len(levels[s]) - 1 for s in SHAPES] == [1, 2, 2, 3, 3]
    assert levels[BENCH_SHAPE] == [1064960, 33280, 1040, 33, 2, 1]
    assert [a.size for a in tree_levels(np.zeros(1064960, dtype=np.float32))] == levels[BENCH_SHAPE]


# ---------------------------------------------------------------- the model
def priority64(td, alpha, eps):
    """(|delta| + eps)^alpha in f64 with the floor at the smallest normal f32 (nan / inf where delta is not finite)"""
    with np.errstate(invalid="ignore", over="ignore"):
        p = np.power(np.abs(td.astype(np.float64)) + np.float64(np.float32(eps)), np.float64(np.float32(alpha)))
    return np.where(np.isfinite(p), np.maximum(p, np.float64(FLT_MIN)), p)


def ulp32(x64):
    return np.spacing(np.abs(np.asarray(x64, dtype=np.float64)).astype(np.float32)).astype(np.float64)


class PriorityModel:
    """Every transition's priority by (T, e) (DESIGN.md §13): a step adds rows at the running max and drops rows older than
    t - t_cap; an update zeroes the valid indices, raises the running max by each finite priority, then sets each index to
    the largest priority among its duplicates (a non-finite delta: the raised running max); indices >= len are ignored; a
    load puts every row at the running max. With alpha in {0, 1} every priority is exact; otherwise a freshly computed
    leaf and the running max must be within 1 f32 ulp of f64, and the model adopts the library's f32 values."""

    def __init__(self, n_envs, t_cap, alpha, eps, t=0):
        self.n, self.t_cap, self.alpha, self.eps = n_envs, t_cap, alpha, eps
        self.exact = alpha in (0.0, 1.0)
        self.mx = np.float32(1.0)
        self.pending, self.round_trips = None, 0
        self.load(t)

    def oldest(self):
        return self.t - self.t_cap if self.t > self.t_cap else 0

    def __len__(self):
        return (self.t - self.oldest()) * self.n

    def step(self, k):
        t1 = self.t + k
        o1 = t1 - self.t_cap if t1 > self.t_cap else 0
        for T in range(max(self.t, o1), t1):
            self.rows[T] = np.full(self.n, self.mx, dtype=np.float32)
        self.t = t1
        self.rows = {T: r for T, r in self.rows.items() if T >= o1}

    def load(self, t):
        self.t, self.rows = t, {}
        for T in range(self.oldest(), t):
            self.rows[T] = np.full(self.n, self.mx, dtype=np.float32)

    def leaves(self):
        if len(self) == 0:
            return np.zeros(0, dtype=np.float32)
        return np.concatenate([self.rows[T] for T in range(self.oldest(), self.t)])

    def _set_leaves(self, flat):
        for r, T in enumerate(range(self.oldest(), self.t)):
            self.rows[T] = flat[r * self.n:(r + 1) * self.n].copy()

    def update(self, idx, td):
        assert self.pending is None                     # check() after every update
        idx = np.asarray(idx, dtype=np.uint64).ravel()
        td = np.asarray(td, dtype=np.float32).ravel()
        ok = idx < np.uint64(len(self))
        idx, td = idx[ok].astype(np.int64), td[ok]
        fin = np.isfinite(td)
        p64 = priority64(td, self.alpha, self.eps)
        p32 = p64.astype(np.float32)
        mx64 = max(float(self.mx), float(p64[fin].max()) if fin.any() else 0.0)
        self.mx = max(self.mx, p32[fin].max()) if fin.any() else self.mx
        flat = self.leaves()
        e64 = np.zeros(flat.size)
        nonfinite = np.zeros(flat.size, dtype=bool)
        np.maximum.at(e64, idx[fin], p64[fin])
        nonfinite[idx[~fin]] = True
        touched = np.unique(idx)
        e32 = e64.astype(np.float32)
        e32[nonfinite] = self.mx
        flat[touched] = e32[touched]
        self._set_leaves(flat)
        self.pending = (touched[~nonfinite[touched]], e64[touched[~nonfinite[touched]]], touched[nonfinite[touched]], mx64)

    def check(self, per, env):
        """per.read() == the model: leaves, root and running max; a pending update's inexact values are adopted here"""
        leaves, total, mx = per.read()
        assert env.time() == self.t
        assert leaves.size == len(self)
        if self.pending is not None:
            fin_idx, fin64, nonfin_idx, mx64 = self.pending
            self.pending = None
            if not self.exact:
                assert abs(float(mx) - mx64) <= ulp32(mx64), (mx, mx64)
                assert np.all(np.abs(leaves[fin_idx].astype(np.float64) - fin64) <= ulp32(fin64))
                self.mx = np.float32(mx)
                flat = self.leaves()
                flat[fin_idx] = leaves[fin_idx]
                flat[nonfin_idx] = self.mx
                self._set_leaves(flat)
        model = self.leaves()
        bad = np.flatnonzero(leaves.view(np.uint32) != model.view(np.uint32))
        assert bad.size == 0, (self.t, bad[:8], leaves[bad[:8]], model[bad[:8]])
        assert np.float32(mx).view(np.uint32) == self.mx.view(np.uint32), (mx, self.mx)
        assert total == tree_levels(self.phys())[-1][0]
        return leaves

    def phys(self):
        return physical_leaves(self.leaves(), self.t, n_envs=self.n, t_cap=self.t_cap)


# ---------------------------------------------------------------- device helpers
def _stream(torch):
    return torch.cuda.current_stream().cuda_stream


def _update(torch, per, idx, td, stream=None):
    i = torch.as_tensor(np.asarray(idx, dtype=np.uint32).view(np.int32), device="cuda")
    d = torch.as_tensor(np.asarray(td, dtype=np.float32), device="cuda")
    per.update_device(i.data_ptr(), d.data_ptr(), i.numel(), stream if stream is not None else _stream(torch))
    torch.cuda.synchronize()


def _sample(torch, per, batch, n_batches, call_index, beta, stream=None):
    i = torch.empty((n_batches, batch), dtype=torch.int32, device="cuda")
    w = torch.empty((n_batches, batch), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    per.sample_device(batch, n_batches, call_index, beta, i.data_ptr(), w.data_ptr(), stream if stream is not None else _stream(torch))
    torch.cuda.synchronize()
    return i.cpu().numpy().view(np.uint32), w.cpu().numpy()


def _check_sample(model, seed, idx, w, batch, n_batches, call_index, beta):
    ref_idx, ref_w, _, _ = reference_sample(model.phys(), model.t, batch, n_batches, call_index, seed, beta, n_envs=model.n, t_cap=model.t_cap)
    assert np.array_equal(idx, ref_idx), (batch, n_batches, call_index, np.argwhere(idx != ref_idx)[:4])
    assert int(idx.max()) < len(model)
    err = np.abs(w.astype(np.float64) - ref_w)
    assert np.all(err <= WEIGHT_RTOL * ref_w + SUB_MIN), (beta, float((err / (WEIGHT_RTOL * ref_w + SUB_MIN)).max()))
    return ref_w


def _step(env, k, how, rng, torch):
    if how == "many":
        env.step_many(rng.integers(0, 3, size=(k, env.n_envs), dtype=np.uint8))
    else:
        env.step_random_device(k, stream=_stream(torch))
        torch.cuda.synchronize()


SPECIAL_TD = np.array([0.0, -0.0, SUB_MIN, 3e-39, FLT_MAX, -FLT_MAX, np.nan, np.inf, -np.inf], dtype=np.float32)


def _random_update(rng, n_len, extreme):
    """indices with duplicates and some >= len; deltas mostly ordinary, some 0, -0, subnormal and (extreme) +-FLT_MAX,
    NaN, +-inf"""
    m = int(rng.integers(1, max(2, min(3 * n_len, 3000))))
    idx = rng.integers(0, n_len + n_len // 8 + 2, size=m).astype(np.uint32)
    idx[rng.random(m) < 0.1] = idx[0]                                # duplicates
    idx[rng.random(m) < 0.02] = 0xFFFFFFFF
    td = (rng.standard_normal(m) * rng.choice([1e-3, 1.0, 50.0], size=m)).astype(np.float32)
    specials = SPECIAL_TD if extreme else SPECIAL_TD[:4]
    k = rng.random(m) < 0.1
    td[k] = rng.choice(specials, size=int(k.sum()))
    return idx, td


def _round_trip(torch, per, env, model, seed, rng):
    """sample, then update exactly the sampled indices with known deltas: exactly the leaves of those (T, e) change"""
    batch, nb, call = 129, 2, int(rng.integers(0, 1 << 40))
    idx, w = _sample(torch, per, batch, nb, call, 0.5)
    _check_sample(model, seed, idx, w, batch, nb, call, 0.5)
    before = model.check(per, env)
    model.round_trips += 1                                           # deltas above every earlier round trip's
    td = (1000.0 * model.round_trips + 0.5 * np.arange(idx.size)).astype(np.float32)
    _update(torch, per, idx.ravel(), td)
    model.update(idx.ravel(), td)
    after = model.check(per, env)
    u = np.unique(idx)
    expect = u[after[u] != before[u]]
    assert np.array_equal(np.flatnonzero(after != before), expect)
    if model.alpha > 0:
        assert expect.size == u.size
        # each changed leaf holds the priority of the largest delta given to it
        best = np.zeros(after.size, dtype=np.float32)
        np.maximum.at(best, idx.ravel().astype(np.int64), td)
        p = priority64(best[u], model.alpha, model.eps)
        assert np.all(np.abs(after[u].astype(np.float64) - p) <= ulp32(p))


# ---------------------------------------------------------------- 1-3. every shape, every catch-up, interleaved calls
@pytest.mark.gpu
@pytest.mark.parametrize("alpha", [0.6, 1.0])
@pytest.mark.parametrize("shape", SHAPES)
def test_interleaved_calls_follow_the_model(qlb, tmp_path, shape, alpha):
    torch = pytest.importorskip("torch")
    n_envs, cap = shape
    t_cap, ts = ring_dims(n_envs, cap)
    seed = (1 << 32) + 37 if n_envs == 37 else 1000 + n_envs          # one env key with a non-zero high word
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=cap)
    per = qlb.PrioritizedReplay(env, alpha=alpha, epsilon=1e-6)
    model = PriorityModel(n_envs, t_cap, alpha, 1e-6)
    model.check(per, env)                                             # the first sync, at t = 0
    rng = np.random.default_rng(n_envs * 7 + int(alpha * 10))
    calls = [0, (1 << 32) - 2, 12345, (1 << 32) - 2, 1 << 33]
    n_samples = n_round_trips = 0
    for k, op in enumerate(schedule(ts, t_cap)):
        if op == "save":
            env.save(str(tmp_path / "ckpt"))
            saved_t = env.time()
            continue
        if op == "load":
            env.load(str(tmp_path / "ckpt"))
            model.load(saved_t)
        else:
            _step(env, op, "many" if k % 2 else "random", rng, torch)
            model.step(op)
        if rng.random() < 0.5:                                        # the catch-up runs inside the next update or sample
            model.check(per, env)
        for _ in range(int(rng.integers(1, 4))):
            if rng.random() < 0.5:
                idx, td = _random_update(rng, len(model), extreme=rng.random() < 0.3)
                _update(torch, per, idx, td)
                model.update(idx, td)
            else:
                batch, nb = int(rng.choice([1, 7, 129, 1000])), int(rng.integers(1, 4))
                call, beta = calls[n_samples % len(calls)], float(rng.choice([0.0, 0.4, 1.0]))
                idx, w = _sample(torch, per, batch, nb, call, beta)
                _check_sample(model, seed, idx, w, batch, nb, call, beta)
                n_samples += 1
            model.check(per, env)
        if model.t > ts and model.oldest() % ts:                      # a ring that has wrapped
            _round_trip(torch, per, env, model, seed, rng)
            n_round_trips += 1
    assert n_samples >= 5 and n_round_trips >= 3
    per.close(); env.close()


@pytest.mark.gpu
def test_alpha_zero_keeps_every_priority_at_one(qlb):
    torch = pytest.importorskip("torch")
    n_envs, cap = 37, 37 * 16
    t_cap, ts = ring_dims(n_envs, cap)
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=5, replay_capacity=cap)
    per = qlb.PrioritizedReplay(env, alpha=0.0, epsilon=1e-6)
    model = PriorityModel(n_envs, t_cap, 0.0, 1e-6)
    rng = np.random.default_rng(0)
    for k, op in enumerate([3, ts - 1, 7, 2, ts + 1, 5]):
        _step(env, op, "many" if k % 2 else "random", rng, torch)
        model.step(op)
        idx, td = _random_update(rng, len(model), extreme=True)
        _update(torch, per, idx, td)
        model.update(idx, td)
        assert np.all(model.check(per, env) == 1.0)
        _round_trip(torch, per, env, model, 5, rng)
    per.close(); env.close()


# ---------------------------------------------------------------- 4. priority edges
@pytest.mark.gpu
def test_priority_floor_and_flt_max(qlb):
    """alpha = 1, epsilon = the smallest f32 subnormal: delta 0 gives the floor (the smallest normal f32), which keeps the
    transition in the replay and in the draws; +-FLT_MAX gives FLT_MAX and a running max of FLT_MAX.

    The sampler cannot draw a floor leaf in the same call as a FLT_MAX leaf: the floor's share of the total (~1e-76) is far
    below the 2^-32 resolution of a draw, so importance weights that underflow to subnormal or zero cannot arise from a
    sample. Weights are checked at the extremes that can arise: a replay of floor leaves only, and FLT_MAX leaves beside
    leaves 2^-8 as large, for beta in {0, 0.5, 1}; beta = 0 gives exactly 1.0."""
    torch = pytest.importorskip("torch")
    n_envs, cap = 37, 37 * 16
    t_cap, ts = ring_dims(n_envs, cap)
    seed = 17
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=cap)
    rng = np.random.default_rng(1)
    _step(env, t_cap + 7, "many", rng, torch)                          # wrapped
    eps = SUB_MIN
    per = qlb.PrioritizedReplay(env, alpha=1.0, epsilon=eps)
    model = PriorityModel(n_envs, t_cap, 1.0, eps, t=env.time())
    n = len(model)
    # every leaf at the floor
    _update(torch, per, np.arange(n), np.where(np.arange(n) % 2, np.float32(0.0), np.float32(-0.0)))
    model.update(np.arange(n), np.zeros(n, dtype=np.float32))
    leaves = model.check(per, env)
    assert np.all(leaves == FLT_MIN) and model.mx == 1.0
    for beta in (0.0, 0.5, 1.0):
        idx, w = _sample(torch, per, 1000, 2, 99, beta)
        _check_sample(model, seed, idx, w, 1000, 2, 99, beta)
        assert np.all(w == 1.0)
    # +-FLT_MAX
    big = np.arange(0, n, 5)
    td = np.where(big % 2, FLT_MAX, -FLT_MAX).astype(np.float32)
    _update(torch, per, big, td)
    model.update(big, td)
    leaves = model.check(per, env)
    assert np.all(leaves[big] == FLT_MAX) and model.mx == FLT_MAX
    assert np.all(leaves[np.setdiff1d(np.arange(n), big)] == FLT_MIN)
    # FLT_MAX beside leaves 2^-8 as large (FLT_MAX * 2^-8 is exact, delta + eps rounds to it); smaller ones are not drawn
    mid = np.arange(1, n, 5)
    tdm = np.full(mid.size, np.float32(FLT_MAX * 2.0 ** -8))
    _update(torch, per, mid, tdm)
    model.update(mid, tdm)
    model.check(per, env)
    seen_small = False
    for beta in (0.0, 0.5, 1.0):
        for call in (0, 1, (1 << 32) - 1):
            idx, w = _sample(torch, per, 129, 3, call, beta)
            ref_w = _check_sample(model, seed, idx, w, 129, 3, call, beta)
            if beta == 0.0:
                assert np.all(w == 1.0)
            seen_small |= bool((ref_w < 1e-2).any())
    assert seen_small                                                  # some minibatch held both magnitudes
    # new transitions enter at FLT_MAX
    _step(env, 2, "random", rng, torch)
    model.step(2)
    assert np.all(model.check(per, env)[-2 * n_envs:] == FLT_MAX)
    per.close(); env.close()


# ---------------------------------------------------------------- 5. the benchmark-size tree
@pytest.mark.gpu
def test_benchmark_size_tree(qlb):
    """4,096 envs, 2^20 transitions, wrapped: 1,064,960 leaves and 5 levels above them (33,280, 1,040, 33 padded to 64, 2,
    1). Every index updated with a distinct delta, then an exact sample of 32,768 x 2 with the Philox counter carrying into
    its high word, an incremental catch-up of 3 steps and a full rewrite of 260."""
    torch = pytest.importorskip("torch")
    n_envs, cap = BENCH_SHAPE
    t_cap, ts = ring_dims(n_envs, cap)
    seed = 77
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=cap)
    s = _stream(torch)
    env.step_random_device(t_cap + 45, stream=s)
    torch.cuda.synchronize()
    per = qlb.PrioritizedReplay(env)
    model = PriorityModel(n_envs, t_cap, 0.6, 1e-6, t=env.time())
    n = len(model)
    assert n == cap and model.oldest() % ts == 45
    td = (np.arange(1, n + 1, dtype=np.float64) * 2.0 ** -10).astype(np.float32)
    td = np.where(np.arange(n) % 3 == 0, -td, td)
    perm = np.random.default_rng(2).permutation(n).astype(np.uint32)
    _update(torch, per, perm, td[perm])
    model.update(perm, td[perm])
    leaves = model.check(per, env)
    assert np.unique(leaves).size > n // 2

    def sample_and_check():
        idx, w = _sample(torch, per, 32768, 2, (1 << 32) - 1, 0.5)
        _check_sample(model, seed, idx, w, 32768, 2, (1 << 32) - 1, 0.5)

    sample_and_check()
    env.step_random_device(3, stream=s)
    torch.cuda.synchronize()
    model.step(3)
    model.check(per, env)
    sample_and_check()
    env.step_random_device(ts, stream=s)
    torch.cuda.synchronize()
    model.step(ts)
    assert np.all(model.check(per, env) == model.mx)
    sample_and_check()
    per.close(); env.close()


# ---------------------------------------------------------------- 6. the learner's chain
@pytest.mark.gpu
@pytest.mark.parametrize("n_batches", [1, 2])
def test_learner_chain_feeds_td_errors_to_the_tree(qlb, n_batches):
    """TensorCoreLearner.train_prioritized (sample, weighted train, update on one stream) against a twin that runs the same
    chain by hand on networks with the same weights: the learner's indices equal the model's sample, its TD errors are
    Q(s)[a] - y of the twin's forward bit for bit (one minibatch per call), the tree holds the model updated with those TD
    errors, and the online weights stay equal to the twin's."""
    torch = pytest.importorskip("torch")
    from importlib import import_module
    torch_io = import_module("q-learning_b200.torch_io")
    n_envs, cap = 37, 37 * 16
    t_cap, ts = ring_dims(n_envs, cap)
    seed = 23
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=cap)
    rb = qlb.ReplayBuffer(env)
    env.step_many(np.random.default_rng(4).integers(0, 3, size=(t_cap - 3, n_envs), dtype=np.uint8))
    w0 = _random_weights(qlb, 31)
    alpha, gamma, batch = 0.6, 0.99, 32
    learner = torch_io.TensorCoreLearner(env, w0, gamma=gamma, per_alpha=alpha)
    online, target = qlb.QNetwork(env, w0), qlb.QNetwork(env, w0)
    online.set_adam(lr=2.5e-4, clipnorm=1.0)
    twin_per = qlb.PrioritizedReplay(env, alpha)
    model = PriorityModel(n_envs, t_cap, alpha, 1e-6, t=env.time())
    s = _stream(torch)
    idx_t = torch.empty((n_batches, batch), dtype=torch.int32, device="cuda")
    w_t = torch.empty((n_batches, batch), dtype=torch.float32, device="cuda")
    td_t = torch.empty((n_batches, batch), dtype=torch.float32, device="cuda")
    for it, k in enumerate([0, 5, 2, 11, ts - 1, 3]):
        if k:
            env.step_random_device(k, stream=s)
            model.step(k)
        call, beta = (1 << 32) - 1 + it, 0.4 + 0.1 * it
        ref_idx, ref_w, _, _ = reference_sample(model.phys(), model.t, batch, n_batches, call, seed, beta, n_envs=n_envs, t_cap=t_cap)
        torch.cuda.synchronize()
        if n_batches == 1:
            q, _, _ = online.forward(ref_idx.ravel(), 0)
            _, _, max_q = target.forward(ref_idx.ravel(), 1)
            smp = rb.get_many(ref_idx.ravel(), want_state=False, want_next=False)
            y = smp.reward + max_q * np.float32(gamma)
            y = np.where(smp.done != 0, smp.reward, y).astype(np.float32)
            ref_td = (q[np.arange(batch), smp.action.astype(np.int64)] - y).astype(np.float32)
        learner.train_prioritized(batch, n_batches, call, beta)
        twin_per.sample_device(batch, n_batches, call, beta, idx_t.data_ptr(), w_t.data_ptr(), s)
        online.train_weighted_device(idx_t.data_ptr(), w_t.data_ptr(), batch, n_batches, None, target, gamma, None, td_t.data_ptr(), s)
        twin_per.update_device(idx_t.data_ptr(), td_t.data_ptr(), batch * n_batches, s)
        torch.cuda.synchronize()
        assert learner.error() == 0 and online.error() == 0
        l_idx, l_w, l_td = (b.cpu().numpy() for b in learner._per_bufs)
        assert np.array_equal(l_idx.view(np.uint32), ref_idx), it
        assert np.all(np.abs(l_w.astype(np.float64) - ref_w) <= WEIGHT_RTOL * ref_w + SUB_MIN)
        assert np.array_equal(idx_t.cpu().numpy(), l_idx) and np.array_equal(w_t.cpu().numpy().view(np.uint32), l_w.view(np.uint32))
        assert np.array_equal(td_t.cpu().numpy().view(np.uint32), l_td.view(np.uint32)), it
        if n_batches == 1:
            assert np.array_equal(l_td.ravel().view(np.uint32), ref_td.view(np.uint32)), it
        model.update(l_idx.view(np.uint32).ravel(), l_td.ravel())
        leaves = model.check(learner.per, env)
        assert np.array_equal(twin_per.read()[0].view(np.uint32), leaves.view(np.uint32))
        wl, wt = learner.get_weights(), online.get_weights()
        for name in qlb.QNET_SHAPES:
            assert np.array_equal(wl[name].view(np.uint32), wt[name].view(np.uint32)), (it, name)
    assert model.oldest() > 0 and model.oldest() % ts                 # the ring wrapped during the chain
    twin_per.close(); online.close(); target.close(); learner.close(); env.close()


# ---------------------------------------------------------------- 7. stream order at creation
@pytest.mark.gpu
def test_first_sample_on_a_side_stream(qlb):
    """The first call of a new PrioritizedReplay is a sample on a fresh non-blocking stream: it must see the initialised
    block (zero leaves, running max 1.0). Run once; a single run cannot show the race reliably."""
    torch = pytest.importorskip("torch")
    n_envs, cap = 37, 37 * 16
    t_cap, _ = ring_dims(n_envs, cap)
    seed = 3
    env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=seed, replay_capacity=cap)
    env.step_many(np.random.default_rng(0).integers(0, 3, size=(t_cap + 5, n_envs), dtype=np.uint8))
    model = PriorityModel(n_envs, t_cap, 0.6, 1e-6, t=env.time())
    side = torch.cuda.Stream()
    per = qlb.PrioritizedReplay(env)
    idx, w = _sample(torch, per, 1000, 3, 7, 0.5, stream=side.cuda_stream)
    _check_sample(model, seed, idx, w, 1000, 3, 7, 0.5)
    assert np.all(w == 1.0)
    model.check(per, env)
    per.close(); env.close()
