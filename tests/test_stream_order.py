"""Stream order between the caller's stream and the library's own: each call must see the work that earlier calls on the same
handle queued (include/ql_cuda.h, "Stream order"). The host-buffer calls run on the env's own non-blocking stream, the
device-pointer calls on the caller's; nothing in CUDA orders the two, so the library does.

How a race becomes a deterministic reorder: on the caller's stream A the test queues a bounded `torch.cuda._sleep`, then the
producer call, then a torch event E. E still pending when the consumer is called is the control: it shows the hazard was
reached. A synchronous host consumer must have waited for E when it returns, and its outputs must equal the values computed
in the safe order (the oracle, or the same network / a twin run with a synchronise in between). Without the ordering the
host consumer runs entirely before the producer, so its results are wrong and nothing runs concurrently. Every case runs
with A = the legacy default stream and A = a torch side stream.

No case lets two launches that write the same env, network or tree overlap even without the ordering: host consumers are
synchronous and warmed up (no buffer growth, which synchronises the device), and every env a consumer steps is below
16 x SMs envs or steps fewer than 8 steps at a time, so none of its launches is cooperative and waits for the SM the
sleep holds."""
import os
import re
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

N, SEED, T_CAP, MAX_EP = 96, 5, 8, 9       # a small wrapped ring (12 time slots); episodes end every few steps
SLEEP_S = 0.1                             # the delay in front of every producer; >= 20 x the slowest consumer (checked)
BIG_N, BIG_T_CAP = 16384, 8               # pipelined submits: above 96 x SMs, so no step launch is cooperative

# ---------------------------------------------------------------- 6. every entry point has an ordering rule
ASYNC = {   # queued on the caller's stream after submitted host steps; caller_done recorded after the launches
    "qlc_env_step", "qlc_env_step_random", "qlc_env_obs", "qlc_obs_gather", "qlc_replay_sample", "qlc_replay_gather",
    "qlc_replay_sample_gather", "qlc_stats_export", "qlc_qnet_forward", "qlc_qnet_train", "qlc_qnet_train_weighted",
    "qlc_per_sample", "qlc_per_update", "qlc_replay_nstep", "qlc_qnet_train_nstep",
}
HOST_ORDERED = {   # host buffers on the env's own stream, which first waits for caller_done
    "qlc_env_step_host", "qlc_env_step_host_submit", "qlc_env_obs_host", "qlc_obs_gather_host", "qlc_replay_sample_host",
    "qlc_replay_gather_host", "qlc_replay_sample_gather_host", "qlc_qnet_forward_host", "qlc_qnet_train_host",
    "qlc_qnet_debug_grads", "qlc_qnet_debug_grads_weighted",
}
SYNCHRONISES = {   # cudaDeviceSynchronize before (and where they write, after) their own work
    "qlc_env_create", "qlc_env_destroy", "qlc_env_reset", "qlc_env_read_state", "qlc_env_lives_host", "qlc_env_error_flags",
    "qlc_replay_action_counts", "qlc_stats_read", "qlc_env_save", "qlc_env_load", "qlc_comm_init", "qlc_comm_destroy",
    "qlc_qnet_create", "qlc_qnet_set_weights", "qlc_qnet_destroy", "qlc_qnet_error", "qlc_qnet_set_adam", "qlc_qnet_get_weights",
    "qlc_per_create", "qlc_per_destroy", "qlc_per_read_host",
}
EXEMPT = {
    "qlc_version": "constant", "qlc_build_info": "constant", "qlc_last_error_string": "host string",
    "qlc_device_count": "no handle", "qlc_host_alloc": "no handle", "qlc_host_free": "no handle",
    "qlc_sync": "synchronises the caller's stream: what it is for",
    "qlc_env_step_host_wait": "waits for the handle's own submitted steps: what it is for",
    "qlc_env_state_view": "returns device pointers; the caller orders its own reads of them",
    "qlc_env_goal_mean": "constant", "qlc_env_time": "host counter", "qlc_replay_len": "host counter",
    "qlc_replay_capacity": "host counter",
    "qlc_stats_push": "host-side reward window", "qlc_stats_mean": "host-side reward window",
    "qlc_stats_min": "host-side reward window", "qlc_stats_window": "host-side reward window",
    "qlc_comm_unique_id": "no handle", "qlc_comm_info": "host fields",
    "qlc_stats_allreduce": "the communicator's side stream, ordered by its own events (tested in test_round2)",
    "qlc_stats_global": "reads the communicator's host mirror",
    "qlc_debug_collision_wall": "debug hook: own buffers, synchronous copies",
    "qlc_debug_collision_rect": "debug hook: own buffers, synchronous copies",
    "qlc_debug_collision_rect_batch": "debug hook: own buffers, synchronous copies",
    "qlc_debug_gemm_bf16": "debug hook: own buffers, synchronous copies",
}


def test_every_entry_point_has_an_ordering_rule():
    """A new qlc_* function in the header must be placed in one of the tables above."""
    text = open(os.path.join(ROOT, "include", "ql_cuda.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    declared = set(re.findall(r"\b(qlc_\w+)\s*\(", text))
    tables = [ASYNC, HOST_ORDERED, SYNCHRONISES, set(EXEMPT)]
    listed = set().union(*tables)
    assert sum(len(t) for t in tables) == len(listed), "an entry point is listed twice"
    assert declared - listed == set(), "entry points without an ordering rule"
    assert listed - declared == set(), "listed entry points the header does not declare"
    assert len(declared) >= 70


# ---------------------------------------------------------------- helpers
@pytest.fixture(scope="module")
def torch():
    t = pytest.importorskip("torch")
    if not t.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return t


@pytest.fixture(scope="module")
def cycles(torch):
    """torch.cuda._sleep cycles for SLEEP_S seconds, measured with CUDA events."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20_000_000
    torch.cuda._sleep(n)
    a.record(); torch.cuda._sleep(n); b.record(); b.synchronize()
    return int(n * SLEEP_S * 1000.0 / a.elapsed_time(b))


@pytest.fixture(params=["legacy", "side"])
def stream(request, torch):
    return torch.cuda.default_stream() if request.param == "legacy" else torch.cuda.Stream()


def timed(f, twin=None):
    """Two warm-up calls of a consumer (the first allocates its staging), each followed by the same call on the twin, if
    any; the sleep must be at least 20 times as long as the second."""
    f()
    if twin:
        twin()
    t0 = time.perf_counter()
    out = f()
    dt = time.perf_counter() - t0
    if twin:
        twin()
    assert_fast(dt)
    return out


def assert_fast(dt):
    assert 20 * dt < SLEEP_S, "consumer takes %.1f ms: too slow for the sleep in front of the producer" % (dt * 1e3)


def timed_step(w, k):
    """Warm-up host steps of k steps on the env and the oracle; the second env step (alone) is timed like a consumer."""
    w.step_host(k)
    a = w.acts(k)
    t0 = time.perf_counter()
    w.env.step_many(a)
    assert_fast(time.perf_counter() - t0)
    w.follow(a)


def queue_producer(torch, A, cycles, producer):
    """sleep, producer, event E on A; returns E, still pending (the control)."""
    torch.cuda.synchronize()
    with torch.cuda.stream(A):
        torch.cuda._sleep(cycles)
    producer(A.cuda_stream or None)
    ev = torch.cuda.Event()
    ev.record(A)
    assert not ev.query(), "control: the producer finished before the consumer was called"
    return ev


def host_after(torch, A, cycles, producer, consumer):
    """The hazard for a synchronous host consumer: (its outputs, whether the producer had finished when it returned). The
    callers compare the outputs first, then assert_waited: a reordered call shows in the values as well."""
    ev = queue_producer(torch, A, cycles, producer)
    out = consumer()
    waited = ev.query()
    torch.cuda.synchronize()
    return out, waited


def assert_waited(waited):
    assert waited, "the host call returned before the work queued ahead of it had finished"


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def assert_same(got, want, what=""):
    assert got.shape == want.shape and np.array_equal(bits(got), bits(want)), what


def assert_sample(g, o, state=True, nxt=True):
    if state:
        assert_same(g.state, o["state"], "state")
    if nxt:
        assert_same(g.state_next, o["state_next"], "state_next")
    assert_same(g.reward, o["reward"], "reward"); assert_same(g.action, o["action"], "action"); assert_same(g.done, o["done"], "done")


class World:
    """An env with a wrapped replay ring and the oracle in lockstep."""

    def __init__(self, qlb, O, n=N, t_cap=T_CAP, seed=SEED, oracle=True):
        self.qlb, self.O, self.n, self.seed = qlb, O, n, seed
        self.env = qlb.BreakoutEnvironment(n_envs=n, seed=seed, replay_capacity=n * t_cap, max_episode_steps=MAX_EP)
        self.ora = O.VecEnv(n, seed=seed, replay_capacity=n * t_cap, max_episode_steps=MAX_EP) if oracle else None
        self.rb = qlb.ReplayBuffer(self.env)
        self.rng = np.random.default_rng(seed)
        self.step_host(t_cap + 5)

    def acts(self, k):
        return self.rng.integers(0, 3, size=(k, self.n), dtype=np.uint8)

    def follow(self, acts):
        out = [self.ora.step(a) for a in acts]
        return np.stack([r for r, _ in out]), np.stack([d for _, d in out])

    def step_host(self, k):
        a = self.acts(k)
        r, d = self.env.step_many(a)
        if self.ora is not None:
            ro, do = self.follow(a)
            assert_same(r, ro); assert_same(d, do)

    def newest(self, n):
        L = self.rb.len()
        return np.arange(L - n, L, dtype=np.uint32)

    def handles(self, t):
        """handles of every env's observation at time t, which the oracle has reached"""
        k = self.ora.state()["episode_step"]
        return np.array([(t, int(k[e]), e) for e in range(self.n)], dtype=self.qlb.OBS_HANDLE_DTYPE)

    def close(self):
        self.env.close()
        if self.ora is not None:
            self.ora.close()


class DeviceStep:
    """Producer: step_device of k steps, or step_random_device. Its actions are known up front (the random phase draws from
    the oracle's 'ACTI' stream), so follow() moves the oracle ahead before the hazard."""

    def __init__(self, torch, w, kind):
        self.w, self.kind = w, kind
        self.k = {"step3": 3, "step40": 40, "random": 5}[kind]
        if kind == "random":
            self.acts = w.O.synthetic_actions(w.seed, 0, w.n, w.env.time(), self.k)
            self.dev = torch.empty((self.k, w.n), dtype=torch.uint8, device="cuda")
        else:
            self.acts = w.acts(self.k)
            self.dev = torch.from_numpy(self.acts).cuda()

    def __call__(self, s):
        if self.kind == "random":
            self.w.env.step_random_device(self.k, self.dev.data_ptr(), None, None, s)
        else:
            self.w.env.step_device(self.dev.data_ptr(), self.k, None, None, s)

    def follow(self):
        self.w.follow(self.acts)

    def check(self):
        if self.kind == "random":
            assert_same(self.dev.cpu().numpy(), self.acts, "the random phase's actions")


def random_weights(qlb, seed):
    rng = np.random.default_rng(seed)
    w = {}
    for name, shape in qlb.QNET_SHAPES.items():
        lim = np.sqrt(6.0 / (int(np.prod(shape[:-1])) + shape[-1])) if name.endswith("kernel") else 0.1
        w[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)
    return w


def assert_weights(a, b):
    for name in a:
        assert_same(a[name], b[name], name)


# ---------------------------------------------------------------- 1. host call after a device step
# each consumer: warm it up, return (call, check); check(got) compares with the oracle, already moved past the producer
def _get_many(layout, n, reuse=False, want_state=True, want_next=True):
    def make(qlb, w):
        idx = w.newest(n)
        f = lambda: w.rb.get_many(idx, layout, want_state=want_state, want_next=want_next, reuse=reuse)
        timed(f)
        o_layout = "u8" if layout == qlb.LAYOUT_U8_BHYX else "f32"
        return f, lambda got: assert_sample(got, w.ora.get_many(idx, o_layout), want_state, want_next)
    return make


def _sample(qlb, w):
    f = lambda: w.rb.sample(32, qlb.LAYOUT_F32_BXYH, call_index=9)
    timed(f)

    def check(got):
        idx, g = got
        assert_same(idx, w.O.sample_distinct(w.seed, 9, w.rb.len(), 32))
        assert_sample(g, w.ora.get_many(idx, "f32"))
    return f, check


def _obs(layout):
    def make(qlb, w):
        f = lambda: w.env.obs(layout)
        timed(f)

        def check(got):
            want = w.ora.obs_u8() if layout == qlb.LAYOUT_U8_BHYX else w.ora.obs_f32()
            assert_same(got, want if layout != qlb.LAYOUT_U8_BXYH else want.astype(np.uint8))
        return f, check
    return make


def _obs_gather(qlb, w):
    timed(lambda: w.env.obs_gather(w.handles(w.env.time()), qlb.LAYOUT_U8_BHYX))
    return None, None          # the handles name the newest time: built once the oracle has moved ahead (see the test)


def _step_many(qlb, w):
    timed_step(w, 3)
    return None, None          # checked against the oracle after the producer's actions (see the test)


CONSUMERS = {
    "get_many_u8": _get_many(0, 40),
    "get_many_u8_pinned": _get_many(0, 40, reuse=True),
    "get_many_f32_32": _get_many(1, 32),
    "get_many_f32_96": _get_many(1, 96),
    "get_many_next_only": _get_many(1, 32, want_state=False),
    "get_many_scalars": _get_many(1, 40, want_state=False, want_next=False),
    "sample": _sample,
    "obs_u8": _obs(0), "obs_f32": _obs(1), "obs_u8_xyh": _obs(2),
    "obs_gather": _obs_gather,
    "step_many": _step_many,
}


@pytest.mark.gpu
@pytest.mark.parametrize("producer", ["step3", "step40", "random"])
@pytest.mark.parametrize("consumer", sorted(CONSUMERS))
def test_host_call_after_device_step(qlb, O, torch, cycles, stream, producer, consumer):
    assert (qlb.LAYOUT_U8_BHYX, qlb.LAYOUT_F32_BXYH, qlb.LAYOUT_U8_BXYH) == (0, 1, 2)
    w = World(qlb, O)
    call, check = CONSUMERS[consumer](qlb, w)
    prod = DeviceStep(torch, w, producer)
    if consumer == "step_many":
        a2 = w.acts(3)
        prod.follow()
        want = w.follow(a2)
        (r, d), waited = host_after(torch, stream, cycles, prod, lambda: w.env.step_many(a2))
        assert_same(r, want[0], "reward"); assert_same(d, want[1], "done")
        assert_same(w.env.obs(0), w.ora.obs_u8(), "observation after the host steps")
    elif consumer == "obs_gather":
        prod.follow()
        h = w.handles(w.env.time() + prod.k)
        got, waited = host_after(torch, stream, cycles, prod, lambda: w.env.obs_gather(h, qlb.LAYOUT_U8_BHYX))
        assert_same(got, w.ora.obs_u8())
    else:
        prod.follow()
        got, waited = host_after(torch, stream, cycles, prod, call)
        check(got)
    assert_waited(waited)
    prod.check()
    assert w.env.error_flags() == 0
    w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("producer", ["step3", "random"])
def test_synchronising_calls_after_device_step(qlb, O, torch, cycles, stream, producer, tmp_path):
    """read_state, stats, lives, error_flags, actions(), save and PrioritizedReplay.read synchronise the device themselves."""
    w = World(qlb, O)
    per = qlb.PrioritizedReplay(w.env)
    per.read()
    calls = {
        "read_state": lambda: w.env.read_state(),
        "stats": lambda: w.env.stats(),
        "lives": lambda: w.env.lives(),
        "error_flags": lambda: w.env.error_flags(),
        "actions": lambda: w.rb.actions(),
        "save": lambda: w.env.save(str(tmp_path / "ckpt")),
        "per_read": lambda: per.read(),
    }
    for name, f in calls.items():
        prod = DeviceStep(torch, w, producer)
        prod.follow()
        got, waited = host_after(torch, stream, cycles, prod, f)
        prod.check()
        st = w.ora.state()
        if name == "read_state":
            for k in ("ball_cx", "ball_cy", "pad_min_x", "bricks", "score", "episode_step", "finished"):
                assert_same(got[k], st[k], k)
        elif name == "stats":
            o = w.ora.stats()
            assert (got["sum_return"], got["episodes"]) == (o["sum_return"], o["episodes"])
        elif name == "lives":
            assert_same(got, (st["finished"] == 0).astype(np.uint8))
        elif name == "error_flags":
            assert got == 0
        elif name == "actions":
            assert_same(got, w.ora.action_histogram())
        elif name == "save":
            twin = qlb.BreakoutEnvironment(n_envs=N, seed=SEED, replay_capacity=N * T_CAP, max_episode_steps=MAX_EP)
            twin.load(str(tmp_path / "ckpt"))
            assert twin.time() == w.env.time()
            assert_same(twin.obs(0), w.ora.obs_u8())
            twin.close()
        else:
            leaves, total, mx = got
            assert leaves.size == w.rb.len() and np.all(leaves == 1.0) and total == leaves.size and mx == 1.0
        assert_waited(waited)
    per.close(); w.close()


# ---------------------------------------------------------------- Q-network consumers
def _nets(qlb, w, k=2):
    wt = random_weights(qlb, 11)
    return [qlb.QNetwork(w.env, wt) for _ in range(k)]


@pytest.mark.gpu
@pytest.mark.parametrize("consumer", ["forward", "forward_next", "train", "debug_grads"])
def test_qnet_host_call_after_device_step(qlb, O, torch, cycles, stream, consumer):
    """QNetwork.forward() (current stacks), forward(idx, 1), train and debug_grads on the newest transitions see the step queued
    before them: compared with the same call (or a twin network) after a synchronise."""
    w = World(qlb, O, oracle=False)
    net, twin = _nets(qlb, w)
    idx = w.newest(32)
    y = np.random.default_rng(1).uniform(-2, 2, 32).astype(np.float32)
    calls = {
        "forward": lambda n: n.forward(),
        "forward_next": lambda n: n.forward(idx, 1),
        "train": lambda n: n.train(idx, y),
        "debug_grads": lambda n: n.debug_grads(idx, y),
    }
    f = calls[consumer]
    timed(lambda: f(net), lambda: f(twin))
    timed(lambda: net.forward(), lambda: twin.forward())            # both forward sizes allocated: no growth inside the hazard
    a = torch.from_numpy(w.acts(3)).cuda()
    got, waited = host_after(torch, stream, cycles, lambda s: w.env.step_device(a.data_ptr(), 3, None, None, s), lambda: f(net))
    want = f(twin if consumer == "train" else net)
    if consumer == "debug_grads":
        assert_weights(got, want)
    elif consumer == "train":
        assert_same(got, want, "loss"); assert_weights(net.get_weights(), twin.get_weights())
    else:
        for g, o in zip(got, want):
            assert_same(g, o)
    assert_waited(waited)
    net.close(); twin.close(); w.close()


# ---------------------------------------------------------------- 2. host call after a device update
@pytest.mark.gpu
@pytest.mark.parametrize("consumer", ["forward", "get_weights", "train", "debug_grads"])
def test_host_call_after_device_update(qlb, O, torch, cycles, stream, consumer):
    """train_device queued on the caller's stream, then a host call of the same network: it must see the updated weights
    (Adam steps do not commute, so a reordered train shows in the bits). Checked against a twin run with a synchronise."""
    w = World(qlb, O, oracle=False)
    net, twin = _nets(qlb, w)
    idx_h = w.newest(64)
    y_h = np.random.default_rng(2).uniform(-2, 2, 64).astype(np.float32)
    idx, y = torch.from_numpy(idx_h[:32].view(np.int32)).cuda(), torch.from_numpy(y_h[:32]).cuda()
    calls = {
        "forward": lambda n: n.forward(),
        "get_weights": lambda n: n.get_weights(),
        "train": lambda n: n.train(idx_h[32:], y_h[32:]),
        "debug_grads": lambda n: n.debug_grads(idx_h[32:], y_h[32:]),
    }
    f = calls[consumer]
    for n in (net, twin):          # warm-up, the same on both: scratch for 32 items, forward buffers for all envs
        n.train(idx_h[:32], y_h[:32]); n.forward(); f(n)
    timed(lambda: f(net), lambda: f(twin))
    upd = lambda n, s: n.train_device(idx.data_ptr(), 32, 1, y.data_ptr(), None, 0.99, None, s)
    got, waited = host_after(torch, stream, cycles, lambda s: upd(net, s), lambda: f(net))
    upd(twin, None); torch.cuda.synchronize()
    want = f(twin)
    if consumer in ("get_weights", "debug_grads"):
        assert_weights(got, want)
    elif consumer == "train":
        assert_same(got, want, "loss"); assert_weights(net.get_weights(), twin.get_weights())
    else:
        for g, o in zip(got, want):
            assert_same(g, o)
    assert_waited(waited)
    net.close(); twin.close(); w.close()


# ---------------------------------------------------------------- 3. host write after a device read
@pytest.mark.gpu
@pytest.mark.parametrize("reader", ["gather_device", "sample_gather_device", "obs_device", "forward_device", "stats_export"])
def test_host_step_after_device_read(qlb, O, torch, cycles, stream, reader):
    """A device call reads the ring (the oldest transitions, the current stacks) or the statistics; a host step_many of 6
    steps then overwrites them. The device outputs must be those from before the host step."""
    w = World(qlb, O)
    timed_step(w, 6)           # before the expected values are taken: these steps move the ring and the oracle too
    ring = torch.empty((64, 4, 84, 84), dtype=torch.uint8, device="cuda")
    ring2 = torch.empty_like(ring)
    sc = [torch.empty(64, dtype=t, device="cuda") for t in (torch.float32, torch.uint8, torch.uint8)]
    if reader in ("gather_device", "sample_gather_device"):
        idx_h = np.arange(64, dtype=np.uint32) if reader == "gather_device" else w.O.sample_distinct(SEED, 4, w.rb.len(), 64)
        idx = torch.from_numpy(idx_h.view(np.int32)).cuda()
        want = w.ora.get_many(idx_h, "u8")
        if reader == "gather_device":
            read = lambda s: w.rb.gather_device(idx.data_ptr(), 64, 0, ring.data_ptr(), ring2.data_ptr(), *[t.data_ptr() for t in sc], stream=s)
        else:
            read = lambda s: w.rb.sample_gather_device(64, 1, 4, 0, idx.data_ptr(), ring.data_ptr(), ring2.data_ptr(), *[t.data_ptr() for t in sc], stream=s)
    elif reader == "obs_device":
        want = w.ora.obs_u8()
        out = torch.empty((N, 4, 84, 84), dtype=torch.uint8, device="cuda")
        read = lambda s: w.env.obs_device(0, out.data_ptr(), s)
    elif reader == "forward_device":
        net = _nets(qlb, w, 1)[0]
        want = net.forward()
        q, act = torch.empty((N, 3), dtype=torch.float32, device="cuda"), torch.empty(N, dtype=torch.uint8, device="cuda")
        read = lambda s: net.forward_device(None, N, 0, q.data_ptr(), act.data_ptr(), None, s)
    else:
        st = w.env.stats()
        want = np.array([st["sum_return"], st["episodes"], st["steps"], -float(st["min_return"]), st["max_return"]], dtype=np.float64)
        ex = torch.empty(5, dtype=torch.float64, device="cuda")
        read = lambda s: w.env.stats_export(ex.data_ptr(), s)
    a = w.acts(6)
    _, waited = host_after(torch, stream, cycles, read, lambda: w.env.step_many(a))
    if reader in ("gather_device", "sample_gather_device"):
        assert_same(ring.cpu().numpy(), want["state"]); assert_same(ring2.cpu().numpy(), want["state_next"])
        for t, k in zip(sc, ("reward", "action", "done")):
            assert_same(t.cpu().numpy(), want[k], k)
        if reader == "sample_gather_device":
            assert_same(idx.cpu().numpy().view(np.uint32), idx_h)
    elif reader == "obs_device":
        assert_same(out.cpu().numpy(), want)
    elif reader == "forward_device":
        assert_same(q.cpu().numpy(), want[0]); assert_same(act.cpu().numpy(), want[1])
        net.close()
    else:
        assert_same(ex.cpu().numpy(), want)
        after = w.env.stats()
        assert after["episodes"] > st["episodes"], "the host steps must change the statistics for this case to mean anything"
    w.follow(a)
    assert_same(w.env.obs(0), w.ora.obs_u8())
    assert_waited(waited)
    w.close()


@pytest.mark.gpu
def test_host_train_after_device_forward(qlb, O, torch, cycles, stream):
    """forward_device of replay transitions, then a host train of the same network: Q comes from the weights before the
    update, and the update equals a twin's."""
    w = World(qlb, O, oracle=False)
    net, twin = _nets(qlb, w)
    idx_h = w.newest(32)
    y = np.random.default_rng(3).uniform(-2, 2, 32).astype(np.float32)
    idx = torch.from_numpy(idx_h.view(np.int32)).cuda()
    timed(lambda: net.train(idx_h, y), lambda: twin.train(idx_h, y))
    want = net.forward(idx_h)
    q = torch.empty((32, 3), dtype=torch.float32, device="cuda")
    loss, waited = host_after(torch, stream, cycles, lambda s: net.forward_device(idx.data_ptr(), 32, 0, q.data_ptr(), None, None, s), lambda: net.train(idx_h, y))
    assert_same(q.cpu().numpy(), want[0])
    assert_same(loss, twin.train(idx_h, y), "loss")
    assert_weights(net.get_weights(), twin.get_weights())
    assert_waited(waited)
    net.close(); twin.close(); w.close()


# ---------------------------------------------------------------- 4. device call after pipelined host steps
@pytest.mark.gpu
@pytest.mark.parametrize("consumer", ["obs_device", "gather_device", "sample_gather_device", "obs_gather_device", "forward_device",
                                      "train_device", "stats_export"])
def test_device_call_after_submitted_steps(qlb, O, torch, stream, consumer):
    """Page-locked steps submitted with step_many_submit (16,384 envs x 32 steps, 6 submits, not waited for), then a device
    call on the caller's stream. It must see all submitted steps: compared with a twin env that steps synchronously. The
    submitted work cannot be delayed from the test, so without the ordering this case fails likely, not certainly."""
    n = BIG_N
    envs = [qlb.BreakoutEnvironment(n_envs=n, seed=SEED, replay_capacity=n * BIG_T_CAP) for _ in range(2)]
    rng = np.random.default_rng(7)
    warm = rng.integers(0, 3, size=(BIG_T_CAP + 5, n), dtype=np.uint8)
    for e in envs:
        e.step_many(warm)
    k, subs = 32, 6
    acts = [qlb.PinnedArray((k, n), np.uint8) for _ in range(subs)]
    outs = [(qlb.PinnedArray((k, n), np.float32), qlb.PinnedArray((k, n), np.uint8)) for _ in range(subs)]
    for a in acts:
        a.array[:] = rng.integers(0, 3, size=(k, n), dtype=np.uint8)
    nets = [qlb.QNetwork(e, random_weights(qlb, 5)) for e in envs] if consumer in ("forward_device", "train_device") else None
    L = qlb.ReplayBuffer(envs[0]).capacity()
    idx = torch.from_numpy(np.arange(L - 256, L, dtype=np.uint32).view(np.int32)).cuda()
    y = torch.from_numpy(np.random.default_rng(8).uniform(-2, 2, 256).astype(np.float32)).cuda()

    handles = [None]

    def make_handles(e):
        """every 64th env's observation at the twin's time (the twin steps synchronously: the states of env 0 once its
        submitted steps have run), copied to the device before anything is submitted"""
        k_ep = e.read_state()["episode_step"]
        h = np.array([(e.time(), int(k_ep[j]), j) for j in range(0, n, 64)], dtype=qlb.OBS_HANDLE_DTYPE)
        handles[0] = torch.from_numpy(h.view(np.uint8)).cuda()

    def run(i, s):
        """the consumer on env i into fresh tensors; returns them"""
        e, rb = envs[i], qlb.ReplayBuffer(envs[i])
        if consumer == "obs_device":
            out = torch.empty((n, 4, 84, 84), dtype=torch.uint8, device="cuda")
            e.obs_device(0, out.data_ptr(), s); return [out]
        if consumer in ("gather_device", "sample_gather_device"):
            st, nx = (torch.empty((256, 4, 84, 84), dtype=torch.uint8, device="cuda") for _ in range(2))
            sc = [torch.empty(256, dtype=t, device="cuda") for t in (torch.float32, torch.uint8, torch.uint8)]
            if consumer == "gather_device":
                rb.gather_device(idx.data_ptr(), 256, 0, st.data_ptr(), nx.data_ptr(), *[t.data_ptr() for t in sc], stream=s)
            else:
                ix = torch.empty(256, dtype=torch.int32, device="cuda")
                rb.sample_gather_device(256, 1, 3, 0, ix.data_ptr(), st.data_ptr(), nx.data_ptr(), *[t.data_ptr() for t in sc], stream=s)
                sc.append(ix)
            return [st, nx] + sc
        if consumer == "obs_gather_device":
            hd = handles[0]
            out = torch.empty((hd.numel() // 16, 4, 84, 84), dtype=torch.uint8, device="cuda")
            e.obs_gather_device(hd.data_ptr(), hd.numel() // 16, 0, out.data_ptr(), s); return [out]
        if consumer == "forward_device":
            q, a = torch.empty((n, 3), dtype=torch.float32, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
            nets[i].forward_device(None, n, 0, q.data_ptr(), a.data_ptr(), None, s); return [q, a]
        if consumer == "train_device":
            loss = torch.empty(1, dtype=torch.float32, device="cuda")
            nets[i].train_device(idx.data_ptr(), 256, 1, y.data_ptr(), None, 0.99, loss.data_ptr(), s); return [loss]
        ex = torch.empty(5, dtype=torch.float64, device="cuda")
        e.stats_export(ex.data_ptr(), s); return [ex]

    # warm-up of the consumer on both envs, the same on both (buffers allocated), then the twin steps synchronously
    make_handles(envs[1])
    for i in range(2):
        run(i, None)
    torch.cuda.synchronize()
    for a in acts:
        envs[1].step_many(a.array)
    make_handles(envs[1])
    want = run(1, None)
    torch.cuda.synchronize()
    for a, (r, d) in zip(acts, outs):
        envs[0].step_many_submit(a.array, r.array, d.array)
    got = run(0, stream.cuda_stream or None)
    torch.cuda.synchronize()
    envs[0].step_many_wait(0)
    for g, o in zip(got, want):
        assert_same(g.cpu().numpy(), o.cpu().numpy(), consumer)
    if consumer == "train_device":
        assert_weights(nets[0].get_weights(), nets[1].get_weights())
    assert envs[0].time() == envs[1].time()
    if nets:
        for net in nets:
            net.close()
    for a in acts:
        a.free()
    for r, d in outs:
        r.free(); d.free()
    for e in envs:
        e.close()


# ---------------------------------------------------------------- 5. load
@pytest.mark.gpu
def test_step_and_export_right_after_load(qlb, O, torch, tmp_path):
    """load, then at once stats_export and a step on a fresh non-blocking stream: the checkpoint's statistics and the oracle's
    trajectory. Run once; a single run cannot show the race reliably."""
    a = World(qlb, O)
    a.step_host(20)
    path = str(tmp_path / "ckpt")
    a.env.save(path)
    want_stats = a.env.stats()
    b = qlb.BreakoutEnvironment(n_envs=N, seed=SEED, replay_capacity=N * T_CAP, max_episode_steps=MAX_EP)
    b.step_many(np.ones((50, N), dtype=np.uint8))
    assert b.stats()["episodes"] != want_stats["episodes"]
    acts = a.acts(4)
    acts_d = torch.from_numpy(acts).cuda()
    reward = torch.empty((4, N), dtype=torch.float32, device="cuda")
    ex = torch.empty(5, dtype=torch.float64, device="cuda")
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    b.load(path)
    b.stats_export(ex.data_ptr(), side.cuda_stream)
    b.step_device(acts_d.data_ptr(), 4, reward.data_ptr(), None, side.cuda_stream)
    side.synchronize()
    e = ex.cpu().numpy()
    assert (e[0], e[1], e[2]) == (want_stats["sum_return"], want_stats["episodes"], want_stats["steps"])
    r, _ = a.follow(acts)
    assert_same(reward.cpu().numpy(), r)
    assert_same(b.obs(0), a.ora.obs_u8())
    b.close(); a.close()
