"""CPU-only checks of n-step returns and double-DQN targets (DESIGN.md §14): the Python defaults, argument validation without
a GPU, and the numpy model of the walk over the record ring that tests/test_nstep_double.py compares the device with, checked
here against answers worked out by hand."""
import ctypes
import importlib
import inspect

import numpy as np
import pytest


def pack_record(action=0, done=False, k=1, reward=0, truncated=False):
    """kernels.cuh pack_record: bits 0-1 action | 2 done | 3-4 k mod 4 | 5-7 min(k,4) | 8-15 reward | 16 truncated"""
    return (action & 3) | (4 if done else 0) | ((k & 3) << 3) | (min(k, 4) << 5) | ((reward & 0xFF) << 8) | (0x10000 if truncated else 0)


def nstep_model(records, t_oldest, t_now, idx, n_step, gamma):
    """(G f32, disc f32, boot u32, terminal bool) of the logical indices idx over records u32 [time_slots][n_envs]. Walks every
    item in lock step; f32 arithmetic one rounding per operation, in the order DESIGN.md §14 defines."""
    ts, n_envs = records.shape
    idx = np.asarray(idx, dtype=np.uint64)
    gamma = np.float32(gamma)
    T = np.uint64(t_oldest) + idx // np.uint64(n_envs)
    e = (idx % np.uint64(n_envs)).astype(np.int64)
    n = idx.size
    G, pw = np.zeros(n, np.float32), np.ones(n, np.float32)
    m, term = np.ones(n, np.uint64), np.zeros(n, bool)
    alive = T < np.uint64(t_now)
    valid = alive.copy()
    for j in range(n_step):
        a = np.nonzero(alive)[0]
        if a.size == 0:
            break
        t = T[a] + np.uint64(j)
        r = records[(t % np.uint64(ts)).astype(np.int64), e[a]].astype(np.uint64)
        G[a] = G[a] + pw[a] * ((r >> np.uint64(8)) & np.uint64(0xFF)).astype(np.float32)
        pw[a] = pw[a] * gamma
        m[a] = j + 1
        done = ((r >> np.uint64(2)) & np.uint64(1)) != 0
        term[a] = done
        stop = done | ((r & np.uint64(0x10000)) != 0) | (j == n_step - 1) | (t == np.uint64(t_now - 1))
        nxt_t = np.minimum(t + np.uint64(1), np.uint64(t_now - 1))      # the record after a stop at the newest time is not read
        nxt = records[(nxt_t % np.uint64(ts)).astype(np.int64), e[a]].astype(np.uint64)
        stop |= ~stop & (((nxt >> np.uint64(5)) & np.uint64(7)) == 0)
        alive[a[stop]] = False
    disc = np.where(term | ~valid, np.float32(0), pw).astype(np.float32)
    G = np.where(valid, G, np.float32(0)).astype(np.float32)
    boot = np.where(valid, idx + (m - np.uint64(1)) * np.uint64(n_envs), idx).astype(np.uint32)
    return G, disc, boot, term & valid


def target_model(G, disc, term, q_boot):
    """y = G where terminal, else G + Q_boot * disc (f32, the product rounded first)"""
    return np.where(term, G, G + np.asarray(q_boot, np.float32) * disc).astype(np.float32)


def test_python_defaults():
    pytest.importorskip("torch")
    tio = importlib.import_module("q-learning_b200.torch_io")
    d = inspect.signature(tio.TensorCoreLearner.__init__).parameters
    assert (d["n_step"].default, d["double_dqn"].default) == (1, False)
    qlb = importlib.import_module("q-learning_b200")
    d = inspect.signature(qlb.QNetwork.train_nstep_device).parameters
    assert (d["n_step"].default, d["double_dqn"].default) == (1, False)


def test_argument_validation_without_gpu(qlb):
    L = qlb.load_library()
    bad = qlb.ERR_INVALID_ARG
    fake_env = ctypes.create_string_buffer(4096)           # zeroed stand-in for an env handle
    other_env = ctypes.create_string_buffer(4096)
    idx = ctypes.create_string_buffer(64)

    def msg():
        return L.qlc_last_error_string()

    # qlc_replay_nstep
    for n_step in (0, 65):
        assert L.qlc_replay_nstep(fake_env, idx, 4, n_step, 0.99, None, None, None, None) == bad
        assert b"n_step" in msg()
    for gamma in (-0.1, 1.5, float("nan"), float("inf")):
        assert L.qlc_replay_nstep(fake_env, idx, 4, 3, gamma, None, None, None, None) == bad
        assert b"gamma" in msg()
    assert L.qlc_replay_nstep(None, idx, 4, 3, 0.99, None, None, None, None) == bad and b"env" in msg()
    assert L.qlc_replay_nstep(fake_env, None, 4, 3, 0.99, None, None, None, None) == bad and b"idx" in msg()

    # qlc_qnet_train_nstep: stand-in networks whose first field (the env pointer) names a stand-in env, so that the checks of
    # the target network's env can be reached without a device
    def fake_qnet(env):
        b = ctypes.create_string_buffer(4096)
        if env is not None:
            ctypes.c_void_p.from_buffer(b).value = ctypes.addressof(env)
        return b

    q, tgt = fake_qnet(fake_env), fake_qnet(fake_env)
    dead, foreign = fake_qnet(None), fake_qnet(other_env)

    def train(qn=q, ix=idx, batch=32, n_batches=1, target=tgt, gamma=0.99, n_step=3, double=1):
        return L.qlc_qnet_train_nstep(qn, ix, None, batch, n_batches, target, gamma, n_step, double, None, None, None, None)

    for n_step, word in ((0, b"n_step"), (65, b"n_step")):
        assert train(n_step=n_step) == bad and word in msg()
    for gamma in (-0.5, 1.0001, float("nan"), float("-inf")):
        assert train(gamma=gamma) == bad and b"gamma" in msg()
    for double in (-1, 2):
        assert train(double=double) == bad and b"double_dqn" in msg()
    assert train(qn=None) == bad and b"qnet" in msg()
    assert train(ix=None) == bad and b"indices" in msg()
    assert train(target=None) == bad and b"target_net" in msg()
    assert train(target=dead) == bad and b"target network has been destroyed" in msg()
    assert train(target=foreign) == bad and b"another environment" in msg()
    assert train(qn=dead) == bad and b"destroyed" in msg()
    assert train(batch=1 << 16, n_batches=1 << 8) == bad and b"too many items" in msg()
    assert train(batch=0) == bad and b"batch" in msg()
    if qlb.device_count() > 0:
        pytest.skip("a GPU is present")
    assert L.qlc_replay_nstep(fake_env, idx, 4, 3, 0.99, None, None, None, None) == qlb.ERR_NO_DEVICE
    for n_step, gamma, double in ((1, 0.0, 0), (64, 1.0, 1)):
        assert train(n_step=n_step, gamma=gamma, double=double) == qlb.ERR_NO_DEVICE


# ---------------------------------------------------------------- the model on hand-built rings
def _ring(rows, ts=None):
    """records [time_slots][n_envs] from rows[t][e] = dict(pack_record args), times 0 .. len(rows) - 1 at slots t % ts"""
    ts = ts or len(rows)
    rec = np.zeros((ts, len(rows[0])), np.uint32)
    for t, row in enumerate(rows):
        for e, kw in enumerate(row):
            rec[t % ts, e] = pack_record(**kw)
    return rec


def _f(x):
    return np.float32(x)


def test_model_done_at_first_record_and_truncation():
    # env 0: done at t=1; env 1: truncated at t=2; rewards 1, 2, 3, 4 over t = 0..3
    rows = [[dict(k=1, reward=1), dict(k=5, reward=1)],
            [dict(k=2, reward=2, done=True), dict(k=6, reward=2)],
            [dict(k=3, reward=3, done=True), dict(k=7, reward=3, truncated=True)],
            [dict(k=0, reward=4), dict(k=0, reward=4)]]
    rec = _ring(rows)
    g = _f(0.5)
    G, disc, boot, term = nstep_model(rec, 0, 4, np.array([0, 1, 2, 3, 4, 5]), 3, g)
    # idx 0 (t0, e0): r 1, then done at t1 (r 2): G = 1 + 0.5 * 2 = 2, terminal, boot = idx 2
    # idx 1 (t0, e1): 1 + 0.5 * 2 + 0.25 * 3 (truncated at t2) = 2.75, disc 0.125, boot 5
    # idx 2 (t1, e0): done at j = 0: G = 2, terminal, boot 2
    # idx 3 (t1, e1): 2 + 0.5 * 3 (truncated) = 3.5, disc 0.25, boot 5
    # idx 4 (t2, e0): done at j = 0 (the record after it starts an episode anyway): G = 3, terminal
    # idx 5 (t2, e1): truncated at j = 0: G = 3, disc 0.5
    assert G.tolist() == [2.0, 2.75, 2.0, 3.5, 3.0, 3.0]
    assert disc.tolist() == [0.0, 0.125, 0.0, 0.25, 0.0, 0.5]
    assert boot.tolist() == [2, 5, 2, 5, 4, 5]
    assert term.tolist() == [True, False, True, False, True, False]


def test_model_reset_by_caller_and_newest_time():
    # one env; t = 0..4; the record at t=3 starts an episode (k = 0): a reset by the caller after t=2, which was not done
    rows = [[dict(k=1, reward=1)], [dict(k=2, reward=1)], [dict(k=3, reward=1)], [dict(k=0, reward=2)], [dict(k=1, reward=2)]]
    rec = _ring(rows, ts=7)
    g = _f(0.5)
    G, disc, boot, term = nstep_model(rec, 0, 5, np.arange(6), 10, g)
    # idx 0: 1 + 0.5 + 0.25, stop before the reset: disc 0.125, boot 2
    # idx 3: 2 + 0.5 * 2 = 3 at the newest time t=4 (n_step 10 is longer than the history): disc 0.25, boot 4
    # idx 4: the newest time itself: G 2, disc 0.5, boot 4; idx 5 >= len: 0, 0, 5
    assert G.tolist() == [1.75, 1.5, 1.0, 3.0, 2.0, 0.0]
    assert disc.tolist() == [0.125, 0.25, 0.5, 0.25, 0.5, 0.0]
    assert boot.tolist() == [2, 2, 2, 4, 4, 5]
    assert not term.any()


def test_model_wrapped_ring_and_gamma_edges():
    # 2 envs, 6 time slots, times 3..8 live (t_oldest 3, t_now 9): time t sits in slot t % 6
    rows = [[dict(k=t + 1, reward=t), dict(k=t + 1, reward=2 * t)] for t in range(9)]
    rec = _ring(rows, ts=6)
    idx = np.arange(12)
    for gamma in (0.0, 1.0):
        G, disc, boot, term = nstep_model(rec, 3, 9, idx, 4, gamma)
        T = 3 + idx // 2
        m = np.minimum(4, 9 - T)
        r = lambda t, e: t * (1 + e)
        if gamma == 1.0:
            want = [sum(r(T[i] + j, i % 2) for j in range(m[i])) for i in idx]
            assert disc.tolist() == [1.0] * 12
        else:
            want = [r(T[i], i % 2) for i in idx]
            assert disc.tolist() == [0.0] * 12
        assert G.tolist() == [float(w) for w in want]
        assert boot.tolist() == (idx + (m - 1) * 2).tolist()
        assert not term.any()


def test_model_one_step_is_the_td_target_inputs():
    rng = np.random.default_rng(0)
    rec = rng.integers(0, 1 << 17, size=(10, 3), dtype=np.uint32)
    G, disc, boot, term = nstep_model(rec, 2, 8, np.arange(18), 1, 0.99)
    for i in range(18):
        r = int(rec[(2 + i // 3) % 10, i % 3])
        assert G[i] == np.float32((r >> 8) & 0xFF) and boot[i] == i and bool(term[i]) == bool(r & 4)
        assert disc[i] == (0.0 if r & 4 else np.float32(0.99))
    y = target_model(G, disc, term, np.full(18, 2.5, np.float32))
    r = ((rec[(2 + np.arange(18) // 3) % 10, np.arange(18) % 3] >> 8) & 0xFF).astype(np.float32)
    want = np.where(term, r, r + np.float32(2.5) * np.float32(0.99)).astype(np.float32)
    assert np.array_equal(y.view(np.uint32), want.view(np.uint32))


def test_nstep_max_in_header_and_rust():
    """QLC_NSTEP_MAX of include/ql_cuda.h and of the Rust ffi.rs agree (test_abi.py checks that both declare the n-step calls)."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(root, "include", "ql_cuda.h")).read(), flags=re.S)
    assert re.search(r"#define QLC_NSTEP_MAX 64\b", hdr)
    rust = open(os.path.join(root, "bindings", "rust", "ql-cuda", "src", "ffi.rs")).read()
    assert "pub const QLC_NSTEP_MAX: u32 = 64;" in rust
