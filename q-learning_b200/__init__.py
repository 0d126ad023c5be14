"""q-learning_b200 — B200-native (sm_100a) Breakout env + DQN replay hot path of bitmagier/q-learning.

Host-side mirror of the reference's interfaces for this path, bound over the C ABI in include/ql_cuda.h:

    reference (Rust)                                         here
    -------------------------------------------------------  ------------------------------------------
    ql::prelude::Environment            prelude.rs:21-63      BreakoutEnvironment (vectorised: N envs per GPU)
    ql::prelude::Action / BreakoutAction prelude.rs:12-18     BreakoutAction
    BreakoutState + ToMultiDimArray     breakout_environment.rs:24-78   BreakoutState
    ReplayBuffer / BufferSample         replay_buffer.rs:53-146          ReplayBuffer / BufferSample
    generate_distinct_random_ids        self_driving_tf_q_learner.rs:276-296   ReplayBuffer.generate_distinct_random_ids

There is NO CPU fallback: everything that computes goes through libqlcuda.so and raises QlError when the
library or a CUDA device is missing. (The package directory name contains a hyphen; import it with
importlib.import_module("q-learning_b200").)
"""
import ctypes as C
import enum
import os

import numpy as np

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))

FRAME_W = 84
FRAME_H = 84
FRAME_BYTES = FRAME_W * FRAME_H
NUM_FRAMES = 4

LAYOUT_U8_BHYX = 0
LAYOUT_F32_BXYH = 1
LAYOUT_U8_BXYH = 2

OK, ERR_INVALID_ARG, ERR_CUDA, ERR_OUT_OF_RANGE, ERR_NO_DEVICE, ERR_NOT_ENOUGH, ERR_COMM = 0, 1, 2, 3, 4, 5, 6
COMM_ID_BYTES = 128

ENVERR_WALL_DISTANCE, ENVERR_APPROX_RANGE, ENVERR_RECURSION, ENVERR_BISECTION, ENVERR_DEGENERATE, ENVERR_ACTION, ENVERR_HANDOVER = 1, 2, 4, 8, 16, 32, 64

# every symbol include/ql_cuda.h declares (checked by tests/test_abi.py against the header and the built library)
ABI_SYMBOLS = [
    "qlc_version", "qlc_build_info", "qlc_last_error_string", "qlc_device_count", "qlc_env_create", "qlc_env_destroy", "qlc_sync",
    "qlc_host_alloc", "qlc_host_free",
    "qlc_env_reset", "qlc_env_step", "qlc_env_step_random", "qlc_env_step_host", "qlc_env_step_host_submit", "qlc_env_step_host_wait", "qlc_env_obs", "qlc_env_obs_host", "qlc_env_state_view",
    "qlc_env_read_state", "qlc_env_goal_mean", "qlc_env_time", "qlc_env_lives_host", "qlc_env_error_flags",
    "qlc_obs_gather", "qlc_obs_gather_host",
    "qlc_replay_len", "qlc_replay_capacity", "qlc_replay_sample", "qlc_replay_gather", "qlc_replay_sample_gather", "qlc_replay_sample_host",
    "qlc_replay_gather_host", "qlc_replay_sample_gather_host", "qlc_replay_action_counts",
    "qlc_comm_unique_id", "qlc_comm_init", "qlc_comm_destroy", "qlc_comm_info", "qlc_stats_allreduce", "qlc_stats_global",
    "qlc_env_save", "qlc_env_load",
    "qlc_stats_read", "qlc_stats_export", "qlc_stats_push", "qlc_stats_mean", "qlc_stats_min", "qlc_stats_window",
    "qlc_debug_collision_wall", "qlc_debug_collision_rect", "qlc_debug_collision_rect_batch", "qlc_debug_gemm_bf16",
    "qlc_qnet_create", "qlc_qnet_set_weights", "qlc_qnet_destroy", "qlc_qnet_error", "qlc_qnet_forward", "qlc_qnet_forward_host",
    "qlc_qnet_set_adam", "qlc_qnet_get_weights", "qlc_qnet_train", "qlc_qnet_train_host", "qlc_qnet_debug_grads",
    "qlc_qnet_train_weighted", "qlc_qnet_debug_grads_weighted", "qlc_replay_nstep", "qlc_qnet_train_nstep",
    "qlc_per_create", "qlc_per_destroy", "qlc_per_sample", "qlc_per_update", "qlc_per_read_host",
]


class QlError(Exception):
    """Mirrors ql::prelude::QlError (prelude.rs:70-86); carries the C status code."""

    def __init__(self, msg, code=ERR_INVALID_ARG):
        super().__init__(msg)
        self.code = code


class QlcConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("n_envs", C.c_uint32), ("env_id_base", C.c_uint32),
        ("frame_w", C.c_uint32), ("frame_h", C.c_uint32), ("seed", C.c_uint64), ("replay_capacity", C.c_uint64),
        ("max_episode_steps", C.c_uint32), ("episode_window", C.c_uint32), ("auto_reset", C.c_uint32), ("reserved", C.c_uint32),
    ]


class QlcStateHost(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "ball_cx", "ball_cy", "ball_dx", "ball_dy", "pad_min_x", "pad_max_x", "pad_speed",
        "bricks", "score", "episode_step", "episode", "err", "finished")]


class QlcStateView(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "ball_cx", "ball_cy", "ball_dx", "ball_dy", "pad_min_x", "pad_max_x", "pad_speed",
        "bricks", "score", "episode_step", "episode", "err", "finished", "frames", "records")] + [
        ("n_envs", C.c_uint32), ("time_slots", C.c_uint32), ("time", C.c_uint64)]


class QlcObsHandle(C.Structure):
    """qlc_obs_handle: the observation of env `env` after `time` env-steps, `k` of them in the current episode."""
    _fields_ = [("time", C.c_uint64), ("k", C.c_uint32), ("env", C.c_uint32)]


OBS_HANDLE_DTYPE = np.dtype([("time", np.uint64), ("k", np.uint32), ("env", np.uint32)])


class QlcQnetWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("conv1_kernel", "conv1_bias", "conv2_kernel", "conv2_bias", "conv3_kernel", "conv3_bias",
                                           "dense1_kernel", "dense1_bias", "dense2_kernel", "dense2_bias")]


class QlcAdamConfig(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("lr", "beta1", "beta2", "epsilon", "clipnorm")]


QNET_SHAPES = {"conv1_kernel": (8, 8, 4, 32), "conv1_bias": (32,), "conv2_kernel": (4, 4, 32, 64), "conv2_bias": (64,),
               "conv3_kernel": (3, 3, 64, 64), "conv3_bias": (64,), "dense1_kernel": (3136, 512), "dense1_bias": (512,),
               "dense2_kernel": (512, 3), "dense2_bias": (3,)}


class QlcEpisodeStats(C.Structure):
    _fields_ = [("sum_return", C.c_uint64), ("episodes", C.c_uint64), ("steps", C.c_uint64),
                ("min_return", C.c_uint32), ("max_return", C.c_uint32)]


_LIB = None


def library_path():
    return _build.SO_PATH


def load_library(build_if_missing=True):
    """dlopen libqlcuda.so (building it first if it is missing or stale). Fails loudly; no fallback."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if build_if_missing:
        _build.build()
    if not os.path.exists(_build.SO_PATH):
        raise QlError("libqlcuda.so is missing (run q-learning_b200/build.py); there is no CPU fallback", ERR_NO_DEVICE)
    L = C.CDLL(_build.SO_PATH)
    vp, i32, u32, u64 = C.c_void_p, C.c_int32, C.c_uint32, C.c_uint64
    sig = {
        "qlc_version": (i32, []),
        "qlc_build_info": (C.c_char_p, []),
        "qlc_last_error_string": (C.c_char_p, []),
        "qlc_device_count": (i32, [vp]),
        "qlc_env_create": (i32, [C.POINTER(QlcConfig), C.POINTER(vp)]),
        "qlc_env_destroy": (i32, [vp]),
        "qlc_sync": (i32, [vp, vp]),
        "qlc_host_alloc": (i32, [C.c_size_t, C.POINTER(vp)]),
        "qlc_host_free": (i32, [vp]),
        "qlc_env_reset": (i32, [vp, vp, vp]),
        "qlc_env_step": (i32, [vp, vp, u32, vp, vp, vp]),
        "qlc_env_step_random": (i32, [vp, u32, vp, vp, vp, vp]),
        "qlc_env_step_host": (i32, [vp, vp, u32, vp, vp]),
        "qlc_env_step_host_submit": (i32, [vp, vp, u32, vp, vp]),
        "qlc_env_step_host_wait": (i32, [vp, u32]),
        "qlc_env_obs": (i32, [vp, i32, vp, vp]),
        "qlc_env_obs_host": (i32, [vp, i32, vp]),
        "qlc_env_state_view": (i32, [vp, C.POINTER(QlcStateView)]),
        "qlc_env_read_state": (i32, [vp, C.POINTER(QlcStateHost)]),
        "qlc_env_goal_mean": (C.c_float, []),
        "qlc_env_time": (i32, [vp, C.POINTER(u64)]),
        "qlc_env_error_flags": (i32, [vp, C.POINTER(u32)]),
        "qlc_env_lives_host": (i32, [vp, vp]),
        "qlc_obs_gather": (i32, [vp, vp, u32, i32, vp, vp]),
        "qlc_obs_gather_host": (i32, [vp, vp, u32, i32, vp]),
        "qlc_replay_sample_gather": (i32, [vp, u32, u32, u64, i32, vp, vp, vp, vp, vp, vp, vp]),
        "qlc_replay_sample_gather_host": (i32, [vp, u32, u64, i32, vp, vp, vp, vp, vp, vp]),
        "qlc_comm_unique_id": (i32, [vp]),
        "qlc_comm_init": (i32, [vp, i32, i32, vp]),
        "qlc_comm_destroy": (i32, [vp]),
        "qlc_comm_info": (i32, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
        "qlc_stats_allreduce": (i32, [vp, vp]),
        "qlc_stats_global": (i32, [vp, C.POINTER(QlcEpisodeStats), i32]),
        "qlc_qnet_error": (i32, [vp, C.POINTER(u32)]),
        "qlc_replay_len": (i32, [vp, C.POINTER(u64)]),
        "qlc_replay_capacity": (i32, [vp, C.POINTER(u64)]),
        "qlc_replay_sample": (i32, [vp, u32, u32, u64, vp, vp]),
        "qlc_replay_gather": (i32, [vp, vp, u32, i32, vp, vp, vp, vp, vp, vp]),
        "qlc_replay_sample_host": (i32, [vp, u32, u64, vp]),
        "qlc_replay_gather_host": (i32, [vp, vp, u32, i32, vp, vp, vp, vp, vp]),
        "qlc_replay_action_counts": (i32, [vp, vp]),
        "qlc_env_save": (i32, [vp, C.c_char_p]),
        "qlc_env_load": (i32, [vp, C.c_char_p]),
        "qlc_stats_read": (i32, [vp, C.POINTER(QlcEpisodeStats)]),
        "qlc_stats_export": (i32, [vp, vp, vp]),
        "qlc_stats_push": (i32, [vp, C.c_float]),
        "qlc_stats_mean": (i32, [vp, C.POINTER(C.c_float)]),
        "qlc_stats_min": (i32, [vp, C.POINTER(C.c_float)]),
        "qlc_stats_window": (i32, [vp, vp, u32, C.POINTER(u32)]),
        "qlc_debug_collision_wall": (i32, [i32] + [C.c_float] * 5 + [vp] * 6),
        "qlc_debug_collision_rect": (i32, [C.c_float] * 9 + [vp] * 6),
        "qlc_debug_collision_rect_batch": (i32, [vp, vp, u32]),
        "qlc_debug_gemm_bf16": (i32, [vp, vp, vp, i32, vp, u32, u32, u32]),
        "qlc_qnet_create": (i32, [vp, C.POINTER(QlcQnetWeights), C.POINTER(vp)]),
        "qlc_qnet_set_weights": (i32, [vp, C.POINTER(QlcQnetWeights)]),
        "qlc_qnet_destroy": (i32, [vp]),
        "qlc_qnet_forward": (i32, [vp, vp, u32, i32, vp, vp, vp, vp]),
        "qlc_qnet_forward_host": (i32, [vp, vp, u32, i32, vp, vp, vp]),
        "qlc_qnet_set_adam": (i32, [vp, C.POINTER(QlcAdamConfig)]),
        "qlc_qnet_get_weights": (i32, [vp, C.POINTER(QlcQnetWeights)]),
        "qlc_qnet_train": (i32, [vp, vp, u32, u32, vp, vp, C.c_float, vp, vp]),
        "qlc_qnet_train_host": (i32, [vp, vp, u32, u32, vp, vp, C.c_float, vp]),
        "qlc_qnet_debug_grads": (i32, [vp, vp, u32, vp, C.POINTER(QlcQnetWeights)]),
        "qlc_qnet_train_weighted": (i32, [vp, vp, vp, u32, u32, vp, vp, C.c_float, vp, vp, vp]),
        "qlc_qnet_debug_grads_weighted": (i32, [vp, vp, u32, vp, vp, C.POINTER(QlcQnetWeights), vp]),
        "qlc_per_create": (i32, [vp, C.c_float, C.c_float, C.POINTER(vp)]),
        "qlc_per_destroy": (i32, [vp]),
        "qlc_per_sample": (i32, [vp, u32, u32, u64, C.c_float, vp, vp, vp]),
        "qlc_per_update": (i32, [vp, vp, vp, u32, vp]),
        "qlc_per_read_host": (i32, [vp, vp, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
        "qlc_replay_nstep": (i32, [vp, vp, u32, u32, C.c_float, vp, vp, vp, vp]),
        "qlc_qnet_train_nstep": (i32, [vp, vp, vp, u32, u32, vp, C.c_float, u32, i32, vp, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)   # AttributeError if the library lacks a declared symbol
        f.restype = res
        f.argtypes = args
    _LIB = L
    return L


def _check(rc):
    if rc != OK:
        msg = load_library().qlc_last_error_string()
        raise QlError((msg or b"").decode() or "ql_cuda error %d" % rc, rc)


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class PinnedArray:
    """numpy view on page-locked host memory from qlc_host_alloc: the *_host entry points copy such buffers in place
    (no internal staging copy). Keep the object alive while the array is in use."""

    def __init__(self, shape, dtype):
        L = load_library()
        self._L = L
        dt = np.dtype(dtype)
        n = int(np.prod(shape)) * dt.itemsize
        p = C.c_void_p()
        _check(L.qlc_host_alloc(max(n, 1), C.byref(p)))
        self._p = p
        buf = (C.c_uint8 * max(n, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._p:
            self.array = None
            self._L.qlc_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def build_info():
    """{'src_hash': ..., 'profiling': '0' | '1'} of the loaded library (profiling = 1: an ablation build that honours QLC_DEBUG_SKIP)."""
    text = load_library().qlc_build_info().decode()
    return dict(kv.split("=", 1) for kv in text.strip(";").split(";"))


def device_count():
    n = C.c_int32(0)
    rc = load_library().qlc_device_count(C.byref(n))
    return n.value if rc == OK else 0


def comm_unique_id():
    """ncclGetUniqueId through the C ABI: 128 bytes for rank 0 to hand to the other ranks."""
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    _check(load_library().qlc_comm_unique_id(buf))
    return bytes(buf)


def _stack_shape(n, layout):
    if layout == LAYOUT_U8_BHYX:
        return (n, NUM_FRAMES, FRAME_H, FRAME_W), np.uint8
    if layout == LAYOUT_F32_BXYH:
        return (n, FRAME_W, FRAME_H, NUM_FRAMES), np.float32
    if layout == LAYOUT_U8_BXYH:
        return (n, FRAME_W, FRAME_H, NUM_FRAMES), np.uint8
    raise QlError("unknown layout")


class BreakoutAction(enum.IntEnum):
    """BreakoutAction (breakout_environment.rs:94-120)."""
    NONE = 0
    LEFT = 1
    RIGHT = 2

    def numeric(self):
        return int(self)

    @staticmethod
    def try_from_numeric(value):
        if value in (0, 1, 2):
            return BreakoutAction(value)
        raise QlError("value out of range", ERR_OUT_OF_RANGE)


BreakoutAction.ACTION_SPACE = 3


class BreakoutState:
    """Cheap handle on the current observation of all envs (BreakoutState, breakout_environment.rs:24-28).
    Clone = copy of (time) — pixels stay in the HBM frame ring until tensorised."""

    def __init__(self, env, time):
        self._env = env
        self.time = time

    def dims(self):
        return [FRAME_W, FRAME_H, NUM_FRAMES]                      # model_dims, breakout_environment.rs:148

    def to_multi_dim_array(self):
        """[n_envs][x][y][slot] f32 (ToMultiDimArray::to_multi_dim_array, breakout_environment.rs:42-54)."""
        if self.time != self._env.time():
            raise QlError("stale BreakoutState handle: the env has stepped since", ERR_INVALID_ARG)
        return self._env.obs(LAYOUT_F32_BXYH)

    def one_line_info(self):                                        # DebugVisualizer, breakout_environment.rs:81-89
        s = self._env.read_state()
        return "Breakout [%d bricks, ball_pos: [%.1f %.1f], panel_pos: [%.1f 570.0]]" % (
            bin(int(s["bricks"][0])).count("1"), s["ball_cx"][0], s["ball_cy"][0], (s["pad_min_x"][0] + s["pad_max_x"][0]) / 2)


class BreakoutEnvironment:
    """N independent Breakout envs on one GPU behind the reference's Environment interface
    (prelude.rs:21-63; BreakoutEnvironment, breakout_environment.rs:131-207)."""

    def __init__(self, n_envs=1, frame_size_x=FRAME_W, frame_size_y=FRAME_H, device=0, seed=0, env_id_base=0,
                 replay_capacity=0, max_episode_steps=0, episode_window=100, auto_reset=True):
        self._L = load_library()
        self.n_envs = int(n_envs)
        self.max_episode_steps = int(max_episode_steps)
        self.auto_reset = bool(auto_reset)
        cfg = QlcConfig(C.sizeof(QlcConfig), device, n_envs, env_id_base, frame_size_x, frame_size_y, seed,
                        replay_capacity, max_episode_steps, episode_window, 1 if auto_reset else 0, 0)
        h = C.c_void_p()
        _check(self._L.qlc_env_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.device = device

    # -- lifecycle
    def close(self):
        if getattr(self, "_h", None):
            self._L.qlc_env_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    # -- Environment trait
    def reset(self, mask=None, dir_x=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        d = None if dir_x is None else np.ascontiguousarray(dir_x, dtype=np.float32)
        if m is not None and m.shape != (self.n_envs,):
            raise QlError("mask must have n_envs entries")
        if d is not None and d.shape != (self.n_envs,):
            raise QlError("dir_x must have n_envs entries")
        _check(self._L.qlc_env_reset(self._h, None if m is None else _np_ptr(m), None if d is None else _np_ptr(d)))

    def state(self):
        return BreakoutState(self, self.time())

    def step(self, actions):
        """One step for all envs with HOST arrays: returns (state handle, reward f32[n], done u8[n])."""
        a = np.ascontiguousarray(actions, dtype=np.uint8).reshape(1, self.n_envs)
        r, d = self.step_many(a)
        return self.state(), r[0], d[0]

    def step_many(self, actions, out=None):
        """actions u8 [n_steps][n_envs] (host) -> reward f32 [n_steps][n_envs], done u8 [n_steps][n_envs].
        `out=(reward, done)` reuses caller arrays (page-locked ones, see PinnedArray, avoid the staging copy)."""
        a = np.ascontiguousarray(actions, dtype=np.uint8)
        if a.ndim != 2 or a.shape[1] != self.n_envs:
            raise QlError("actions must be [n_steps][n_envs]")
        k = a.shape[0]
        if out is not None:
            reward, done = out
            if reward.shape != (k, self.n_envs) or reward.dtype != np.float32 or done.shape != (k, self.n_envs) or done.dtype != np.uint8 \
                    or not reward.flags.c_contiguous or not done.flags.c_contiguous:
                raise QlError("out arrays must be C-contiguous f32 / u8 [n_steps][n_envs]")
        else:
            reward = np.empty((k, self.n_envs), dtype=np.float32)
            done = np.empty((k, self.n_envs), dtype=np.uint8)
        _check(self._L.qlc_env_step_host(self._h, _np_ptr(a), k, _np_ptr(reward), _np_ptr(done)))
        return reward, done

    def step_many_submit(self, actions, reward, done):
        """Pipelined step_many for action streams that do not depend on the previous result: queues the step and returns.
        All three arrays must be page-locked (PinnedArray(...).array) and stay untouched until step_many_wait()."""
        k = actions.shape[0]
        if actions.dtype != np.uint8 or actions.ndim != 2 or actions.shape[1] != self.n_envs or not actions.flags.c_contiguous:
            raise QlError("actions must be C-contiguous u8 [n_steps][n_envs]")
        if reward.shape != (k, self.n_envs) or reward.dtype != np.float32 or done.shape != (k, self.n_envs) or done.dtype != np.uint8 \
                or not reward.flags.c_contiguous or not done.flags.c_contiguous:
            raise QlError("out arrays must be C-contiguous f32 / u8 [n_steps][n_envs]")
        _check(self._L.qlc_env_step_host_submit(self._h, _np_ptr(actions), k, _np_ptr(reward), _np_ptr(done)))

    def step_many_wait(self, max_pending=0):
        """Blocks until at most `max_pending` of the submitted steps are still running (0 = all results are in)."""
        _check(self._L.qlc_env_step_host_wait(self._h, max_pending))

    def step_device(self, actions_ptr, n_steps, reward_ptr=None, done_ptr=None, stream=None):
        """Asynchronous step on device buffers (raw device pointers, e.g. torch tensor .data_ptr())."""
        _check(self._L.qlc_env_step(self._h, actions_ptr, n_steps, reward_ptr, done_ptr, stream))

    def step_random_device(self, n_steps, actions_out_ptr=None, reward_ptr=None, done_ptr=None, stream=None):
        """The learner's pure-random phase: the step kernel draws the uniform action of every env and step itself (Philox 'ACTI'
        stream); no action buffer, no policy kernel. Asynchronous, device pointers."""
        _check(self._L.qlc_env_step_random(self._h, n_steps, actions_out_ptr, reward_ptr, done_ptr, stream))

    def episode_reward_goal_mean(self):
        return float(self._L.qlc_env_goal_mean())

    # -- state access
    def time(self):
        t = C.c_uint64(0)
        _check(self._L.qlc_env_time(self._h, C.byref(t)))
        return t.value

    def obs(self, layout=LAYOUT_U8_BHYX):
        shape, dt = _stack_shape(self.n_envs, layout)
        out = np.empty(shape, dtype=dt)
        _check(self._L.qlc_env_obs_host(self._h, layout, _np_ptr(out)))
        return out

    def obs_device(self, layout, out_ptr, stream=None):
        _check(self._L.qlc_env_obs(self._h, layout, out_ptr, stream))

    def read_state(self):
        n = self.n_envs
        f = {k: np.empty(n, dtype=np.float32) for k in ("ball_cx", "ball_cy", "ball_dx", "ball_dy", "pad_min_x", "pad_max_x", "pad_speed")}
        f["bricks"] = np.empty(n, dtype=np.uint64)
        for k in ("score", "episode_step", "episode", "err"):
            f[k] = np.empty(n, dtype=np.uint32)
        f["finished"] = np.empty(n, dtype=np.uint8)
        sh = QlcStateHost(*[f[name].ctypes.data for name, _ in QlcStateHost._fields_])
        _check(self._L.qlc_env_read_state(self._h, C.byref(sh)))
        f["lives"] = (f["finished"] == 0).astype(np.uint8)      # one life per episode (mechanics.rs:131-135)
        return f

    def state_view(self):
        v = QlcStateView()
        _check(self._L.qlc_env_state_view(self._h, C.byref(v)))
        return v

    def lives(self):
        """u8 [n_envs]: 1 while an env's episode runs, 0 once it is over (the reference game ends with the first miss,
        mechanics.rs:131-135: there is no lives counter to decrement)."""
        out = np.empty(self.n_envs, dtype=np.uint8)
        _check(self._L.qlc_env_lives_host(self._h, _np_ptr(out)))
        return out

    def obs_gather(self, handles, layout=LAYOUT_F32_BXYH):
        """Stacks of state handles (numpy array of OBS_HANDLE_DTYPE: time, k, env) into a host array."""
        h = np.ascontiguousarray(handles, dtype=OBS_HANDLE_DTYPE)
        shape, dt = _stack_shape(h.size, layout)
        out = np.empty(shape, dtype=dt)
        _check(self._L.qlc_obs_gather_host(self._h, _np_ptr(h), h.size, layout, _np_ptr(out)))
        return out

    def obs_gather_device(self, handles_ptr, n, layout, out_ptr, stream=None):
        _check(self._L.qlc_obs_gather(self._h, handles_ptr, n, layout, out_ptr, stream))

    # -- statistics reduction over the env shards, NCCL behind the C ABI (one process per GPU)
    def comm_init(self, rank, world, unique_id=None):
        """unique_id: the 128 bytes rank 0 got from comm_unique_id(), handed to every rank by the host's own channel
        (torch.distributed broadcast, a file, ...). world == 1 without an id needs no NCCL."""
        buf = None if unique_id is None else (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(bytes(unique_id))
        _check(self._L.qlc_comm_init(self._h, rank, world, buf))

    def comm_info(self):
        r, w, v, n = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
        _check(self._L.qlc_comm_info(self._h, C.byref(r), C.byref(w), C.byref(v), C.byref(n)))
        return dict(rank=r.value, world=w.value, nccl_version=v.value, nccl_ranks=n.value)

    def stats_allreduce(self, stream=None):
        """Enqueue one reduction on the communicator's side stream (only an event record touches `stream`)."""
        _check(self._L.qlc_stats_allreduce(self._h, stream))

    def stats_global(self, wait=True):
        s = QlcEpisodeStats()
        _check(self._L.qlc_stats_global(self._h, C.byref(s), 1 if wait else 0))
        return dict(sum_return=s.sum_return, episodes=s.episodes, steps=s.steps, min_return=s.min_return, max_return=s.max_return)

    def error_flags(self):
        e = C.c_uint32(0)
        _check(self._L.qlc_env_error_flags(self._h, C.byref(e)))
        return e.value

    def sync(self, stream=None):
        _check(self._L.qlc_sync(self._h, stream))

    def save(self, path):
        """Checkpoint the env shard + replay ring (SoA state, records, frames, statistics, episode window)."""
        _check(self._L.qlc_env_save(self._h, os.fsencode(path)))

    def load(self, path):
        """Resume from a checkpoint taken with the same configuration; the run continues bit-identically."""
        _check(self._L.qlc_env_load(self._h, os.fsencode(path)))

    # -- shard statistics
    def stats(self):
        s = QlcEpisodeStats()
        _check(self._L.qlc_stats_read(self._h, C.byref(s)))
        return dict(sum_return=s.sum_return, episodes=s.episodes, steps=s.steps, min_return=s.min_return, max_return=s.max_return)

    def stats_export(self, out_ptr, stream=None):
        _check(self._L.qlc_stats_export(self._h, out_ptr, stream))


class BufferSample:
    """BufferSample (replay_buffer.rs:140-146)."""

    def __init__(self, state, state_next, reward, action, done):
        self.state, self.state_next, self.reward, self.action, self.done = state, state_next, reward, action, done


class ReplayBuffer:
    """The replay shard of a BreakoutEnvironment behind ReplayBuffer's method set (replay_buffer.rs:53-137).
    Frames are written once, by the step kernel, straight into the HBM frame ring; a transition is a 4-byte record."""

    def __init__(self, env):
        self._env = env
        self._L = env._L
        self._calls = 0

    def len(self):
        n = C.c_uint64(0)
        _check(self._L.qlc_replay_len(self._env._h, C.byref(n)))
        return n.value

    __len__ = len

    def capacity(self):
        n = C.c_uint64(0)
        _check(self._L.qlc_replay_capacity(self._env._h, C.byref(n)))
        return n.value

    def add(self, action=None, state=None, state_next=None, reward=None, done=None):
        """ReplayBuffer::add (:85-98). The step kernel has already appended the transition(s) on the device
        (frame ring + record); this keeps the reference's call site valid and checks the handles it is given."""
        if state_next is not None and isinstance(state_next, BreakoutState) and state_next.time != self._env.time():
            raise QlError("ReplayBuffer.add: state_next is not the env's latest state")

    def add_episode_reward(self, episode_reward):
        _check(self._L.qlc_stats_push(self._env._h, float(episode_reward)))

    def avg_episode_reward(self):
        v = C.c_float(0)
        _check(self._L.qlc_stats_mean(self._env._h, C.byref(v)))
        return v.value

    def min_episode_reward(self):
        v = C.c_float(0)
        _check(self._L.qlc_stats_min(self._env._h, C.byref(v)))
        return v.value

    def episode_rewards(self):
        n = C.c_uint32(0)
        _check(self._L.qlc_stats_window(self._env._h, None, 0, C.byref(n)))
        out = np.empty(max(n.value, 1), dtype=np.float32)
        _check(self._L.qlc_stats_window(self._env._h, _np_ptr(out), out.size, C.byref(n)))
        return out[:n.value]

    def actions(self):
        """Histogram of the stored actions (what the learner's log derives from actions(): :242-245)."""
        out = np.zeros(3, dtype=np.uint64)
        _check(self._L.qlc_replay_action_counts(self._env._h, _np_ptr(out)))
        return out

    @staticmethod
    def should_sample(step_count, length, batch, update_after_actions=4):
        """The learner's sample gate (self_driving_tf_q_learner.rs:181): every n-th step once len > BATCH_SIZE."""
        return step_count % update_after_actions == 0 and length > batch

    def generate_distinct_random_ids(self, batch, call_index=None):
        """BATCH distinct uniform indices in 0..len (self_driving_tf_q_learner.rs:276-296), host copy."""
        if call_index is None:
            call_index = self._calls
            self._calls += 1
        out = np.empty(batch, dtype=np.uint32)
        _check(self._L.qlc_replay_sample_host(self._env._h, batch, call_index, _np_ptr(out)))
        return out

    def get_many(self, indices, layout=LAYOUT_F32_BXYH, want_state=True, want_next=True, reuse=False):
        """get_many (:126-137) + batch_to_multi_dim_array for state and state_next, into host arrays.
        reuse=True returns views on page-locked buffers owned by this object (the device copies straight into them; valid
        until the next get_many(reuse=True) of the same size) instead of fresh pageable arrays."""
        idx = np.ascontiguousarray(indices, dtype=np.uint32)
        n = idx.size
        shape, dt = _stack_shape(n, layout)
        if reuse:
            key = (n, layout)
            if getattr(self, "_pinned_key", None) != key:
                self._pinned = (PinnedArray(shape, dt), PinnedArray(shape, dt))
                self._pinned_key = key
            s = self._pinned[0].array if want_state else None
            sn = self._pinned[1].array if want_next else None
        else:
            s = np.empty(shape, dtype=dt) if want_state else None
            sn = np.empty(shape, dtype=dt) if want_next else None
        reward = np.empty(n, dtype=np.float32)
        action = np.empty(n, dtype=np.uint8)
        done = np.empty(n, dtype=np.uint8)
        _check(self._L.qlc_replay_gather_host(self._env._h, _np_ptr(idx), n, layout, None if s is None else _np_ptr(s),
                                              None if sn is None else _np_ptr(sn), _np_ptr(reward), _np_ptr(action), _np_ptr(done)))
        return BufferSample(s, sn, reward, action, done)

    def sample(self, batch, layout=LAYOUT_F32_BXYH, call_index=None, want_state=True, want_next=True):
        """generate_distinct_random_ids + get_many + batch_to_multi_dim_array as ONE kernel launch (the kernel draws the indices
        itself), into host arrays: (indices u32[batch], BufferSample)."""
        if call_index is None:
            call_index = self._calls
            self._calls += 1
        shape, dt = _stack_shape(batch, layout)
        s = np.empty(shape, dtype=dt) if want_state else None
        sn = np.empty(shape, dtype=dt) if want_next else None
        idx = np.empty(batch, dtype=np.uint32)
        reward = np.empty(batch, dtype=np.float32)
        action = np.empty(batch, dtype=np.uint8)
        done = np.empty(batch, dtype=np.uint8)
        _check(self._L.qlc_replay_sample_gather_host(self._env._h, batch, call_index, layout, _np_ptr(idx), None if s is None else _np_ptr(s),
                                                     None if sn is None else _np_ptr(sn), _np_ptr(reward), _np_ptr(action), _np_ptr(done)))
        return idx, BufferSample(s, sn, reward, action, done)

    # device-buffer forms
    def sample_gather_device(self, batch, n_batches, call_index, layout, idx_out_ptr, state_ptr, next_ptr, reward_ptr=None, action_ptr=None, done_ptr=None,
                             stream=None):
        """sample + gather in one launch on device buffers (idx_out_ptr may be None)."""
        _check(self._L.qlc_replay_sample_gather(self._env._h, batch, n_batches, call_index, layout, idx_out_ptr, state_ptr, next_ptr, reward_ptr, action_ptr,
                                                done_ptr, stream))

    def sample_device(self, batch, n_batches, call_index, idx_ptr, stream=None):
        _check(self._L.qlc_replay_sample(self._env._h, batch, n_batches, call_index, idx_ptr, stream))

    def gather_device(self, idx_ptr, n, layout, state_ptr, next_ptr, reward_ptr=None, action_ptr=None, done_ptr=None, stream=None):
        _check(self._L.qlc_replay_gather(self._env._h, idx_ptr, n, layout, state_ptr, next_ptr, reward_ptr, action_ptr, done_ptr, stream))

    def nstep_device(self, idx_ptr, n, n_step, gamma, ret_ptr=None, disc_ptr=None, boot_ptr=None, stream=None):
        """n-step returns of the n transitions idx_ptr (u32 logical indices): G f32 at ret_ptr, discount f32 at disc_ptr (gamma^m,
        0 where terminal), and the logical index whose state_next bootstraps, u32 at boot_ptr (any may be None). Asynchronous."""
        _check(self._L.qlc_replay_nstep(self._env._h, idx_ptr, n, n_step, gamma, ret_ptr, disc_ptr, boot_ptr, stream))


def debug_collision_wall(which, center, radius, mv):
    """Run the DEVICE wall test on the GPU: (some, way, approximation, nx, ny, err)."""
    L = load_library()
    some, err = C.c_int32(0), C.c_uint32(0)
    f = [C.c_float(0) for _ in range(4)]
    _check(L.qlc_debug_collision_wall({"left": 0, "right": 1, "top": 2}[which], center[0], center[1], radius, mv[0], mv[1],
                                      C.addressof(some), *[C.addressof(x) for x in f], C.addressof(err)))
    return some.value, f[0].value, f[1].value, f[2].value, f[3].value, err.value


def debug_collision_rect(center, radius, mv, rmin, rmax):
    """Run the DEVICE ball-vs-rectangle sweep on the GPU: (some, way, approximation, nx, ny, err)."""
    L = load_library()
    some, err = C.c_int32(0), C.c_uint32(0)
    f = [C.c_float(0) for _ in range(4)]
    _check(L.qlc_debug_collision_rect(center[0], center[1], radius, mv[0], mv[1], rmin[0], rmin[1], rmax[0], rmax[1],
                                      C.addressof(some), *[C.addressof(x) for x in f], C.addressof(err)))
    return some.value, f[0].value, f[1].value, f[2].value, f[3].value, err.value


def debug_collision_rect_batch(cases):
    """cases f32 [n][9] (cx, cy, radius, mvx, mvy, min_x, min_y, max_x, max_y) -> (some u8[n], surf f32[n][4], err u32[n])
    from the DEVICE sweep routine."""
    a = np.ascontiguousarray(cases, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] != 9:
        raise QlError("cases must be [n][9]")
    out = np.empty((a.shape[0], 6), dtype=np.float32)
    _check(load_library().qlc_debug_collision_rect_batch(_np_ptr(a), _np_ptr(out), a.shape[0]))
    return (out[:, 0] != 0).astype(np.uint8), out[:, 1:5].copy(), out[:, 5].copy().view(np.uint32)


def debug_gemm_bf16(a, w, bias, relu=False):
    """out[m][n] = act(bf16(a)[m][k] @ bf16(w)[n][k].T + bias) on the tcgen05 tensor-core kernel (f32 host arrays)."""
    a = np.ascontiguousarray(a, dtype=np.float32); w = np.ascontiguousarray(w, dtype=np.float32); bias = np.ascontiguousarray(bias, dtype=np.float32)
    m, k = a.shape
    n = w.shape[0]
    out = np.empty((m, n), dtype=np.float32)
    _check(load_library().qlc_debug_gemm_bf16(_np_ptr(a), _np_ptr(w), _np_ptr(bias), 1 if relu else 0, _np_ptr(out), m, n, k))
    return out


class QNetwork:
    """Q-network on the tensor cores (tcgen05) for a BreakoutEnvironment: the reference's DeepQLearningModel
    (ml_model/model.rs:29-77) — predict_action for every env, batch_predict_max_future_reward for replay samples, and
    train on replay minibatches — reading the u8 frames straight from the frame ring. `weights`: dict of f32 arrays in the
    Keras layouts (QNET_SHAPES); bf16 operands, f32 accumulation; f32 master weights and Adam moments for training."""

    def __init__(self, env, weights):
        self._env = env
        self._L = env._L
        h = C.c_void_p()
        w, self._keep = self._pack(weights)
        _check(self._L.qlc_qnet_create(env._h, C.byref(w), C.byref(h)))
        self._h = h

    @staticmethod
    def _pack(weights):
        keep = []
        vals = []
        for name, _ in QlcQnetWeights._fields_:
            a = np.ascontiguousarray(weights[name], dtype=np.float32)
            if a.shape != QNET_SHAPES[name]:
                raise QlError("%s must have shape %s" % (name, QNET_SHAPES[name]))
            keep.append(a)
            vals.append(a.ctypes.data)
        return QlcQnetWeights(*vals), keep

    def set_weights(self, weights):
        w, keep = self._pack(weights)
        _check(self._L.qlc_qnet_set_weights(self._h, C.byref(w)))

    def close(self):
        if getattr(self, "_h", None):
            self._L.qlc_qnet_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def forward(self, indices=None, which=0):
        """indices None: current observation of every env; else replay transitions (which = 0 state / 1 state_next).
        Returns (q f32 [n][3], action u8 [n], max_q f32 [n]) on the host."""
        if indices is None:
            n, idx = self._env.n_envs, None
        else:
            idx = np.ascontiguousarray(indices, dtype=np.uint32)
            n = idx.size
        q = np.empty((n, 3), dtype=np.float32)
        a = np.empty(n, dtype=np.uint8)
        m = np.empty(n, dtype=np.float32)
        _check(self._L.qlc_qnet_forward_host(self._h, None if idx is None else _np_ptr(idx), n, which, _np_ptr(q), _np_ptr(a), _np_ptr(m)))
        return q, a, m

    def error(self):
        """Synchronise and return (then clear) the sticky time-out flag of the asynchronous forward_device passes."""
        e = C.c_uint32(0)
        _check(self._L.qlc_qnet_error(self._h, C.byref(e)))
        return e.value

    def forward_device(self, idx_ptr, n, which, q_ptr=None, action_ptr=None, max_q_ptr=None, stream=None):
        _check(self._L.qlc_qnet_forward(self._h, idx_ptr, n, which, q_ptr, action_ptr, max_q_ptr, stream))

    def get_weights(self):
        """The f32 master weights as a dict of arrays in the Keras layouts (QNET_SHAPES)."""
        out = {name: np.empty(shape, dtype=np.float32) for name, shape in QNET_SHAPES.items()}
        w, _ = self._pack(out)
        _check(self._L.qlc_qnet_get_weights(self._h, C.byref(w)))
        return out

    def set_adam(self, lr=2.5e-4, beta1=0.9, beta2=0.999, epsilon=1e-7, clipnorm=1.0):
        """Adam + per-variable clipnorm settings (clipnorm <= 0: no clipping); resets the moments and the step count."""
        _check(self._L.qlc_qnet_set_adam(self._h, C.byref(QlcAdamConfig(lr, beta1, beta2, epsilon, clipnorm))))

    def train(self, indices, targets=None, target_net=None, gamma=0.99, n_batches=1):
        """`n_batches` successive updates on the replay transitions `indices` ([n_batches * batch], minibatch j = the j-th
        slice). Targets: f32 [n_batches * batch], or None for y = r + max Q_target(state_next) * gamma (y = r where done)
        from `target_net`. Returns the Huber loss of each minibatch (before its update) as f32 [n_batches]."""
        idx = np.ascontiguousarray(indices, dtype=np.uint32).ravel()
        if n_batches < 1 or idx.size % n_batches:
            raise QlError("the number of indices must be a multiple of n_batches")
        batch = idx.size // n_batches
        tgt = None
        if targets is not None:
            tgt = np.ascontiguousarray(targets, dtype=np.float32).ravel()
            if tgt.size != idx.size:
                raise QlError("targets must have one value per index")
        loss = np.empty(n_batches, dtype=np.float32)
        _check(self._L.qlc_qnet_train_host(self._h, _np_ptr(idx), batch, n_batches, None if tgt is None else _np_ptr(tgt),
                                           None if target_net is None else target_net._h, gamma, _np_ptr(loss)))
        return loss

    def train_device(self, idx_ptr, batch, n_batches, target_ptr=None, target_net=None, gamma=0.99, loss_ptr=None, stream=None):
        """Device-pointer form of train (asynchronous on `stream`; time-outs surface through error())."""
        _check(self._L.qlc_qnet_train(self._h, idx_ptr, batch, n_batches, target_ptr, None if target_net is None else target_net._h,
                                      gamma, loss_ptr, stream))

    def debug_grads(self, indices, targets):
        """Forward + backward only: the unclipped f32 gradients of the loss on (indices, targets), Keras layouts."""
        idx = np.ascontiguousarray(indices, dtype=np.uint32).ravel()
        tgt = np.ascontiguousarray(targets, dtype=np.float32).ravel()
        if tgt.size != idx.size:
            raise QlError("targets must have one value per index")
        out = {name: np.empty(shape, dtype=np.float32) for name, shape in QNET_SHAPES.items()}
        w, _ = self._pack(out)
        _check(self._L.qlc_qnet_debug_grads(self._h, _np_ptr(idx), idx.size, _np_ptr(tgt), C.byref(w)))
        return out

    def train_weighted_device(self, idx_ptr, weight_ptr, batch, n_batches, target_ptr=None, target_net=None, gamma=0.99, loss_ptr=None, td_ptr=None,
                              stream=None):
        """train_device with per-item loss weights (weight_ptr None = 1: train_device's arithmetic) and, if td_ptr is given, the
        TD errors Q(s)[a] - y of every item written there (what PrioritizedReplay.update_device takes)."""
        _check(self._L.qlc_qnet_train_weighted(self._h, idx_ptr, weight_ptr, batch, n_batches, target_ptr, None if target_net is None else target_net._h,
                                               gamma, loss_ptr, td_ptr, stream))

    def train_nstep_device(self, idx_ptr, weight_ptr, batch, n_batches, target_net, gamma=0.99, n_step=1, double_dqn=False, loss_ptr=None,
                           td_ptr=None, y_ptr=None, stream=None):
        """train_weighted_device with n-step targets (ReplayBuffer.nstep_device) bootstrapped from `target_net`: max_a Q_target,
        or with `double_dqn` Q_target at the online network's greedy action. y_ptr (may be None) gets every item's target.
        n_step=1, double_dqn=False is train_weighted_device's arithmetic."""
        _check(self._L.qlc_qnet_train_nstep(self._h, idx_ptr, weight_ptr, batch, n_batches, target_net._h, gamma, n_step, 1 if double_dqn else 0,
                                            loss_ptr, td_ptr, y_ptr, stream))

    def debug_grads_weighted(self, indices, targets, weights):
        """Forward + backward only of the loss mean(w * Huber): (gradients in the Keras layouts, TD errors f32 [n])."""
        idx = np.ascontiguousarray(indices, dtype=np.uint32).ravel()
        tgt = np.ascontiguousarray(targets, dtype=np.float32).ravel()
        wt = np.ascontiguousarray(weights, dtype=np.float32).ravel()
        if tgt.size != idx.size or wt.size != idx.size:
            raise QlError("targets and weights must have one value per index")
        out = {name: np.empty(shape, dtype=np.float32) for name, shape in QNET_SHAPES.items()}
        w, _ = self._pack(out)
        td = np.empty(idx.size, dtype=np.float32)
        _check(self._L.qlc_qnet_debug_grads_weighted(self._h, _np_ptr(idx), idx.size, _np_ptr(tgt), _np_ptr(wt), C.byref(w), _np_ptr(td)))
        return out, td


class PrioritizedReplay:
    """Proportional prioritized replay (Schaul et al., ICLR 2016) over the replay ring of a BreakoutEnvironment: a sum tree on the
    device, p = (|delta| + epsilon)^alpha, new transitions at the running maximum priority. Sampling is stratified with
    replacement and returns logical replay indices (the ones QNetwork.train_device takes) and importance weights."""

    def __init__(self, env, alpha=0.6, epsilon=1e-6):
        self._env = env
        self._L = env._L
        self.alpha, self.epsilon = float(alpha), float(epsilon)
        h = C.c_void_p()
        _check(self._L.qlc_per_create(env._h, self.alpha, self.epsilon, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.qlc_per_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sample_device(self, batch, n_batches, call_index, beta, idx_ptr, weight_ptr=None, stream=None):
        """n_batches minibatches of `batch` indices (u32 [n_batches][batch] at idx_ptr) and weights (f32, weight_ptr may be None).
        Asynchronous on `stream`."""
        _check(self._L.qlc_per_sample(self._h, batch, n_batches, call_index, beta, idx_ptr, weight_ptr, stream))

    def update_device(self, idx_ptr, td_ptr, n, stream=None):
        """New priorities of the n transitions idx_ptr (u32) from their TD errors td_ptr (f32). Asynchronous on `stream`."""
        _check(self._L.qlc_per_update(self._h, idx_ptr, td_ptr, n, stream))

    def read(self):
        """(leaves f32 [len] in logical order, total f64 = the root, running max priority f32); synchronises."""
        n = C.c_uint64(0)
        _check(self._L.qlc_replay_len(self._env._h, C.byref(n)))
        leaves = np.empty(n.value, dtype=np.float32)
        total, mx = C.c_double(0), C.c_float(0)
        _check(self._L.qlc_per_read_host(self._h, _np_ptr(leaves) if leaves.size else None, C.byref(total), C.byref(mx)))
        return leaves, total.value, mx.value
