"""CPU-only checks of the prioritized-replay ABI: the Python defaults, and argument validation without a GPU (out-of-range
alpha / epsilon / beta and null handles are rejected; a valid call that would compute fails with QLC_ERR_NO_DEVICE)."""
import ctypes
import importlib
import inspect

import pytest


def test_python_defaults():
    qlb = importlib.import_module("q-learning_b200")
    d = inspect.signature(qlb.PrioritizedReplay.__init__).parameters
    assert (d["alpha"].default, d["epsilon"].default) == (0.6, 1e-6)
    pytest.importorskip("torch")
    tio = importlib.import_module("q-learning_b200.torch_io")
    d = inspect.signature(tio.TensorCoreLearner.__init__).parameters
    assert (d["per_alpha"].default, d["per_epsilon"].default) == (None, 1e-6)


def test_argument_validation_without_gpu(qlb):
    lib = qlb.load_library()
    h = ctypes.c_void_p()
    # a zeroed stand-in for an env handle: every check below fails before anything reads it
    fake_env = ctypes.create_string_buffer(4096)
    assert lib.qlc_per_create(None, 0.6, 1e-6, ctypes.byref(h)) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_create(fake_env, 0.6, 1e-6, None) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_create(fake_env, 1.5, 1e-6, ctypes.byref(h)) == qlb.ERR_INVALID_ARG
    assert b"alpha" in lib.qlc_last_error_string()
    assert lib.qlc_per_create(fake_env, -0.1, 1e-6, ctypes.byref(h)) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_create(fake_env, 0.6, 0.0, ctypes.byref(h)) == qlb.ERR_INVALID_ARG
    assert b"epsilon" in lib.qlc_last_error_string()
    assert lib.qlc_per_create(fake_env, 0.6, float("inf"), ctypes.byref(h)) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_sample(None, 32, 1, 0, -0.1, None, None, None) == qlb.ERR_INVALID_ARG
    assert b"beta" in lib.qlc_last_error_string()
    assert lib.qlc_per_sample(None, 0, 1, 0, 0.4, None, None, None) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_sample(None, 32, 1, 0, 0.4, None, None, None) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_sample(None, 1 << 16, 1 << 15, 0, 0.4, None, None, None) == qlb.ERR_INVALID_ARG     # too many items
    assert lib.qlc_per_update(None, None, None, 4, None) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_read_host(None, None, None, None) == qlb.ERR_INVALID_ARG
    assert lib.qlc_per_destroy(None) == qlb.OK
    assert lib.qlc_qnet_train_weighted(None, None, None, 32, 1, None, None, 0.99, None, None, None) == qlb.ERR_INVALID_ARG
    assert lib.qlc_qnet_debug_grads_weighted(None, None, 4, None, None, None, None) == qlb.ERR_INVALID_ARG
    if qlb.device_count() > 0:
        pytest.skip("a GPU is present")
    assert lib.qlc_per_create(fake_env, 0.6, 1e-6, ctypes.byref(h)) == qlb.ERR_NO_DEVICE
    assert h.value is None
