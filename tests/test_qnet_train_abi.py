"""CPU-only checks of the training ABI: the Adam settings struct is declared alike in the C header, the ctypes binding
and the Rust ffi, and the Python defaults are the Keras model's."""
import inspect
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["lr", "beta1", "beta2", "epsilon", "clipnorm"]


def test_adam_config_layout_matches_across_bindings(qlb):
    header = open(os.path.join(ROOT, "include", "ql_cuda.h")).read()
    m = re.search(r"typedef struct qlc_adam_config \{ float ([^;]*); \} qlc_adam_config;", header)
    assert m and [f.strip() for f in m.group(1).split(",")] == FIELDS
    assert [n for n, _ in qlb.QlcAdamConfig._fields_] == FIELDS
    ffi = open(os.path.join(ROOT, "bindings", "rust", "ql-cuda", "src", "ffi.rs")).read()
    body = re.search(r"pub struct qlc_adam_config \{(.*?)\}", ffi, re.S).group(1)
    assert re.findall(r"pub (\w+): f32", body) == FIELDS


def test_python_adam_defaults_are_the_keras_models():
    import importlib
    qlb = importlib.import_module("q-learning_b200")
    d = inspect.signature(qlb.QNetwork.set_adam).parameters
    assert (d["lr"].default, d["beta1"].default, d["beta2"].default, d["epsilon"].default, d["clipnorm"].default) == (2.5e-4, 0.9, 0.999, 1e-7, 1.0)
    assert inspect.signature(qlb.QNetwork.train).parameters["gamma"].default == 0.99
