"""The training half of the C++ TensorCoreQModel (include/ql_cuda.hpp: weights(), train_replay()): compiles and links on the
CPU; on the GPU tests/cpp/test_train_facade.cpp checks the weight round trip and one update."""
import os
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(qlb, out_dir):
    qlb.load_library()
    so_dir = os.path.dirname(qlb.library_path())
    exe = os.path.join(out_dir, "test_train_facade")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_train_facade.cpp"),
           "-o", exe, "-L", so_dir, "-lqlcuda", "-Wl,-rpath," + so_dir]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def test_train_facade_compiles_and_links(qlb):
    with tempfile.TemporaryDirectory() as d:
        assert os.path.exists(_build(qlb, d))


@pytest.mark.gpu
def test_train_facade_round_trip_and_update(qlb):
    with tempfile.TemporaryDirectory() as d:
        res = subprocess.run([_build(qlb, d)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "train facade ok" in res.stdout
