"""The C++ mirror of the reference interfaces (include/ql_cuda.hpp): compiles and links on CPU; on the GPU box it is
driven like SelfDrivingQLearner::learn_episode drives Environment + ReplayBuffer (tests/cpp/test_facade.cpp)."""
import os
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(qlb, out_dir):
    """builds tests/cpp/test_facade.cpp into out_dir (a temporary directory: the repository tree may be read-only)"""
    qlb.load_library()
    so_dir = os.path.dirname(qlb.library_path())
    exe = os.path.join(out_dir, "test_facade")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_facade.cpp"),
           "-o", exe, "-L", so_dir, "-lqlcuda", "-Wl,-rpath," + so_dir]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def test_facade_compiles_and_links(qlb):
    with tempfile.TemporaryDirectory() as d:
        exe = _build(qlb, d)
        assert os.path.exists(exe)
        if qlb.device_count() == 0:
            res = subprocess.run([exe], capture_output=True, text=True)
            assert res.returncode == 2 and "no CUDA device" in res.stdout      # loud failure, no fallback


@pytest.mark.gpu
def test_facade_learn_episode_loop(qlb):
    with tempfile.TemporaryDirectory() as d:
        res = subprocess.run([_build(qlb, d)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "facade ok" in res.stdout
