"""CPU: the C-ABI shared library loads, exports every symbol include/flexgpu.h declares, its
struct layout matches the Python binding, and it refuses to run without a GPU (no fallback).
No compute calls are made here."""
import ctypes as C
import os
import re

import pytest

from flexgpu import _lib
from flexgpu.config import DEFAULT_ENV_ARGS, make_fp_config, normalize_args
from flexgpu.network import Network, create_network

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "flexgpu.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fp_[a-z0-9_]+)\s*\(", src)))


def test_library_is_built_in_tree():
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    assert os.path.dirname(_lib.LIB_PATH).startswith(ROOT)


def test_every_declared_symbol_is_exported_and_bound():
    syms = declared_symbols()
    assert len(syms) >= 19
    raw = C.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(raw, s), f"{s} declared in flexgpu.h but not exported"
    assert set(syms) == set(_lib.EXPORTED_SYMBOLS), "python binding and header disagree"


def test_struct_layout_matches_library():
    l = _lib.lib()
    assert l.fp_sizeof_config() == C.sizeof(_lib.FpConfig)


def test_header_constants_match_binding():
    src = open(HEADER).read()
    for name, val in (("FP_MAX_BUS", _lib.FP_MAX_BUS), ("FP_MAX_AGENTS", _lib.FP_MAX_AGENTS),
                      ("FP_INFO_STRIDE", _lib.FP_INFO_STRIDE), ("FP_NSTATS", _lib.FP_NSTATS),
                      ("FP_REC_STRIDE", _lib.FP_REC_STRIDE)):
        m = re.search(rf"#define\s+{name}\s+(\d+)", src)
        assert m and int(m.group(1)) == val
    for name, val in (("FP_REC_E_INIT", _lib.REC_E_INIT), ("FP_REC_E_CUR", _lib.REC_E_CUR), ("FP_REC_CUM", _lib.REC_CUM),
                      ("FP_REC_TIME", _lib.REC_TIME), ("FP_REC_HIST", _lib.REC_HIST), ("FP_REC_VMASK", _lib.REC_VMASK),
                      ("FP_REC_COUNTS", _lib.REC_COUNTS), ("FP_REC_LINES", _lib.REC_LINES)):
        m = re.search(rf"{name}\s*=\s*(\d+)", src)
        assert m and int(m.group(1)) == val


def test_no_cpu_fallback():
    """Without a CUDA device fp_create must fail loudly (skipped on a GPU box)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    l = _lib.lib()
    args = normalize_args(None)
    cfg = make_fp_config(args, Network(create_network(DEFAULT_ENV_ARGS)))
    h = C.c_void_p()
    rc = l.fp_create(C.byref(cfg), 4, 0, C.byref(h))
    assert rc == -2 and not h.value
    assert b"no CUDA device" in l.fp_last_error(None)
    from flexgpu import BatchedFlexProvisionEnv, FlexGpuError
    with pytest.raises(FlexGpuError):
        BatchedFlexProvisionEnv(None, n_envs=2)


def test_null_handle_calls_are_rejected():
    l = _lib.lib()
    assert l.fp_step(None, None, 0, None, None, None, None, None) == -1
    assert l.fp_n_envs(None) == 0 and l.fp_launch_count(None) == 0
    assert l.fp_destroy(None) == 0
    assert l.fp_policy_act(None, None, 0, 0, 0, None, None, None, 0, None, None, None, None, 0, 0, 1.0, 0, None) == -1
    assert l.fp_policy_load(None, *[None] * 10) == -1 and l.fp_critic_load(None, *[None] * 8) == -1
    assert l.fp_critic_value(None, None, 0, 0, 0, None, None, None) == -1
    assert l.fp_policy_rows_to_ring(None, None, 0, 0, None, 0, 0, None) == -1
    assert l.fp_learner_feed(None, None, None, None, 0, None, None, None) == -1
    assert l.fp_policy_launch_count(None) == 0 and l.fp_policy_destroy(None) == 0
    assert l.fp_replay_write(None, 0, 0, 0, None, None) == -1
    assert l.fp_replay_sample(None, 0, 0, None, None) == -1
    assert l.fp_replay_reserve(None, 0, None) == -1 and l.fp_replay_clear(None) == -1
    assert l.fp_replay_len(None) == 0 and l.fp_replay_destroy(None) == 0
    assert l.fp_predict(None, 0, None, None, None, None, 0, 0, 0, None) == -1
