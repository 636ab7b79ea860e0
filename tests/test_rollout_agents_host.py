"""Host side of the device rollout's agent count: the Transition widths, the exported entry point and the checks that
need no device."""
import ctypes as C

import numpy as np
import pytest


def test_transition_fields_widths():
    from flexgpu.policy import TRANSITION_FIELDS, transition_fields
    assert transition_fields(5) == TRANSITION_FIELDS
    for na in range(1, 6):
        f = transition_fields(na)
        assert list(f) == list(TRANSITION_FIELDS)
        assert f == {"state": 144 * na, "action": 4 * na, "log_prob_a": 4 * na, "value": na, "next_value": na, "reward": na,
                     "next_state": 144 * na, "done": 1, "last_step": 1, "action_avail": 4 * na, "last_hid": 64 * na,
                     "hid": 64 * na}


def test_weight_shapes_follow_the_agent_count():
    from flexgpu.policy import _CRITIC_SHAPES, _WEIGHT_SHAPES, critic_shapes, weight_shapes
    assert weight_shapes(5) == _WEIGHT_SHAPES and critic_shapes(5) == _CRITIC_SHAPES
    assert weight_shapes(2)[0] == (64, 146) and critic_shapes(2)[0] == (64, 298) and critic_shapes(5)[0] == (64, 745)


def test_create_agents_is_exported():
    import subprocess
    from flexgpu import _lib
    syms = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert " T fp_policy_create_agents\n" in syms                      # the built library's dynamic symbol table
    lib = _lib.lib()
    assert lib.fp_policy_create_agents.argtypes[1] is C.c_int32
    p = C.c_void_p()
    assert lib.fp_policy_create_agents(0, 0, C.byref(p)) == -1             # FP_EINVAL before any device is touched
    assert b"n_agents must be in [1, 5]" in lib.fp_policy_last_error(None)


def test_policy_agent_count_checks_before_the_device():
    from flexgpu.policy import DevicePolicy
    for na in (0, 6):
        with pytest.raises(ValueError, match=r"\[1, 5\]"):
            DevicePolicy(None, n_agents=na)
    sd = {"fc1.weight": np.zeros((64, 147), np.float32)}
    with pytest.raises(ValueError, match="conflicts"):
        DevicePolicy(sd, n_agents=4)
    with pytest.raises(ValueError, match="fc1.weight"):
        DevicePolicy({"fc1.weight": np.zeros((64, 150), np.float32)})
