"""CPU: the gradient-clipping entry points reject malformed arguments with VINE_ERR_INVALID_ARG before any CUDA call, so these
run without a GPU (the pointers are never dereferenced on the host)."""
import ctypes as C

import pytest

from vine_robot_isaacgymenvs_b200 import abi, build as vbuild

F = C.c_void_p(4096)          # stand-in device pointers: validation returns before anything is launched
NULL = None


@pytest.fixture(scope="module")
def lib():
    vbuild.build()
    return abi.load_library()


def test_grad_clip_symbols_are_declared(lib):
    for name in ("vine_grad_clip", "vine_ppo_adam_clipped", "vine_lstm_adam_clipped"):
        assert name in abi.EXPORTED_SYMBOLS and getattr(lib, name) is not None
    assert (abi.PPO_STATE_CLIP_COEF, abi.PPO_STATE_GRAD_NORM) == (9, 10) and abi.PPO_STATE_GRAD_NORM < abi.PPO_STATE_FLOATS


@pytest.mark.parametrize("args", [
    # flat, count, length, flat2, count2, length2, scale, max_norm, state, workspace, ch, ch2
    (NULL, 10, 14, NULL, 0, 0, 1.0, 1.0, F, F, NULL, NULL),             # no gradient vector
    (F, 10, 14, NULL, 0, 0, 1.0, 1.0, NULL, F, NULL, NULL),             # no state block
    (F, 10, 14, NULL, 0, 0, 1.0, 1.0, F, NULL, NULL, NULL),             # no workspace
    (F, 0, 14, NULL, 0, 0, 1.0, 1.0, F, F, NULL, NULL),                 # count < 1
    (F, 15, 14, NULL, 0, 0, 1.0, 1.0, F, F, NULL, NULL),                # count above the vector length
    (F, 10, 14, F, 0, 20, 1.0, 1.0, F, F, NULL, NULL),                  # second vector: count < 1
    (F, 10, 14, F, 21, 20, 1.0, 1.0, F, F, NULL, NULL),                 # second vector: count above its length
    (F, 10, 14, NULL, 5, 0, 1.0, 1.0, F, F, NULL, NULL),                # a count without a second vector
    (F, 10, 14, NULL, 0, 0, 1.0, 1.0, F, F, NULL, F),                   # a channel without a second vector
    (F, 10, 14, NULL, 0, 0, 1.0, float("inf"), F, F, NULL, NULL),       # max_norm not finite
    (F, 10, 14, NULL, 0, 0, 1.0, float("nan"), F, F, NULL, NULL),
], ids=["flat", "state", "workspace", "count0", "count_gt_len", "count2_0", "count2_gt_len2", "count2_without_flat2",
        "channel2_without_flat2", "max_norm_inf", "max_norm_nan"])
def test_grad_clip_rejects_malformed_arguments(lib, args):
    assert lib.vine_grad_clip(*args, NULL) == abi.ERR_INVALID_ARG


def test_clipped_adam_entry_points_reject_malformed_arguments(lib):
    common = (0.9, 0.999, 1e-8)
    assert lib.vine_ppo_adam_clipped(NULL, 1.0, F, F, F, F, F, 18, *common, 1, F, NULL, NULL) == abi.ERR_INVALID_ARG
    assert lib.vine_ppo_adam_clipped(F, 1.0, NULL, F, F, F, F, 18, *common, 1, F, NULL, NULL) == abi.ERR_INVALID_ARG
    assert lib.vine_ppo_adam_clipped(F, 1.0, F, F, F, F, F, 0, *common, 1, F, NULL, NULL) == abi.ERR_INVALID_ARG
    assert lib.vine_ppo_adam_clipped(F, 1.0, F, F, F, F, F, 32, *common, 1, F, NULL, NULL) == abi.ERR_INVALID_ARG
    assert lib.vine_lstm_adam_clipped(NULL, 1.0, F, F, F, F, F, 18, *common, F, NULL, NULL) == abi.ERR_INVALID_ARG
    assert lib.vine_lstm_adam_clipped(F, 1.0, F, F, F, NULL, F, 18, *common, F, NULL, NULL) == abi.ERR_INVALID_ARG
    assert lib.vine_lstm_adam_clipped(F, 1.0, F, F, F, F, F, 0, *common, F, NULL, NULL) == abi.ERR_INVALID_ARG
