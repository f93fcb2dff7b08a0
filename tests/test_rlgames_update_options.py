"""CPU: the rl_games keys lr_schedule, schedule_type, max_epochs, clip_value, schedule_entropy and reward_shaper are parsed and
checked on a plain train-config dict (PPOAgent.update_options) before any agent or GPU exists: a value the update paths cannot
honour raises instead of being ignored, and the reference configuration passes unchanged."""
import copy
import json
import math
import os

import pytest

from conftest import REPO
from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent


def reference_train_cfg():
    with open(os.path.join(REPO, "tests", "golden", "reference_cfg.json")) as f:
        return json.load(f)["train"]


def with_keys(**keys):
    cfg = copy.deepcopy(reference_train_cfg())
    cfg["params"]["config"].update(keys)
    return cfg


def test_reference_config_is_accepted_unchanged():
    cfg = reference_train_cfg()
    before = copy.deepcopy(cfg)
    o = PPOAgent.update_options(cfg)
    assert cfg == before
    assert o == {"adaptive": True, "linear": False, "standard": False, "max_epochs": 500, "clip_value": True,
                 "reward_scale": 0.01, "reward_shift": 0.0, "reward_min": -math.inf, "reward_max": math.inf}


def test_unknown_schedule_type_raises():
    with pytest.raises(ValueError, match="schedule_type"):
        PPOAgent.update_options(with_keys(schedule_type="cosine"))


@pytest.mark.parametrize("max_epochs", [0, -1])
def test_linear_schedule_needs_positive_max_epochs(max_epochs):
    with pytest.raises(ValueError, match="max_epochs"):
        PPOAgent.update_options(with_keys(lr_schedule="linear", max_epochs=max_epochs))
    # the same max_epochs is fine for the other schedules, which do not read it
    assert not PPOAgent.update_options(with_keys(lr_schedule="adaptive", max_epochs=max_epochs))["linear"]


def test_schedule_entropy_raises_not_implemented():
    with pytest.raises(NotImplementedError, match="schedule_entropy"):
        PPOAgent.update_options(with_keys(lr_schedule="linear", schedule_entropy=True))
    assert PPOAgent.update_options(with_keys(schedule_entropy=False))["adaptive"]


def test_reward_shaper_log_val_raises_not_implemented():
    with pytest.raises(NotImplementedError, match="log_val"):
        PPOAgent.update_options(with_keys(reward_shaper={"scale_value": 0.01, "log_val": True}))


def test_new_keys_are_parsed():
    o = PPOAgent.update_options(with_keys(lr_schedule="linear", schedule_type="standard", max_epochs=7, clip_value=False,
                                          reward_shaper={"scale_value": 0.5, "shift_value": -2.0, "min_val": -1, "max_val": 3}))
    assert o == {"adaptive": False, "linear": True, "standard": True, "max_epochs": 7, "clip_value": False,
                 "reward_scale": 0.5, "reward_shift": -2.0, "reward_min": -1.0, "reward_max": 3.0}
    # any other lr_schedule is a constant learning rate, as in rl_games
    o = PPOAgent.update_options(with_keys(lr_schedule=None))
    assert not o["adaptive"] and not o["linear"]
