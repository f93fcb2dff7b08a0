"""CPU: the Hydra-free config surface (resolvers, overrides, FSTR command line) and that the built-in defaults equal the
reference's own YAML files (composed and stored by tests/golden/generate_golden.py as reference_cfg.json)."""
import json
import os

import pytest

from conftest import GOLDEN_DIR
from vine_robot_isaacgymenvs_b200 import abi, config as vcfg


def test_defaults_resolve_like_the_reference_resolvers():
    cfg = vcfg.compose()
    env = cfg["task"]["env"]
    assert env["numEnvs"] == 4096 and env["controlFrequencyInv"] == 4
    assert env["RANDOM_INIT_CART_MIN_Y"] == -0.1 * 0.3 and env["RANDOM_INIT_CART_MAX_Y"] == 0.3   # ${eval:...}, ${.X}
    assert cfg["task"]["sim"]["use_gpu_pipeline"] is True                                             # ${eq:...}
    assert cfg["task"]["sim"]["physx"]["use_gpu"] is True                                             # ${contains:...}
    assert cfg["task"]["sim"]["physx"]["num_threads"] == 4                                            # ${....x}
    assert cfg["task"]["physics_engine"] == "physx" and cfg["task_name"] == "Vine5LinkMovingBase"
    assert cfg["train"]["params"]["config"]["num_actors"] == 4096
    assert cfg["train"]["params"]["load_checkpoint"] is False                                         # ${if:...}
    assert cfg["train"]["params"]["config"]["minibatch_size"] == 32768


def test_cli_overrides_and_root_forwards():
    cfg = vcfg.compose(["num_envs=64", "RAIL_P_GAIN=30", "task.env.RAIL_SOFT_LIMIT=0.25", "pipeline=cpu",
                        "sim_device=cpu", "checkpoint=runs/x.pth", "vine_randomize=False"])
    env = cfg["task"]["env"]
    assert env["numEnvs"] == 64 and env["RAIL_P_GAIN"] == 30 and env["RAIL_SOFT_LIMIT"] == 0.25
    assert env["RANDOM_INIT_CART_MIN_Y"] == -0.1 * 0.25 and env["RANDOM_INIT_CART_MAX_Y"] == 0.25
    assert cfg["task"]["sim"]["use_gpu_pipeline"] is False and cfg["task"]["sim"]["physx"]["use_gpu"] is False
    assert cfg["train"]["params"]["load_checkpoint"] is True and cfg["train"]["params"]["load_path"] == "runs/x.pth"
    assert cfg["task"]["task"]["vine_randomize"] is False


def test_fstr_command_line():
    """README.md:63 incl. the undeclared ACCEL_TARGET_SCALING_* keys (SURVEY 0.1)."""
    t = vcfg.fstr_task_config(["num_envs=4096"])
    vc = vcfg.task_cfg_to_vine_config(t)
    assert vc.observation_type == abi.OBSERVATION_TYPES["TIP_AND_CART_AND_OBJ_INFO"]
    assert (vc.rail_p_gain, vc.rail_acceleration, vc.action_delay, vc.max_episode_length) == (30, 6, 1, 100)
    assert (vc.create_shelf, vc.create_pipe, vc.vine_randomize) == (0, 0, 1)
    assert (vc.accel_target_scaling_min, vc.accel_target_scaling_max) == (0.99, 1.05)
    assert (vc.dynamics_scaling_min, vc.action_noise_std, vc.success_dist) == (0.999999, 0.001, 0.04)
    assert vcfg.num_observations(t["env"]["OBSERVATION_TYPE"]) == 18


def test_unknown_observation_type_raises_keyerror_like_the_reference():
    t = vcfg.task_config(["OBSERVATION_TYPE=NOPE"])
    with pytest.raises(KeyError):
        vcfg.task_cfg_to_vine_config(t)


def test_builtin_defaults_equal_the_reference_yaml_files():
    ours = vcfg.compose(["task=Vine5LinkMovingBase"])
    with open(os.path.join(GOLDEN_DIR, "reference_cfg.json")) as f:
        theirs = json.load(f)          # without the author's wandb_* settings
    assert ours["task"] == theirs["task"]
    assert ours["train"] == theirs["train"]
    for k, v in theirs.items():
        assert ours[k] == v, k
