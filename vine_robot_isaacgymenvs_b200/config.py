"""Configuration surface of the Vine5LinkMovingBase path.

The reference composes its config with Hydra/OmegaConf (neither is installed here):
``isaacgymenvs/cfg/config.yaml`` (root), ``cfg/task/Vine5LinkMovingBase.yaml`` and
``cfg/train/Vine5LinkMovingBasePPO.yaml``, using the custom resolvers of
``isaacgymenvs/__init__.py:8-12`` (eq, contains, if, resolve_default, eval).  The env
constructor finally receives a *plain nested dict* (``utils/rlgames_utils.py:78-86``).

This module provides
  * the same key set with the same defaults (as Python data, SURVEY Appendix C),
  * a small interpolation engine for those five resolvers + relative node references, so
    ``compose(["task.env.RAIL_P_GAIN=30", "num_envs=4096"])`` behaves like the reference CLI
    and a user's own ``cfg/`` YAML files load unchanged (``compose(cfg_dir=...)``),
  * ``task_cfg_to_vine_config``: plain dict -> ``VineConfig`` for the C ABI.
Unknown keys are accepted (the FSTR command line of README.md:63 passes
``ACCEL_TARGET_SCALING_MIN/MAX`` which this snapshot's YAML does not declare).
"""
import copy
import ctypes as C
import os
import re

import yaml

from . import abi

# --------------------------------------------------------------------------------------------
# Defaults (key names/values: cfg/config.yaml:13-49, cfg/task/Vine5LinkMovingBase.yaml:2-134)
# --------------------------------------------------------------------------------------------
ROOT_DEFAULTS = {
    "task_name": "${task.name}",
    "experiment": "",
    "num_envs": "", "horizon_length": "", "minibatch_size": "", "control_frequency_inv": "",
    "vine_randomize": "", "CAPTURE_VIDEO": "", "RAIL_VELOCITY_SCALE": "", "RAIL_SOFT_LIMIT": "",
    "RAIL_P_GAIN": "", "OBSERVATION_TYPE": "", "RAIL_ACCELERATION": "",
    "enable_viewer_sync_at_start": True,
    "wandb_group": "", "wandb_name": "${train.params.config.name}", "wandb_entity": "",
    "wandb_project": "isaacgymenvs", "capture_video_freq": 1464, "capture_video_len": 100,
    "seed": 42, "torch_deterministic": False, "max_iterations": "",
    "physics_engine": "physx", "pipeline": "gpu", "sim_device": "cuda:0", "rl_device": "cuda:0",
    "graphics_device_id": 0,
    "num_threads": 4, "solver_type": 1, "num_subscenes": 4,
    "test": False, "checkpoint": "", "multi_gpu": False,
    "wandb_activate": False, "capture_video": False, "force_render": True, "headless": False,
}


def _rd(default, knob):
    return "${resolve_default:%s,${...%s}}" % (default, knob)


TASK_DEFAULTS = {
    "name": "Vine5LinkMovingBase",
    "physics_engine": "${..physics_engine}",
    "env": {
        "numEnvs": _rd(4096, "num_envs"), "envSpacing": 6.0,
        "clipObservations": 5.0, "clipActions": 1.0,
        "maxEpisodeLength": 500,
        "controlFrequencyInv": _rd(4, "control_frequency_inv"),
        "enableCameraSensors": False,
        "USE_MOVING_BASE": True, "USE_SMOOTHED_FPAM": True,
        "FORCE_U_FPAM": False, "FORCE_U_RAIL_VELOCITY": False,
        "SMOOTHING_ALPHA_INFLATE": 0.81, "SMOOTHING_ALPHA_DEFLATE": 0.86,
        "CAPTURE_VIDEO": _rd(True, "CAPTURE_VIDEO"),
        "CREATE_SHELF": False, "CREATE_PIPE": True, "CREATE_HISTOGRAMS_PERIODICALLY": False,
        "MAT_FILE": "",
        "FPAM_MIN": -0.1, "FPAM_MAX": 3.0, "RAIL_VELOCITY_SCALE": _rd(1.0, "RAIL_VELOCITY_SCALE"),
        "DAMPING": 2e-2, "STIFFNESS": 0.0,
        "RAIL_SOFT_LIMIT": _rd(0.3, "RAIL_SOFT_LIMIT"),
        "RAIL_P_GAIN": _rd(10.0, "RAIL_P_GAIN"), "RAIL_D_GAIN": 0.0,
        "RAIL_ACCELERATION": _rd(8.0, "RAIL_ACCELERATION"),
        "OBSERVATION_TYPE": _rd("POS_AND_FD_VEL_AND_OBJ_INFO", "OBSERVATION_TYPE"),
        "RANDOMIZE_DOF_INIT": True,
        "RANDOM_INIT_CART_MIN_Y": "${eval:'-0.1 * ${.RAIL_SOFT_LIMIT}'}",
        "RANDOM_INIT_CART_MAX_Y": "${.RAIL_SOFT_LIMIT}",
        "RANDOMIZE_TARGETS": True,
        "SUCCESS_DIST": 0.08,
        "MIN_TARGET_DEPTH_IN_OBSTACLE": -0.05, "MAX_TARGET_DEPTH_IN_OBSTACLE": 0.2,
        "MIN_TARGET_Y": -0.48, "MAX_TARGET_Y": -0.4, "MIN_TARGET_Z": 0.58, "MAX_TARGET_Z": 0.67,
        "POSITION_REWARD_WEIGHT": 0.0, "CONST_NEGATIVE_REWARD_WEIGHT": 0.0,
        "POSITION_SUCCESS_REWARD_WEIGHT": 1.0, "VELOCITY_SUCCESS_REWARD_WEIGHT": 0,
        "VELOCITY_REWARD_WEIGHT": 0.1, "U_RAIL_VELOCITY_CONTROL_REWARD_WEIGHT": 0.0,
        "U_FPAM_CONTROL_REWARD_WEIGHT": 0.0, "RAIL_VELOCITY_CHANGE_REWARD_WEIGHT": 0.0,
        "U_FPAM_CHANGE_REWARD_WEIGHT": 0.0, "RAIL_LIMIT_REWARD_WEIGHT": 1.0,
        "CART_Y_REWARD_WEIGHT": 0.0, "TIP_Y_REWARD_WEIGHT": 0.0,
        "CONTACT_FORCE_REWARD_WEIGHT": 0.10,
        "USE_TARGET_REACHED_RESET": True, "USE_TIP_LIMIT_HIT_RESET": False,
        "USE_NONZERO_CONTACT_FORCE_RESET": False,
        "SCALE_OBSERVATIONS": True,
        "ACTION_DELAY": 1,
    },
    "sim": {
        "dt": 0.00833, "substeps": 10, "up_axis": "z",
        "use_gpu_pipeline": '${eq:${...pipeline},"gpu"}',
        "gravity": [0.0, 0.0, -9.81],
        "enable_viewer_sync_at_start": _rd(True, "enable_viewer_sync_at_start"),
        "physx": {
            "num_threads": "${....num_threads}", "solver_type": "${....solver_type}",
            "use_gpu": '${contains:"cuda",${....sim_device}}',
            "num_position_iterations": 8, "num_velocity_iterations": 4,
            "contact_offset": 0.02, "rest_offset": 0.001,
            "bounce_threshold_velocity": 0.2, "max_depenetration_velocity": 100.0,
            "default_buffer_size_multiplier": 2.0, "max_gpu_contact_pairs": 1048576,
            "num_subscenes": "${....num_subscenes}", "contact_collection": 0,
        },
    },
    "task": {
        "vine_randomize": _rd(True, "vine_randomize"),
        "randomization_parameters": {
            "DYNAMICS_SCALING_MIN": 0.999, "DYNAMICS_SCALING_MAX": 1.001,
            "OBSERVATION_NOISE_STD": 0.0, "ACTION_NOISE_STD": 0.0,
        },
    },
}

# cfg/train/Vine5LinkMovingBasePPO.yaml (rl_games a2c_continuous)
TRAIN_DEFAULTS = {
    "params": {
        "seed": "${...seed}",
        "algo": {"name": "a2c_continuous"},
        "model": {"name": "continuous_a2c_logstd"},
        "network": {
            "name": "actor_critic", "separate": False,
            "space": {"continuous": {
                "mu_activation": "None", "sigma_activation": "None",
                "mu_init": {"name": "default"},
                "sigma_init": {"name": "const_initializer", "val": 0},
                "fixed_sigma": True}},
            "mlp": {"units": [256, 128, 64], "activation": "elu", "d2rl": False,
                    "initializer": {"name": "default"}, "regularizer": {"name": "None"}},
            "rnn": {"name": "lstm", "units": 256, "layers": 1, "before_mlp": False,
                    "concat_input": True, "layer_norm": True},
        },
        "load_checkpoint": "${if:${...checkpoint},True,False}",
        "load_path": "${...checkpoint}",
        "config": {
            "name": "${resolve_default:Vine5LinkMovingBase,${....experiment}}",
            "full_experiment_name": "${.name}",
            "env_name": "rlgpu", "device": "${....rl_device}", "multi_gpu": "${....multi_gpu}",
            "ppo": True, "mixed_precision": True, "normalize_input": True,
            "normalize_value": True, "value_bootstrap": True,
            "num_actors": "${....task.env.numEnvs}",
            "reward_shaper": {"scale_value": 0.01},
            "normalize_advantage": True, "gamma": 0.99, "tau": 0.95,
            "learning_rate": 3e-4, "lr_schedule": "adaptive", "schedule_type": "legacy",
            "kl_threshold": 0.008, "score_to_win": 20000000000,
            "max_epochs": "${resolve_default:500,${....max_iterations}}",
            "save_best_after": 50, "save_frequency": 50, "grad_norm": 1.0,
            "entropy_coef": 0.0, "truncate_grads": False, "e_clip": 0.2,
            "horizon_length": "${resolve_default:16,${....horizon_length}}",
            "minibatch_size": "${resolve_default:32768,${....minibatch_size}}",
            "mini_epochs": 4, "critic_coef": 2, "clip_value": True, "seq_len": 4,
            "bounds_loss_coef": 0.0001,
        },
    }
}

# The FSTR command line (README.md:63), as overrides for compose().
FSTR_OVERRIDES = [
    "task=Vine5LinkMovingBase", "wandb_activate=False",
    "task.env.RAIL_SOFT_LIMIT=0.25", "RAIL_P_GAIN=30", "RAIL_ACCELERATION=6", "RAIL_VELOCITY_SCALE=1",
    "task.env.CREATE_SHELF=False", "task.env.CREATE_PIPE=False", "vine_randomize=True",
    "OBSERVATION_TYPE=TIP_AND_CART_AND_OBJ_INFO", "task.env.ACTION_DELAY=1",
    "task.env.maxEpisodeLength=100", "task.env.SUCCESS_DIST=0.04",
    "task.env.MIN_TARGET_Y=-0.4", "task.env.MAX_TARGET_Y=0.4",
    "task.env.MIN_TARGET_Z=0.55", "task.env.MAX_TARGET_Z=0.7",
    "task.env.MIN_TARGET_DEPTH_IN_OBSTACLE=0.0", "task.env.MAX_TARGET_DEPTH_IN_OBSTACLE=0.0",
    "task.env.CONTACT_FORCE_REWARD_WEIGHT=0.0",
    "task.task.randomization_parameters.DYNAMICS_SCALING_MIN=0.999999",
    "task.task.randomization_parameters.DYNAMICS_SCALING_MAX=1.000001",
    "task.task.randomization_parameters.ACTION_NOISE_STD=0.001",
    "task.task.randomization_parameters.OBSERVATION_NOISE_STD=0.0",
    "+task.task.randomization_parameters.ACCEL_TARGET_SCALING_MIN=0.99",
    "+task.task.randomization_parameters.ACCEL_TARGET_SCALING_MAX=1.05",
    "max_iterations=600",
]

# BASELINE configs[2]: shelf target reaching (README.md:71 + contact-force resets on), SURVEY §8(d) C3
SHELF_OVERRIDES = [
    "task=Vine5LinkMovingBase", "wandb_activate=False", "task.env.CREATE_SHELF=True", "task.env.CREATE_PIPE=False",
    "task.env.MIN_TARGET_DEPTH_IN_OBSTACLE=-0.05", "task.env.MAX_TARGET_DEPTH_IN_OBSTACLE=0.2",
    "task.env.USE_NONZERO_CONTACT_FORCE_RESET=True", "vine_randomize=True",
    "task.task.randomization_parameters.ACTION_NOISE_STD=0.01",
]
# BASELINE configs[3]: pipe obstacle with full domain randomization (widened ranges), SURVEY §8(d) C4
PIPE_DR_OVERRIDES = [
    "task=Vine5LinkMovingBase", "wandb_activate=False", "task.env.CREATE_SHELF=False", "task.env.CREATE_PIPE=True",
    "vine_randomize=True",
    "task.task.randomization_parameters.DYNAMICS_SCALING_MIN=0.9",
    "task.task.randomization_parameters.DYNAMICS_SCALING_MAX=1.1",
    "task.task.randomization_parameters.ACTION_NOISE_STD=0.01",
    "task.task.randomization_parameters.OBSERVATION_NOISE_STD=0.01",
    "+task.task.randomization_parameters.ACCEL_TARGET_SCALING_MIN=0.9",
    "+task.task.randomization_parameters.ACCEL_TARGET_SCALING_MAX=1.1",
]


# --------------------------------------------------------------------------------------------
# Interpolation engine (OmegaConf subset)
# --------------------------------------------------------------------------------------------
def _resolver_eq(x, y):
    return str(x).lower() == str(y).lower()


def _resolver_contains(x, y):
    return str(x).lower() in str(y).lower()


def _resolver_if(pred, a, b):
    return a if pred else b


def _resolver_resolve_default(default, arg):
    return default if arg == "" else arg


RESOLVERS = {
    "eq": _resolver_eq, "contains": _resolver_contains, "if": _resolver_if,
    "resolve_default": _resolver_resolve_default, "eval": lambda s: eval(s),  # noqa: S307 (reference does the same)
}


class _Loader(yaml.SafeLoader):
    """SafeLoader that reads ``2e-2`` / ``3e-4`` as floats like OmegaConf does (YAML 1.1, which
    PyYAML implements, demands a dot in the mantissa; the reference's YAMLs rely on OmegaConf)."""


_Loader.add_implicit_resolver(
    "tag:yaml.org,2002:float",
    re.compile(r"""^(?:[-+]?(?:[0-9][0-9_]*)\.[0-9_]*(?:[eE][-+]?[0-9]+)?
                   |[-+]?(?:[0-9][0-9_]*)(?:[eE][-+]?[0-9]+)
                   |\.[0-9_]+(?:[eE][-+][0-9]+)?
                   |[-+]?\.(?:inf|Inf|INF)|\.(?:nan|NaN|NAN))$""", re.X),
    list("-+0123456789."))


def _yaml_load(stream):
    return yaml.load(stream, Loader=_Loader)  # noqa: S506 - subclass of SafeLoader


def _primitive(text):
    t = text.strip()
    if t == "":
        return ""
    try:
        v = _yaml_load(t)
    except yaml.YAMLError:
        return t
    return t if isinstance(v, (dict, list)) else v


_ROOT = object()   # sentinel: "start at the root" (None is a legal node value, e.g. ``rnn=null``)


class _Resolver:
    def __init__(self, root):
        self.root = root

    def get(self, path):
        node = self.root
        for k in path:
            node = node[int(k)] if isinstance(node, list) else node[k]
        return node

    def resolve_node(self, path):
        v = self.get(path)
        if isinstance(v, str) and "${" in v:
            return self.resolve_str(v, path[:-1])
        return v

    def resolve_str(self, s, parent):
        parts, i, only = [], 0, None
        while i < len(s):
            j = s.find("${", i)
            if j < 0:
                parts.append(s[i:])
                break
            if j > i:
                parts.append(s[i:j])
            end = self._match(s, j)
            val = self.resolve_interp(s[j + 2:end], parent)
            parts.append(val)
            only = val
            i = end + 1
        if len(parts) == 1 and only is not None and not isinstance(parts[0], str):
            return parts[0]
        if len(parts) == 1:
            return parts[0]
        return "".join(str(p) for p in parts)

    @staticmethod
    def _match(s, start):
        depth, i, quote = 0, start, None
        while i < len(s):
            ch = s[i]
            if quote:
                if ch == quote:
                    quote = None
            elif ch in "'\"":
                quote = ch
            elif s.startswith("${", i):
                depth += 1
                i += 1
            elif ch == "}":
                depth -= 1
                if depth == 0:
                    return i
            i += 1
        raise ValueError(f"unbalanced interpolation in {s!r}")

    def _split_args(self, s):
        args, depth, quote, cur = [], 0, None, []
        i = 0
        while i < len(s):
            ch = s[i]
            if quote:
                cur.append(ch)
                if ch == quote:
                    quote = None
            elif ch in "'\"":
                quote = ch
                cur.append(ch)
            elif s.startswith("${", i):
                depth += 1
                cur.append("${")
                i += 1
            elif ch == "}":
                depth -= 1
                cur.append(ch)
            elif ch == "," and depth == 0:
                args.append("".join(cur))
                cur = []
            else:
                cur.append(ch)
            i += 1
        args.append("".join(cur))
        return args

    def _arg(self, text, parent):
        t = text.strip()
        if len(t) >= 2 and t[0] in "'\"" and t[-1] == t[0]:
            inner = t[1:-1]
            return self.resolve_str(inner, parent) if "${" in inner else inner
        if "${" in t:
            return self.resolve_str(t, parent)
        return _primitive(t)

    def resolve_interp(self, body, parent):
        # resolver call?  name:args  (node paths never contain ':')
        colon = body.find(":")
        head = body[:colon] if colon >= 0 else ""
        if colon >= 0 and head.replace("_", "").isalnum() and head in RESOLVERS:
            args = [self._arg(a, parent) for a in self._split_args(body[colon + 1:])]
            return RESOLVERS[head](*args)
        ref = body.strip()
        if ref.startswith("."):
            ndots = len(ref) - len(ref.lstrip("."))
            base = list(parent)
            for _ in range(ndots - 1):
                base = base[:-1]
            keys = [k for k in ref.lstrip(".").split(".") if k]
            return self.resolve_node(base + keys)
        return self.resolve_node(ref.split("."))

    def resolve_all(self, node=_ROOT, path=()):
        node = self.root if node is _ROOT else node
        if isinstance(node, dict):
            return {k: self.resolve_all(v, path + (k,)) for k, v in node.items()}
        if isinstance(node, list):
            return [self.resolve_all(v, path + (str(i),)) for i, v in enumerate(node)]
        if isinstance(node, str) and "${" in node:
            return self.resolve_str(node, list(path[:-1]))
        return node


def _set_path(root, dotted, value, create=True):
    keys = dotted.split(".")
    node = root
    for k in keys[:-1]:
        if k not in node:
            if not create:
                raise KeyError(dotted)
            node[k] = {}
        node = node[k]
    node[keys[-1]] = value


def compose(overrides=None, cfg_dir=None, task="Vine5LinkMovingBase", train=None):
    """Hydra-like composition: root + task + train, CLI-style ``a.b=c`` overrides, then resolve.

    ``cfg_dir``: optional path to a reference-style ``cfg/`` directory (config.yaml, task/*.yaml,
    train/*.yaml) to load instead of the built-in defaults.
    Returns a plain nested dict; ``cfg["task"]`` is what the env constructor takes.
    """
    overrides = list(overrides or [])
    for o in overrides:
        if o.startswith("task=") and "." not in o.split("=", 1)[0]:
            task = o.split("=", 1)[1]
        if o.startswith("train=") and "." not in o.split("=", 1)[0]:
            train = o.split("=", 1)[1]
    if cfg_dir is not None:
        with open(os.path.join(cfg_dir, "config.yaml")) as f:
            root = _yaml_load(f)
        root.pop("defaults", None)
        root.pop("hydra", None)
        with open(os.path.join(cfg_dir, "task", task + ".yaml")) as f:
            root["task"] = _yaml_load(f)
        tname = train or (task + "PPO")
        tpath = os.path.join(cfg_dir, "train", tname + ".yaml")
        if os.path.exists(tpath):
            with open(tpath) as f:
                root["train"] = _yaml_load(f)
    else:
        if task != "Vine5LinkMovingBase":
            raise ValueError(f"built-in defaults exist only for Vine5LinkMovingBase, not {task!r}")
        root = copy.deepcopy(ROOT_DEFAULTS)
        root["task"] = copy.deepcopy(TASK_DEFAULTS)
        root["train"] = copy.deepcopy(TRAIN_DEFAULTS)
    for o in overrides:
        key, _, val = o.partition("=")
        key = key.lstrip("+")
        if key in ("task", "train"):
            continue
        _set_path(root, key, _primitive(val))
    return _Resolver(root).resolve_all()


def task_config(overrides=None, **kw):
    """The plain dict the env constructor takes (``cfg["task"]`` of compose())."""
    return compose(overrides, **kw)["task"]


def fstr_task_config(extra_overrides=None, **kw):
    """BASELINE configs[1]: the README.md:63 free-space target reaching (FSTR) command line."""
    return task_config(FSTR_OVERRIDES + list(extra_overrides or []), **kw)


# --------------------------------------------------------------------------------------------
# plain dict -> VineConfig
# --------------------------------------------------------------------------------------------
def num_observations(observation_type):
    """numObservations from OBSERVATION_TYPE (Vine5LinkMovingBase.py:152-171)."""
    return abi.NUM_OBSERVATIONS[abi.OBSERVATION_TYPES[observation_type]]


def task_cfg_to_vine_config(cfg):
    """Map cfg["env"|"sim"|"task"] (reference key names) onto the C struct.

    Extension keys (all optional): env.TORQUE_LAW_INTEGRATION ("implicit"|"zoh"),
    env.EMULATE_STALE_BODY_STATE_ON_RESET, env.ARMATURE, env.DOF_LOWER/UPPER_*,
    sim.vine_contact.{stiffness,damping}.
    """
    env, sim = cfg["env"], cfg["sim"]
    task = cfg.get("task", {})
    rp = task.get("randomization_parameters", {})
    c = abi.VineConfig()
    c.struct_size = C.sizeof(abi.VineConfig)
    c.substeps = int(sim.get("substeps", 2))
    c.dt = float(sim["dt"])
    c.gravity_z = float(sim.get("gravity", [0.0, 0.0, -9.81])[2])
    c.control_freq_inv = int(env.get("controlFrequencyInv", 1))
    c.max_episode_length = int(env["maxEpisodeLength"])
    c.clip_observations = float(env.get("clipObservations", float("inf")))
    c.clip_actions = float(env.get("clipActions", float("inf")))
    ot = env["OBSERVATION_TYPE"]
    if ot not in abi.OBSERVATION_TYPES:
        raise KeyError(ot)  # ObservationType[...] raises KeyError in the reference too (V5:152)
    c.observation_type = abi.OBSERVATION_TYPES[ot]
    c.scale_observations = int(bool(env["SCALE_OBSERVATIONS"]))
    c.create_shelf = int(bool(env["CREATE_SHELF"]))
    c.create_pipe = int(bool(env["CREATE_PIPE"]))
    c.use_smoothed_fpam = int(bool(env["USE_SMOOTHED_FPAM"]))
    c.force_u_fpam = int(bool(env["FORCE_U_FPAM"]))
    c.force_u_rail_velocity = int(bool(env["FORCE_U_RAIL_VELOCITY"]))
    c.action_delay = int(env["ACTION_DELAY"])
    c.smoothing_alpha_inflate = float(env["SMOOTHING_ALPHA_INFLATE"])
    c.smoothing_alpha_deflate = float(env["SMOOTHING_ALPHA_DEFLATE"])
    c.fpam_min = float(env["FPAM_MIN"])
    c.fpam_max = float(env["FPAM_MAX"])
    c.rail_velocity_scale = float(env["RAIL_VELOCITY_SCALE"])
    c.damping = float(env["DAMPING"])
    c.stiffness = float(env["STIFFNESS"])
    c.rail_soft_limit = float(env["RAIL_SOFT_LIMIT"])
    c.rail_p_gain = float(env["RAIL_P_GAIN"])
    c.rail_d_gain = float(env["RAIL_D_GAIN"])
    c.rail_acceleration = float(env["RAIL_ACCELERATION"])
    c.randomize_dof_init = int(bool(env["RANDOMIZE_DOF_INIT"]))
    c.randomize_targets = int(bool(env["RANDOMIZE_TARGETS"]))
    c.random_init_cart_min_y = float(env["RANDOM_INIT_CART_MIN_Y"])
    c.random_init_cart_max_y = float(env["RANDOM_INIT_CART_MAX_Y"])
    c.success_dist = float(env["SUCCESS_DIST"])
    c.min_target_depth_in_obstacle = float(env["MIN_TARGET_DEPTH_IN_OBSTACLE"])
    c.max_target_depth_in_obstacle = float(env["MAX_TARGET_DEPTH_IN_OBSTACLE"])
    c.min_target_y = float(env["MIN_TARGET_Y"])
    c.max_target_y = float(env["MAX_TARGET_Y"])
    c.min_target_z = float(env["MIN_TARGET_Z"])
    c.max_target_z = float(env["MAX_TARGET_Z"])
    for i, k in enumerate(abi.REWARD_WEIGHT_KEYS):
        c.reward_weights[i] = float(env[k])
    c.use_target_reached_reset = int(bool(env["USE_TARGET_REACHED_RESET"]))
    c.use_tip_limit_hit_reset = int(bool(env["USE_TIP_LIMIT_HIT_RESET"]))
    c.use_nonzero_contact_force_reset = int(bool(env["USE_NONZERO_CONTACT_FORCE_RESET"]))
    c.vine_randomize = int(bool(task.get("vine_randomize", False)))
    c.dynamics_scaling_min = float(rp.get("DYNAMICS_SCALING_MIN", 1.0))
    c.dynamics_scaling_max = float(rp.get("DYNAMICS_SCALING_MAX", 1.0))
    c.observation_noise_std = float(rp.get("OBSERVATION_NOISE_STD", 0.0))
    c.action_noise_std = float(rp.get("ACTION_NOISE_STD", 0.0))
    c.accel_target_scaling_min = float(rp.get("ACCEL_TARGET_SCALING_MIN", 1.0))
    c.accel_target_scaling_max = float(rp.get("ACCEL_TARGET_SCALING_MAX", 1.0))
    c.torque_law_integration = abi.TORQUE_LAW_INTEGRATION[
        str(env.get("TORQUE_LAW_INTEGRATION", "implicit")).lower()]
    c.emulate_stale_body_state = int(bool(env.get("EMULATE_STALE_BODY_STATE_ON_RESET", True)))
    c.armature = float(env.get("ARMATURE", 0.0))
    big = 3.4e38  # what Isaac Gym reports for limit-less URDF joints (V5:568 docstring)
    c.revolute_lower = float(env.get("DOF_LOWER_REVOLUTE", -big))
    c.revolute_upper = float(env.get("DOF_UPPER_REVOLUTE", big))
    c.prismatic_lower = float(env.get("DOF_LOWER_PRISMATIC", -big))
    c.prismatic_upper = float(env.get("DOF_UPPER_PRISMATIC", big))
    vc = sim.get("vine_contact", {})
    c.contact_stiffness = float(vc.get("stiffness", 2000.0))
    c.contact_damping = float(vc.get("damping", 2.0))
    c.contact_rest_offset = float(sim.get("physx", {}).get("rest_offset", 0.001))
    # launch tuning of the library (no counterpart in the reference; results do not depend on it)
    c.contact_cull_slack = float(vc.get("cull_slack", 0.01))
    b = vc.get("binning", 1)                    # 0 = one launch in identity order, 1 = routed from 4096 envs, 2 = always routed
    c.contact_binning = int(b) if not isinstance(b, bool) else int(b)
    return c
