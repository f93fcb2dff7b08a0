"""Time one PPO iteration of the reference network (MLP -> LSTM 256 -> LayerNorm) at FSTR, N envs, CUDA-graph replay:
python tools/ppo_time.py [N] [--mlp] [--no-pdl] [--no-arena] [--pad K] [--truncate-grads [--grad-norm X]]
Prints ms per iteration / rollout / update (CUDA events, best of 3 x 20).  --truncate-grads also builds a second agent with
gradient-norm clipping (truncate_grads=True, grad_norm X, default 1.0) and times the two update graphs alternately."""
import sys

import torch

sys.path.insert(0, ".")
import vine_robot_isaacgymenvs_b200 as vine  # noqa: E402
from vine_robot_isaacgymenvs_b200 import config as vcfg  # noqa: E402
from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent  # noqa: E402

args = [a for a in sys.argv[1:]]
n = int(args[0]) if args and args[0].isdigit() else 4096
extra = ["train.params.network.rnn=null"] if "--mlp" in args else []
if "--no-pdl" in args:
    PPOAgent.PDL_MAX_ENVS = 0
if "--no-arena" in args:
    from vine_robot_isaacgymenvs_b200.ppo.lstm_native import NativeLstmPath
    NativeLstmPath.ARENA = False
if "--pad" in args:   # perturb the caching allocator's placement of the agent's buffers (placement-sensitivity experiment)
    k = int(args[args.index("--pad") + 1])
    _g = torch.Generator().manual_seed(k)
    _pads = [torch.empty(int(torch.randint(1, 64, (1,), generator=_g)) * 524288 + 512 * k, dtype=torch.uint8, device="cuda") for _ in range(k)]
    del _pads[::2]
cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True"] + extra)
env = vine.make(cfg=cfg)
agent = PPOAgent(env, cfg["train"], device="cuda:0", seed=42, use_graphs=True, use_fused_update=True)
for _ in range(5):
    agent.train_epoch()
torch.cuda.synchronize()
clip_agent = None
if "--truncate-grads" in args:
    gn = float(args[args.index("--grad-norm") + 1]) if "--grad-norm" in args else 1.0
    ccfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True", "train.params.config.truncate_grads=True",
                                               f"train.params.config.grad_norm={gn}"] + extra)
    clip_agent = PPOAgent(vine.make(cfg=ccfg), ccfg["train"], device="cuda:0", seed=42, use_graphs=True, use_fused_update=True)
    for _ in range(5):
        clip_agent.train_epoch()
    torch.cuda.synchronize()


def best(fn, reps=3, iters=20):
    b = 1e9
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        b = min(b, e0.elapsed_time(e1) / iters)
    return b


it = best(agent.train_epoch)
ro = best(agent.play_steps)
up = best(agent._g_update.replay if agent._g_update is not None else agent._update_any)
st = agent.pop_stats()
print(f"n={n} {' '.join(args[1:])}: iteration {it:.3f} ms  rollout {ro:.3f}  update {up:.3f}  frames/s {n * agent.T / it * 1e3:.4g}  "
      f"kl {st['kl']:.4g} a_loss {st['a_loss']:.4g} c_loss {st['c_loss']:.4g}", flush=True)
if clip_agent is not None:   # update graph without / with clipping, alternating; the card and its power limit of this run
    import subprocess
    off, on = [], []
    for _ in range(5):
        off.append(best(agent._g_update.replay))
        on.append(best(clip_agent._g_update.replay))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    coef = float(clip_agent.ppo_state[9])
    print(f"n={n} {'mlp' if extra else 'reference network'}: update {min(off):.3f} ms without clipping, {min(on):.3f} ms with "
          f"(+{(min(on) - min(off)) * 1e3:.1f} us per update, {(min(on) - min(off)) * 1e3 / (agent.mini_epochs * (agent.n // agent.mb_envs)):.2f} "
          f"us per minibatch; spread off {min(off):.3f}-{max(off):.3f}, on {min(on):.3f}-{max(on):.3f}); last coefficient {coef:.4g}; "
          f"{q.stdout.strip() or torch.cuda.get_device_name(0)}", flush=True)
