"""Multi-GPU check of the linear learning-rate schedule with schedule_type standard in the kernel update (run under torchrun,
one rank per GPU):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29543 tools/lr_schedule_multi_check.py
For both networks and both gradient all-reduces (p2p, nccl) PPO trains a few iterations with lr_schedule linear, schedule_type
standard, then reports whether the parameters and the learning rate (state slot 0) are bit-identical on all ranks, the lr and
the closed form it should equal.  Prints one JSON line on rank 0."""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vine_robot_isaacgymenvs_b200 as vine  # noqa: E402
from vine_robot_isaacgymenvs_b200 import config as vcfg, distributed as vd  # noqa: E402
from vine_robot_isaacgymenvs_b200.ppo.ppo import LR_MIN, PPOAgent  # noqa: E402

MAX_EPOCHS, ITERS, LR0 = 8, 6, 3e-4


def make_agent(extra, mode, rank, dev, n=4096):
    over = ["train.params.config.lr_schedule=linear", "train.params.config.schedule_type=standard",
            f"train.params.config.max_epochs={MAX_EPOCHS}", f"train.params.config.learning_rate={LR0}"]
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True", f"sim_device={dev}", f"rl_device={dev}"] + extra + over)
    env = vine.make(cfg=cfg, global_env_offset=rank * n)
    return PPOAgent(env, cfg["train"], device=dev, seed=42 + rank, use_graphs=True, grad_allreduce=mode)


def identical_across_ranks(x, world):
    gathered = [torch.empty_like(x) for _ in range(world)]
    dist.all_gather(gathered, x)
    return all(torch.equal(gathered[0].view(torch.uint8), g.view(torch.uint8)) for g in gathered)


def main():
    rank, world, local = vd.rank_world()
    dev = f"cuda:{local}"
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=torch.device(dev))
    out = {"world": world, "gpu": torch.cuda.get_device_name(dev)}
    for name, extra in (("mlp", ["train.params.network.rnn=null"]), ("lstm", [])):
        res = {}
        for mode in ("p2p", "nccl"):
            agent = make_agent(extra, mode, rank, dev)
            while agent.epoch < ITERS:
                agent.train_epoch()
            torch.cuda.synchronize()
            flat = torch.cat([q.detach().reshape(-1) for q in agent.model.parameters()])
            lr = agent.ppo_state[0:1].clone()
            # the last Adam step of iteration e (4 mini-epochs) ran with f(e)
            e = agent.epoch
            res[mode] = {"params_bit_identical_across_ranks": identical_across_ranks(flat, world),
                         "lr_bit_identical_across_ranks": identical_across_ranks(lr, world),
                         "finite": bool(torch.isfinite(flat).all()), "lr": float(lr), "epoch": e,
                         "lr_expected": LR_MIN + (float(torch.tensor(LR0)) - LR_MIN) * max(0, MAX_EPOCHS - e) / MAX_EPOCHS}
            del agent
            torch.cuda.empty_cache()
        out[name] = res
    if rank == 0:
        print(json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
