"""Multi-GPU check of gradient-norm clipping in the kernel update (truncate_grads=True; run under torchrun, one rank per GPU):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 tools/grad_clip_multi_check.py
For both networks and both gradient all-reduces (p2p: vine_grad_clip consumes the peer-memory channels; nccl: it runs after
the all-reduce) PPO trains a few iterations with a grad_norm that clips, then reports whether the parameters and the clipping
coefficient (state slot 9) are bit-identical on all ranks, whether a peer-memory wait timed out, and the loss statistics.
With p2p it also times the update graph with clipping off and on (alternating, CUDA events, max over ranks).
Prints one JSON line on rank 0."""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vine_robot_isaacgymenvs_b200 as vine  # noqa: E402
from vine_robot_isaacgymenvs_b200 import abi, config as vcfg, distributed as vd  # noqa: E402
from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent  # noqa: E402

GRAD_NORM = 0.01


def make_agent(extra, mode, rank, dev, clip, n=4096):
    over = [f"train.params.config.truncate_grads={clip}", f"train.params.config.grad_norm={GRAD_NORM}"]
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True", f"sim_device={dev}", f"rl_device={dev}"] + extra + over)
    env = vine.make(cfg=cfg, global_env_offset=rank * n)
    return PPOAgent(env, cfg["train"], device=dev, seed=42 + rank, use_graphs=True, grad_allreduce=mode)


def max_over_ranks(x, dev):
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def identical_across_ranks(x, world):
    gathered = [torch.empty_like(x) for _ in range(world)]
    dist.all_gather(gathered, x)
    return all(torch.equal(gathered[0].view(torch.uint8), g.view(torch.uint8)) for g in gathered)


def time_update(agent, dev, iters=20):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        agent._g_update.replay()
    e1.record()
    torch.cuda.synchronize()
    return max_over_ranks(e0.elapsed_time(e1) / iters, dev)


def main():
    rank, world, local = vd.rank_world()
    dev = f"cuda:{local}"
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=torch.device(dev))
    out = {"world": world, "gpu": torch.cuda.get_device_name(dev), "grad_norm": GRAD_NORM}
    for name, extra in (("mlp", ["train.params.network.rnn=null"]), ("lstm", [])):
        res = {}
        for mode in ("p2p", "nccl"):
            agent = make_agent(extra, mode, rank, dev, True)
            for _ in range(6):
                agent.train_epoch()
            torch.cuda.synchronize()
            flat = torch.cat([q.detach().reshape(-1) for q in agent.model.parameters()])
            coef = agent.ppo_state[abi.PPO_STATE_CLIP_COEF:abi.PPO_STATE_CLIP_COEF + 1].clone()
            st = agent.pop_stats()
            r = {"params_bit_identical_across_ranks": identical_across_ranks(flat, world),
                 "coef_bit_identical_across_ranks": identical_across_ranks(coef, world),
                 "finite": bool(torch.isfinite(flat).all()), "coef": float(coef),
                 "grad_norm_seen": float(agent.ppo_state[abi.PPO_STATE_GRAD_NORM]),
                 "kl": st["kl"], "a_loss": st["a_loss"], "c_loss": st["c_loss"]}
            if mode == "p2p":
                chans = [c for c in (agent._p2p_mlp, agent._p2p_lstm) if c is not None]
                stats = [c.status() for c in chans]
                r.update({"exchanges": min(s[0] for s in stats), "timed_out": any(s[1] for s in stats)})
                # update time, clipping off vs on, alternating (same shapes, same world)
                plain = make_agent(extra, mode, rank, dev, False)
                for _ in range(4):
                    plain.train_epoch()
                torch.cuda.synchronize()
                off, on = [], []
                for _ in range(3):
                    off.append(time_update(plain, dev))
                    on.append(time_update(agent, dev))
                r.update({"update_ms_clip_off": min(off), "update_ms_clip_on": min(on)})
                del plain
            res[mode] = r
            del agent
            torch.cuda.empty_cache()
        out[name] = res
    if rank == 0:
        print(json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
