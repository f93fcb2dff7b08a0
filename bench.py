#!/usr/bin/env python
"""bench.py — env-steps/s of the Vine5LinkMovingBase hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on host cores
    python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/<name>.npy

Workload (config.workload): the FSTR command line of the reference's README.md:63 (BASELINE
configs[1] knobs) driven with synthetic U(-1,1)^2 actions, env-step only, ``--num-envs`` envs per
GPU (default 1,048,576: the top of BASELINE configs[4]'s sweep; state + I/O ~ 400 MB > the 126 MB
L2, so no L2 flush is needed between steps).  A "step" = one control step of every env = ONE
fused kernel launch.  Weak scaling: per-GPU env count fixed, envs sharded by contiguous global
env id, no collective in the step.

Printed JSON (one line, rank 0): the contract keys + ``roofline`` (HBM, SURVEY §8d bytes),
``roofline_fp32`` (the binding resource: FP32 FMA, against an FFMA peak measured in the same run),
``cpu_baseline``, ``e2e`` (through the public env class with pinned HOST buffers, H2D + D2H
every step), ``clocks``, ``gpu_launches``, ``sweep`` (smaller env counts, same kernel).
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

OUT = sys.stdout
METRIC = "env-steps/s (whole box, device-timed)"
WORKLOAD = "FSTR (README.md:63 / BASELINE configs[1] knobs) env step, U(-1,1) actions, env-step only"
UNIT = "env-steps/s"
# Algorithmic work per env-step of the FSTR workload (derivations: DESIGN.md §6)
HBM_BYTES_PER_ENV_STEP = 273.0      # SURVEY.md §8(d): O=18, ACTION_DELAY=1
FLOPS_PER_ENV_STEP = 17.61e3        # fallback; the shipped kernels' counts are read from profiles/flops_per_env_step.json
DESYNC_STEPS = 130                  # untimed steps before every timed region: episodes (<= 100 steps in FSTR) are out of phase,
                                    # so the in-kernel reset branch, and with obstacles contacts, are inside the timed steps


def profile_json(name, default=None):
    """A small measured record committed under profiles/ (ncu-derived counts, build-container CPU baselines)."""
    path = os.path.join(REPO, "profiles", name)
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return default


def flops_per_env_step(key):
    """Algorithmic FP32 work of one env-step of a workload = 2 x FFMA + FMUL + FADD thread-instructions of all kernels of a
    control step / envs, counted by ncu on the shipped kernels (tools/ncu_flops.sh -> profiles/flops_per_env_step.json)."""
    rec = profile_json("flops_per_env_step.json", {})
    return float(rec.get(key, {}).get("flops_per_env_step", FLOPS_PER_ENV_STEP if key == "fstr_1048576" else 0.0)) or None


def fstr_cfg(num_envs, extra=()):
    from vine_robot_isaacgymenvs_b200 import config as vcfg
    return vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={num_envs}", "headless=True"] + list(extra))


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.stop_flag, self.ok = [], False, True
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), sm, reasons))
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self, t0, t1):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml_unavailable"]}
        nv = self.nv
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        clocks = sorted(s[1] for s in inside)
        bits = 0
        for s in inside:
            bits |= s[2]
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        return {"sm_mhz": clocks[len(clocks) // 2], "sm_max_mhz": mx, "samples": len(inside),
                "reasons": [k for k, b in names.items() if bits & b]}


def cpu_oracle_rate(num_envs, budget_s, nthreads=0, min_steps=2, max_steps=64, fixed_steps=None, warmup=1):
    """env-steps/s of the CPU oracle (f32 dynamics, OpenMP over envs) on a bounded FSTR sample."""
    import numpy as np
    from oracle import oracle as O
    from vine_robot_isaacgymenvs_b200 import config as vcfg
    vc = vcfg.task_cfg_to_vine_config(fstr_cfg(num_envs)["task"])
    # explicit thread count: torchrun exports OMP_NUM_THREADS=1, which would silently serialise the CPU arm
    env = O.OracleEnv(vc, num_envs, seed=42, use_f64=False, nthreads=nthreads or host_threads())
    rng = np.random.default_rng(42)
    acts = rng.uniform(-1, 1, (4, num_envs, 2)).astype(np.float32)
    for i in range(max(warmup, 1)):
        env.step(acts[i % 4])
    t0 = time.perf_counter()
    env.step(acts[0])
    one = time.perf_counter() - t0
    steps = fixed_steps if fixed_steps is not None else int(min(max_steps, max(min_steps, budget_s / max(one, 1e-6))))
    t0 = time.perf_counter()
    for i in range(steps):
        env.step(acts[i % 4])
    dt = time.perf_counter() - t0
    return num_envs * steps / dt, steps, dt


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, rank):
    """The reference's CPU implementation of the path, timed on the box's host cores.  The reference's
    own arithmetic for this path is closed PhysX + torch (not installable here), so this arm runs the
    oracle port (kind "port"), which is pinned bit-exactly to the reference's step logic."""
    if rank != 0:
        return
    cores = host_threads()
    # size the per-step sample so the whole run ends within ~2 minutes
    probe_n = 4096
    rate, _, _ = cpu_oracle_rate(probe_n, 0.0, fixed_steps=2)
    total_steps = args.steps + args.warmup
    n = int(max(256, min(args.num_envs, rate * 100.0 / max(total_steps, 1))))
    n = 1 << (n.bit_length() - 1)
    value, steps, dt = cpu_oracle_rate(n, 0.0, fixed_steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_envs_per_step": n,
                   "note": "same workload as the CUDA arm; each step is a bounded sample of it on the host cores"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{n} envs x {steps} control steps, oracle f32 dynamics, OpenMP x{cores}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=OUT, flush=True)


def timed_steps(env, lib, pool, steps, use_graph):
    """Device time (ms) of `steps` control steps, rotating through the action pool."""
    import torch
    dev = env.device
    s = torch.cuda.Stream(dev)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def launch(stream_ptr):
        for i in range(steps):
            env._bind(pool[i % len(pool)])
            env._check(lib.vine_step(env._h, stream_ptr))

    torch.cuda.synchronize(dev)
    if use_graph:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(s):
            with torch.cuda.graph(g, stream=s):
                launch(C.c_void_p(s.cuda_stream))
        torch.cuda.synchronize(dev)
        return g, s, start, end
    return launch, s, start, end


def dump_outputs(env, out_dir, max_bytes=64e6):
    """Write what a caller of ``env.step()`` receives after the last timed step -- clamped observations, rewards, resets
    and time-outs -- as float32 ``<out_dir>/<name>.npy``, one row per env, with the env ids of the rows in ``env_ids.npy``
    (float64).  Above ``max_bytes`` in all, the rows are a fixed seeded sample of the envs, so that two builds run with
    the same arguments can be compared output for output."""
    import numpy as np
    import torch
    arrays = {"obs": env._obs_clamped, "rew": env.rew_buf, "reset": env.reset_buf, "time_outs": env.timeout_buf}
    n = env.num_envs
    row_bytes = 4 * sum(a[0].numel() for a in arrays.values()) + 8
    ids = np.arange(n)
    if n * row_bytes > max_bytes - 4096:              # 4096: room for the .npy headers
        ids = np.sort(np.random.default_rng(0).choice(n, int((max_bytes - 4096) // row_bytes), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    rows = torch.from_numpy(ids).to(env.device)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[rows].float().cpu().numpy())
    np.save(os.path.join(out_dir, "env_ids.npy"), (ids + env._global_env_offset).astype(np.float64))


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    import vine_robot_isaacgymenvs_b200 as vine
    from vine_robot_isaacgymenvs_b200 import abi

    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    n = args.num_envs
    lib = abi.load_library()

    def make_env(num_envs, preset=None):
        from vine_robot_isaacgymenvs_b200 import config as vcfg
        extra = [f"sim_device={dev}", f"rl_device={dev}"]
        cfg = fstr_cfg(num_envs, extra) if preset is None else vcfg.compose(preset + [f"num_envs={num_envs}", "headless=True"] + extra)
        return vine.make(cfg=cfg, global_env_offset=rank * num_envs), cfg

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def measure(num_envs, steps, warmup, sampler=None, preset=None):
        env, cfg = make_env(num_envs, preset)
        gen = torch.Generator(device=dev).manual_seed(42 + rank)
        pool = [torch.rand(num_envs, 2, device=dev, generator=gen) * 2 - 1 for _ in range(4)]
        for i in range(max(warmup, 3) + DESYNC_STEPS):
            env._bind(pool[i % 4])
            env._check(lib.vine_step(env._h, env._stream()))
        runner, s, start, end = timed_steps(env, lib, pool, steps, not args.no_graph)
        barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(s):
            start.record()
            if args.no_graph:
                runner(C.c_void_p(s.cuda_stream))
            else:
                runner.replay()
            end.record()
        torch.cuda.synchronize(dev)
        barrier()
        t1 = time.perf_counter()
        ms = max_over_ranks(start.elapsed_time(end))
        assert torch.isfinite(env.obs_buf).all() and torch.isfinite(env.rew_buf).all()
        env._bind()
        return env, cfg, ms, (t0, t1)

    sampler = ClockSampler(local_rank)
    sampler.start()
    env, cfg, ms, window = measure(n, args.steps, args.warmup)
    clocks = sampler.summary(*window)
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs)           # before the e2e steps below advance the same env
    value = n * world * args.steps / (ms * 1e-3)
    ms_per_step = ms / args.steps

    # ---- e2e: public env.step() with pinned host buffers, H2D + D2H inside the timed region ----
    O = env.num_obs
    e2e_steps = max(3, min(args.steps, args.e2e_steps))
    a_host = [torch.empty(n, 2).uniform_(-1, 1).pin_memory() for _ in range(4)]
    obs_h = torch.empty(n, O).pin_memory()
    rew_h = torch.empty(n).pin_memory()
    rst_h = torch.empty(n, dtype=torch.long).pin_memory()
    to_h = torch.empty(n, dtype=torch.bool).pin_memory()
    stream = torch.cuda.current_stream(dev)

    def e2e_step(i):
        od, rew, rst, extras = env.step(a_host[i % 4])          # H2D of the actions happens inside
        obs_h.copy_(od["obs"], non_blocking=True)
        rew_h.copy_(rew, non_blocking=True)
        rst_h.copy_(rst, non_blocking=True)
        to_h.copy_(extras["time_outs"], non_blocking=True)
        stream.synchronize()                                   # a policy needs the result before acting

    def e2e_step_pipelined(i):
        # same contract, one call: chunked H2D -> step -> D2H on rotating streams (env.step_host)
        env.step_host(a_host[i % 4], obs_h, rew_h, rst_h, to_h, chunks=args.e2e_chunks)

    def time_e2e(fn):
        for i in range(3):
            fn(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            fn(i)
        barrier()
        return n * world * e2e_steps / max_over_ranks(time.perf_counter() - t0)

    e2e_simple = time_e2e(e2e_step)
    e2e_value = time_e2e(e2e_step_pipelined)
    sampler.stop_flag = True

    # ---- PPO frames/s (second half of BASELINE.json's metric): BASELINE configs[1] literally ----
    # FSTR, 4096 envs per GPU, horizon 16, minibatch 32768, 4 mini-epochs; one iteration = rollout
    # (16 x {policy, fused env step}) + GAE + update; frames = T * N * ranks per iteration.
    def measure_ppo(num_envs, iters, warmup, extra, use_graphs=True, fused_update=True, preset=None):
        from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent
        from vine_robot_isaacgymenvs_b200 import config as vcfg
        devs = [f"sim_device={dev}", f"rl_device={dev}"]
        pcfg = (fstr_cfg(num_envs, devs + list(extra)) if preset is None else
                vcfg.compose(preset + [f"num_envs={num_envs}", "headless=True"] + devs + list(extra)))
        penv = vine.make(cfg=pcfg, global_env_offset=rank * num_envs)
        exchange = "none" if world == 1 else "p2p"
        try:
            agent = PPOAgent(penv, pcfg["train"], device=dev, seed=42 + rank, use_graphs=use_graphs, use_fused_update=fused_update)
        except RuntimeError as err:   # no CUDA IPC / peer access on this box: every rank gets the same error (P2PChannel agrees first)
            if "vine_p2p" not in str(err):
                raise
            exchange = "nccl (peer-memory channel unavailable: %s)" % str(err)[:120]
            agent = PPOAgent(penv, pcfg["train"], device=dev, seed=42 + rank, use_graphs=use_graphs, use_fused_update=fused_update,
                             grad_allreduce="nccl")
        if world > 1 and not agent.fused_update:
            exchange = "nccl"
        for _ in range(max(warmup, 3)):
            agent.train_epoch()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            agent.train_epoch()
        e1.record()
        barrier()
        ms_it = max_over_ranks(e0.elapsed_time(e1)) / iters
        # split of one iteration, timed separately (same graphs / launches): rollout+GAE vs update
        parts = {}
        for name, fn in (("rollout_ms", agent.play_steps), ("update_ms", (agent._g_update.replay if agent._g_update is not None
                                                                          else agent._update_any))):
            barrier()
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            barrier()
            parts[name] = max_over_ranks(e0.elapsed_time(e1)) / iters
        stats = agent.pop_stats()
        assert all(x == x for x in (stats["a_loss"], stats["c_loss"], stats["kl"])), stats
        upd_tf = (6 * (392448 if agent.has_rnn else 45760) * agent.T * num_envs * agent.mini_epochs / (parts["update_ms"] * 1e-3) / 1e12)
        bf16_peak = measured_peaks()[0].get("bf16_tflops_sustained", 1395.8)
        return {"value": agent.T * num_envs * world / (ms_it * 1e-3), "unit": "frames/s", "ms_per_iteration": ms_it,
                "num_envs_per_gpu": num_envs, "horizon": agent.T, "minibatch": agent.minibatch,
                "mini_epochs": agent.mini_epochs, "iterations": iters, **parts,
                # algorithmic tensor work of the update: 3 x forward MACs x 2 per sample per mini-epoch (MLP: 18*256+256*128+128*64+64*3 = 45,760 MAC)
                # algorithmic tensor work of the update per sample and mini-epoch = 3 GEMM passes (forward, backward data,
                # weight gradients) x 2 FLOP x MACs; MLP: 18*256+256*128+128*64+64*3 = 45,760 MAC; reference network:
                # MLP body 45,568 + LSTM (64+18)*1024 + 256*1024 = 346,112 + heads 768 = 392,448 MAC
                "update_tflops": upd_tf,
                "update_roofline": {"bound": "tensor", "achieved": upd_tf, "peak": bf16_peak, "unit": "TFLOP/s", "frac": upd_tf / bf16_peak,
                                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernels timed inside a long step)"},
                "trained_policy_band": "parity unpinned: no reference checkpoint or learning curve exists in this image (README.md:63-66 "
                                       "links to wandb); this trainer's own FSTR success rate (0.82-0.89 at 400 iterations) shows "
                                       "learnability, not parity with the reference policy",
                "network": "mlp[256,128,64]+lstm256+ln" if agent.has_rnn else "mlp[256,128,64]",
                "cuda_graphs": agent.use_graphs,
                "update": ("vine_lstm_* + vine_ppo_minibatch (tcgen05, hand-written; ppo/lstm_native.py)" if agent.native_lstm else
                           "vine_ppo_minibatch/reduce/adam (tcgen05, hand-written)" if agent.fused_update
                           else "torch autograd + cuBLAS/cuDNN + torch Adam"),
                "policy_forward": ("vine_policy_act + vine_lstm_step/head (tcgen05)" if agent.native_lstm else
                                   "vine_policy_act (tcgen05)" if agent.fused else "torch"),
                "collectives": "none" if world == 1 else (
                    "gradients + loss statistics per minibatch and running-statistics moments per iteration over NVLink peer memory "
                    "inside the reduce / Adam kernels (csrc/vine_p2p.cuh); NCCL only for the start-up broadcast" if exchange == "p2p"
                    else "NCCL all-reduce: grads+KL per minibatch, running stats per iteration [%s]" % exchange)}

    # ---- HBM-bound PPO helper kernels (SURVEY §8d: GAE 24 B per (t, env)), timed alone against the measured copy bandwidth ----
    def measure_gae(num_envs, T=16, reps=200):
        peaks_hbm = measured_peaks()[0]["hbm_gbs"]
        f = lambda *sh: torch.rand(*sh, device=dev)  # noqa: E731
        r, v, d, lv, ld = f(T, num_envs), f(T, num_envs), (f(T, num_envs) < 0.05).float(), f(num_envs), f(num_envs)
        adv, ret = torch.empty(T, num_envs, device=dev), torch.empty(T, num_envs, device=dev)
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        call = lambda: lib.vine_gae(p(r), p(v), p(d), p(lv), p(ld), T, num_envs, 0.99, 0.95, p(adv), p(ret), st)  # noqa: E731
        for _ in range(5):
            assert call() == 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        torch.cuda.synchronize(dev)
        us = e0.elapsed_time(e1) / reps * 1e3
        gbs = 24.0 * T * num_envs / (us * 1e-6) / 1e9
        return {"kernel": "vine_gae_kernel", "num_envs": num_envs, "horizon": T, "us": us,
                "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks_hbm, "unit": "GB/s", "frac": gbs / peaks_hbm,
                             "note": "24 algorithmic B per (t, env); 25 MB at 65,536 envs fits the 126 MB L2 when timed back to back"
                                     if num_envs * T * 24 < 126e6 else "24 algorithmic B per (t, env); larger than L2"}}

    ppo = None
    if not args.no_ppo:
        del env
        env = None
        torch.cuda.empty_cache()
        ppo = {"config": "BASELINE configs[1]: FSTR num_envs=4096 rollout+PPO",
               "hbm_kernels": [measure_gae(65536), measure_gae(1 << 20)],
               "reference_network": measure_ppo(4096, args.ppo_iters, 5, []),
               "reference_network_torch_update": measure_ppo(4096, max(3, args.ppo_iters // 2), 3, [], fused_update=False),
               "mlp_only": measure_ppo(4096, args.ppo_iters, 5, ["train.params.network.rnn=null"]),
               "mlp_only_torch_update": measure_ppo(4096, args.ppo_iters, 5, ["train.params.network.rnn=null"],
                                                    fused_update=False)}
        if not args.no_sweep:
            from vine_robot_isaacgymenvs_b200.config import SHELF_OVERRIDES as shelf_preset
            ppo["reference_network_65536_envs"] = measure_ppo(65536, max(3, args.ppo_iters // 4), 3,
                                                              ["train.params.config.minibatch_size=131072"])
            # BASELINE configs[2]: shelf + contact-force resets at its own env count (minibatch = the whole 16384 x 16 batch / 2)
            ppo["reference_network_configs2_shelf_16384_envs"] = measure_ppo(
                16384, max(3, args.ppo_iters // 2), 3, ["train.params.config.minibatch_size=131072"], preset=shelf_preset)
            ppo["mlp_only_65536_envs"] = measure_ppo(65536, max(3, args.ppo_iters // 4), 3,
                                                     ["train.params.network.rnn=null",
                                                      "train.params.config.minibatch_size=131072"])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the (only) kernel in the timed region: the binding resource is FP32 (SURVEY §8d) ----
    peaks, peaks_kind = measured_peaks()
    fp32_peak = None
    try:
        pk = C.CDLL(os.path.join(REPO, "vine_robot_isaacgymenvs_b200", "csrc", "libvine_benchpeak.so"))
        pk.vine_bench_ffma_tflops.restype = C.c_double
        fp32_peak = pk.vine_bench_ffma_tflops(5)
    except OSError:
        pass
    fp32_source = "FFMA microbenchmark (shared multiplier/addend operands) measured in this run; nominal 74.4"
    if not fp32_peak:
        fp32_peak, fp32_source = 74.4, "nominal 148 SM x 128 FMA x 2 x 1.965 GHz (microbenchmark library missing)"
    traffic = profile_json("traffic_bytes_per_env_step.json", {}).get("bytes_per_env_step")

    def fp32_roofline(key, num_envs, ms_step, kernel):
        f = flops_per_env_step(key)
        if not f:
            return None
        ach = f * num_envs / (ms_step * 1e-3) / 1e12
        return {"bound": "fp32_fma", "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach / fp32_peak,
                "traffic": None, "peak_source": fp32_source, "kernel": kernel, "flops_per_env_step": f,
                "flops_source": "ncu 2*ffma+fmul+fadd thread-instructions of every kernel of a control step / envs "
                                "(profiles/flops_per_env_step.json)"}

    roofline = fp32_roofline("fstr_1048576", n, ms_per_step, "vine_step_kernel<false>")
    roofline["traffic"] = traffic * n if traffic else None
    roofline["traffic_unit"] = "bytes per launch (dram read+write, ncu)"
    roofline["note"] = ("register-operand bandwidth, not issue slots, caps this instruction mix at ~0.68 of the FFMA peak: a stream of "
                        "FFMAs with three distinct register operands measures 50 TFLOP/s on B200 and the packed f32x2 variant of the "
                        "kernel (half the issue slots) runs at the same FMA-pipe occupancy (profiles/README.md, r02a)")
    hbm_achieved = HBM_BYTES_PER_ENV_STEP * n / (ms_per_step * 1e-3) / 1e9
    roofline_hbm = {"bound": "hbm", "achieved": hbm_achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": hbm_achieved / peaks["hbm_gbs"], "traffic": traffic * n if traffic else None, "peak_source": peaks_kind,
                    "kernel": "vine_step_kernel<false>", "note": "not the binding resource (273 algorithmic B per env-step, SURVEY §8d)"}

    # ---- smaller env counts, same kernel (BASELINE configs[1] literal size and the configs[4] sweep) ----
    sweep = []
    if world == 1 and not args.no_sweep:
        env = None
        torch.cuda.empty_cache()
        for m in (4096, 65536, 262144):
            if m >= n:
                continue
            _, _, ms_m, _ = measure(m, args.steps, args.warmup)
            sweep.append({"num_envs": m, "value": m * args.steps / (ms_m * 1e-3), "ms_per_step": ms_m / args.steps,
                          "l2_resident": True, "roofline": fp32_roofline("fstr_1048576", m, ms_m / args.steps, "vine_step_kernel<false>")})

        # the contact kernels (same fused launch, CONTACT=true template): BASELINE configs[2] and [3] at their env counts
        from vine_robot_isaacgymenvs_b200 import config as vcfg
        for label, preset, m in (("configs[2] shelf, contact-force resets", vcfg.SHELF_OVERRIDES, 16384),
                                 ("configs[3] pipe + full DR (per-GPU share of 65536)", vcfg.PIPE_DR_OVERRIDES, 8192),
                                 ("shelf", vcfg.SHELF_OVERRIDES, 1 << 20), ("pipe + full DR", vcfg.PIPE_DR_OVERRIDES, 1 << 20)):
            _, _, ms_m, _ = measure(m, args.steps, args.warmup, preset=preset)
            key = ("shelf_" if preset is vcfg.SHELF_OVERRIDES else "pipe_dr_") + str(m)
            sweep.append({"workload": label, "num_envs": m, "value": m * args.steps / (ms_m * 1e-3), "ms_per_step": ms_m / args.steps,
                          "roofline": fp32_roofline(key, m, ms_m / args.steps,
                                                    "routed step: vine_bin + vine_step_far + vine_step_kernel<true> (near, redo)")})

    # ---- CPU baseline (oracle port) on a bounded sample, rank 0, N=1 only ----
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores = host_threads()
        cn = 65536
        rate, steps, dt = cpu_oracle_rate(cn, budget_s=12.0, max_steps=512)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{cn} envs x {steps} control steps ({dt:.1f} s), oracle f32 dynamics, OpenMP x{cores}"}

    # BASELINE.md §4-2a: the reference's unmodified Python step (torch CPU) + port dynamics, configs[0]; needs /root/reference,
    # which exists only in the build container: live there, the committed build-container record elsewhere
    cpu_c1 = None
    if world == 1 and not args.no_cpu_baseline:
        if os.path.isdir("/root/reference"):
            sys.path.insert(0, os.path.join(REPO, "tools"))
            import cpu_baseline_c1
            cpu_c1 = cpu_baseline_c1.measure()
            cpu_c1["measured_on"] = "this run"
        else:
            cpu_c1 = profile_json("cpu_baseline_c1.json")

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "num_envs_per_gpu": n, "global_envs": n * world,
                   "obs": cfg["task"]["env"]["OBSERVATION_TYPE"], "substeps_per_step":
                       cfg["task"]["sim"]["substeps"] * cfg["task"]["env"]["controlFrequencyInv"],
                   "parallelism": f"env-sharded x{world}, no collective in the step",
                   "l2": "inputs larger than L2 (no flush)" if n * 400 > 126e6 else "L2-resident",
                   "untimed_steps_before_timing": max(args.warmup, 3) + DESYNC_STEPS,
                   "cuda_graph": not args.no_graph},
        "roofline": roofline, "roofline_hbm": roofline_hbm, "cpu_baseline": cpu, "cpu_baseline_c1": cpu_c1,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 2 * 4,
                "d2h_bytes_per_step": n * (O * 4 + 4 + 8 + 1), "steps": e2e_steps,
                "api": f"env.step_host(pinned host buffers, chunks={args.e2e_chunks}): H2D, step and D2H of different "
                       "env chunks overlap on separate streams; returns after all results are on the host",
                "unpipelined_value": e2e_simple,
                "note": "bounded by the HOST side (pinned-memory writes of 85 B/env of results), not by a kernel or one PCIe link: "
                        "8 ranks reach the same ~1.1e9 env-steps/s (~95 GB/s aggregate D2H) as 2 on these one-NUMA-node VMs; the "
                        "reference keeps the policy on the device, so this is the only case that pays it"},
        "clocks": clocks, "gpu_launches": args.steps, "sweep": sweep,
        # second half of BASELINE.json's metric: PPO frames/s at configs[1] with the reference's own network
        "ppo_frames_per_s": (ppo or {}).get("reference_network", {}).get("value"), "ppo": ppo,
    }
    print(json.dumps(line), file=OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def _quiet_stdout():
    """The contract is ONE JSON line on stdout: libraries that write to fd 1 (NCCL prints its version banner or its
    NCCL_DEBUG log there) are sent to stderr; the returned stream is the real stdout for the JSON line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    global OUT
    OUT = _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--num-envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--e2e-steps", type=int, default=30)
    ap.add_argument("--e2e-chunks", type=int, default=8)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ppo", action="store_true")
    ap.add_argument("--ppo-iters", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0's envs) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the CUDA arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
