"""Dense-contact states of the obstacle variants (test infrastructure, no GPU).

The f64 oracle evaluates every (link, rectangle) pair of every env with no culling, so it decides which random states touch
an obstacle.  ``select`` draws candidates the way ``test_gpu_parity.test_simulate_matches_f64_oracle`` does (chain bent
toward -y, the same efforts, u and dynamics-scaling draws; targets and object info from the config's ranges) and keeps
  * touched envs: the oracle's sim step with the obstacles differs from the same step without them (max |dqd| > 1e-3), or
    the lip force is > 0;
  * fillers: free-space envs, untouched and without candidate pairs;
and of both only the well-conditioned ones, whose sim step in the oracle's own f32 build agrees with f64 (|dq| < 1e-5,
|dqd| < 1e-3); a touched env must also stay within the tolerance the
kernel is held to in 64 f64 runs from q and qd perturbed by up to 32 ulps.

``pair_masks`` restates the kernel's cull (vine_device.cuh ``chain_obstacle_gap`` + ``cull_pairs``) in numpy at the start
state.  It only shows which load a layout puts on the warp's pooled narrow phase (passes of VINE_PAIR_PASS items, envs whose
pairs straddle a pass boundary); the kernel is never checked against it.
"""
import functools

import numpy as np

from vine_robot_isaacgymenvs_b200 import abi

PAIR_PASS = 64                      # VINE_PAIR_PASS: work items of the warp's narrow phase per pass
WARP = 32
LINK_LEN, PIVOT_Z, BASE_ANGLE = 0.0885, 0.965, 3.1415
FPAM_REACH = 0.055 + 0.0169         # VINE_FPAM_OFFSET + VINE_FPAM_RADIUS: the widest cross-section of a link
CULL_SLACK = 0.01                   # VineConfig.contact_cull_slack default
PROBES = 64                         # perturbed f64 runs of the conditioning probe

CONFIGS = {"shelf": (1, 0), "pipe": (0, 1), "shelf_pipe": (1, 1)}


def obstacle_config(oracle, name):
    vc = oracle.default_config()
    vc.create_shelf, vc.create_pipe = CONFIGS[name]
    return vc


def _copy(vc):
    return type(vc).from_buffer_copy(vc)


def pipe_angle(tz):
    """V5:854-885 as the oracle's reset computes it: polyval of 1 - target z in f64, degrees -> radians in f32."""
    ez = (np.float32(1.0) - np.asarray(tz, np.float32)).astype(np.float64)
    y = np.zeros_like(ez)
    for c in (1.0e4 * 1.3199, 1.0e4 * -1.2276, 1.0e4 * 0.4045, 1.0e4 * -0.0447):
        y = y * ez + c
    return y.astype(np.float32) * np.float32(np.pi / 180.0)


def draw_candidates(vc, n, rng):
    f = np.float32
    q = rng.normal(0, 0.15, (n, 6)).astype(f)
    q[:, 0] = rng.uniform(-0.3, 0.3, n)
    q[:, 1:] -= 0.12                                   # bent toward -y where the obstacles are
    qd = rng.normal(0, 0.5, (n, 6)).astype(f)
    tz = rng.uniform(vc.min_target_z, vc.max_target_z, n).astype(f)
    target = np.stack([np.zeros(n), rng.uniform(vc.min_target_y, vc.max_target_y, n), tz], 1).astype(f)
    depth = rng.uniform(vc.min_target_depth_in_obstacle, vc.max_target_depth_in_obstacle, n)
    obj = np.stack([depth, pipe_angle(tz) if vc.create_pipe else np.zeros(n)], 1).astype(f)
    eff = np.concatenate([rng.uniform(-4, 4, (n, 1)), rng.normal(0, 0.05, (n, 5))], 1).astype(f)
    scale = rng.uniform(0.9, 1.1, (n, 5, 4)).astype(f)
    u = rng.uniform(-0.1, 3, n).astype(f)
    return {"dof_pos": q, "dof_vel": qd, "dof_efforts": eff, "dynamics_scaling": scale, "u_fpam_to_use": u,
            "target_positions": target, "object_info": obj}


def simulate(oracle, vc, st, use_f64=True):
    """One sim step of the oracle from the states ``st``; returns the simulate outputs."""
    n = len(st["dof_pos"])
    f = np.float32
    out = {k: np.array(v, copy=True) for k, v in st.items()}
    out.update({"tip_positions": np.zeros((n, 3), f), "tip_velocities": np.zeros((n, 3), f), "shelf_contact_force": np.zeros(n, f)})
    oracle.call_io("oracle_simulate", vc, n, abi.VineSimulateIO, out, int(use_f64))
    return out


def take(st, idx):
    return {k: v[idx] for k, v in st.items()}


def concat(*sts):
    return {k: np.concatenate([s[k] for s in sts]) for k in sts[0]}


def rects(vc, target, obj):
    """[n, rects, 6] = centre y, z, unit axis y, z, half extents along the axis and the normal (for_each_obstacle_rect)."""
    ty, tz, depth, theta = (np.asarray(a, np.float64) for a in (target[:, 1], target[:, 2], obj[:, 0], obj[:, 1]))
    one, zero = np.ones_like(ty), np.zeros_like(ty)
    out = []
    if vc.create_shelf:
        ry, rz = ty - 0.2 + depth, tz - 0.01
        out += [(ry - 0.001, rz, one, zero, 0.1995 * one, 0.005 * one), (ry, rz + 0.2, one, zero, 0.2 * one, 0.005 * one),
                (ry + 0.199, rz, one, zero, 0.001 * one, 0.005 * one)]
    if vc.create_pipe:
        st, ct = np.sin(theta), np.cos(theta)
        off, win, wout = 0.0735 - 0.0777, 0.07232816, 0.07758640
        ey, ez = ty + depth * ct + off * st, tz + depth * st - off * ct
        ay, az = -ct, -st
        ny, nz = -az, ay
        mid, hn, ha = 0.5 * (win + wout), 0.5 * (wout - win), 0.5 * 0.34125
        for s in (-1, 1):
            out.append((ey + ay * ha + s * mid * ny, ez + az * ha + s * mid * nz, ay, az, ha * one, hn * one))
    return np.stack([np.stack(r, 1) for r in out], 1)


def joints(q):
    """[n, 6] y and z of the cart pivot and the five link ends."""
    q = np.asarray(q, np.float64)
    phi = BASE_ANGLE + np.cumsum(q[:, 1:], 1)
    py = q[:, :1] + np.concatenate([np.zeros((len(q), 1)), np.cumsum(-LINK_LEN * np.sin(phi), 1)], 1)
    pz = PIVOT_Z + np.concatenate([np.zeros((len(q), 1)), np.cumsum(LINK_LEN * np.cos(phi), 1)], 1)
    return py, pz


def chain_gap(vc, st):
    """The chain's bounding box (inflated by the widest cross-section + rest + slack) against the obstacles' box."""
    py, pz = joints(st["dof_pos"])
    R = rects(vc, st["target_positions"], st["object_info"])
    ey = np.abs(R[..., 2]) * R[..., 4] + np.abs(R[..., 3]) * R[..., 5]
    ez = np.abs(R[..., 3]) * R[..., 4] + np.abs(R[..., 2]) * R[..., 5]
    lo_y, hi_y = (R[..., 0] - ey).min(1), (R[..., 0] + ey).max(1)
    lo_z, hi_z = (R[..., 1] - ez).min(1), (R[..., 1] + ez).max(1)
    m = FPAM_REACH + vc.contact_rest_offset + 1e-3 + CULL_SLACK
    return np.maximum(np.maximum(py.min(1) - m - hi_y, lo_y - (py.max(1) + m)),
                      np.maximum(pz.min(1) - m - hi_z, lo_z - (pz.max(1) + m)))


def pair_masks(vc, st):
    """Candidate (link j, rectangle r) pairs at the start state, bit 5 r + j: the link's midpoint against the rectangle
    inflated by 0.09 + rest + slack in the rectangle's frame; none while the boxes have a gap."""
    py, pz = joints(st["dof_pos"])
    my, mz = 0.5 * (py[:, :-1] + py[:, 1:]), 0.5 * (pz[:, :-1] + pz[:, 1:])
    R = rects(vc, st["target_positions"], st["object_info"])
    reach = 0.09 + vc.contact_rest_offset + CULL_SLACK
    mask = np.zeros(len(py), np.int64)
    for r in range(R.shape[1]):
        cy, cz, ay, az, ha, hn = (R[:, r, k:k + 1] for k in range(6))
        dy, dz = my - cy, mz - cz
        hit = (np.abs(dy * ay + dz * az) <= ha + reach) & (np.abs(dz * ay - dy * az) <= hn + reach)
        mask |= (hit * (1 << (5 * r + np.arange(5)))).sum(1)
    return np.where(chain_gap(vc, st) > 0, 0, mask)


def pair_counts(vc, st):
    m = pair_masks(vc, st)
    return np.array([bin(int(x)).count("1") for x in m])


def warp_load(counts):
    """Per warp of a layout (lanes in order, ragged tail allowed): total pairs, passes, and per env whether its pairs
    straddle a pass boundary of the warp's work list."""
    counts = np.asarray(counts)
    n = len(counts)
    padded = np.zeros(-(-n // WARP) * WARP, np.int64)
    padded[:n] = counts
    w = padded.reshape(-1, WARP)
    start = np.cumsum(w, 1) - w
    end = start + w - 1
    straddle = ((w > 0) & (start // PAIR_PASS != end // PAIR_PASS)).reshape(-1)[:n]
    total = w.sum(1)
    return total, -(-total // PAIR_PASS), straddle


def perturb(st, rng, ulps=16):
    """``st`` with q and qd multiplied by 1 + U(-ulps, ulps) 2^-23: input changes of the size of the kernel's own roundings
    (approximate sin/cos and reciprocals, contracted products), which exceed an ulp"""
    p = dict(st)
    for k in ("dof_pos", "dof_vel"):
        v = np.asarray(st[k], np.float64)
        p[k] = (v * (1 + rng.uniform(-ulps, ulps, v.shape) * 2.0 ** -23)).astype(np.float32)
    return p


def _agree(a, b):
    return (np.abs(a["dof_pos"] - b["dof_pos"]).max(1) < 1e-5) & (np.abs(a["dof_vel"] - b["dof_vel"]).max(1) < 1e-3)


def within_tolerance(a, b):
    """per env: within the contact tolerances of test_simulate_matches_f64_oracle (q 1e-3 rel + 1e-5, qd 1e-2 rel + 2e-3)"""
    return (np.abs(a["dof_pos"] - b["dof_pos"]) <= 1e-5 + 1e-3 * np.abs(b["dof_pos"])).all(1) \
        & (np.abs(a["dof_vel"] - b["dof_vel"]) <= 2e-3 + 1e-2 * np.abs(b["dof_vel"])).all(1)


def _well(oracle, vc, st, ref, rng, probes=PROBES):
    """The oracle's f32 build agrees with f64, and ``probes`` f64 runs from perturbed inputs stay within the tolerance the
    kernel is held to.  The f32 build alone passes envs whose step jumps under input changes of a few ulps (a contact feature
    switching at a face/corner boundary): it agrees with f64 by chance."""
    well = _agree(simulate(oracle, vc, st, use_f64=False), ref)
    idx = np.flatnonzero(well)
    sub, sub_ref = take(st, idx), take(ref, idx)
    for _ in range(probes):
        well[idx[~within_tolerance(simulate(oracle, vc, perturb(sub, rng, 32)), sub_ref)]] = False
    return well


@functools.lru_cache(maxsize=None)
def _select_cached(oracle, name, seed, n_touched, n_fillers, batch):
    vc = obstacle_config(oracle, name)
    free = _copy(vc)
    free.create_shelf = free.create_pipe = 0
    rng = np.random.default_rng(seed)
    touched, fillers = [], []
    n_drawn = n_t = n_f = 0
    while n_t < n_touched or n_f < n_fillers:
        st = draw_candidates(vc, batch, rng)
        n_drawn += batch
        ref, ref_free = simulate(oracle, vc, st), simulate(oracle, free, st)
        dqd = np.abs(ref["dof_vel"] - ref_free["dof_vel"]).max(1)
        hit = (dqd > 1e-3) | (ref["shelf_contact_force"] > 0)
        t = np.flatnonzero(hit)
        t = t[_well(oracle, vc, take(st, t), take(ref, t), rng)]
        fl = np.flatnonzero(~hit & (dqd == 0) & (pair_counts(vc, st) == 0))
        fl = fl[_agree(simulate(oracle, vc, take(st, fl), use_f64=False), take(ref, fl))]
        touched.append(take(st, t)); fillers.append(take(st, fl))
        n_t += len(t); n_f += len(fl)
    touched = take(concat(*touched), np.arange(n_touched))
    fillers = take(concat(*fillers), np.arange(n_fillers))
    return {"vc": vc, "touched": touched, "fillers": fillers, "counts": pair_counts(vc, touched),
            "acceptance": n_t / n_drawn, "filler_rate": n_f / n_drawn, "drawn": n_drawn}


def select(oracle, name, seed=0, n_touched=1024, n_fillers=2048, batch=4096):
    """Touched and filler states of one obstacle config (cached per arguments); prints the acceptance rate.  About 20 % of
    the candidates are touched and well-conditioned and 70 % are fillers with every config, so two or three batches of
    4096 candidates do."""
    s = _select_cached(oracle, name, seed, n_touched, n_fillers, batch)
    print(f"\n[dense contact {name}] drew {s['drawn']}: touched and well-conditioned {100 * s['acceptance']:.1f} %, "
          f"fillers {100 * s['filler_rate']:.1f} %; pairs per touched env mean {s['counts'].mean():.1f} max {s['counts'].max()}")
    return s


def layouts(n_touched, n_fillers, seed=0):
    """Batch layouts of the same envs for ``vine_simulate``, as indices into touched (0 .. n_touched) followed by fillers:
      dense     every lane of every warp is a touched env (pass after pass of the pooled work list, envs straddling passes);
      isolated  one touched env per warp among 31 fillers, at lane k % 32 (its column of the warp's scratch moves);
      shuffled  a random permutation of the touched envs and most fillers, ragged n (offsets in the work list move);
      tail_<n>  32 k + 1 and 32 k + 31 envs with a touched env in the last slot: the ghost lanes run on copies of it."""
    assert n_touched % WARP == 0 and n_fillers >= WARP - 1
    rng = np.random.default_rng(seed)
    T = n_touched
    out = {"dense": np.arange(T)}
    iso = T + (np.arange(T)[:, None] * (WARP - 1) + np.arange(WARP - 1)) % n_fillers
    out["isolated"] = np.array([np.insert(iso[k], k % WARP, k) for k in range(T)]).reshape(-1)
    out["shuffled"] = rng.permutation(np.concatenate([np.arange(T), T + np.arange(n_fillers - 13)]))
    for k, last in ((1, 0), (3, T // 2), (1, T - 1)):
        for n in (WARP * k + 1, WARP * k + WARP - 1):
            out[f"tail_{n}_{last}"] = np.append((last + 1 + np.arange(n - 1)) % T, last)
    return out
