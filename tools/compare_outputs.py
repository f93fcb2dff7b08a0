"""Compare two `bench.py --dump-outputs DIR` runs of different builds, output for output.

    python tools/compare_outputs.py DIR_A DIR_B [--rel 2e-4]

A row (one env) agrees when every observation and the reward differ by at most rel * (1 + |a|) and the reset and time-out
flags are equal. Rows whose reset flag differs are counted apart: a reset decided by a threshold (target reached, tip
limit) flips when the state sits within rounding of it, and the env then continues from a fresh episode in one build only.
Prints one JSON line.
"""
import argparse
import json
import os

import numpy as np


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--rel", type=float, default=2e-4)
    args = ap.parse_args()
    load = lambda d, k: np.load(os.path.join(d, k + ".npy"))  # noqa: E731
    ids_a, ids_b = load(args.a, "env_ids"), load(args.b, "env_ids")
    if not np.array_equal(ids_a, ids_b):
        raise SystemExit("the two dumps hold different envs (different bench.py arguments?)")
    obs_a, obs_b = load(args.a, "obs").astype(np.float64), load(args.b, "obs").astype(np.float64)
    rew_a, rew_b = load(args.a, "rew").astype(np.float64), load(args.b, "rew").astype(np.float64)
    flags_same = (load(args.a, "reset") == load(args.b, "reset")) & (load(args.a, "time_outs") == load(args.b, "time_outs"))
    d_obs, d_rew = np.abs(obs_a - obs_b), np.abs(rew_a - rew_b)
    close = (d_obs <= args.rel * (1 + np.abs(obs_a))).all(1) & (d_rew <= args.rel * (1 + np.abs(rew_a)))
    rows = len(ids_a)
    agree = close & flags_same
    print(json.dumps({
        "rows": rows, "rel": args.rel,
        "rows_within_bound": float(agree.mean()),
        "rows_reset_flipped": int((~flags_same).sum()),
        "rows_outside_bound_same_flags": int((~close & flags_same).sum()),
        "bitwise_equal_rows": float(((obs_a == obs_b).all(1) & (rew_a == rew_b) & flags_same).mean()),
        "max_abs_diff_obs": float(d_obs.max()), "max_abs_diff_rew": float(d_rew.max()),
        "max_abs_diff_obs_same_flags": float(d_obs[flags_same].max()) if flags_same.any() else 0.0,
        "median_abs_diff_obs": float(np.median(d_obs)),
        "mean_obs_shift": float((obs_b - obs_a).mean()),
    }))


if __name__ == "__main__":
    main()
