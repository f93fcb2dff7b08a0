"""The integrator evaluates sin/cos of every link angle afresh in each substep (MUFU.SIN/COS), so its accuracy has no bound
on the link rate. These tests spin the links at 50-150 rad/s, where rotating (sin, cos) incrementally by h*w per substep
with a truncated series would no longer be exact to f32 (that held below 36 rad/s).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from vine_robot_isaacgymenvs_b200 import abi

pytestmark = pytest.mark.gpu


def fast_states(n, seed):
    """joint positions and velocities [n, 6] (relative coordinates) whose absolute link rates are 50-150 rad/s either way"""
    rng = np.random.default_rng(seed)
    f = np.float32
    q = rng.normal(0, 0.15, (n, 6)).astype(f)
    q[:, 0] = rng.uniform(-0.3, 0.3, n)
    w = rng.uniform(50, 150, (n, 5)) * rng.choice([-1.0, 1.0], (n, 5))
    qd = np.empty((n, 6), f)
    qd[:, 0] = rng.normal(0, 0.5, n)
    qd[:, 1] = w[:, 0]
    qd[:, 2:] = np.diff(w, axis=1)
    return q, qd


def test_simulate_at_fast_link_rates_matches_f64_oracle(oracle_lib):
    """vine_simulate (one sim step = 10 substeps) from states spinning at 50-150 rad/s against the f64 oracle, with the
    free-space tolerances of test_gpu_parity.py::test_simulate_matches_f64_oracle."""
    vc = oracle_lib.default_config()
    vc.create_pipe = 0
    vc.create_shelf = 0
    n = 4096
    q, qd = fast_states(n, 11)
    rng = np.random.default_rng(12)
    f = np.float32
    eff = np.concatenate([rng.uniform(-4, 4, (n, 1)), rng.normal(0, 0.05, (n, 5))], 1).astype(f)
    scale = rng.uniform(0.9, 1.1, (n, 5, 4)).astype(f)
    u = rng.uniform(-0.1, 3, n).astype(f)
    zeros3 = np.zeros((n, 3), f)
    ref = {"dof_pos": q.copy(), "dof_vel": qd.copy(), "dof_efforts": eff, "dynamics_scaling": scale, "u_fpam_to_use": u,
           "target_positions": zeros3.copy(), "object_info": np.zeros((n, 2), f), "tip_positions": zeros3.copy(),
           "tip_velocities": zeros3.copy(), "shelf_contact_force": np.zeros(n, f)}
    oracle_lib.call_io("oracle_simulate", vc, n, abi.VineSimulateIO, ref, 1)
    lib = abi.load_library()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    t = {k: dev(v) for k, v in ref.items() if k not in ("dof_pos", "dof_vel")}
    t["dof_pos"], t["dof_vel"] = dev(q), dev(qd)
    for k in ("tip_positions", "tip_velocities", "shelf_contact_force"):
        t[k].zero_()
    h = C.c_void_p()
    assert lib.vine_create(C.byref(vc), n, 0, 0, 42, C.byref(h)) == 0, lib.vine_last_error(None)
    io = abi.VineSimulateIO()
    for name, ftype in io._fields_:
        if name in t:
            setattr(io, name, C.cast(t[name].data_ptr(), ftype))
    rc = lib.vine_simulate(h, C.byref(io), None)
    torch.cuda.synchronize()
    assert rc == 0, lib.vine_last_error(h)
    lib.vine_destroy(h)
    got_q, got_qd = t["dof_pos"].cpu().numpy(), t["dof_vel"].cpu().numpy()
    assert np.isfinite(got_q).all() and np.isfinite(got_qd).all()
    assert np.abs(ref["dof_vel"][:, 1:].cumsum(1)).max() > 50     # still spinning fast after the sim step
    np.testing.assert_allclose(got_q, ref["dof_pos"], rtol=1e-3, atol=1e-5)
    np.testing.assert_allclose(got_qd, ref["dof_vel"], rtol=1e-2, atol=1e-4)
    np.testing.assert_allclose(t["tip_positions"].cpu().numpy(), ref["tip_positions"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(t["tip_velocities"].cpu().numpy(), ref["tip_velocities"], rtol=1e-2, atol=2e-3)

