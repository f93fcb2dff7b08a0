"""The dense-contact generator (tests/dense_contact.py) and the load its layouts put on the warp's pooled narrow phase, checked
without a GPU, so that a generator that stops producing that load fails here and not only on a B200."""
import numpy as np
import pytest

import dense_contact as D


@pytest.fixture(scope="module", params=sorted(D.CONFIGS))
def selected(request, oracle_lib):
    return request.param, D.select(oracle_lib, request.param)


def test_touched_envs_touch_and_fillers_do_not(selected, oracle_lib):
    name, s = selected
    vc, t, fl = s["vc"], s["touched"], s["fillers"]
    free = type(vc).from_buffer_copy(vc)
    free.create_shelf = free.create_pipe = 0
    for st, touched in ((t, True), (fl, False)):
        ref, ref_free = D.simulate(oracle_lib, vc, st), D.simulate(oracle_lib, free, st)
        dqd = np.abs(ref["dof_vel"] - ref_free["dof_vel"]).max(1)
        hit = (dqd > 1e-3) | (ref["shelf_contact_force"] > 0)
        assert hit.all() if touched else (dqd == 0).all()
        r32 = D.simulate(oracle_lib, vc, st, use_f64=False)
        assert (np.abs(r32["dof_pos"] - ref["dof_pos"]).max() < 1e-5) and (np.abs(r32["dof_vel"] - ref["dof_vel"]).max() < 1e-3)
    assert (D.pair_counts(vc, fl) == 0).all() and (s["counts"] > 0).all()
    ref, rng = D.simulate(oracle_lib, vc, t), np.random.default_rng(123)
    for _ in range(16):         # conditioning: fresh perturbed f64 runs stay within the tolerance the kernel is held to
        assert D.within_tolerance(D.simulate(oracle_lib, vc, D.perturb(t, rng, 16)), ref).all()
    if vc.create_shelf:
        assert (D.simulate(oracle_lib, vc, t)["shelf_contact_force"] > 0).sum() > 10
    again = D._select_cached.__wrapped__(oracle_lib, name, 0, len(s["counts"]), len(fl["dof_pos"]), 4096)   # uncached
    assert again["touched"]["dof_pos"] is not t["dof_pos"]
    for k in t:                                                                                  # seeded: the same states
        assert np.array_equal(again["touched"][k], t[k]) and np.array_equal(again["fillers"][k], fl[k]), k


def test_dense_layouts_load_the_narrow_phase_pass_after_pass(selected):
    """Dense layout: > 64 candidate pairs in >= 90 % of the warps; every config has envs whose pairs straddle a 64-item
    boundary of the work list; shelf + pipe (25-bit pair mask) has warps that need three or more passes."""
    name, s = selected
    counts = np.concatenate([s["counts"], np.zeros(len(s["fillers"]["dof_pos"]), np.int64)])
    lay = D.layouts(len(s["counts"]), len(s["fillers"]["dof_pos"]))
    total, passes, straddle = D.warp_load(counts[lay["dense"]])
    _, _, straddle_shuffled = D.warp_load(counts[lay["shuffled"]])
    print(f"\n[dense contact {name}] dense layout: {len(total)} warps, pairs per warp min {total.min()} mean {total.mean():.0f} "
          f"max {total.max()}, passes per warp {np.bincount(passes).tolist()}, envs straddling a pass "
          f"boundary {straddle.sum()} (shuffled layout {straddle_shuffled.sum()})")
    assert (total > D.PAIR_PASS).mean() >= 0.9
    assert straddle.sum() > 0
    if name == "shelf_pipe":
        assert (passes >= 3).any()
        assert (D.pair_masks(s["vc"], s["touched"]) >> 15).any()          # pair bits 15..24: rectangles 3 and 4 (the pipe)


def test_layouts_place_the_same_envs():
    T, F = 64, 40
    lay = D.layouts(T, F)
    assert np.array_equal(np.sort(lay["dense"]), np.arange(T))
    iso = lay["isolated"].reshape(-1, D.WARP)
    assert len(iso) == T and ((iso < T).sum(1) == 1).all()
    assert np.array_equal(np.argmax(iso < T, 1), np.arange(T) % D.WARP) and np.array_equal(iso[iso < T], np.arange(T))
    assert len(lay["shuffled"]) % D.WARP != 0 and set(range(T)) <= set(lay["shuffled"].tolist())
    tails = [k for k in lay if k.startswith("tail_")]
    assert {len(lay[k]) % D.WARP for k in tails} == {1, D.WARP - 1}
    assert all(lay[k][-1] < T and (lay[k] < T).all() for k in tails)
