"""5x5 angular search windows (an = 2) on the host side: the static window plan (lfbm5d_step_plan) against the schedule the
CPU oracle's step driver takes. No GPU needed."""
import numpy as np
import pytest

import lfdata


@pytest.mark.parametrize("aw,ah,holes,major", [
    (17, 17, (), "row"),
    (7, 7, (), "row"),
    (6, 9, (), "row"),
    (7, 7, (10, 24, 38), "row"),
    (7, 7, (24,), "col"),
    (6, 9, (4, 31), "col"),
])
def test_step_plan_an2_matches_the_oracle_schedule(oracle, aw, ah, holes, major):
    """Same windows in the same order as the oracle's step driver at an = 2; windows of one plan level share no SAI; every SAI is
    covered; the sticky dct -> sadct switch starts at the first window that holds an empty SAI."""
    import lfbm5d_b200 as L
    am = L.ROWMAJOR if major == "row" else L.COLMAJOR
    clean = lfdata.synth_lf(aw, ah, 12, 12)
    noisy = oracle.add_noise(clean, 10.0)
    mask = np.ones(aw * ah, np.uint32)
    for h in holes:
        mask[h] = 0
    _, _, sched = oracle.run_step1(noisy, mask, 10.0, 2.7, aw, ah, 2, 2, 2, 1, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR, ang_major=am)
    prm = L.make_params(10.0, 2.7, aw, ah, 2, 12, 12, 3, 2, 2, 1, 8, 4, L.ID, L.DCT, L.HAAR, ang_major=am)
    plan = L.step_plan(prm, mask)
    assert len(plan) == len(sched)
    assert np.array_equal(plan[:, 2:4], sched[:, 1:3])
    if (aw, ah, holes) == (17, 17, ()):
        assert len(plan) == 25
    seen = np.zeros(aw * ah, bool)
    for lvl in lfdata.plan_levels(plan):
        used = []
        for w in lvl:
            used += lfdata.window_sais(w, prm, mask)
        assert len(used) == len(set(used))
        seen[used] = True
    assert np.array_equal(seen, mask.astype(bool))
    with_hole = [i for i, w in enumerate(plan) if any(not mask[st] for st in lfdata.window_sais(w, prm))]
    expect = np.zeros(len(plan), np.uint32)
    if with_hole:
        expect[min(with_hole):] = 1
    assert np.array_equal(plan[:, 5], expect)
