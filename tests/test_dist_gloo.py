"""world_size-2 gloo test of the multi-GPU host logic (SAI sharding, gather, max-over-ranks timing)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from lfbm5d_b200 import dist as D
    asize = 9
    full = np.arange(asize * 6, dtype=np.float32).reshape(asize, 2, 3)
    lo, hi = D.shard_sais(asize, world, rank)
    mask = D.shard_mask(np.ones(asize), world, rank)
    assert mask.sum() == hi - lo and mask[lo:hi].all()
    out = D.gather_shards(full[lo:hi] * 2.0, asize, dist)
    ok = bool(np.array_equal(out.numpy(), full * 2.0))
    t = D.max_over_ranks(1.0 + rank, dist)
    ret[rank] = (ok, t, lo, hi)
    dist.destroy_process_group()


def test_shard_gather_max_over_ranks():
    from lfbm5d_b200 import dist as D
    for asize in (1, 9, 289):
        for world in (1, 2, 4, 8):
            cover = []
            for r in range(world):
                lo, hi = D.shard_sais(asize, world, r)
                cover += list(range(lo, hi))
            assert cover == list(range(asize))
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, 2, 29613, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert ret[0][0] and ret[1][0] and ret[0][1] == 2.0 and ret[1][1] == 2.0
    assert (ret[0][2], ret[0][3], ret[1][2], ret[1][3]) == (0, 5, 5, 9)


def test_window_plan_matches_the_sequential_schedule(oracle):
    """lfbm5d_step_plan (static form of the reference's window selection) against the schedule the oracle's step driver takes
    (itself bit-identical to the reference), with and without empty SAIs; windows of one level share no SAI."""
    import lfbm5d_b200 as L
    import lfdata
    for (aw, ah, holes, major) in [(5, 5, (), L.ROWMAJOR), (7, 5, (3, 17), L.ROWMAJOR), (6, 4, (23,), L.COLMAJOR)]:
        clean = lfdata.synth_lf(aw, ah, 12, 12)
        noisy = oracle.add_noise(clean, 10.0)
        mask = np.ones(aw * ah, np.uint32)
        for h in holes:
            mask[h] = 0
        _, _, sched = oracle.run_step1(noisy, mask, 10.0, 2.7, aw, ah, 1, 2, 2, 1, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR, ang_major=major)
        prm = L.make_params(10.0, 2.7, aw, ah, 1, 12, 12, 3, 2, 2, 1, 8, 4, L.ID, L.DCT, L.HAAR, ang_major=major)
        plan = L.step_plan(prm, mask)
        assert len(plan) == len(sched)
        assert np.array_equal(plan[:, 2:4], sched[:, 1:3])                       # same windows in the same order
        seen = np.zeros(aw * ah, bool)
        for lvl in lfdata.plan_levels(plan):
            used = []
            for w in lvl:
                used += lfdata.window_sais(w, prm, mask)
            assert len(used) == len(set(used))                                   # windows of a level are disjoint
            seen[used] = True
        assert np.array_equal(seen, mask.astype(bool))
        if holes:                                                               # sticky dct -> sadct switch from the first window with a hole
            first = min(i for i, w in enumerate(plan) if any(not mask[st] for st in lfdata.window_sais(w, prm)))
            assert np.array_equal(plan[:, 5], (np.arange(len(plan)) >= first).astype(np.uint32))


def _band_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import lfbm5d_b200 as L
    p1 = L.make_params(10.0, 2.7, 17, 17, 1, 1024, 1024, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    mine = torch.tensor(L.plan_band(world, rank, 1, p1), dtype=torch.int64)
    allb = [torch.zeros(3, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(allb, mine)
    ret[rank] = [tuple(int(x) for x in b) for b in allb]
    dist.destroy_process_group()


def test_team_bands_tile_the_light_field():
    """Row bands of the team path (lfbm5d_team_plan_band; csrc/team.cuh): for every world size the owned interior rows tile [0, H)
    in rank order, every rank keeps its band plus the rows it shares with the next rank (halo = 2 n + k - p rows), ranks that would
    break the two-ranks-per-pixel-row rule get nothing. Host logic only (no GPU); the world-2 part runs over gloo."""
    import lfbm5d_b200 as L
    for (H, k, N, t2) in ((1024, 16, 8, L.ID), (1024, 8, 16, L.DCT), (256, 16, 8, L.ID), (434, 8, 8, L.DCT)):
        prm = L.make_params(10.0, 2.7, 17, 17, 1, 640, H, 3, N, 18, 6, k, 4, t2, L.SADCT, L.HAAR)
        for world in (1, 2, 3, 4, 8, 16):
            bands = [L.plan_band(world, r, 1, prm) for r in range(world)]
            assert bands[0][0] == 0
            active = [b for b in bands if b[1] > b[0]]
            assert active and active[-1][1] == H
            for a, b in zip(bands[:-1], bands[1:]):
                assert a[1] == b[0] or b[1] == b[0]                      # contiguous in rank order (idle ranks own nothing)
            for b in active[:-1]:
                assert b[2] - b[1] == 2 * 24 + k - 4 or b[2] == H        # rows shared with the next rank: 2 n + k - p (search radius each way + patch)
            if H == 256:
                assert len(active) <= 4                                   # 61 reference rows: at most 4 ranks get rows
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_band_worker, args=(r, 2, 29617, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert ret[0] == ret[1] and ret[0][0][0] == 0 and ret[0][0][1] == ret[0][1][0] and ret[0][1][1] == 1024


def test_step2_bands_nest_in_step1_bands_or_need_the_late_gather():
    """LF_basic may stay band-resident between the steps of a team (lfbm5d_team_step, gather = 0): rank g then holds the rows
    [lo, keep) of its step-1 band. That is enough for step 2 only if its bands lie inside; otherwise team_step_begin sends the step-1
    bands around first. Host logic of that decision, from the planned bands (no GPU): the README parameters on 1024-row SAIs nest
    on every world size the bench runs; BASELINE config 2 (434 rows) on 8 ranks does not (step 1 gives rows to 7 ranks, step 2
    to 8) — the case that produced 11 dB before the fix."""
    import lfbm5d_b200 as L

    def nests(world, p1, p2):
        b1 = [L.plan_band(world, r, 1, p1) for r in range(world)]
        b2 = [L.plan_band(world, r, 2, p2) for r in range(world)]
        return all(b2[r][2] <= b2[r][0] or (b2[r][0] >= b1[r][0] and b2[r][2] <= b1[r][2]) for r in range(world)), b1, b2
    p1 = L.make_params(10.0, 2.7, 17, 17, 1, 1024, 1024, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(10.0, 0.0, 17, 17, 1, 1024, 1024, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    for world in (1, 2, 4, 8):
        ok, b1, b2 = nests(world, p1, p2)
        assert ok, (world, b1, b2)
    q1 = L.make_params(10.0, 2.7, 15, 15, 1, 625, 434, 3, 1, 18, 3, 16, 3, L.BIOR, L.SADCT, L.HAAR)
    q2 = L.make_params(10.0, 0.0, 15, 15, 1, 625, 434, 3, 8, 18, 3, 8, 3, L.DCT, L.SADCT, L.HAAR)
    assert nests(2, q1, q2)[0] and nests(4, q1, q2)[0]
    ok, b1, b2 = nests(8, q1, q2)
    assert not ok
    assert sum(1 for b in b1 if b[1] > b[0]) == 7 and sum(1 for b in b2 if b[1] > b[0]) == 8
