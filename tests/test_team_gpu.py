"""One light field on a team of ranks that split every window pass (csrc/team.cuh), emulated on ONE GPU: `world` contexts on the
same device, exchanges as device copies. The band logic — plane-parallel block matching with merged candidate lists, row-band
groups, the chained border sums of the ordered aggregation — must reproduce the single-context result BIT FOR BIT: basic,
denoised, the colour-round-tripped inputs and the window schedule. (tests/dist_team_gpu.py runs the same check over NCCL.)"""
import numpy as np
import pytest

import lfdata
from gpucheck import run_single, run_team

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("world,aw,ah,H,W,C,masked", [(2, 3, 3, 200, 72, 3, False), (3, 4, 3, 330, 64, 3, True), (4, 3, 3, 340, 56, 3, False),
                                                       (8, 3, 3, 620, 48, 3, False), (2, 3, 3, 150, 60, 1, False)])
def test_team_bit_identical_to_single(world, aw, ah, H, W, C, masked, oracle):
    import torch
    import lfbm5d_b200 as L
    dev = torch.device("cuda", 0)
    clean = lfdata.synth_lf(aw, ah, H, W)[:, :C]
    noisy = torch.from_numpy(oracle.add_noise(np.ascontiguousarray(clean), 15.0)).to(dev)
    mask = np.ones(aw * ah, np.uint32)
    if masked:
        mask[5] = 0
    p1 = L.make_params(15.0, 2.7, aw, ah, 1, W, H, C, 8, 18, 6, 16, 4, L.ID, L.DCT if masked else L.SADCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, aw, ah, 1, W, H, C, 16, 18, 6, 8, 4, L.DCT, L.DCT if masked else L.SADCT, L.HAAR)
    eng = L.LFBM5D(0)
    w0, b0, o0, s0 = run_single(L, eng, torch, noisy, mask, p1, p2)
    eng.close()
    # complete results on every rank (gather) ...
    ws, bs, outs, bands1, bands2, st = run_team(L, torch, world, noisy, mask, p1, p2, gather=1)
    assert st["bytes_exchanged"] > 0
    assert bands2[0][0] == 0 and bands2[-1][1] == H and all(bands2[g][1] == bands2[g + 1][0] for g in range(world - 1))
    for g in range(world):
        assert torch.equal(outs[g], o0), "denoised differs on rank %d" % g
        assert torch.equal(ws[g], w0), "noisy round trip differs on rank %d" % g
    # ... and band-resident results (no gather): every rank holds its band and the rows it shares with the next rank
    ws, bs, outs, bands1, bands2, st = run_team(L, torch, world, noisy, mask, p1, p2, gather=0)
    for g in range(world):
        lo, hi, keep = bands1[g]
        assert torch.equal(bs[g][:, :, lo:keep], b0[:, :, lo:keep]), "basic differs on rank %d" % g
        lo, hi, keep = bands2[g]
        assert torch.equal(outs[g][:, :, lo:keep], o0[:, :, lo:keep]), "denoised differs on rank %d" % g


def test_team_exact_distance_ties(oracle):
    """Quantised, partly flat light field: reference patches with exact distance ties among their selected self matches need the
    complete candidate sequence (the re-implemented libstdc++ partial_sort). With the peer view of the other ranks' sums they are
    redone in place; without it the team exchanges the complete sums and redoes the pass. Bit-identical to one GPU either way."""
    import torch
    import lfbm5d_b200 as L
    dev = torch.device("cuda", 0)
    aw = ah = 3
    H, W = 200, 64
    clean = np.round(lfdata.synth_lf(aw, ah, H, W) / 64.0) * 64.0
    clean[:, :, 60:140, 10:50] = 64.0
    noisy = torch.from_numpy(clean.astype(np.float32)).to(dev)
    mask = np.ones(9, np.uint32)
    p1 = L.make_params(15.0, 2.7, aw, ah, 1, W, H, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, aw, ah, 1, W, H, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    eng = L.LFBM5D(0)
    w0, b0, o0, s0 = run_single(L, eng, torch, noisy, mask, p1, p2)
    eng.close()
    for peer_view in (True, False):
        ws, bs, outs, bands1, bands2, st = run_team(L, torch, 3, noisy, mask, p1, p2, gather=1, peer_view=peer_view)
        assert st["peer_view"] == peer_view
        assert (st["tie_patches"] > 0 and st["passes_redone"] == 0) if peer_view else st["passes_redone"] > 0
        for g in range(3):
            assert torch.equal(outs[g], o0) and torch.equal(ws[g], w0)


@pytest.mark.parametrize("world,lanes", [(2, 2), (3, 3), (1, 4)])
def test_team_lanes_run_independent_windows_concurrently(world, lanes, oracle):
    """Several lanes: the windows of one level of the static plan (no shared SAI) run concurrently, one per lane, in level order
    instead of the sequential order. A 6 x 5 light field (12 windows, several levels, one empty SAI with the sticky dct -> sadct
    switch): still bit-identical to the sequential single-context run."""
    import torch
    import lfbm5d_b200 as L
    dev = torch.device("cuda", 0)
    aw, ah, H, W = 6, 5, 170, 60
    clean = lfdata.synth_lf(aw, ah, H, W)
    noisy = torch.from_numpy(oracle.add_noise(clean, 15.0)).to(dev)
    mask = np.ones(aw * ah, np.uint32)
    mask[9] = 0
    p1 = L.make_params(15.0, 2.7, aw, ah, 1, W, H, 3, 8, 18, 6, 16, 4, L.ID, L.DCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, aw, ah, 1, W, H, 3, 16, 18, 6, 8, 4, L.DCT, L.DCT, L.HAAR)
    plan = L.step_plan(p1, mask)
    assert len(plan) >= 6 and int(plan[:, 4].max()) + 1 < len(plan)          # some level holds more than one window
    eng = L.LFBM5D(0)
    w0, b0, o0, s0 = run_single(L, eng, torch, noisy, mask, p1, p2)
    eng.close()
    assert np.array_equal(plan[:, 2:4], s0[:, 1:3])                           # the plan's windows are the sequential schedule's
    ws, bs, outs, bands1, bands2, st = run_team(L, torch, world, noisy, mask, p1, p2, gather=1, lanes=lanes)
    for g in range(world):
        assert torch.equal(outs[g], o0), "denoised differs on rank %d" % g
        assert torch.equal(ws[g], w0), "noisy round trip differs on rank %d" % g


@pytest.mark.parametrize("world,params", [(4, "config2"), (8, "config2"), (4, "config3")])
def test_team_band_resident_basic_with_other_step2_bands(world, params, oracle):
    """Step 1 without a gather (LF_basic stays band-resident), then step 2 on the same team, with more ranks than row bands: the
    two steps cut different bands (other patch size / step, another number of ranks that get rows at all), so step 2 reads rows of
    LF_basic a rank did not keep. The team has to send the step-1 bands around first (team_step_begin). BASELINE config-2 parameters
    (`1 18 3 16 3 bior / 8 18 3 8 3 dct`) and the README parameters, twice on the same team object; bit-identical to one context."""
    import torch
    import lfbm5d_b200 as L
    dev = torch.device("cuda", 0)
    aw, ah, H, W = 4, 3, 217, 157
    clean = lfdata.synth_lf(aw, ah, H, W)
    noisy = torch.from_numpy(oracle.add_noise(clean, 10.0)).to(dev)
    mask = np.ones(aw * ah, np.uint32)
    if params == "config2":
        p1 = L.make_params(10.0, 2.7, aw, ah, 1, W, H, 3, 1, 18, 3, 16, 3, L.BIOR, L.SADCT, L.HAAR)
        p2 = L.make_params(10.0, 0.0, aw, ah, 1, W, H, 3, 8, 18, 3, 8, 3, L.DCT, L.SADCT, L.HAAR)
    else:
        p1 = L.make_params(10.0, 2.7, aw, ah, 1, W, H, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
        p2 = L.make_params(10.0, 0.0, aw, ah, 1, W, H, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    b1 = [L.plan_band(world, g, 1, p1) for g in range(world)]
    b2 = [L.plan_band(world, g, 2, p2) for g in range(world)]
    assert any(b2[g][2] > b2[g][0] and (b2[g][0] < b1[g][0] or b2[g][2] > b1[g][2]) for g in range(world)), "bands nest: the case is not exercised"
    eng = L.LFBM5D(0)
    w0, b0, o0, s0 = run_single(L, eng, torch, noisy, mask, p1, p2)
    eng.close()
    team = L.Team.emulated(0, world)
    for rep in range(2):
        ws = [noisy.clone() for _ in range(world)]
        bs = [torch.zeros_like(noisy) for _ in range(world)]
        outs = [torch.zeros_like(noisy) for _ in range(world)]
        team.step(1, p1, [t.data_ptr() for t in ws], None, mask, [t.data_ptr() for t in bs], gather=0)
        team.step(2, p2, [t.data_ptr() for t in ws], [t.data_ptr() for t in bs], mask, [t.data_ptr() for t in outs], gather=1)
        torch.cuda.synchronize()
        for g in range(world):
            assert torch.equal(outs[g], o0), "denoised differs on rank %d (repetition %d)" % (g, rep)
    team.close()
