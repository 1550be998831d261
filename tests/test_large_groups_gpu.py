"""k = 16 groups of 3x3 windows that do not fit the shared memory of one CTA (N = 32 in step 1, N = 16 and 32 in step 2) run on
clusters of 2 or 4 CTAs that share the group through distributed shared memory (k_groups_cl). GPU against the CPU oracle through
the C ABI. The oracle is generic in N but pinned against the reference only at the N values of the other tests, so these results
are checked GPU vs oracle: match lists, disparity argmin and shape flags bit-exact; step 1 accumulators and LF_basic bit-identical;
complete runs within 0.01 dB; step 2 within the rounding bound of the oracle's group sums (gpucheck.wiener_tol)."""
import os

import numpy as np
import pytest

import golden_inputs as gi
import lfdata
from gpucheck import (LIBDIR, assert_team_matches_single, check_complete_run, check_pass, check_pngs, eng, estimate, psnr_on,
                      run_cli, wiener_tol, write_lf)  # noqa: F401 (eng is the engine fixture)

pytestmark = pytest.mark.gpu
K = 16


def expected_cluster(step, N):
    """CTAs per group: one channel of the group is N * 9 * 16 * RS * 4 B (RS = 16 for id, 17 otherwise), twice that in step 2."""
    return {(1, 32): 2, (2, 16): 2, (2, 32): 4}[(step, N)]


def spread_inputs(H=40, W=48):
    """Noisy padded SAIs with a flat region (every candidate matches, with exact distance ties: groups of N patches) and a region
    of strong noise (only the reference patch matches: the duplicated single match, groups of 2 patches)."""
    _, _, sym = gi.pad_inputs(H, W, 25.0)
    rng = np.random.default_rng(7)
    sym[:, :, 24:44, 24:56] = 100.0
    sym[:, :, 44:64, 40:72] += rng.normal(0.0, 120.0, (9, 3, 20, 32)).astype(np.float32)
    return sym


def check_pass_cl(eng, oracle, step, sym, basic, num0, den0, mask, proc, N, t2, t4, t5, lam=2.7, useSD=0, pst=4, cst=None, spread=False):
    """check_pass at k = 16 on the cluster size the group needs, step 2 and useSD within wiener_tol."""
    import lfbm5d_b200 as L
    A, C, hb, wb = sym.shape
    prm = L.make_params(25.0, lam, 3, 3, 1, wb - 48, hb - 48, C, N, 18, 6, K, 4, t2, t4, t5, useSD=int(useSD))
    cl, occ = eng.group_cluster(step, prm)
    assert cl == expected_cluster(step, N) and occ > 0, (cl, occ)
    on, od, gn, gd, gdbg = check_pass(eng, oracle, step, sym, basic, num0, den0, mask, proc, K, N, t2, t4, t5, pst=pst, cst=cst, lam=lam,
                                      useSD=useSD, rel=wiener_tol(N, useSD), est=False)
    if spread:
        # every CTA of the cluster holds patches (nSx = N), and the CTAs hold one patch each or, on 4-CTA clusters, two of them
        # hold none (nSx = 2, the smallest group: a single match is duplicated)
        cnt = gdbg[0][gdbg[0] > 0]
        assert (cnt == N).any() and (cnt == 2).any(), np.unique(cnt)
    return on, od, gn, gd


@pytest.mark.parametrize("t2", ["id", "dct", "bior"])
def test_single_passes_cluster(eng, oracle, t2):
    """Step 1 at N = 32 (2-CTA clusters) and step 2 at N = 16 (2 CTAs) and N = 32 (4 CTAs), every angular / 1-D transform."""
    T2 = {"id": oracle.ID, "dct": oracle.DCT, "bior": oracle.BIOR}[t2]
    sym = spread_inputs()
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    on, od, _, _ = check_pass_cl(eng, oracle, 1, sym, None, z, z, mask, proc, 32, oracle.ID, oracle.SADCT, oracle.HAAR, spread=True)
    basic = estimate(on, od, sym)
    for t4 in (oracle.DCT, oracle.SADCT, oracle.ID):
        for t5 in (oracle.HAAR, oracle.HADAMARD, oracle.DCT):
            check_pass_cl(eng, oracle, 1, sym, None, z, z, mask, proc, 32, T2, t4, t5)
            for N in (16, 32):
                check_pass_cl(eng, oracle, 2, sym, basic, z, z, mask, proc, N, T2, t4, t5, lam=0.0, spread=t4 == oracle.SADCT)


def test_single_passes_cluster_sd_ties_and_second_pass(eng, oracle):
    """useSD in both steps (group-wide sums over the cluster), quantised input with exact distance ties, and a second pass of
    step 1 on top of the first pass's accumulators."""
    sym = spread_inputs()
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    on, od, _, _ = check_pass_cl(eng, oracle, 1, sym, None, z, z, mask, proc, 32, oracle.DCT, oracle.SADCT, oracle.HAAR)
    basic = estimate(on, od, sym)
    check_pass_cl(eng, oracle, 1, sym, None, z, z, mask, proc, 32, oracle.ID, oracle.SADCT, oracle.HAAR, useSD=1, spread=True)
    for N in (16, 32):
        check_pass_cl(eng, oracle, 2, sym, basic, z, z, mask, proc, N, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, useSD=1, spread=True)
    check_pass_cl(eng, oracle, 1, sym, None, on, od, mask, proc, 32, oracle.DCT, oracle.SADCT, oracle.HAAR)
    q = (np.round(sym / 64.0) * 64.0).astype(np.float32)
    qn, qd, _, _ = check_pass_cl(eng, oracle, 1, q, None, z, z, mask, proc, 32, oracle.ID, oracle.SADCT, oracle.HAAR)
    check_pass_cl(eng, oracle, 2, q, estimate(qn, qd, q), z, z, mask, proc, 32, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0)


def test_single_passes_cluster_masked_processed_and_partial(eng, oracle):
    sym = spread_inputs()
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    mask[2] = 0
    proc[2] = proc[7] = 1
    on, od, gn, gd = check_pass_cl(eng, oracle, 1, sym, None, z, z, mask, proc, 32, oracle.DCT, oracle.SADCT, oracle.HAAR, spread=True)
    assert not gd[7].any() and not gd[2].any()
    basic = estimate(on, od, sym)
    for N in (16, 32):
        check_pass_cl(eng, oracle, 2, sym, basic, z, z, mask, proc, N, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, spread=True)
    # partial-window branch (pst != cst) on accumulators with holes: skipped groups are skipped by every CTA of their cluster
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    num, den = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, K, 32, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    basic = estimate(num, den, sym)
    num, den = gi.partial_holes(num, den)
    proc[4] = 1
    for pst in (1, 6):
        pon, _, _, _ = check_pass_cl(eng, oracle, 1, sym, None, num, den, mask, proc, 32, oracle.ID, oracle.SADCT, oracle.HAAR, pst=pst, cst=4)
        assert not np.array_equal(pon, num)
        for N in (16, 32):
            check_pass_cl(eng, oracle, 2, sym, basic, num, den, mask, proc, N, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, pst=pst, cst=4)


@pytest.mark.parametrize("aw,C,masked,N1,N2", [(3, 3, False, 8, 16), (3, 3, False, 32, 32), (5, 3, False, 32, 32), (3, 1, True, 32, 32)])
def test_complete_runs_cluster(eng, oracle, aw, C, masked, N1, N2):
    """Both steps with the group sizes `8 / 16` and `32 / 32` at k = 16 (an = 1) through the host-buffer and the device-resident
    entry points, with the oracle's window schedule; grayscale with an empty centre SAI takes the partial-window branch."""
    import lfbm5d_b200 as L
    H, W = 32, 36
    clean = np.ascontiguousarray(lfdata.synth_lf(aw, aw, H, W)[:, :C])
    m = np.ones(aw * aw, np.uint32)
    if masked:
        m[(aw * aw) // 2] = 0
    p1 = L.make_params(25.0, 2.7, aw, aw, 1, W, H, C, N1, 18, 6, K, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, aw, aw, 1, W, H, C, N2, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
    assert eng.group_cluster(1, p1)[0] == (1 if N1 == 8 else 2) and eng.group_cluster(2, p2)[0] == expected_cluster(2, N2)
    noisy, sched, _, d, _, _ = check_complete_run(eng, oracle, clean, m, p1, p2)
    if masked:
        assert sched[:, 3].max() > 1
    psnr = psnr_on(clean, m)
    assert psnr(d) > psnr(noisy) + 3.0


@pytest.mark.parametrize("world,H,W", [(2, 200, 72), (3, 330, 64)])
def test_team_bit_identical_to_single_cluster(eng, oracle, world, H, W):
    """Emulated teams run the cluster kernel on their row bands; its sums are reduced in a fixed order, so the results are
    bit-identical to one GPU."""
    import lfbm5d_b200 as L
    p1 = L.make_params(15.0, 2.7, 3, 3, 1, W, H, 3, 32, 18, 6, K, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, 3, 3, 1, W, H, 3, 32, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
    assert eng.group_cluster(1, p1)[0] == 2 and eng.group_cluster(2, p2)[0] == 4
    assert_team_matches_single(oracle, world, p1, p2)


def test_command_line_cluster(tmp_path):
    """LFBM5Ddenoising with kWien = 16 and NWien = 16 (step 2 on 2-CTA clusters): the files are what the library gives."""
    import lfbm5d_b200 as L
    H, W = 40, 44
    clean = lfdata.synth_lf(3, 3, H, W)
    src = write_lf(tmp_path, clean, 3)
    dirs = [str(tmp_path / d) for d in ("noisyLF", "basicLF", "denoisedLF", "diffLF")]
    head = [os.path.join(LIBDIR, "LFBM5Ddenoising"), str(src), "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "25", "2.7"] + dirs
    tail = ["8", "18", "6", "16", "4", "id", "sadct", "haar", "0", "16", "18", "6", "16", "4", "dct", "sadct", "haar", "0"]
    run_cli(head + tail + ["opp", "0", str(tmp_path / "objectiveResults.txt")])
    src8 = np.clip(np.floor(clean + 0.5), 0, 255).astype(np.float32)
    noisy = L.add_noise(src8, 25.0, seed0=20171016)
    mask = np.ones(9, np.uint32)
    e = L.LFBM5D(0)
    p1 = L.make_params(25.0, 2.7, 3, 3, 1, W, H, 3, 8, 18, 6, K, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, 3, 3, 1, W, H, 3, 16, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
    assert e.group_cluster(2, p2)[0] == 2
    basic, n1 = e.step1(p1, noisy, mask)
    den, _, _ = e.step2(p2, n1, basic, mask)
    e.close()
    check_pngs(tmp_path, (("noisyLF", noisy), ("basicLF", basic), ("denoisedLF", den)), 3)


def test_group_cluster_query(eng):
    """Groups that fit one CTA report a cluster size of 1; the others the smallest cluster that holds them."""
    import lfbm5d_b200 as L
    for step, N, t2, want in [(1, 8, L.ID, 1), (1, 16, L.DCT, 1), (2, 8, L.DCT, 1), (1, 32, L.ID, 2), (1, 32, L.BIOR, 2),
                              (2, 16, L.ID, 2), (2, 16, L.DCT, 2), (2, 32, L.ID, 4), (2, 32, L.DCT, 4)]:
        prm = L.make_params(25.0, 2.7 if step == 1 else 0.0, 3, 3, 1, 64, 64, 3, N, 18, 6, K, 4, t2, L.SADCT, L.HAAR)
        cl, occ = eng.group_cluster(step, prm)
        assert cl == want and (occ > 0) == (want > 1), (step, N, t2, cl, occ)
    # k = 8 and an = 0 groups always fit one CTA
    assert eng.group_cluster(2, L.make_params(25.0, 0.0, 3, 3, 1, 64, 64, 3, 32, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR))[0] == 1
    assert eng.group_cluster(2, L.make_params(25.0, 0.0, 3, 3, 0, 64, 64, 3, 32, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR))[0] == 1
