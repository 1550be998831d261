"""12 x 12 patches (k = 12) on the GPU, through the C ABI against the CPU oracle. The oracle is generic in k but pinned against the
reference only at k = 8 and 16, so these results are checked GPU vs oracle. Tolerances are those of gpucheck.py: match lists,
disparity argmin and shape flags bit-exact; step 1 accumulators and LF_basic bit-identical; step 2 within 2e-5 relative per pass
(1e-4 with useSD); complete runs within 0.01 dB."""
import os

import numpy as np
import pytest

import golden_inputs as gi
import lfdata
from gpucheck import (LIBDIR, assert_rejected, assert_team_matches_single, channel0_planes, check_bm, check_complete_run, check_pass,
                      check_pngs, eng, estimate, psnr_on, run_cli, write_lf)  # noqa: F401 (eng is the engine fixture)

pytestmark = pytest.mark.gpu
K = 12


@pytest.mark.parametrize("nDisp", [6, 12])
def test_block_matching_k12(eng, oracle, nDisp):
    """Self and disparity matching at k = 12 on planes of 300+ rows (the 128-row source ring wraps), with a padded row pitch that is a
    multiple of 16 B and one that is not, noisy and quantised noise-free input (tied minima)."""
    n = 18 + nDisp
    H = 300
    w16 = 64 - (2 * n) % 4                    # (w16 + 2 n) floats per padded row: a multiple of 16 B
    for W in (w16, w16 + 1):
        check_bm(eng, oracle, channel0_planes(oracle, H, W, 10.0, 3, n=n), 1, K, 16, 3000.0, nDisp=nDisp)
        q = channel0_planes(oracle, H, W, 0.0, 3, n=n, quantise=True)
        assert check_bm(eng, oracle, q, 2, K, 16, 2000.0, nDisp=nDisp)[1] > 0


def test_single_passes_k12(eng, oracle):
    """Every 2-D / angular / 1-D transform combination at k = 12, both steps, and a second pass on top of the first's accumulators."""
    import lfbm5d_b200 as L
    _, _, sym = gi.pad_inputs(40, 48, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    on, od, _, _, _ = check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, K, 16, oracle.ID, oracle.SADCT, oracle.HAAR)
    basic = estimate(on, od, sym)
    prm = L.make_params(25.0, 0.0, 3, 3, 1, 48, 40, 3, 16, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
    assert eng.group_kernel(1, prm) == "k_groups12<1,3>" and eng.group_kernel(2, prm) == "k_groups12<2,3>"
    for t2 in (oracle.ID, oracle.DCT):
        for t4 in (oracle.DCT, oracle.SADCT, oracle.ID):
            for t5 in (oracle.HAAR, oracle.HADAMARD, oracle.DCT):
                check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, K, 8, t2, t4, t5)
                check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, K, 16, t2, t4, t5, lam=0.0)
    check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, K, 32, oracle.DCT, oracle.SADCT, oracle.HAAR)     # largest step-1 group
    check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, K, 16, oracle.ID, oracle.SADCT, oracle.HAAR, useSD=1)
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, K, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, useSD=1)
    # second pass of step 1 on top of the first pass's accumulators (block matching on num / den)
    check_pass(eng, oracle, 1, sym, None, on, od, mask, proc, K, 16, oracle.ID, oracle.SADCT, oracle.HAAR)


def test_single_passes_k12_masked_processed_and_partial(eng, oracle):
    _, _, sym = gi.pad_inputs(32, 40, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    mask[2] = 0
    proc[2] = proc[7] = 1
    on, od, gn, gd, _ = check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, K, 16, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert not gd[7].any() and not gd[2].any()
    basic = estimate(on, od, sym)
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, K, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0)
    # partial-window branch (pst != cst) on accumulators with holes
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    num, den = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, K, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    basic = estimate(num, den, sym)
    num, den = gi.partial_holes(num, den)
    proc[4] = 1
    for pst in (1, 6):
        pon = check_pass(eng, oracle, 1, sym, None, num, den, mask, proc, K, 16, oracle.ID, oracle.SADCT, oracle.HAAR, pst=pst, cst=4)[0]
        assert not np.array_equal(pon, num)
        check_pass(eng, oracle, 2, sym, basic, num, den, mask, proc, K, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, pst=pst, cst=4)


@pytest.mark.parametrize("aw,an,C,masked,t2", [(3, 1, 3, False, "id"), (3, 1, 3, False, "dct"), (3, 0, 3, False, "dct"),
                                                (3, 1, 1, True, "id")])
def test_complete_runs_k12(eng, oracle, aw, an, C, masked, t2):
    """Both steps at k = 12 through the host-buffer and the device-resident entry points, with the oracle's window schedule;
    grayscale with an empty centre SAI takes the partial-window branch."""
    import lfbm5d_b200 as L
    H, W = 32, 36
    clean = np.ascontiguousarray(lfdata.synth_lf(aw, aw, H, W)[:, :C])
    m = np.ones(aw * aw, np.uint32)
    if masked:
        m[(aw * aw) // 2] = 0
    T1 = L.ID if t2 == "id" else L.DCT
    p1 = L.make_params(25.0, 2.7, aw, aw, an, W, H, C, 8, 18, 6, K, 4, T1, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, aw, aw, an, W, H, C, 16, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
    noisy, sched, _, d, _, _ = check_complete_run(eng, oracle, clean, m, p1, p2)
    if masked:
        assert sched[:, 3].max() > 1
    psnr = psnr_on(clean, m)
    assert psnr(d) > psnr(noisy) + 3.0


@pytest.mark.parametrize("world,H,W", [(2, 200, 72), (3, 330, 64)])
def test_team_bit_identical_to_single_k12(oracle, world, H, W):
    import lfbm5d_b200 as L
    p1 = L.make_params(15.0, 2.7, 3, 3, 1, W, H, 3, 8, 18, 6, K, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, 3, 3, 1, W, H, 3, 16, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
    assert_team_matches_single(oracle, world, p1, p2)


def test_lfbm3d_k12(eng, oracle):
    """Per-SAI BM3D with kHard = kWien = 12 (dct / dct, the 12 x 12 Kaiser window in the aggregation) and a masked SAI."""
    import lfbm5d_b200 as L
    clean = lfdata.synth_lf(2, 2, 40, 48)
    noisy = oracle.add_noise(clean, 10.0)
    mask = np.ones(4, np.uint32)
    mask[3] = 0
    with oracle.sum_mode(1):
        ob, od, on = oracle.run_bm3d_lf(noisy, mask, 10.0, 16, 16, K, K, 16, 32, 3, 3, L.DCT, L.DCT, 2.7)
    prm = L.make_params3d(10.0, 4, 48, 40, 3, 16, 16, K, K, 16, 32, 3, 3, L.DCT, L.DCT, 2.7)
    gb, gd, gn = eng.bm3d(prm, noisy, mask)
    assert np.array_equal(gn, on)
    assert np.array_equal(gb[:3], ob[:3])                  # step 1: bit-exact
    assert np.abs(gd[:3] - od[:3]).max() <= 1e-3
    assert not gb[3].any() and not gd[3].any()
    assert oracle.psnr(gd[:3], clean[:3])[0] > oracle.psnr(noisy[:3], clean[:3])[0] + 4.0


@pytest.mark.parametrize("prog", ["LFBM5Ddenoising", "LFBM3Ddenoising"])
def test_command_lines_k12(tmp_path, prog):
    """Both command lines with k = 12 in both steps on a 3x3 light field of PNGs: the files are what the library gives."""
    import lfbm5d_b200 as L
    H, W = 40, 44
    clean = lfdata.synth_lf(3, 3, H, W)
    src = write_lf(tmp_path, clean, 3)
    dirs = [str(tmp_path / d) for d in ("noisyLF", "basicLF", "denoisedLF", "diffLF")]
    head = [os.path.join(LIBDIR, prog), str(src), "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "25", "2.7"] + dirs
    if prog == "LFBM5Ddenoising":
        tail = ["8", "18", "6", "12", "4", "id", "sadct", "haar", "0", "16", "18", "6", "12", "4", "dct", "sadct", "haar", "0"]
    else:
        tail = ["16", "16", "12", "3", "dct", "0", "32", "16", "12", "3", "dct", "0"]
    run_cli(head + tail + ["opp", "0", str(tmp_path / "objectiveResults.txt")])
    src8 = np.clip(np.floor(clean + 0.5), 0, 255).astype(np.float32)
    noisy = L.add_noise(src8, 25.0, seed0=20171016)
    mask = np.ones(9, np.uint32)
    e = L.LFBM5D(0)
    if prog == "LFBM5Ddenoising":
        p1 = L.make_params(25.0, 2.7, 3, 3, 1, W, H, 3, 8, 18, 6, K, 4, L.ID, L.SADCT, L.HAAR)
        p2 = L.make_params(25.0, 0.0, 3, 3, 1, W, H, 3, 16, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
        basic, n1 = e.step1(p1, noisy, mask)
        den, _, _ = e.step2(p2, n1, basic, mask)
    else:
        prm = L.make_params3d(25.0, 9, W, H, 3, 16, 16, K, K, 16, 32, 3, 3, L.DCT, L.DCT, 2.7)
        basic, den, _ = e.bm3d(prm, noisy, mask)
    e.close()
    check_pngs(tmp_path, (("noisyLF", noisy), ("basicLF", basic), ("denoisedLF", den)), 3)


def test_k12_parameter_errors_launch_nothing(eng):
    import lfbm5d_b200 as L
    noisy = np.zeros((25, 3, 40, 44), np.float32)
    mask = np.ones(25, np.uint32)
    assert_rejected(eng, [
        (lambda: eng.step1(L.make_params(25.0, 2.7, 3, 3, 1, 44, 40, 3, 8, 18, 6, K, 4, L.BIOR, L.SADCT, L.HAAR), noisy[:9], mask[:9]),
         "bior needs a power-of-two patch size"),
        (lambda: eng.step1(L.make_params(25.0, 2.7, 5, 5, 2, 44, 40, 3, 2, 18, 6, K, 4, L.ID, L.SADCT, L.HAAR), noisy, mask),
         "an = 2 is not supported at k = 12"),
        (lambda: eng.step2(L.make_params(25.0, 0.0, 3, 3, 1, 44, 40, 3, 32, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR), noisy[:9], noisy[:9], mask[:9]),
         "k = 12 needs N"),
        (lambda: eng.step1(L.make_params(25.0, 2.7, 3, 3, 1, 44, 40, 3, 8, 18, 6, 10, 4, L.ID, L.SADCT, L.HAAR), noisy[:9], mask[:9]),
         "patch size must be 8, 12 or 16"),
        (lambda: eng.bm3d(L.make_params3d(25.0, 9, 44, 40, 3, 16, 16, K, K, 16, 32, 3, 3, L.BIOR, L.DCT, 2.7), noisy[:9], mask[:9]),
         "bior needs a power-of-two patch size")])
