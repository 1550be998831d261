"""5x5 angular search windows (an = 2) on the GPU, through the C ABI against the CPU oracle (which runs the same asw-generic code
that is pinned against the reference at an = 1, with its asw = 5 tables pinned). Tolerances are those of gpucheck.py: match lists,
disparity argmin and shape flags bit-exact; step 1 bit-identical (ordered aggregation); step 2 within 2e-5 relative, 1e-3
absolute after normalisation (reduction order of the Wiener weight sum); with useSD 1e-4 relative (the group's standard deviation
is reduced over 25 N k^2 values in another order than the oracle's serial sum). Complete runs: LF_basic bit-identical; LF_denoised
within 0.01 dB, and within 1e-3 absolute for a single core call (later core calls block-match on a running estimate that differs in
the last bits and match lists flip, as in test_gpu_parity.py)."""
import os

import numpy as np
import pytest

import lfdata
from gpucheck import (EST_ABS, LIBDIR, assert_rejected, assert_team_matches_single, check_complete_run, check_pass, check_pngs,
                      eng, estimate, pad_inputs5, run_cli, write_lf)  # noqa: F401 (eng is the engine fixture)

pytestmark = pytest.mark.gpu


def test_an2_single_passes(eng, oracle):
    import lfbm5d_b200 as L
    prm = L.make_params(25.0, 0.0, 5, 5, 2, 48, 40, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    assert eng.group_kernel(1, prm) == "k_groups25<1>" and eng.group_kernel(2, prm) == "k_groups25<2>"
    sym = pad_inputs5(oracle, 40, 48, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(25, np.uint32), np.zeros(25, np.uint32)
    on, od, _, _, _ = check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, an=2)
    for (k, N, t2, t4, t5) in [(8, 16, oracle.DCT, oracle.DCT, oracle.HADAMARD), (16, 1, oracle.BIOR, oracle.SADCT, oracle.HAAR),
                               (8, 32, oracle.BIOR, oracle.DCT, oracle.HAAR), (16, 8, oracle.ID, oracle.SADCT, oracle.DCT)]:
        check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, k, N, t2, t4, t5, an=2)
    check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, 8, 16, oracle.DCT, oracle.DCT, oracle.DCT, useSD=1, an=2)
    basic = estimate(on, od, sym)
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, an=2)
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, 16, 4, oracle.BIOR, oracle.DCT, oracle.HADAMARD, lam=0.0, an=2)
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.DCT, lam=0.0, useSD=1, an=2)
    # second pass of step 1 on top of the accumulators of the first
    check_pass(eng, oracle, 1, sym, None, on, od, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, an=2)


def test_an2_empty_and_processed_sais(eng, oracle):
    """Empty SAIs anywhere in the 5x5 window force 25-bit SA-DCT shapes in every group; processed SAIs are matched, not aggregated."""
    sym = pad_inputs5(oracle, 32, 40, 25.0)
    sym[3][:, :, :40] += 120.0          # a brightness step: some disparity matches fail tauMatch (shape flag 0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(25, np.uint32), np.zeros(25, np.uint32)
    mask[[2, 11, 23]] = 0
    proc[[2, 7, 19]] = 1
    on, od, _, _, _ = check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, an=2)
    assert not od[7].any() and not od[2].any() and od[12].any()
    basic = estimate(on, od, sym)
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, an=2)


def test_an2_pass_large_sais(eng, oracle):
    """SAIs of 256 x 320: the strip ring of the summed-area planes wraps, several strips per plane."""
    sym = pad_inputs5(oracle, 256, 320, 20.0, C=1)
    z = np.zeros_like(sym)
    mask, proc = np.ones(25, np.uint32), np.zeros(25, np.uint32)
    check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, sigma=20.0, an=2)


@pytest.mark.parametrize("aw,H,W,C,masked", [(5, 24, 28, 3, False), (7, 24, 28, 3, False), (7, 24, 28, 1, True)])
def test_an2_complete_runs(eng, oracle, aw, H, W, C, masked):
    """Both steps through the host-buffer entry points and the device-resident ones. Grayscale with an empty centre SAI takes the
    partial-window branch (several core calls per window)."""
    import lfbm5d_b200 as L
    clean = np.ascontiguousarray(lfdata.synth_lf(aw, aw, H, W)[:, :C])
    m = np.ones(aw * aw, np.uint32)
    if masked:
        m[(aw * aw) // 2] = 0
    p1 = L.make_params(25.0, 2.7, aw, aw, 2, W, H, C, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, aw, aw, 2, W, H, C, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    _, sched, sched2, d, dd, od = check_complete_run(eng, oracle, clean, m, p1, p2, calls_only=True)
    if masked:
        assert sched[:, 3].max() > 1
    if len(sched2) == 1 and sched2[0, 3] == 1:
        assert np.abs(d[m == 1] - od[m == 1]).max() <= EST_ABS
        assert np.abs(dd[m == 1] - od[m == 1]).max() <= EST_ABS


@pytest.mark.parametrize("world,H,W", [(2, 200, 64), (3, 330, 56)])
def test_an2_team_bit_identical_to_single(oracle, world, H, W):
    import lfbm5d_b200 as L
    p1 = L.make_params(15.0, 2.7, 5, 5, 2, W, H, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, 5, 5, 2, W, H, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    assert_team_matches_single(oracle, world, p1, p2)


def test_an2_command_line(tmp_path):
    """LFBM5Ddenoising with asw_size_ht = asw_size_wien = 2 on a 5x5 light field of PNGs: the files are what the library gives."""
    import lfbm5d_b200 as L
    clean = lfdata.synth_lf(5, 5, 48, 56)
    src = write_lf(tmp_path, clean, 5)
    run_cli([os.path.join(LIBDIR, "LFBM5Ddenoising"), str(src), "SAI", "_", "5", "5", "1", "1", "2", "2", "row", "25", "2.7",
             str(tmp_path / "noisyLF"), str(tmp_path / "basicLF"), str(tmp_path / "denoisedLF"), str(tmp_path / "diffLF"),
             "8", "18", "6", "16", "4", "id", "sadct", "haar", "0", "16", "18", "6", "8", "4", "dct", "sadct", "haar", "0",
             "opp", "0", str(tmp_path / "objectiveResults.txt")])
    src8 = np.clip(np.floor(clean + 0.5), 0, 255).astype(np.float32)
    noisy = L.add_noise(src8, 25.0, seed0=20171016)
    mask = np.ones(25, np.uint32)
    e = L.LFBM5D(0)
    p1 = L.make_params(25.0, 2.7, 5, 5, 2, 56, 48, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, 5, 5, 2, 56, 48, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    basic, n1 = e.step1(p1, noisy, mask)
    den, _, _ = e.step2(p2, n1, basic, mask)
    e.close()
    check_pngs(tmp_path, (("noisyLF", noisy), ("basicLF", basic), ("denoisedLF", den)), 5)


def test_an2_parameter_errors_launch_nothing(eng):
    import lfbm5d_b200 as L
    noisy = np.zeros((49, 3, 24, 28), np.float32)
    mask = np.ones(49, np.uint32)
    p = L.make_params(25.0, 2.7, 7, 7, 3, 28, 24, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, 7, 7, 2, 28, 24, 3, 8, 18, 6, 16, 4, L.DCT, L.SADCT, L.HAAR)
    assert_rejected(eng, [(lambda: eng.step1(p, noisy, mask), "an > 2"), (lambda: eng.step2(p2, noisy, noisy, mask), "2048")])
