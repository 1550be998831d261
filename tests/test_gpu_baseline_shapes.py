"""GPU parity at the shapes BASELINE.json names (run with -m gpu): block matching on full 1072x1072 planes (17x17x1024^2
configs: every strip hand-off, every wrap of the 128-row shared-memory ring, full-length candidate lists), teacher-forced
window passes at the config-1 size and on a wide plane, and the reference's own fixture (configs[0]) against vectors produced
by the unmodified reference. Bars as in gpucheck.py: match lists / disparity matches / step-1 accumulators bit-exact,
step 2 within 2e-5 relative per pass, complete single-window runs within 1e-3 absolute and 0.01 dB."""
import os

import numpy as np
import pytest

from gpucheck import channel0_planes, check_bm, check_pass, eng, estimate  # noqa: F401 (eng is the engine fixture)

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_block_matching_full_planes(eng, oracle):
    """1072x1072 planes, both README parameter sets (k = 16 / N = 8 / tau 3000 and k = 8 / N = 16 / tau 2000): counts, ordered
    lists, argmin and shape flags bit-exact; 64,009 / 65,025 reference patches as SURVEY 8 states."""
    H = W = 1024
    planes = channel0_planes(oracle, H, W, 10.0, 3)
    assert planes.shape == (3, 1072, 1072)
    r1, _ = check_bm(eng, oracle, planes, 1, 16, 8, 3000.0)
    r2, _ = check_bm(eng, oracle, planes, 2, 8, 16, 2000.0)
    assert (r1, r2) == (64009, 65025)
    # quantised input without noise: exact distance ties along the mirror axes and in flat regions, resolved like libstdc++'s
    # partial_sort / sort (rare at this size: the float32 summed-area sums of a flat patch are not exactly equal)
    q = channel0_planes(oracle, H, W, 0.0, 2, quantise=True)
    _, nties = check_bm(eng, oracle, q, 1, 16, 8, 3000.0)
    assert nties > 0


def test_pass_ring_wrap_and_strips(eng, oracle):
    """SAIs of 120 x 150: 168 padded rows (the 128-row ring of k_sat2 wraps, K mirror slots in use), 5 / 6 strips with CTA-to-CTA
    hand-off, several chunks with the boundary prefetch; teacher-forced both steps."""
    import golden_inputs as gi
    _, _, sym = gi.pad_inputs(120, 150, 25.0)
    assert sym.shape[2] >= 160
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    on, od = check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR)[:2]
    basic = estimate(on, od, sym)
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0)
    # narrow search window with a large patch: more self strips than disparity strips share the hand-off buffers
    _, _, sym2 = gi.pad_inputs(40, 65, 25.0, n=7)
    z2 = np.zeros_like(sym2)
    check_pass(eng, oracle, 1, sym2, None, z2, z2, mask, proc, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR, nSim=2, nDisp=5)
    check_pass(eng, oracle, 1, sym2, None, z2, z2, mask, proc, 8, 2, oracle.DCT, oracle.DCT, oracle.HAAR, nSim=3, nDisp=4)


def test_pass_config1_shape_and_wide_plane(eng, oracle):
    """Teacher-forced passes of both steps at the config-1 size (3x3 SAIs of 256^2, sigma 25) and on 1024-wide SAIs (33 strips,
    the full row length of configs[2], 208 padded rows), README parameters."""
    import golden_inputs as gi
    for (H, W, sigma) in ((256, 256, 25.0), (160, 1024, 10.0)):
        _, _, sym = gi.pad_inputs(H, W, sigma)
        z = np.zeros_like(sym)
        mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
        on, od = check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, sigma=sigma)[:2]
        basic = estimate(on, od, sym)
        check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, sigma=sigma, lam=0.0)


def test_pass_full_size_window(eng, oracle):
    """One teacher-forced window pass per step on 3x3 SAIs of 1024^2 (configs[2] / configs[3] SAI size; 9 x 3 planes of 1072^2,
    64,009 / 65,025 groups): match tables and step-1 accumulators bit-exact, step 2 within 2e-5 relative."""
    import golden_inputs as gi
    _, _, sym = gi.pad_inputs(1024, 1024, 10.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    on, od = check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, sigma=10.0)[:2]
    basic = estimate(on, od, sym)
    del on, od
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, sigma=10.0, lam=0.0)


def test_config1_fixture_against_reference(eng, oracle):
    """BASELINE.json configs[0]: the reference's fixture testing/sourceLF with mt19937ar noise (seed 20171016 + st), README.md:50
    parameters, through the host-buffer entry points; against tiles and PSNRs produced by the unmodified reference
    (tests/make_golden_config1.py)."""
    import golden_inputs as gi
    import lfbm5d_b200 as L
    g = np.load(os.path.join(GOLD, "config1.npz"))
    clean = gi.config1_fixture().astype(np.float32)
    noisy = oracle.add_noise(clean, 25.0)
    mask = np.ones(9, np.uint32)
    p1 = L.make_params(25.0, 2.7, 3, 3, 1, 256, 256, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, 3, 3, 1, 256, 256, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    b, nrt = eng.step1(p1, noisy, mask)
    assert len(eng.schedule()) == 1
    d, _, _ = eng.step2(p2, nrt, b, mask)
    tiles = {"centre": (slice(96, 160), slice(96, 160)), "corner": (slice(0, 40), slice(0, 40)), "edge": (slice(216, 256), slice(100, 164))}
    sais = [0, 4, 8]
    assert np.array_equal(nrt[sais][:, :, 96:160, 96:160], g["noisy_rt_centre"])
    for name, (ys, xs) in tiles.items():
        assert np.array_equal(b[sais][:, :, ys, xs], g["basic_" + name]), name      # step 1 is bit-identical to the reference's
        # step 2: the Wiener weight sum is reduced in another order (last-bit weights); one window, no re-matching
        assert np.abs(d[sais][:, :, ys, xs] - g["denoised_" + name]).max() <= 1e-3, name
    dp_b = oracle.psnr(b, clean)[0] - float(g["psnr_basic"])
    dp_d = oracle.psnr(d, clean)[0] - float(g["psnr_denoised"])
    assert abs(dp_b) <= 1e-6 and abs(dp_d) <= 0.01, (dp_b, dp_d)
