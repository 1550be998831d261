"""The CPU oracle against golden vectors produced by the unmodified reference (tests/make_golden.py): bit-exact."""
import os

import numpy as np

import golden_inputs as gi

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_block_matching_golden(oracle):
    g = np.load(os.path.join(GOLD, "bm_40x48.npz"))
    _, _, sym = gi.pad_inputs(40, 48, 25.0)
    img = sym[4, 0]
    for tag, (k, N, tau) in {"s1": (16, 8, 3000.0), "s2": (8, 16, 2000.0)}.items():
        cnt, idx = oracle.bm_self(img, k, N, 24, 18, 4, tau)
        sel = np.nonzero(cnt)[0]
        assert np.array_equal(sel, g["bm_%s_pos" % tag]) and np.array_equal(cnt[sel], g["bm_%s_cnt" % tag])
        m = np.arange(N + 1)[None, :] < cnt[sel][:, None]
        assert np.array_equal(idx[sel] * m, g["bm_%s_idx" % tag] * m)
        first, shape, _ = oracle.bm_stereo(img, sym[0, 0], k, 24, 6, tau)
        assert np.array_equal(first, g["st_%s_first" % tag]) and np.array_equal(shape.astype(np.uint8), g["st_%s_shape" % tag])


def test_pass_golden(oracle):
    g = np.load(os.path.join(GOLD, "pass_40x48.npz"))
    _, _, sym = gi.pad_inputs(40, 48, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9), np.zeros(9)
    crop = (slice(None), slice(None), slice(24, -24), slice(24, -24))
    on, od = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(on[crop], g["p1_num"]) and np.array_equal(od[crop], g["p1_den"])
    est = np.where(od != 0, on / np.where(od != 0, od, 1), sym).astype(np.float32)
    on2, od2 = oracle.run_pass(2, sym, est, z, z, mask, proc, 4, 3, 25.0, 0.0, 18, 6, 8, 16, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(on2[crop], g["p2_num"]) and np.array_equal(od2[crop], g["p2_den"])
    on3, od3 = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, 16, 1, 4, oracle.BIOR, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(on3[crop], g["p1bior_num"]) and np.array_equal(od3[crop], g["p1bior_den"])


def test_runs_golden(oracle):
    for tag, npass in (("3x3", 1), ("5x5", 5)):
        g = np.load(os.path.join(GOLD, "runs_%s.npz" % tag))
        aw, clean, noisy = gi.run_inputs(tag)
        mask = np.ones(aw * aw)
        b, nrt, sch = oracle.run_step1(noisy, mask, 25.0, 2.7, aw, aw, 1, 8, 18, 6, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
        assert len(sch) == npass and all(int(e[3]) == 1 for e in sch)      # one core call per window (SURVEY A1)
        assert np.array_equal(b, g["basic_" + tag]) and np.array_equal(nrt, g["noisy_rt_" + tag])
        d, b2, _, sch2 = oracle.run_step2(nrt, b, mask, 25.0, aw, aw, 1, 16, 18, 6, 8, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
        assert np.array_equal(d, g["denoised_" + tag]) and np.array_equal(b2, g["basic_rt_" + tag])
        assert np.array_equal(sch, sch2)


def test_partial_window_golden(oracle):
    """`pst != cst` branch (core:531-821 / :1332-1658) against vectors of the unmodified reference: single calls on
    accumulators with holes, and a complete grayscale run (several core calls per window)."""
    import lfdata
    g = np.load(os.path.join(GOLD, "partial.npz"))
    _, _, sym = gi.pad_inputs(32, 40, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9), np.zeros(9)
    num, den = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    basic = np.where(den != 0, num / np.where(den != 0, den, 1), sym).astype(np.float32)
    num, den = gi.partial_holes(num, den)
    p2 = proc.copy(); p2[4] = 1
    for pst in (1, 6):
        on, od = oracle.run_pass(1, sym, None, num, den, mask, p2, pst, 3, 25.0, 2.7, 18, 6, 16, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR, cst=4)
        assert np.array_equal(on[pst], g["s1_pst%d_num" % pst]) and np.array_equal(od[pst], g["s1_pst%d_den" % pst])
        on, od = oracle.run_pass(2, sym, basic, num, den, mask, p2, pst, 3, 25.0, 0.0, 18, 6, 8, 16, 4, oracle.DCT, oracle.SADCT, oracle.HAAR, cst=4)
        assert np.array_equal(on[pst], g["s2_pst%d_num" % pst]) and np.array_equal(od[pst], g["s2_pst%d_den" % pst])
    clean = np.ascontiguousarray(lfdata.synth_lf(3, 3, 28, 32)[:, :1])
    noisy = oracle.add_noise(clean, 25.0)
    b, nrt, sch = oracle.run_step1(noisy, np.ones(9), 25.0, 2.7, 3, 3, 1, 8, 18, 6, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert int(sch[0][3]) == 2
    assert np.array_equal(b, g["basic_g3x3"])
    d, _, _, _ = oracle.run_step2(nrt, b, np.ones(9), 25.0, 3, 3, 1, 16, 18, 6, 8, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(d, g["denoised_g3x3"])


def test_schedule_pass_counts(oracle):
    """Window passes per step with an = 1 (SURVEY A1): 1 (3x3), 16 (9x9) — exercised on tiny SAIs for speed."""
    import lfdata
    clean = lfdata.synth_lf(9, 9, 12, 12)
    noisy = oracle.add_noise(clean, 10.0)
    b, nrt, sch = oracle.run_step1(noisy, np.ones(81), 10.0, 2.7, 9, 9, 1, 2, 2, 1, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert len(sch) == 16 and int(sch[0][0]) == 40 and int(sch[1][0]) == 80
    assert sorted(set(int(e[0]) for e in sch)) == sorted(int(e[0]) for e in sch)


def test_config1_fixture_golden(oracle):
    """BASELINE.json configs[0] (the reference's fixture, README.md:50 parameters): the oracle reproduces the unmodified reference's
    basic and denoised estimates bit for bit (tiles + PSNRs of tests/golden/config1.npz, tests/make_golden_config1.py). The fixture's
    pixels are stored losslessly as tests/golden/sourceLF/SAI_<s>_<t>.png."""
    g = np.load(os.path.join(GOLD, "config1.npz"))
    clean = gi.config1_fixture().astype(np.float32)
    noisy = oracle.add_noise(clean, 25.0)
    mask = np.ones(9)
    b, nrt, sched = oracle.run_step1(noisy, mask, 25.0, 2.7, 3, 3, 1, 8, 18, 6, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    d, _, _, _ = oracle.run_step2(nrt, b, mask, 25.0, 3, 3, 1, 16, 18, 6, 8, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
    assert len(sched) == 1
    sais = [0, 4, 8]
    tiles = {"centre": (slice(96, 160), slice(96, 160)), "corner": (slice(0, 40), slice(0, 40)), "edge": (slice(216, 256), slice(100, 164))}
    for name, (ys, xs) in tiles.items():
        assert np.array_equal(b[sais][:, :, ys, xs], g["basic_" + name]), name
        assert np.array_equal(d[sais][:, :, ys, xs], g["denoised_" + name]), name
    assert oracle.psnr(b, clean)[0] == float(g["psnr_basic"]) and oracle.psnr(d, clean)[0] == float(g["psnr_denoised"])
    # the reference's own sensitivity to the unpinned FFTW arithmetic (double-accumulating stand-in): the noise floor of dPSNR
    assert abs(float(g["psnr_denoised_f64dct"]) - float(g["psnr_denoised"])) < 0.01
