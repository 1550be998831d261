"""Pins the CPU oracle (oracle/lfbm5d_oracle.c) against the UNMODIFIED reference: every comparison here is bit-exact. Where
oracle/_ref is built (oracle/Makefile) the reference runs live; elsewhere the oracle's values are checked against the stored
digests of the reference's values on the same seeded inputs (tests/golden/ref_pins.json, refapi.Pinned)."""
import ctypes as C

import numpy as np
import pytest

import golden_inputs as gi
import lfdata

pytestmark = pytest.mark.filterwarnings("ignore")


def prep(oracle, H, W, sigma=25.0, n=24, aw=3, ah=3):
    clean = lfdata.synth_lf(aw, ah, H, W)
    noisy = oracle.add_noise(clean, sigma)
    y = noisy.copy()
    for st in range(aw * ah):
        oracle.lib().orc_color_space_transform(oracle.fp(y[st]), oracle.OPP, W, H, 3, 1)
    return clean, noisy, np.stack([oracle.symetrize(y[st], n) for st in range(aw * ah)])


def masked(cnt, idx):
    """Self-match lists with the entries past each count zeroed (they are not part of the result)."""
    return cnt, idx * (np.arange(idx.shape[1])[None, :] < cnt[:, None])


def test_rng_and_noise(oracle, ref):
    oracle.lib().orc_mt_seed(20171016)
    got = np.array([oracle.lib().orc_mt_res53() for _ in range(3000)])

    def want(R):
        R.lib().ref_mt_seed(20171016)
        return np.array([R.lib().ref_mt_res53() for _ in range(3000)])
    ref.check("rng", got, want)


def test_small_helpers(oracle, ref):
    for (m, N, s) in [(289, 24, 4), (1057, 24, 4), (652, 21, 3), (100, 6, 1), (300, 16, 3)]:
        b = np.zeros(2000, np.uint32)
        nb = oracle.lib().orc_ind_initialize(oracle.up(b), m, N, s)

        def want(R):
            a = np.zeros(2000, np.uint32)
            na = R.lib().ref_ind_initialize(R.up(a), m, N, s)
            return na, a[:na]
        ref.check("ind_initialize_%d_%d_%d" % (m, N, s), (nb, b[:nb]), want)
    for k in (4, 8, 12, 16):
        o = [np.zeros(k * k, np.float32) for _ in range(3)]
        oracle.lib().orc_preProcess(*[oracle.fp(x) for x in o], k)

        def want(R):
            r = [np.zeros(k * k, np.float32) for _ in range(3)]
            R.lib().ref_preProcess(*[R.fp(x) for x in r], k)
            return r
        ref.check("preProcess_%d" % k, o, want)
    for a in (1, 3, 5):
        o = [np.zeros(a * a, np.float32) for _ in range(2)]
        oracle.lib().orc_preProcess_4d(oracle.fp(o[0]), oracle.fp(o[1]), a, a)

        def want(R):
            r = [np.zeros(a * a, np.float32) for _ in range(2)]
            R.lib().ref_preProcess_4d(R.fp(r[0]), R.fp(r[1]), a, a)
            return r
        ref.check("preProcess_4d_%d" % a, o, want)
        if a > 1:
            o = [np.zeros(a * a, np.float32) for _ in range(2)]
            oracle.lib().orc_preProcess_4d_sadct(oracle.fp(o[0]), oracle.fp(o[1]), a)

            def want(R):
                r = [np.zeros(a * a, np.float32) for _ in range(2)]
                R.lib().ref_preProcess_4d_sadct(R.fp(r[0]), R.fp(r[1]), a)
                return r
            ref.check("preProcess_4d_sadct_%d" % a, o, want)
    for cs in (oracle.YUV, oracle.YCBCR, oracle.OPP, oracle.RGB):
        o = np.zeros(3, np.float32)
        oracle.lib().orc_estimate_sigma(C.c_float(10.0), oracle.fp(o), 3, cs)

        def want(R):
            r = np.zeros(3, np.float32)
            R.lib().ref_estimate_sigma(C.c_float(10.0), R.fp(r), 3, cs)
            return r
        ref.check("estimate_sigma_%d" % cs, o, want)
    rng = np.random.RandomState(1)
    img = (rng.rand(3, 20, 24) * 255).astype(np.float32)
    for cs in (oracle.YUV, oracle.YCBCR, oracle.OPP):
        for fwd in (1, 0):
            b = img.copy()
            oracle.lib().orc_color_space_transform(oracle.fp(b), cs, 24, 20, 3, fwd)

            def want(R):
                a = img.copy()
                R.lib().ref_color_space_transform(R.fp(a), cs, 24, 20, 3, fwd)
                return a
            ref.check("color_space_transform_%d_%d" % (cs, fwd), b, want)

    def want(R):
        s1 = np.zeros((3, 20 + 14, 24 + 14), np.float32)
        R.lib().ref_symetrize(R.fp(img), R.fp(s1), 24, 20, 3, 7)
        return s1
    ref.check("symetrize", oracle.symetrize(img, 7), want)
    for (aidx, asize) in [(0, 17), (8, 17), (16, 17), (1, 3), (4, 5)]:
        oa = [C.c_int() for _ in range(3)]
        oracle.lib().orc_angular_search_window(*[C.byref(x) for x in oa], aidx, asize, 1)

        def want(R):
            ra = [C.c_int() for _ in range(3)]
            R.lib().ref_angular_search_window(*[C.byref(x) for x in ra], aidx, asize, 1)
            return np.array([x.value for x in ra])
        ref.check("angular_search_window_%d_%d" % (aidx, asize), np.array([x.value for x in oa]), want)


def test_transform_primitives(oracle, ref):
    rng = np.random.RandomState(2)
    for N in (2, 4, 8, 16, 32):
        v = rng.randn(N).astype(np.float32) * 50
        for fr, fo in (("ref_haar_forward", "orc_haar_forward"), ("ref_haar_inverse", "orc_haar_inverse"), ("ref_hadamard", "orc_hadamard")):
            b = v.copy()
            getattr(oracle.lib(), fo)(oracle.fp(b), N)

            def want(R):
                a = v.copy()
                getattr(R.lib(), fr)(R.fp(a), N)
                return a
            ref.check("%s_%d" % (fr, N), b, want)
    for k in (8, 16):
        p = (rng.rand(k * k) * 255).astype(np.float32)
        b = np.zeros_like(p)
        oracle.lib().orc_bior_2d_forward(oracle.fp(p), oracle.fp(b), k)
        b_fwd = b.copy()
        oracle.lib().orc_bior_2d_inverse(oracle.fp(b), k)

        def want(R):
            a = np.zeros_like(p)
            R.lib().ref_bior_2d_forward(R.fp(p), R.fp(a), k)
            a_fwd = a.copy()
            R.lib().ref_bior_2d_inverse(R.fp(a), k)
            return a_fwd, a
        ref.check("bior_2d_%d" % k, (b_fwd, b), want)     # (the reference's bior pair is not a perfect-reconstruction pair on random data)
        for mode in (0, 1):
            oracle.set_dct_mode(mode)
            b = np.zeros_like(p)
            oracle.lib().orc_dct_2d_forward(oracle.fp(p), oracle.fp(b), k)
            b_fwd = b.copy()
            oracle.lib().orc_dct_2d_inverse(oracle.fp(b), k)
            assert np.abs(b - p).max() < 1e-2     # known answer: round trip

            def want(R):
                R.lib().ref_set_dct_mode(mode)
                a = np.zeros_like(p)
                R.lib().ref_dct_2d_patch(R.fp(p), R.fp(a), k)
                a_fwd = a.copy()
                R.lib().ref_dct_2d_inverse_patch(R.fp(a), k)
                R.lib().ref_set_dct_mode(0)
                return a_fwd, a
            ref.check("dct_2d_%d_mode%d" % (k, mode), (b_fwd, b), want)
        oracle.set_dct_mode(0)


def test_block_matching_lists_bit_exact(oracle, ref):
    clean, noisy, sym = prep(oracle, 128, 144)
    img = sym[4, 0]
    c2, i2 = oracle.bm_self(img, 16, 8, 24, 18, 4, 3000.0)
    ref.check("bm_self", masked(c2, i2), lambda R: masked(*R.precompute_bm(img, 16, 8, 24, 18, 4, 3000.0)))
    assert (c2 > 0).sum() > 500
    # flat image: every distance ties -> libstdc++ heap/sort order decides
    flat = np.full_like(img, 7.0)
    c2, i2 = oracle.bm_self(flat, 8, 16, 24, 18, 4, 2000.0)
    ref.check("bm_self_flat", masked(c2, i2), lambda R: masked(*R.precompute_bm(flat, 8, 16, 24, 18, 4, 2000.0)))
    nties = 0
    for st in (0, 8):
        f2, s2, ties = oracle.bm_stereo(img, sym[st, 0], 16, 24, 6, 3000.0)
        ref.check("bm_stereo_%d" % st, (f2, s2), lambda R: R.precompute_bm_stereo(img, sym[st, 0], 16, 24, 6, 3000.0)[:2])
        nties += int(ties.sum())
    f2, s2, ties = oracle.bm_stereo(flat, flat, 8, 24, 6, 2000.0)
    ref.check("bm_stereo_flat", (f2, s2), lambda R: R.precompute_bm_stereo(flat, flat, 8, 24, 6, 2000.0)[:2])
    assert ties.sum() > 1000


def test_std_sort_emulation(oracle, ref):
    # ties everywhere: quantised distances
    rng = np.random.RandomState(3)
    img1 = np.round(rng.rand(70, 80) * 3).astype(np.float32)
    img2 = np.round(rng.rand(70, 80) * 3).astype(np.float32)
    f2, s2, ties = oracle.bm_stereo(img1, img2, 8, 24, 6, 2000.0)
    assert ties.sum() > 100
    ref.check("sort_bm_stereo", (f2, s2), lambda R: R.precompute_bm_stereo(img1, img2, 8, 24, 6, 2000.0, want_all=True)[:2])
    c2, i2 = oracle.bm_self(img1, 8, 16, 24, 18, 4, 2000.0)
    ref.check("sort_bm_self", masked(c2, i2), lambda R: masked(*R.precompute_bm(img1, 8, 16, 24, 18, 4, 2000.0)))


@pytest.mark.parametrize("mode", [0, 1])
def test_single_pass_bit_exact(oracle, ref, mode):
    clean, noisy, sym = prep(oracle, 40, 48)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9), np.zeros(9)
    O = oracle

    def live(fn):
        def want(R):
            R.lib().ref_set_dct_mode(mode)
            try:
                return fn(R)
            finally:
                R.lib().ref_set_dct_mode(0)
        return want
    oracle.set_dct_mode(mode)
    try:
        for (k, N, t2, t4, t5) in [(16, 8, O.ID, O.SADCT, O.HAAR), (16, 1, O.BIOR, O.SADCT, O.HAAR),
                                   (8, 16, O.DCT, O.DCT, O.HADAMARD), (8, 8, O.ID, O.ID, O.HAAR)]:
            on, od = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, k, N, 4, t2, t4, t5)
            ref.check("pass1_m%d_%d_%d_%d_%d_%d" % (mode, k, N, t2, t4, t5), (on, od),
                      live(lambda R: R.pass_step1(sym, z, z, mask, proc, 4, 4, 3, 25.0, 2.7, 18, 6, k, N, 4, t2, t4, t5)))
        est = np.where(od != 0, on / np.where(od != 0, od, 1), sym).astype(np.float32)
        for t5 in (O.HAAR, O.HADAMARD):
            on2, od2 = oracle.run_pass(2, sym, est, z, z, mask, proc, 4, 3, 25.0, 0.0, 18, 6, 8, 16, 4, O.DCT, O.SADCT, t5)
            ref.check("pass2_m%d_%d" % (mode, t5), (on2, od2),
                      live(lambda R: R.pass_step2(sym, est, z, z, mask, proc, 4, 4, 3, 25.0, 18, 6, 8, 16, 4, O.DCT, O.SADCT, t5)))
        # an empty SAI in the window forces the shape-adaptive path for every group; a processed SAI is not aggregated
        mask2, proc2 = mask.copy(), proc.copy()
        mask2[2] = 0
        proc2[2] = 1
        proc2[7] = 1
        on, od = oracle.run_pass(1, sym, None, z, z, mask2, proc2, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, O.ID, O.SADCT, O.HAAR)
        ref.check("pass1_m%d_masked" % mode, (on, od),
                  live(lambda R: R.pass_step1(sym, z, z, mask2, proc2, 4, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, O.ID, O.SADCT, O.HAAR)))
        on2, od2 = oracle.run_pass(2, sym, est, on, od, mask2, proc2, 4, 3, 25.0, 0.0, 18, 6, 8, 16, 4, O.DCT, O.SADCT, O.HAAR)
        ref.check("pass2_m%d_masked" % mode, (on2, od2),
                  live(lambda R: R.pass_step2(sym, est, on, od, mask2, proc2, 4, 4, 3, 25.0, 18, 6, 8, 16, 4, O.DCT, O.SADCT, O.HAAR)))
    finally:
        oracle.set_dct_mode(0)


def test_full_run_multi_pass_bit_exact(oracle, ref):
    clean = lfdata.synth_lf(5, 5, 32, 40)
    noisy = oracle.add_noise(clean, 25.0)
    mask = np.ones(25)
    ob, on, sch = oracle.run_step1(noisy, mask, 25.0, 2.7, 5, 5, 1, 8, 18, 6, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert len(sch) == 5
    ref.check("run_step1_5x5", (ob, on), lambda R: R.run_step1(noisy, mask, 25.0, 2.7, 5, 5, 1, 8, 18, 6, 16, 4, R.ID, R.SADCT, R.HAAR))
    od, ob2, on2, sch = oracle.run_step2(on, ob, mask, 25.0, 5, 5, 1, 16, 18, 6, 8, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
    ref.check("run_step2_5x5", (od, ob2, on2), lambda R: R.run_step2(on, ob, mask, 25.0, 5, 5, 1, 16, 18, 6, 8, 4, R.DCT, R.SADCT, R.HAAR))
    assert oracle.psnr(od, clean)[0] > oracle.psnr(ob, clean)[0] > oracle.psnr(noisy, clean)[0] + 5


def test_lfbm3d_bit_exact(oracle, ref):
    """bm3d_LF path (config 4 parameters): A = 1 specialisation with BM3D's thresholds."""
    clean = lfdata.synth_lf(2, 1, 36, 44)
    noisy = oracle.add_noise(clean, 10.0)
    mask = np.ones(2)
    for (t2h, t2w) in ((oracle.BIOR, oracle.DCT), (oracle.DCT, oracle.BIOR)):
        got = oracle.run_bm3d_lf(noisy, mask, 10.0, 16, 16, 8, 8, 16, 32, 3, 3, t2h, t2w, 2.7)
        ref.check("bm3d_lf_%d_%d" % (t2h, t2w), got, lambda R: R.run_bm3d_lf(noisy, mask, 10.0, 16, 16, 8, 8, 16, 32, 3, 3, t2h, t2w, 2.7))


def test_partial_window_branch_bit_exact(oracle, ref):
    """`pst != cst` (core:531-821 / :1332-1658): single calls on accumulators with holes, and a complete grayscale run where
    every window takes several core calls (LF_denoised_percent < 100 after the first SAI when C == 1)."""
    _, _, sym = gi.pad_inputs(32, 40, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    num, den = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    basic = np.where(den != 0, num / np.where(den != 0, den, 1), sym).astype(np.float32)
    num, den = gi.partial_holes(num, den)
    p2 = proc.copy(); p2[4] = 1
    for pst in (1, 6, 3):
        on, od = oracle.run_pass(1, sym, None, num, den, mask, p2, pst, 3, 25.0, 2.7, 18, 6, 8, 4, 4, oracle.BIOR, oracle.DCT, oracle.HAAR, cst=4)
        ref.check("partial_s1_pst%d" % pst, (on, od),
                  lambda R: R.pass_step1(sym, num, den, mask, p2, 4, pst, 3, 25.0, 2.7, 18, 6, 8, 4, 4, R.BIOR, R.DCT, R.HAAR))
        assert np.array_equal(on, num) == (pst == 3)          # SAI 3 has no holes: nothing to do
        on, od = oracle.run_pass(2, sym, basic, num, den, mask, p2, pst, 3, 25.0, 0.0, 18, 6, 8, 8, 4, oracle.DCT, oracle.SADCT, oracle.HAAR, cst=4)
        ref.check("partial_s2_pst%d" % pst, (on, od),
                  lambda R: R.pass_step2(sym, basic, num, den, mask, p2, 4, pst, 3, 25.0, 18, 6, 8, 8, 4, R.DCT, R.SADCT, R.HAAR))
    clean = np.ascontiguousarray(lfdata.synth_lf(3, 3, 24, 28)[:, :1])
    noisy = oracle.add_noise(clean, 25.0)
    m = np.ones(9, np.uint32)
    m[4] = 0                                                      # empty centre SAI: already the first call is partial
    ob, on_, sched = oracle.run_step1(noisy, m, 25.0, 2.7, 3, 3, 1, 8, 18, 6, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert int(sched[0][3]) > 1
    ref.check("partial_gray_run_step1", ob, lambda R: R.run_step1(noisy, m, 25.0, 2.7, 3, 3, 1, 8, 18, 6, 16, 4, R.ID, R.SADCT, R.HAAR)[0])


def test_5d_dct_and_sd_weighting_bit_exact(oracle, ref):
    """tau_5D = dct (core:2524-2700 / :2943-3130) and useSD (core:3140-3173; bm3d.cpp:1345-1372 incl. its channel-0 quirk)."""
    _, _, sym = gi.pad_inputs(28, 32, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    num, den = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    basic = np.where(den != 0, num / np.where(den != 0, den, 1), sym).astype(np.float32)
    for (step, k, N, t2, t4, t5, sd) in [(1, 16, 8, oracle.ID, oracle.SADCT, oracle.DCT, 0), (2, 8, 16, oracle.DCT, oracle.SADCT, oracle.DCT, 0),
                                         (1, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, 1), (2, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, 1)]:
        oracle.lib().orc_set_use_sd(sd)
        try:
            on, od = oracle.run_pass(step, sym, basic if step == 2 else None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, k, N, 4, t2, t4, t5)
        finally:
            oracle.lib().orc_set_use_sd(0)

        def want(R):
            if step == 1:
                return R.pass_step1(sym, z, z, mask, proc, 4, 4, 3, 25.0, 2.7, 18, 6, k, N, 4, t2, t4, t5, useSD=bool(sd))
            return R.pass_step2(sym, basic, z, z, mask, proc, 4, 4, 3, 25.0, 18, 6, k, N, 4, t2, t4, t5, useSD=bool(sd))
        ref.check("pass%d_tau5_%d_sd%d" % (step, t5, sd), (on, od), want)
    clean = lfdata.synth_lf(1, 1, 36, 40)
    noisy = oracle.add_noise(clean, 20.0)
    one = np.ones(1, np.uint32)
    oracle.lib().orc_set_use_sd(1)
    try:
        ob, od, _ = oracle.run_bm3d_lf(noisy, one, 20.0, 16, 16, 8, 8, 16, 32, 3, 3, oracle.BIOR, oracle.DCT, 2.7)
    finally:
        oracle.lib().orc_set_use_sd(0)

    def want(R):
        n = noisy.copy(); rb = np.zeros_like(n); rden = np.zeros_like(n)
        assert R.lib().ref_run_bm3d_LF(C.c_float(20.0), R.fp(n), R.up(R.u32(one)), R.fp(rb), R.fp(rden), 1, 40, 36, 3, 16, 16, 8, 8, 16, 32, 3, 3,
                                       1, 1, R.BIOR, R.DCT, C.c_float(2.7), R.OPP, 1) == 0
        return rb, rden
    ref.check("bm3d_lf_sd", (ob, od), want)
