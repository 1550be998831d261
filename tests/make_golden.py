"""Generates tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref) in the build container.
Inputs are re-creatable anywhere from tests/lfdata.py + the oracle's mt19937ar noise, so only outputs are stored.
Run:  python tests/make_golden.py      (needs oracle/_ref built from the reference's sources; see oracle/Makefile)"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import lfdata  # noqa: E402
import oracleapi as O  # noqa: E402
import refapi as R  # noqa: E402

GOLD = os.path.join(HERE, "golden")


def pad_inputs(H, W, sigma, n=24):
    clean = lfdata.synth_lf(3, 3, H, W)
    noisy = O.add_noise(clean, sigma)
    y = noisy.copy()
    for st in range(9):
        O.lib().orc_color_space_transform(O.fp(y[st]), O.OPP, W, H, 3, 1)
    return clean, noisy, np.stack([O.symetrize(y[st], n) for st in range(9)])


def partial_holes(num, den):
    """Accumulators of a first core call with the weights of SAI 1 and 6 removed in places."""
    num, den = num.copy(), den.copy()
    num[1][:, 30:52, 28:70] = 0; den[1][:, 30:52, 28:70] = 0
    num[1][:, 60:, :40] = 0; den[1][:, 60:, :40] = 0
    num[6][:, :, 60:] = 0; den[6][:, :, 60:] = 0
    return num, den


def main():
    os.makedirs(GOLD, exist_ok=True)
    R.lib().ref_set_dct_mode(0)
    # 1. block matching on one padded channel-0 plane (README parameters of both steps)
    clean, noisy, sym = pad_inputs(40, 48, 25.0)
    img = sym[4, 0]
    out = {}
    for tag, (k, N, tau) in {"s1": (16, 8, 3000.0), "s2": (8, 16, 2000.0)}.items():
        cnt, idx = R.precompute_bm(img, k, N, 24, 18, 4, tau)
        sel = np.nonzero(cnt)[0]
        out["bm_%s_pos" % tag] = sel.astype(np.uint32)
        out["bm_%s_cnt" % tag] = cnt[sel]
        out["bm_%s_idx" % tag] = idx[sel]
        first, shape, _ = R.precompute_bm_stereo(img, sym[0, 0], k, 24, 6, tau)
        out["st_%s_first" % tag] = first
        out["st_%s_shape" % tag] = shape.astype(np.uint8)
    np.savez_compressed(os.path.join(GOLD, "bm_40x48.npz"), **out)
    # 2. one teacher-forced window pass per step, accumulators cropped to the unpadded interior
    z = np.zeros_like(sym)
    mask, proc = np.ones(9), np.zeros(9)
    n = 24
    crop = (slice(None), slice(None), slice(n, -n), slice(n, -n))
    out = {}
    rn, rd = R.pass_step1(sym, z, z, mask, proc, 4, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, R.ID, R.SADCT, R.HAAR)
    out["p1_num"], out["p1_den"] = rn[crop], rd[crop]
    est = np.where(rd != 0, rn / np.where(rd != 0, rd, 1), sym).astype(np.float32)
    rn2, rd2 = R.pass_step2(sym, est, z, z, mask, proc, 4, 4, 3, 25.0, 18, 6, 8, 16, 4, R.DCT, R.SADCT, R.HAAR)
    out["p2_num"], out["p2_den"] = rn2[crop], rd2[crop]
    rn3, rd3 = R.pass_step1(sym, z, z, mask, proc, 4, 4, 3, 25.0, 2.7, 18, 6, 16, 1, 4, R.BIOR, R.SADCT, R.HAAR)
    out["p1bior_num"], out["p1bior_den"] = rn3[crop], rd3[crop]
    np.savez_compressed(os.path.join(GOLD, "pass_40x48.npz"), **out)
    # 3. complete runs: 3x3 (one window pass per step) and 5x5 (five passes per step), README parameters; one file per run
    for tag, (aw, H, W) in {"3x3": (3, 32, 40), "5x5": (5, 24, 28)}.items():
        clean = lfdata.synth_lf(aw, aw, H, W)
        noisy = O.add_noise(clean, 25.0)
        mask = np.ones(aw * aw)
        b, nrt = R.run_step1(noisy, mask, 25.0, 2.7, aw, aw, 1, 8, 18, 6, 16, 4, R.ID, R.SADCT, R.HAAR)
        d, b2, _ = R.run_step2(nrt, b, mask, 25.0, aw, aw, 1, 16, 18, 6, 8, 4, R.DCT, R.SADCT, R.HAAR)
        out = {"basic_" + tag: b, "noisy_rt_" + tag: nrt, "denoised_" + tag: d, "basic_rt_" + tag: b2}
        np.savez_compressed(os.path.join(GOLD, "runs_%s.npz" % tag), **out)
    # 4. partial-window branch (pst != cst): one call per step on accumulators with holes, and complete grayscale runs
    #    (several core calls per window: LF_denoised_percent stays below 100 after the first SAI when C == 1)
    _, _, sym = pad_inputs(32, 40, 25.0)
    z = np.zeros_like(sym)
    out = {}
    num, den = R.pass_step1(sym, z, z, mask, proc, 4, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, R.ID, R.SADCT, R.HAAR)
    basic = np.where(den != 0, num / np.where(den != 0, den, 1), sym).astype(np.float32)
    num, den = partial_holes(num, den)
    p2 = proc.copy(); p2[4] = 1
    for pst in (1, 6):
        rn, rd = R.pass_step1(sym, num, den, mask, p2, 4, pst, 3, 25.0, 2.7, 18, 6, 16, 8, 4, R.ID, R.SADCT, R.HAAR)
        out["s1_pst%d_num" % pst], out["s1_pst%d_den" % pst] = rn[pst], rd[pst]
        rn, rd = R.pass_step2(sym, basic, num, den, mask, p2, 4, pst, 3, 25.0, 18, 6, 8, 16, 4, R.DCT, R.SADCT, R.HAAR)
        out["s2_pst%d_num" % pst], out["s2_pst%d_den" % pst] = rn[pst], rd[pst]
    for tag, (aw, H, W) in {"g3x3": (3, 28, 32), "g5x5": (5, 24, 28)}.items():
        clean = np.ascontiguousarray(lfdata.synth_lf(aw, aw, H, W)[:, :1])
        noisy = O.add_noise(clean, 25.0)
        m = np.ones(aw * aw)
        b, nrt = R.run_step1(noisy, m, 25.0, 2.7, aw, aw, 1, 8, 18, 6, 16, 4, R.ID, R.SADCT, R.HAAR)
        d, _, _ = R.run_step2(nrt, b, m, 25.0, aw, aw, 1, 16, 18, 6, 8, 4, R.DCT, R.SADCT, R.HAAR)
        out["basic_" + tag], out["denoised_" + tag] = b, d
    np.savez_compressed(os.path.join(GOLD, "partial.npz"), **out)
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == "__main__":
    main()
