"""Noise-level estimate (lfbm5d_estimate_sigma, csrc/noise_estimate.cuh) on the GPU: bit-exact against the NumPy restatement of
its definition, through the host and the device entry points; its accuracy on synthetic light fields; `sigma = auto` on both
command lines; and the rejected arguments."""
import os
import re

import numpy as np
import pytest

import lfdata
from gpucheck import LIBDIR, assert_rejected, check_pngs, eng, run_cli, write_lf  # noqa: F401

SIGMA_DIV = np.float32(0.6744897501960817)


# -- the definition, restated ---------------------------------------------------------------------------------------------------

def keys(lf):
    """|finest diagonal Haar detail| of every 2 x 2 block: [..., H/2, W/2] float32 (an odd last row / column is dropped)."""
    h2, w2 = lf.shape[-2] // 2 * 2, lf.shape[-1] // 2 * 2
    x = lf[..., :h2, :w2]
    return np.abs(((x[..., 0::2, 0::2] - x[..., 0::2, 1::2]) - (x[..., 1::2, 0::2] - x[..., 1::2, 1::2])) * np.float32(0.5))


def mad_sigma(k):
    """Lower median (rank (n - 1) / 2) of the keys over 0.6744897501960817f, one float division."""
    k = k.ravel()
    r = (k.size - 1) // 2
    return np.float32(np.partition(k, r)[r]) / SIGMA_DIV


def expected(lf, mask):
    k = keys(np.ascontiguousarray(lf, np.float32))
    on = np.asarray(mask) != 0
    chnl = np.array([mad_sigma(k[on][:, c]) for c in range(lf.shape[1])], np.float32)
    sai = np.array([mad_sigma(k[st]) if on[st] else 0.0 for st in range(lf.shape[0])], np.float32)
    return mad_sigma(k[on]), chnl, sai


# -- checks ---------------------------------------------------------------------------------------------------------------------

def check_exact(eng, lf, mask):
    """Host and device entry points equal the restatement bit for bit (pooled, per channel, per SAI), leave their input as it was and
    launch their kernels through the context (6 per call)."""
    import torch
    lf = np.ascontiguousarray(lf, np.float32)
    mask = np.asarray(mask, np.uint32)
    want = expected(lf, mask)
    before = lf.copy()
    eng.reset_stats()
    got = eng.estimate_sigma(lf, mask)
    assert eng.stats().kernel_launches == 6
    assert np.array_equal(lf, before)
    d = torch.from_numpy(lf).cuda()
    dgot = eng.estimate_sigma_device(d.data_ptr(), mask, *lf.shape[:2], lf.shape[3], lf.shape[2])
    assert torch.equal(d.cpu(), torch.from_numpy(before))
    for g in (got, dgot):
        assert np.float32(g[0]) == want[0], (g[0], want[0])
        assert np.array_equal(g[1], want[1]), (g[1], want[1])
        assert np.array_equal(g[2], want[2])
    return got


def noisy_lf(aw, h, w, sigma, c=3, seed=12345):
    import lfbm5d_b200 as L
    return L.add_noise(lfdata.synth_lf(aw, aw, h, w, C=c, seed=seed), sigma)


@pytest.mark.gpu
@pytest.mark.parametrize("aw,h,w,c", [(5, 37, 53, 3), (3, 64, 64, 1), (17, 24, 20, 3), (3, 1024, 1024, 3)])
def test_bit_exact_shapes(eng, aw, h, w, c):
    """Odd sizes (a row and a column dropped), grey, many SAIs of a few blocks each, and planes of 512^2 blocks whose pooled and
    per-channel segments are fed by hundreds of CTAs."""
    lf = noisy_lf(aw, h, w, 10.0, c)
    check_exact(eng, lf, np.ones(aw * aw, np.uint32))


@pytest.mark.gpu
def test_bit_exact_masks_ties_constant_and_range(eng):
    lf = noisy_lf(5, 40, 48, 15.0)
    mask = np.ones(25, np.uint32)
    mask[[0, 7, 12, 24]] = 0                          # the centre among them
    _, _, sai = check_exact(eng, lf, mask)
    assert (sai[mask == 0] == 0).all() and (sai[mask == 1] > 0).all()
    # integer-valued input (what the command lines read): keys are multiples of 0.5, massive ties at every rank
    q = np.clip(np.floor(lf + np.float32(0.5)), 0, 255).astype(np.float32)
    s, _, _ = check_exact(eng, q, np.ones(25, np.uint32))
    m = np.float32(s) * SIGMA_DIV
    assert m * 2 == np.round(m * 2)
    # a constant light field: every key is 0
    s, chnl, sai = check_exact(eng, np.full((9, 3, 16, 16), 77.0, np.float32), np.ones(9, np.uint32))
    assert s == 0 and (chnl == 0).all() and (sai == 0).all()
    # unclipped values far below 0 and above 255
    wide = noisy_lf(3, 32, 40, 30.0) * np.float32(4) - np.float32(500)
    assert wide.min() < -300 and wide.max() > 400
    check_exact(eng, wide, np.ones(9, np.uint32))


@pytest.mark.gpu
def test_sai_permutation(eng):
    """Permuting the SAIs permutes sigma_sai and changes neither the pooled nor the per-channel values."""
    lf = noisy_lf(5, 32, 32, 12.0)
    mask = np.ones(25, np.uint32)
    mask[3] = 0
    perm = np.random.default_rng(5).permutation(25)
    s0, c0, a0 = eng.estimate_sigma(lf, mask)
    s1, c1, a1 = eng.estimate_sigma(lf[perm], mask[perm])
    assert s0 == s1 and np.array_equal(c0, c1) and np.array_equal(a0[perm], a1)


@pytest.mark.gpu
@pytest.mark.parametrize("sigma", [5, 10, 25, 50])
def test_accuracy(eng, sigma):
    """Within 5 % on 5x5x128^2 with the reference's noise, as floats and as 8-bit PNGs hold them (rounded, clipped). Measured with the
    restatement: +2.2 / +0.6 / +0.1 / -0.0 % for floats and +3.8 / +3.8 / +0.8 / -2.2 % for 8-bit at sigma 5 / 10 / 25 / 50 (texture
    biases low sigmas up, clipping biases sigma 50 down)."""
    lf = noisy_lf(5, 128, 128, float(sigma))
    q = np.clip(np.floor(lf + np.float32(0.5)), 0, 255).astype(np.float32)
    mask = np.ones(25, np.uint32)
    for x in (lf, q):
        s, chnl, sai = eng.estimate_sigma(x, mask)
        assert abs(s / sigma - 1) < 0.05, (sigma, s)
        assert np.float32(s) == expected(x, mask)[0]


def cli_args(driver, src, tmp_path):
    dirs = [str(src)] + [str(tmp_path / d) for d in ("basicLF", "denoisedLF", "diffLF")]
    args = [os.path.join(LIBDIR, driver), "none", "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "auto", "2.7"] + dirs
    if driver == "LFBM5Ddenoising":
        args += ["8", "18", "6", "16", "4", "id", "sadct", "haar", "0", "16", "18", "6", "8", "4", "dct", "sadct", "haar", "0"]
    else:
        args += ["16", "16", "8", "3", "bior", "0", "32", "16", "8", "3", "dct", "0"]
    return args + ["opp", "0", str(tmp_path / "results.txt")]


@pytest.mark.gpu
@pytest.mark.parametrize("driver", ["LFBM5Ddenoising", "LFBM3Ddenoising"])
def test_cli_sigma_auto(eng, tmp_path, driver):
    """`sigma = auto` without ground truth: the printed sigma is estimate_sigma of the 8-bit light field the command line read, and
    the written basic and denoised light fields are what the library gives at that float."""
    import lfbm5d_b200 as L
    noisy8 = np.clip(np.floor(noisy_lf(3, 64, 72, 20.0) + np.float32(0.5)), 0, 255).astype(np.float32)
    src = write_lf(tmp_path, noisy8, 3)
    out = run_cli(cli_args(driver, src, tmp_path))
    mask = np.ones(9, np.uint32)
    s, chnl, _ = eng.estimate_sigma(noisy8, mask)
    m = re.search(r"Estimated noise level: sigma = (\S+) \(per channel: (\S+) (\S+) (\S+)\)", out)
    assert m, out[-2000:]
    assert np.float32(m.group(1)) == np.float32(s) and [np.float32(v) for v in m.groups()[1:]] == list(chnl)
    assert abs(s / 20.0 - 1) < 0.05
    if driver == "LFBM5Ddenoising":
        p1 = L.make_params(s, 2.7, 3, 3, 1, 72, 64, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
        p2 = L.make_params(s, 0.0, 3, 3, 1, 72, 64, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
        basic, n1 = eng.step1(p1, noisy8, mask)
        den, _, _ = eng.step2(p2, n1, basic, mask)
    else:
        basic, den, _ = eng.bm3d(L.make_params3d(s, 9, 72, 64, 3, 16, 16, 8, 8, 16, 32, 3, 3, L.BIOR, L.DCT, 2.7), noisy8, mask)
    check_pngs(tmp_path, (("basicLF", basic), ("denoisedLF", den)), 3)


@pytest.mark.gpu
def test_rejections(eng):
    import torch
    d = torch.zeros(9 * 3 * 8 * 8, device="cuda")
    ones, z = np.ones(9, np.uint32), np.zeros((9, 3, 8, 8), np.float32)
    assert_rejected(eng, [
        (lambda: eng.estimate_sigma(np.zeros((9, 2, 8, 8), np.float32), ones), "chnls must be 1 or 3"),
        (lambda: eng.estimate_sigma(np.zeros((9, 3, 8, 1), np.float32), ones), "at least 2 x 2"),
        (lambda: eng.estimate_sigma(np.zeros((9, 3, 1, 8), np.float32), ones), "at least 2 x 2"),
        (lambda: eng.estimate_sigma(np.zeros((0, 3, 8, 8), np.float32), np.zeros(0, np.uint32)), "asize = 0"),
        (lambda: eng.estimate_sigma(z, np.zeros(9, np.uint32)), "every SAI is masked"),
        (lambda: eng.estimate_sigma_device(d.data_ptr(), ones, 9, 4, 8, 6), "chnls must be 1 or 3"),
        (lambda: eng.estimate_sigma_device(d.data_ptr(), ones, 9, 3, 1, 64), "at least 2 x 2"),
        (lambda: eng.estimate_sigma_device(d.data_ptr(), ones, 9, 3, 64, 1), "at least 2 x 2"),
        (lambda: eng.estimate_sigma_device(d.data_ptr(), np.zeros(0, np.uint32), 0, 3, 8, 8), "asize = 0"),
        (lambda: eng.estimate_sigma_device(d.data_ptr(), np.zeros(9, np.uint32), 9, 3, 8, 8), "every SAI is masked"),
        (lambda: eng.estimate_sigma_device(0, ones, 9, 3, 8, 8), "null argument"),
    ])
