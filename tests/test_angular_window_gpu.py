"""5x5 angular search windows (an = 2) on the GPU, through the C ABI against the CPU oracle (which runs the same asw-generic code
that is pinned against the reference at an = 1, with its asw = 5 tables pinned). Tolerances as in test_gpu_parity.py: match lists,
disparity argmin and shape flags bit-exact; step 1 bit-identical (ordered aggregation); step 2 within 2e-5 relative, 1e-3
absolute after normalisation (reduction order of the Wiener weight sum); with useSD 1e-4 relative (the group's standard deviation
is reduced over 25 N k^2 values in another order than the oracle's serial sum). Complete runs: LF_basic bit-identical; LF_denoised
within 0.01 dB, and within 1e-3 absolute for a single core call (later core calls block-match on a running estimate that differs in
the last bits and match lists flip, as in test_gpu_parity.py)."""
import os
import subprocess

import numpy as np
import pytest

import lfdata

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "lfbm5d_b200", "_lib")


@pytest.fixture(scope="module")
def eng():
    import lfbm5d_b200 as L
    e = L.LFBM5D(0)
    yield e
    e.close()


def estimate(num, den, sub):
    return np.where(den != 0, num / np.where(den != 0, den, 1), sub).astype(np.float32)


def pad_inputs5(oracle, H, W, sigma, n=24, C=3):
    clean = lfdata.synth_lf(5, 5, H, W)[:, :C]
    noisy = oracle.add_noise(np.ascontiguousarray(clean), sigma)
    y = noisy.copy()
    if C == 3:
        for st in range(25):
            oracle.lib().orc_color_space_transform(oracle.fp(y[st]), oracle.OPP, W, H, 3, 1)
    return np.stack([oracle.symetrize(y[st], n) for st in range(25)])


def check_pass5(eng, oracle, step, sym, basic, num0, den0, mask, proc, k, N, t2, t4, t5, sigma=25.0, lam=2.7, nSim=18, nDisp=6, p=4,
                useSD=0):
    import lfbm5d_b200 as L
    A, C, hb, wb = sym.shape
    H, W = hb - 2 * (nSim + nDisp), wb - 2 * (nSim + nDisp)
    oracle.lib().orc_set_use_sd(int(useSD))
    try:
        on, od, odbg = oracle.run_pass(step, sym, basic, num0, den0, mask, proc, 12, 5, sigma, lam, nSim, nDisp, k, N, p, t2, t4, t5, debug=True)
    finally:
        oracle.lib().orc_set_use_sd(0)
    prm = L.make_params(sigma, lam, 5, 5, 2, W, H, C, N, nSim, nDisp, k, p, t2, t4, t5, useSD=int(useSD))
    gn, gd, gdbg = eng.debug_pass(step, prm, sym, basic, num0, den0, mask, proc, 12, debug=True)
    assert np.array_equal(odbg[0], gdbg[0]), "self-match counts differ"
    m = np.arange(N + 1)[None, :] < odbg[0][:, None]
    assert np.array_equal(odbg[1] * m, gdbg[1] * m), "self-match lists differ"
    assert np.array_equal(odbg[2], gdbg[2]), "disparity argmin differs"
    assert np.array_equal(odbg[3], gdbg[3]), "shape flags differ"
    if step == 1 and not useSD:
        assert np.array_equal(gn, on) and np.array_equal(gd, od)
    else:
        assert np.array_equal(od != 0, gd != 0)
        sub = sym if step == 1 else basic
        assert np.abs(estimate(on, od, sub) - estimate(gn, gd, sub)).max() <= 1e-3
        rel = 1e-4 if useSD else 2e-5
        assert np.abs(gn - on).max() <= rel * np.abs(on).max() and np.abs(gd - od).max() <= rel * np.abs(od).max()
    return on, od


def test_an2_single_passes(eng, oracle):
    sym = pad_inputs5(oracle, 40, 48, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(25, np.uint32), np.zeros(25, np.uint32)
    on, od = check_pass5(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR)
    for (k, N, t2, t4, t5) in [(8, 16, oracle.DCT, oracle.DCT, oracle.HADAMARD), (16, 1, oracle.BIOR, oracle.SADCT, oracle.HAAR),
                               (8, 32, oracle.BIOR, oracle.DCT, oracle.HAAR), (16, 8, oracle.ID, oracle.SADCT, oracle.DCT)]:
        check_pass5(eng, oracle, 1, sym, None, z, z, mask, proc, k, N, t2, t4, t5)
    check_pass5(eng, oracle, 1, sym, None, z, z, mask, proc, 8, 16, oracle.DCT, oracle.DCT, oracle.DCT, useSD=1)
    basic = estimate(on, od, sym)
    check_pass5(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0)
    check_pass5(eng, oracle, 2, sym, basic, z, z, mask, proc, 16, 4, oracle.BIOR, oracle.DCT, oracle.HADAMARD, lam=0.0)
    check_pass5(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.DCT, lam=0.0, useSD=1)
    # second pass of step 1 on top of the accumulators of the first
    check_pass5(eng, oracle, 1, sym, None, on, od, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR)


def test_an2_empty_and_processed_sais(eng, oracle):
    """Empty SAIs anywhere in the 5x5 window force 25-bit SA-DCT shapes in every group; processed SAIs are matched, not aggregated."""
    sym = pad_inputs5(oracle, 32, 40, 25.0)
    sym[3][:, :, :40] += 120.0          # a brightness step: some disparity matches fail tauMatch (shape flag 0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(25, np.uint32), np.zeros(25, np.uint32)
    mask[[2, 11, 23]] = 0
    proc[[2, 7, 19]] = 1
    on, od = check_pass5(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert not od[7].any() and not od[2].any() and od[12].any()
    basic = estimate(on, od, sym)
    check_pass5(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0)


def test_an2_pass_large_sais(eng, oracle):
    """SAIs of 256 x 320: the strip ring of the summed-area planes wraps, several strips per plane."""
    sym = pad_inputs5(oracle, 256, 320, 20.0, C=1)
    z = np.zeros_like(sym)
    mask, proc = np.ones(25, np.uint32), np.zeros(25, np.uint32)
    check_pass5(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, sigma=20.0)


@pytest.mark.parametrize("aw,H,W,C,masked", [(5, 24, 28, 3, False), (7, 24, 28, 3, False), (7, 24, 28, 1, True)])
def test_an2_complete_runs(eng, oracle, aw, H, W, C, masked):
    """Both steps through the host-buffer entry points and the device-resident ones. Grayscale with an empty centre SAI takes the
    partial-window branch (several core calls per window)."""
    import torch
    import lfbm5d_b200 as L
    clean = np.ascontiguousarray(lfdata.synth_lf(aw, aw, H, W)[:, :C])
    noisy = oracle.add_noise(clean, 25.0)
    m = np.ones(aw * aw, np.uint32)
    if masked:
        m[(aw * aw) // 2] = 0
    p1 = L.make_params(25.0, 2.7, aw, aw, 2, W, H, C, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, aw, aw, 2, W, H, C, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    b, nrt = eng.step1(p1, noisy, m)
    ob, onrt, sched = oracle.run_step1(noisy, m, 25.0, 2.7, aw, aw, 2, 8, 18, 6, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert len(eng.schedule()) == len(sched) and np.array_equal(eng.schedule()[:, 3], sched[:, 3])
    if masked:
        assert sched[:, 3].max() > 1
    assert np.array_equal(nrt[m == 1], onrt[m == 1])
    assert np.array_equal(b[m == 1], ob[m == 1])                                 # step 1 is bit-identical
    d, _, _ = eng.step2(p2, nrt, b, m)
    # both sides start step 2 from the same colour-round-tripped noisy light field and the same basic estimate
    od, _, _, sched2 = oracle.run_step2(nrt, ob, m, 25.0, aw, aw, 2, 16, 18, 6, 8, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
    assert len(eng.schedule()) == len(sched2) and np.array_equal(eng.schedule()[:, 3], sched2[:, 3])
    c1 = clean[m == 1]
    psnr = lambda x: 10.0 * np.log10(255.0 ** 2 / np.mean((x - c1) ** 2))
    diff = np.abs(d[m == 1] - od[m == 1])
    assert abs(psnr(d[m == 1]) - psnr(od[m == 1])) <= 0.01, (psnr(d[m == 1]), psnr(od[m == 1]))
    if len(sched2) == 1 and sched2[0, 3] == 1:
        assert diff.max() <= 1e-3, diff.max()
    # device-resident entry points (the light field travels in place: noisy comes back colour-round-tripped after step 1)
    dev = torch.device("cuda", 0)
    w = torch.from_numpy(noisy.copy()).to(dev)
    bd, dd = torch.zeros_like(w), torch.zeros_like(w)
    eng.step1_device(p1, w.data_ptr(), m, bd.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(bd.cpu().numpy()[m == 1], ob[m == 1])
    eng.step2_device(p2, w.data_ptr(), bd.data_ptr(), m, dd.data_ptr())
    dd = dd.cpu().numpy()
    assert abs(psnr(dd[m == 1]) - psnr(od[m == 1])) <= 0.01
    if len(sched2) == 1 and sched2[0, 3] == 1:
        assert np.abs(dd[m == 1] - od[m == 1]).max() <= 1e-3


@pytest.mark.parametrize("world,H,W", [(2, 200, 64), (3, 330, 56)])
def test_an2_team_bit_identical_to_single(oracle, world, H, W):
    import torch
    import lfbm5d_b200 as L
    from test_team_gpu import run_single, run_team
    dev = torch.device("cuda", 0)
    clean = lfdata.synth_lf(5, 5, H, W)
    noisy = torch.from_numpy(oracle.add_noise(np.ascontiguousarray(clean), 15.0)).to(dev)
    mask = np.ones(25, np.uint32)
    p1 = L.make_params(15.0, 2.7, 5, 5, 2, W, H, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, 5, 5, 2, W, H, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    e = L.LFBM5D(0)
    w0, b0, o0, s0 = run_single(L, e, torch, noisy, mask, p1, p2)
    e.close()
    ws, bs, outs, bands1, bands2, st = run_team(L, torch, world, noisy, mask, p1, p2, gather=1)
    assert st["bytes_exchanged"] > 0
    for g in range(world):
        assert torch.equal(bs[g], b0) and torch.equal(outs[g], o0) and torch.equal(ws[g], w0)


def test_an2_command_line(tmp_path):
    """LFBM5Ddenoising with asw_size_ht = asw_size_wien = 2 on a 5x5 light field of PNGs: the files are what the library gives."""
    from PIL import Image
    import lfbm5d_b200 as L
    clean = lfdata.synth_lf(5, 5, 48, 56)
    src = tmp_path / "sourceLF"
    for d in ("sourceLF", "noisyLF", "basicLF", "denoisedLF", "diffLF"):
        (tmp_path / d).mkdir()
    for s in range(5):
        for t in range(5):
            img = np.clip(np.floor(clean[s * 5 + t] + 0.5), 0, 255).astype(np.uint8).transpose(1, 2, 0)
            Image.fromarray(img).save(str(src / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))
    report = tmp_path / "objectiveResults.txt"
    args = [os.path.join(LIBDIR, "LFBM5Ddenoising"), str(src), "SAI", "_", "5", "5", "1", "1", "2", "2", "row", "25", "2.7",
            str(tmp_path / "noisyLF"), str(tmp_path / "basicLF"), str(tmp_path / "denoisedLF"), str(tmp_path / "diffLF"),
            "8", "18", "6", "16", "4", "id", "sadct", "haar", "0", "16", "18", "6", "8", "4", "dct", "sadct", "haar", "0",
            "opp", "0", str(report)]
    env = dict(os.environ, LFBM5D_SEED="20171016")
    p = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, timeout=300)
    out = p.stdout.decode()
    assert p.returncode == 0, out[-2000:]
    src8 = np.clip(np.floor(clean + 0.5), 0, 255).astype(np.float32)
    noisy = L.add_noise(src8, 25.0, seed0=20171016)
    mask = np.ones(25, np.uint32)
    e = L.LFBM5D(0)
    p1 = L.make_params(25.0, 2.7, 5, 5, 2, 56, 48, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, 5, 5, 2, 56, 48, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    basic, n1 = e.step1(p1, noisy, mask)
    den, _, _ = e.step2(p2, n1, basic, mask)
    e.close()
    for s in range(5):
        for t in range(5):
            st = s * 5 + t
            for d, arr in (("noisyLF", noisy), ("basicLF", basic), ("denoisedLF", den)):
                img = np.asarray(Image.open(str(tmp_path / d / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))).transpose(2, 0, 1)
                assert np.array_equal(img, np.clip(np.floor(arr[st] + np.float32(0.5)), 0, 255).astype(np.uint8)), (d, st)


def test_an2_parameter_errors_launch_nothing(eng):
    import lfbm5d_b200 as L
    noisy = np.zeros((49, 3, 24, 28), np.float32)
    mask = np.ones(49, np.uint32)
    eng.reset_stats()
    p = L.make_params(25.0, 2.7, 7, 7, 3, 28, 24, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    with pytest.raises(RuntimeError, match="an > 2"):
        eng.step1(p, noisy, mask)
    p2 = L.make_params(25.0, 0.0, 7, 7, 2, 28, 24, 3, 8, 18, 6, 16, 4, L.DCT, L.SADCT, L.HAAR)
    with pytest.raises(RuntimeError, match="2048"):
        eng.step2(p2, noisy, noisy, mask)
    assert eng.stats().kernel_launches == 0
