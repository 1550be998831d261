"""Disparity search windows wider than nDisp = 6 (up to 16) on the GPU, through the C ABI against the CPU oracle. The oracle's
disparity matching is generic in nDisp but pinned against the reference only at nDisp = 6, so these results are checked GPU vs
oracle. Tolerances are those of test_gpu_parity.py / test_angular_window_gpu.py: match lists, disparity argmin and shape flags
bit-exact; step 1 bit-identical; step 2 within 2e-5 relative per pass; complete runs: LF_basic bit-identical, LF_denoised within
0.01 dB, and within 1e-3 where the run is one window of one core call (later windows block-match on a running estimate that
differs in the last bits, so match lists flip).

Above nDisp = 6 the disparity sums buffer holds fewer slots than a window has (csrc/lfbm5d_cuda.cu, stereo_buffer_slots) and a pass
runs its slots in chunks. The parity, complete-run and team tests assert that their passes cross at least one chunk boundary."""
import os
import subprocess

import numpy as np
import pytest

import lfdata
from test_angular_window_gpu import check_pass5, pad_inputs5
from test_gpu_baseline_shapes import channel0_planes
from test_gpu_parity import check_pass, estimate

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "lfbm5d_b200", "_lib")


def buffer_slots(an, nDisp):
    """Stereo slots of the sums buffer: floor((A - 1) * 169 / (2 nDisp + 1)^2), at least 1, at most A - 1."""
    a1 = (2 * an + 1) ** 2 - 1
    return min(a1, max(1, a1 * 169 // (2 * nDisp + 1) ** 2))


@pytest.fixture(scope="module")
def eng():
    import lfbm5d_b200 as L
    e = L.LFBM5D(0)
    yield e
    e.close()


# README parameter sets per step: (k, N, tauMatch); the library derives tauMatch from the step (RGB, sigma < 35, core:146 / :915)
BM_STEP = {1: (16, 8, 3000.0), 2: (8, 16, 2000.0)}


def check_bm(eng, oracle, planes, nDisp, W, H, step=1, self_too=True):
    """debug_block_matching against orc_bm_self / orc_bm_stereo; returns the number of tied disparity minima the oracle saw."""
    import lfbm5d_b200 as L
    k, N, tau = BM_STEP[step]
    n = 18 + nDisp
    prm = L.make_params(10.0, 2.7, 3, 3, 1, W, H, 3, N, 18, nDisp, k, 4, L.ID if step == 1 else L.DCT, L.SADCT, L.HAAR)
    cnt, idx, first, shape = eng.debug_block_matching(step, prm, planes)
    if self_too:
        ocnt, oidx = oracle.bm_self(planes[0], k, N, n, 18, 4, tau)
        assert np.array_equal(cnt, ocnt), "self-match counts differ"
        m = np.arange(N + 1)[None, :] < ocnt[:, None]
        assert np.array_equal(idx * m, oidx * m), "self-match lists differ"
    nties = 0
    for s in range(1, planes.shape[0]):
        of, osh, oties = oracle.bm_stereo(planes[0], planes[s], k, n, nDisp, tau)
        assert np.array_equal(first[s], of), "disparity argmin differs (nDisp %d, plane %d)" % (nDisp, s)
        assert np.array_equal(shape[s], osh), "shape flags differ (nDisp %d, plane %d)" % (nDisp, s)
        nties += int(oties.sum())
    return nties


@pytest.mark.parametrize("nDisp", [7, 8, 12, 16])
def test_block_matching_wide_disparity(eng, oracle, nDisp):
    """Nine planes (eight disparity slots, one to four chunks), a padded row pitch that is a multiple of 16 B (TMA loads) and one
    that is not (cp.async), noisy and quantised noise-free input (tied minima along the mirror axes and in flat regions)."""
    n = 18 + nDisp
    assert buffer_slots(1, nDisp) < 8
    w_tma = 48 - (2 * n) % 4                 # (w_tma + 2 n) floats per padded row: a multiple of 16 B
    for W in (w_tma, w_tma + 1):
        H = 40
        check_bm(eng, oracle, channel0_planes(oracle, H, W, 10.0, 9, n=n), nDisp, W, H, step=1)
        q = channel0_planes(oracle, H, W, 0.0, 9, n=n, quantise=True)
        assert check_bm(eng, oracle, q, nDisp, W, H, step=2) > 0


def test_block_matching_full_plane_ndisp16(eng, oracle):
    """One 1072 x 1072 plane pair at nDisp = 16: 33 disparity strips with CTA-to-CTA hand-off, the 128-row ring wraps, and each of
    the 33 row offsets takes three groups of 11 column offsets."""
    H = W = 1004
    planes = channel0_planes(oracle, H, W, 10.0, 2, n=34)
    assert planes.shape == (2, 1072, 1072)
    check_bm(eng, oracle, planes, 16, W, H, self_too=False)


@pytest.mark.parametrize("nDisp", [8, 12])
def test_single_passes_an1(eng, oracle, nDisp):
    import golden_inputs as gi
    n = 18 + nDisp
    assert buffer_slots(1, nDisp) < 8
    _, _, sym = gi.pad_inputs(40, 48, 25.0, n=n)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    on, od, gn, gd = check_pass(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, nDisp=nDisp)
    assert np.array_equal(gn, on) and np.array_equal(gd, od)              # step 1: bit-identical
    basic = estimate(on, od, sym)
    check_pass(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, nDisp=nDisp)
    # partial-window branch (pst != cst): holes in the accumulators of SAI 1 and 6
    num, den = gi.partial_holes(on, od)
    pr = proc.copy()
    pr[4] = 1
    import lfbm5d_b200 as L
    prm = L.make_params(25.0, 2.7, 3, 3, 1, 48, 40, 3, 8, 18, nDisp, 16, 4, L.ID, L.SADCT, L.HAAR)
    for pst in (1, 6):
        pon, pod = oracle.run_pass(1, sym, None, num, den, mask, pr, pst, 3, 25.0, 2.7, 18, nDisp, 16, 8, 4, oracle.ID, oracle.SADCT,
                                   oracle.HAAR, cst=4)
        pgn, pgd = eng.debug_pass(1, prm, sym, None, num, den, mask, pr, pst, cst=4)
        assert not np.array_equal(pgn, num)
        assert np.array_equal(pgn, pon) and np.array_equal(pgd, pod)


@pytest.mark.parametrize("nDisp", [8, 12])
def test_single_passes_an2(eng, oracle, nDisp):
    n = 18 + nDisp
    assert buffer_slots(2, nDisp) < 24
    sym = pad_inputs5(oracle, 32, 40, 25.0, n=n)
    z = np.zeros_like(sym)
    mask, proc = np.ones(25, np.uint32), np.zeros(25, np.uint32)
    on, od = check_pass5(eng, oracle, 1, sym, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR, nDisp=nDisp)
    basic = estimate(on, od, sym)
    check_pass5(eng, oracle, 2, sym, basic, z, z, mask, proc, 8, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, nDisp=nDisp)


@pytest.mark.parametrize("aw,an,C,masked", [(3, 1, 3, False), (7, 2, 3, False), (3, 1, 1, True)])
def test_complete_runs_ndisp10(eng, oracle, aw, an, C, masked):
    """Both steps at nDisp = 10 through the host-buffer and the device-resident entry points; grayscale with an empty centre SAI
    takes the partial-window branch."""
    import torch
    import lfbm5d_b200 as L
    nDisp, H, W = 10, 32, 36
    assert buffer_slots(an, nDisp) < (2 * an + 1) ** 2 - 1
    clean = np.ascontiguousarray(lfdata.synth_lf(aw, aw, H, W)[:, :C])
    noisy = oracle.add_noise(clean, 25.0)
    m = np.ones(aw * aw, np.uint32)
    if masked:
        m[(aw * aw) // 2] = 0
    p1 = L.make_params(25.0, 2.7, aw, aw, an, W, H, C, 8, 18, nDisp, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, aw, aw, an, W, H, C, 16, 18, nDisp, 8, 4, L.DCT, L.SADCT, L.HAAR)
    b, nrt = eng.step1(p1, noisy, m)
    ob, onrt, sched = oracle.run_step1(noisy, m, 25.0, 2.7, aw, aw, an, 8, 18, nDisp, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(eng.schedule(), sched)
    if masked:
        assert sched[:, 3].max() > 1
    assert np.array_equal(nrt[m == 1], onrt[m == 1])
    assert np.array_equal(b[m == 1], ob[m == 1])                                 # step 1 is bit-identical
    d, _, _ = eng.step2(p2, nrt, b, m)
    od, _, _, sched2 = oracle.run_step2(nrt, ob, m, 25.0, aw, aw, an, 16, 18, nDisp, 8, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(eng.schedule(), sched2)
    c1 = clean[m == 1]
    psnr = lambda x: 10.0 * np.log10(255.0 ** 2 / np.mean((x - c1) ** 2))
    # one window of one core call: nothing re-matches on a running estimate that differs in the last bits (test_gpu_parity.py)
    single = len(sched2) == 1 and int(sched2[0, 3]) == 1
    assert abs(psnr(d[m == 1]) - psnr(od[m == 1])) <= 0.01, (psnr(d[m == 1]), psnr(od[m == 1]))
    if single:
        assert np.abs(d[m == 1] - od[m == 1]).max() <= 1e-3
    dev = torch.device("cuda", 0)
    w = torch.from_numpy(noisy.copy()).to(dev)
    bd, dd = torch.zeros_like(w), torch.zeros_like(w)
    eng.step1_device(p1, w.data_ptr(), m, bd.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(bd.cpu().numpy()[m == 1], ob[m == 1])
    eng.step2_device(p2, w.data_ptr(), bd.data_ptr(), m, dd.data_ptr())
    dd = dd.cpu().numpy()
    assert abs(psnr(dd[m == 1]) - psnr(od[m == 1])) <= 0.01
    if single:
        assert np.abs(dd[m == 1] - od[m == 1]).max() <= 1e-3


@pytest.mark.parametrize("world,an,H,W", [(2, 1, 200, 72), (3, 1, 330, 64), (2, 2, 200, 64), (3, 2, 330, 56)])
def test_team_bit_identical_to_single_ndisp12(oracle, world, an, H, W):
    """Each rank chunks its own share of the slots, so the chunks start at other slots than on one GPU."""
    import torch
    import lfbm5d_b200 as L
    from test_team_gpu import run_single, run_team
    nDisp = 12
    aw = 2 * an + 1
    assert buffer_slots(an, nDisp) < aw * aw - 1
    dev = torch.device("cuda", 0)
    clean = lfdata.synth_lf(aw, aw, H, W)
    noisy = torch.from_numpy(oracle.add_noise(np.ascontiguousarray(clean), 15.0)).to(dev)
    mask = np.ones(aw * aw, np.uint32)
    p1 = L.make_params(15.0, 2.7, aw, aw, an, W, H, 3, 8, 18, nDisp, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, aw, aw, an, W, H, 3, 16, 18, nDisp, 8, 4, L.DCT, L.SADCT, L.HAAR)
    e = L.LFBM5D(0)
    w0, b0, o0, s0 = run_single(L, e, torch, noisy, mask, p1, p2)
    e.close()
    ws, bs, outs, bands1, bands2, st = run_team(L, torch, world, noisy, mask, p1, p2, gather=1)
    assert st["bytes_exchanged"] > 0
    for g in range(world):
        assert torch.equal(bs[g], b0) and torch.equal(outs[g], o0) and torch.equal(ws[g], w0)


def wide_lf(H=64, W=64, d=9):
    """3x3 RGB light field with d px of disparity per view (the corner views are d px away from the centre along both axes)."""
    return lfdata.synth_lf(3, 3, H, W, disparity=d)


def test_disparity_found_only_with_a_wide_enough_window(eng):
    """Noise free, 9 px of disparity per view: at nDisp = 10 the argmin of >= 95 % of the interior positions of every non-centre SAI
    is the true offset; at nDisp = 6 the true offset is outside the window for every non-centre SAI."""
    import lfbm5d_b200 as L
    import oracleapi as O
    H = W = 64
    d, k = 9, 16
    clean = wide_lf(H, W, d)
    order = [4] + [st for st in range(9) if st != 4]          # plane 0 = the centre SAI, the reference
    for nDisp, expect in ((10, True), (6, False)):
        n = 18 + nDisp
        planes = np.stack([O.symetrize(clean[st][:1], n)[0] for st in order])
        prm = L.make_params(10.0, 2.7, 3, 3, 1, W, H, 3, 8, 18, nDisp, k, 4, L.ID, L.SADCT, L.HAAR)
        _, _, first, _ = eng.debug_block_matching(1, prm, planes)
        wb = W + 2 * n
        ii, jj = np.mgrid[n + d:n + H - k + 1 - d, n + d:n + W - k + 1 - d]
        k_r = (ii * wb + jj).ravel()
        for a, st in enumerate(order[1:], start=1):
            s, t = divmod(st, 3)
            di, dj = -d * (s - 1), -d * (t - 1)
            hit = np.mean(first[a][k_r] == k_r + di * wb + dj)
            if expect:
                assert hit >= 0.95, (nDisp, st, hit)
            else:
                assert hit == 0.0, (nDisp, st, hit)


def test_wide_window_denoises_better(eng, oracle):
    """Same light field with noise: step 1 at nDisp = 10 groups the true correspondences and beats nDisp = 6 in PSNR."""
    import lfbm5d_b200 as L
    H = W = 64
    clean = wide_lf(H, W, 9)
    noisy = oracle.add_noise(clean, 25.0)
    mask = np.ones(9, np.uint32)
    out = {}
    for nDisp in (6, 10):
        p1 = L.make_params(25.0, 2.7, 3, 3, 1, W, H, 3, 8, 18, nDisp, 16, 4, L.ID, L.SADCT, L.HAAR)
        b, _ = eng.step1(p1, noisy, mask)
        out[nDisp] = oracle.psnr(b, clean)[0]
    print("step-1 PSNR, 9 px disparity per view: nDisp 6 %.3f dB, nDisp 10 %.3f dB" % (out[6], out[10]))
    assert out[10] > out[6], out


def test_command_line_ndisp10(tmp_path):
    """LFBM5Ddenoising with nDisp = 10 for both steps on a 3x3 light field of PNGs: the files are what the library gives."""
    from PIL import Image
    import lfbm5d_b200 as L
    H, W = 40, 44
    clean = wide_lf(H, W, 4)
    src = tmp_path / "sourceLF"
    for dname in ("sourceLF", "noisyLF", "basicLF", "denoisedLF", "diffLF"):
        (tmp_path / dname).mkdir()
    for s in range(3):
        for t in range(3):
            img = np.clip(np.floor(clean[s * 3 + t] + 0.5), 0, 255).astype(np.uint8).transpose(1, 2, 0)
            Image.fromarray(img).save(str(src / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))
    report = tmp_path / "objectiveResults.txt"
    args = [os.path.join(LIBDIR, "LFBM5Ddenoising"), str(src), "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "25", "2.7",
            str(tmp_path / "noisyLF"), str(tmp_path / "basicLF"), str(tmp_path / "denoisedLF"), str(tmp_path / "diffLF"),
            "8", "18", "10", "16", "4", "id", "sadct", "haar", "0", "16", "18", "10", "8", "4", "dct", "sadct", "haar", "0",
            "opp", "0", str(report)]
    env = dict(os.environ, LFBM5D_SEED="20171016")
    p = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, timeout=300)
    out = p.stdout.decode()
    assert p.returncode == 0, out[-2000:]
    src8 = np.clip(np.floor(clean + 0.5), 0, 255).astype(np.float32)
    noisy = L.add_noise(src8, 25.0, seed0=20171016)
    mask = np.ones(9, np.uint32)
    e = L.LFBM5D(0)
    p1 = L.make_params(25.0, 2.7, 3, 3, 1, W, H, 3, 8, 18, 10, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, 3, 3, 1, W, H, 3, 16, 18, 10, 8, 4, L.DCT, L.SADCT, L.HAAR)
    basic, n1 = e.step1(p1, noisy, mask)
    den, _, _ = e.step2(p2, n1, basic, mask)
    e.close()
    for s in range(3):
        for t in range(3):
            st = s * 3 + t
            for dname, arr in (("noisyLF", noisy), ("basicLF", basic), ("denoisedLF", den)):
                img = np.asarray(Image.open(str(tmp_path / dname / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))).transpose(2, 0, 1)
                assert np.array_equal(img, np.clip(np.floor(arr[st] + np.float32(0.5)), 0, 255).astype(np.uint8)), (dname, st)


def test_parameter_errors_launch_nothing(eng):
    import lfbm5d_b200 as L
    noisy = np.zeros((9, 3, 40, 44), np.float32)
    mask = np.ones(9, np.uint32)
    eng.reset_stats()
    with pytest.raises(RuntimeError, match="nDisp > 16"):
        eng.step1(L.make_params(25.0, 2.7, 3, 3, 1, 44, 40, 3, 8, 18, 17, 16, 4, L.ID, L.SADCT, L.HAAR), noisy, mask)
    with pytest.raises(RuntimeError, match="nDisp > 16"):
        eng.step2(L.make_params(25.0, 0.0, 3, 3, 1, 44, 40, 3, 16, 18, 17, 8, 4, L.DCT, L.SADCT, L.HAAR), noisy, noisy, mask)
    small = np.zeros((9, 3, 30, 44), np.float32)      # 30 rows < nSim + nDisp = 18 + 16
    with pytest.raises(RuntimeError, match="image smaller than the padding nSim \\+ nDisp"):
        eng.step1(L.make_params(25.0, 2.7, 3, 3, 1, 44, 30, 3, 8, 18, 16, 16, 4, L.ID, L.SADCT, L.HAAR), small, mask)
    assert eng.stats().kernel_launches == 0
