"""12 x 12 patches (k = 12) on the GPU, through the C ABI against the CPU oracle. The oracle is generic in k but pinned against the
reference only at k = 8 and 16, so these results are checked GPU vs oracle. Tolerances are those of test_gpu_parity.py /
test_angular_window_gpu.py: match lists, disparity argmin and shape flags bit-exact; step 1 accumulators and LF_basic
bit-identical; step 2 within 2e-5 relative per pass (1e-4 with useSD); complete runs within 0.01 dB."""
import os
import subprocess

import numpy as np
import pytest

import golden_inputs as gi
import lfdata
from test_gpu_baseline_shapes import channel0_planes
from test_gpu_parity import estimate

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "lfbm5d_b200", "_lib")
K = 12


@pytest.fixture(scope="module")
def eng():
    import lfbm5d_b200 as L
    e = L.LFBM5D(0)
    yield e
    e.close()


def check_bm(eng, oracle, planes, step, N, tau, W, H, nDisp):
    import lfbm5d_b200 as L
    n = 18 + nDisp
    prm = L.make_params(10.0, 2.7, 3, 3, 1, W, H, 3, N, 18, nDisp, K, 4, L.ID if step == 1 else L.DCT, L.SADCT, L.HAAR)
    cnt, idx, first, shape = eng.debug_block_matching(step, prm, planes)
    ocnt, oidx = oracle.bm_self(planes[0], K, N, n, 18, 4, tau)
    assert np.array_equal(cnt, ocnt), "self-match counts differ"
    m = np.arange(N + 1)[None, :] < ocnt[:, None]
    assert np.array_equal(idx * m, oidx * m), "self-match lists differ"
    nties = 0
    for s in range(1, planes.shape[0]):
        of, osh, oties = oracle.bm_stereo(planes[0], planes[s], K, n, nDisp, tau)
        assert np.array_equal(first[s], of), "disparity argmin differs (plane %d)" % s
        assert np.array_equal(shape[s], osh), "shape flags differ (plane %d)" % s
        nties += int(oties.sum())
    return nties


@pytest.mark.parametrize("nDisp", [6, 12])
def test_block_matching_k12(eng, oracle, nDisp):
    """Self and disparity matching at k = 12 on planes of 300+ rows (the 128-row source ring wraps), with a padded row pitch that is a
    multiple of 16 B and one that is not, noisy and quantised noise-free input (tied minima)."""
    n = 18 + nDisp
    H = 300
    w16 = 64 - (2 * n) % 4                    # (w16 + 2 n) floats per padded row: a multiple of 16 B
    for W in (w16, w16 + 1):
        check_bm(eng, oracle, channel0_planes(oracle, H, W, 10.0, 3, n=n), 1, 16, 3000.0, W, H, nDisp)
        q = channel0_planes(oracle, H, W, 0.0, 3, n=n, quantise=True)
        assert check_bm(eng, oracle, q, 2, 16, 2000.0, W, H, nDisp) > 0


def check_pass12(eng, oracle, step, sym, basic, num0, den0, mask, proc, N, t2, t4, t5, lam=2.7, useSD=0, pst=4, cst=None):
    import lfbm5d_b200 as L
    A, C, hb, wb = sym.shape
    H, W = hb - 48, wb - 48
    oracle.lib().orc_set_use_sd(int(useSD))
    try:
        on, od, odbg = oracle.run_pass(step, sym, basic, num0, den0, mask, proc, pst, 3, 25.0, lam, 18, 6, K, N, 4, t2, t4, t5, debug=True,
                                       cst=cst)
    finally:
        oracle.lib().orc_set_use_sd(0)
    prm = L.make_params(25.0, lam, 3, 3, 1, W, H, C, N, 18, 6, K, 4, t2, t4, t5, useSD=int(useSD))
    gn, gd, gdbg = eng.debug_pass(step, prm, sym, basic, num0, den0, mask, proc, pst, debug=True, cst=cst)
    assert np.array_equal(odbg[0], gdbg[0]), "self-match counts differ"
    m = np.arange(N + 1)[None, :] < odbg[0][:, None]
    assert np.array_equal(odbg[1] * m, gdbg[1] * m), "self-match lists differ"
    assert np.array_equal(odbg[2], gdbg[2]), "disparity argmin differs"
    assert np.array_equal(odbg[3], gdbg[3]), "shape flags differ"
    assert np.array_equal(od != 0, gd != 0)
    if step == 1 and not useSD:
        assert np.array_equal(gn, on) and np.array_equal(gd, od)                     # step 1: bit-identical
    else:
        tol = 1e-4 if useSD else 2e-5
        assert np.abs(gn - on).max() <= tol * np.abs(on).max() and np.abs(gd - od).max() <= tol * np.abs(od).max()
    return on, od, gn, gd


def test_single_passes_k12(eng, oracle):
    """Every 2-D / angular / 1-D transform combination at k = 12, both steps, and a second pass on top of the first's accumulators."""
    _, _, sym = gi.pad_inputs(40, 48, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    on, od, _, _ = check_pass12(eng, oracle, 1, sym, None, z, z, mask, proc, 16, oracle.ID, oracle.SADCT, oracle.HAAR)
    basic = estimate(on, od, sym)
    for t2 in (oracle.ID, oracle.DCT):
        for t4 in (oracle.DCT, oracle.SADCT, oracle.ID):
            for t5 in (oracle.HAAR, oracle.HADAMARD, oracle.DCT):
                check_pass12(eng, oracle, 1, sym, None, z, z, mask, proc, 8, t2, t4, t5)
                check_pass12(eng, oracle, 2, sym, basic, z, z, mask, proc, 16, t2, t4, t5, lam=0.0)
    check_pass12(eng, oracle, 1, sym, None, z, z, mask, proc, 32, oracle.DCT, oracle.SADCT, oracle.HAAR)     # largest step-1 group
    check_pass12(eng, oracle, 1, sym, None, z, z, mask, proc, 16, oracle.ID, oracle.SADCT, oracle.HAAR, useSD=1)
    check_pass12(eng, oracle, 2, sym, basic, z, z, mask, proc, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, useSD=1)
    # second pass of step 1 on top of the first pass's accumulators (block matching on num / den)
    check_pass12(eng, oracle, 1, sym, None, on, od, mask, proc, 16, oracle.ID, oracle.SADCT, oracle.HAAR)


def test_single_passes_k12_masked_processed_and_partial(eng, oracle):
    _, _, sym = gi.pad_inputs(32, 40, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    mask[2] = 0
    proc[2] = proc[7] = 1
    on, od, gn, gd = check_pass12(eng, oracle, 1, sym, None, z, z, mask, proc, 16, oracle.ID, oracle.SADCT, oracle.HAAR)
    assert not gd[7].any() and not gd[2].any()
    basic = estimate(on, od, sym)
    check_pass12(eng, oracle, 2, sym, basic, z, z, mask, proc, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0)
    # partial-window branch (pst != cst) on accumulators with holes
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    num, den = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, K, 16, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    basic = estimate(num, den, sym)
    num, den = gi.partial_holes(num, den)
    proc[4] = 1
    for pst in (1, 6):
        gn, _, _, _ = check_pass12(eng, oracle, 1, sym, None, num, den, mask, proc, 16, oracle.ID, oracle.SADCT, oracle.HAAR, pst=pst, cst=4)
        assert not np.array_equal(gn, num)
        check_pass12(eng, oracle, 2, sym, basic, num, den, mask, proc, 16, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0, pst=pst, cst=4)


def psnr_on(clean, m):
    c1 = clean[m == 1]
    return lambda x: 10.0 * np.log10(255.0 ** 2 / np.mean((x[m == 1] - c1) ** 2))


@pytest.mark.parametrize("aw,an,C,masked,t2", [(3, 1, 3, False, "id"), (3, 1, 3, False, "dct"), (3, 0, 3, False, "dct"),
                                                (3, 1, 1, True, "id")])
def test_complete_runs_k12(eng, oracle, aw, an, C, masked, t2):
    """Both steps at k = 12 through the host-buffer and the device-resident entry points, with the oracle's window schedule;
    grayscale with an empty centre SAI takes the partial-window branch."""
    import torch
    import lfbm5d_b200 as L
    H, W = 32, 36
    clean = np.ascontiguousarray(lfdata.synth_lf(aw, aw, H, W)[:, :C])
    noisy = oracle.add_noise(clean, 25.0)
    m = np.ones(aw * aw, np.uint32)
    if masked:
        m[(aw * aw) // 2] = 0
    T1 = L.ID if t2 == "id" else L.DCT
    p1 = L.make_params(25.0, 2.7, aw, aw, an, W, H, C, 8, 18, 6, K, 4, T1, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, aw, aw, an, W, H, C, 16, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
    b, nrt = eng.step1(p1, noisy, m)
    ob, onrt, sched = oracle.run_step1(noisy, m, 25.0, 2.7, aw, aw, an, 8, 18, 6, K, 4, T1, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(eng.schedule(), sched)
    if masked:
        assert sched[:, 3].max() > 1
    assert np.array_equal(nrt[m == 1], onrt[m == 1])
    assert np.array_equal(b[m == 1], ob[m == 1])                                  # step 1 is bit-identical
    d, _, _ = eng.step2(p2, nrt, b, m)
    od, _, _, sched2 = oracle.run_step2(nrt, ob, m, 25.0, aw, aw, an, 16, 18, 6, K, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(eng.schedule(), sched2)
    psnr = psnr_on(clean, m)
    assert abs(psnr(d) - psnr(od)) <= 0.01, (psnr(d), psnr(od))
    assert psnr(d) > psnr(noisy) + 3.0
    dev = torch.device("cuda", 0)
    w = torch.from_numpy(noisy.copy()).to(dev)
    bd, dd = torch.zeros_like(w), torch.zeros_like(w)
    eng.step1_device(p1, w.data_ptr(), m, bd.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(bd.cpu().numpy()[m == 1], ob[m == 1])
    eng.step2_device(p2, w.data_ptr(), bd.data_ptr(), m, dd.data_ptr())
    assert abs(psnr(dd.cpu().numpy()) - psnr(od)) <= 0.01


@pytest.mark.parametrize("world,H,W", [(2, 200, 72), (3, 330, 64)])
def test_team_bit_identical_to_single_k12(oracle, world, H, W):
    import torch
    import lfbm5d_b200 as L
    from test_team_gpu import run_single, run_team
    dev = torch.device("cuda", 0)
    clean = lfdata.synth_lf(3, 3, H, W)
    noisy = torch.from_numpy(oracle.add_noise(np.ascontiguousarray(clean), 15.0)).to(dev)
    mask = np.ones(9, np.uint32)
    p1 = L.make_params(15.0, 2.7, 3, 3, 1, W, H, 3, 8, 18, 6, K, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(15.0, 0.0, 3, 3, 1, W, H, 3, 16, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR)
    e = L.LFBM5D(0)
    w0, b0, o0, s0 = run_single(L, e, torch, noisy, mask, p1, p2)
    e.close()
    ws, bs, outs, bands1, bands2, st = run_team(L, torch, world, noisy, mask, p1, p2, gather=1)
    assert st["bytes_exchanged"] > 0
    for g in range(world):
        assert torch.equal(bs[g], b0) and torch.equal(outs[g], o0) and torch.equal(ws[g], w0)


def test_lfbm3d_k12(eng, oracle):
    """Per-SAI BM3D with kHard = kWien = 12 (dct / dct, the 12 x 12 Kaiser window in the aggregation) and a masked SAI."""
    import lfbm5d_b200 as L
    clean = lfdata.synth_lf(2, 2, 40, 48)
    noisy = oracle.add_noise(clean, 10.0)
    mask = np.ones(4, np.uint32)
    mask[3] = 0
    ob, od, on = oracle.run_bm3d_lf(noisy, mask, 10.0, 16, 16, K, K, 16, 32, 3, 3, L.DCT, L.DCT, 2.7)
    prm = L.make_params3d(10.0, 4, 48, 40, 3, 16, 16, K, K, 16, 32, 3, 3, L.DCT, L.DCT, 2.7)
    gb, gd, gn = eng.bm3d(prm, noisy, mask)
    assert np.array_equal(gn, on)
    assert np.array_equal(gb[:3], ob[:3])                  # step 1: bit-exact
    assert np.abs(gd[:3] - od[:3]).max() <= 1e-3
    assert not gb[3].any() and not gd[3].any()
    assert oracle.psnr(gd[:3], clean[:3])[0] > oracle.psnr(noisy[:3], clean[:3])[0] + 4.0


def write_lf(tmp_path, clean, aw):
    from PIL import Image
    src = tmp_path / "sourceLF"
    for dname in ("sourceLF", "noisyLF", "basicLF", "denoisedLF", "diffLF"):
        (tmp_path / dname).mkdir()
    for s in range(aw):
        for t in range(aw):
            img = np.clip(np.floor(clean[s * aw + t] + 0.5), 0, 255).astype(np.uint8).transpose(1, 2, 0)
            Image.fromarray(img).save(str(src / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))
    return src


def check_files(tmp_path, arrays, aw):
    from PIL import Image
    for s in range(aw):
        for t in range(aw):
            st = s * aw + t
            for dname, arr in arrays:
                img = np.asarray(Image.open(str(tmp_path / dname / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))).transpose(2, 0, 1)
                assert np.array_equal(img, np.clip(np.floor(arr[st] + np.float32(0.5)), 0, 255).astype(np.uint8)), (dname, st)


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
    args = head + tail + ["opp", "0", str(tmp_path / "objectiveResults.txt")]
    env = dict(os.environ, LFBM5D_SEED="20171016")
    p = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, timeout=300)
    out = p.stdout.decode()
    assert p.returncode == 0, out[-2000:]
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
    check_files(tmp_path, (("noisyLF", noisy), ("basicLF", basic), ("denoisedLF", den)), 3)


def test_k12_parameter_errors_launch_nothing(eng):
    import lfbm5d_b200 as L
    noisy = np.zeros((25, 3, 40, 44), np.float32)
    mask = np.ones(25, np.uint32)
    eng.reset_stats()
    with pytest.raises(RuntimeError, match="bior needs a power-of-two patch size"):
        eng.step1(L.make_params(25.0, 2.7, 3, 3, 1, 44, 40, 3, 8, 18, 6, K, 4, L.BIOR, L.SADCT, L.HAAR), noisy[:9], mask[:9])
    with pytest.raises(RuntimeError, match="an = 2 is not supported at k = 12"):
        eng.step1(L.make_params(25.0, 2.7, 5, 5, 2, 44, 40, 3, 2, 18, 6, K, 4, L.ID, L.SADCT, L.HAAR), noisy, mask)
    with pytest.raises(RuntimeError, match="k = 12 needs N"):
        eng.step2(L.make_params(25.0, 0.0, 3, 3, 1, 44, 40, 3, 32, 18, 6, K, 4, L.DCT, L.SADCT, L.HAAR), noisy[:9], noisy[:9], mask[:9])
    with pytest.raises(RuntimeError, match="patch size must be 8, 12 or 16"):
        eng.step1(L.make_params(25.0, 2.7, 3, 3, 1, 44, 40, 3, 8, 18, 6, 10, 4, L.ID, L.SADCT, L.HAAR), noisy[:9], mask[:9])
    with pytest.raises(RuntimeError, match="bior needs a power-of-two patch size"):
        eng.bm3d(L.make_params3d(25.0, 9, 44, 40, 3, 16, 16, K, K, 16, 32, 3, 3, L.BIOR, L.DCT, 2.7), noisy[:9], mask[:9])
    assert eng.stats().kernel_launches == 0
