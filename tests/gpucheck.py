"""What the GPU tests share: the engine fixture, the input builders and the checks of the GPU against the CPU oracle. Every GPU test
module imports `eng` from here (pytest registers an imported fixture per module, so each module gets its own engine).

The parity contract (DESIGN.md section 2) is written here once: self-match lists, disparity argmin and shape flags bit-exact; step-1
accumulators bit-identical (ordered aggregation, integer-valued weights), hence LF_basic bit-identical; step-2 accumulators within
STEP2_REL of the pass's largest value (only the Wiener weight sum is reduced in another order than the reference's serial float sum),
STEP2_REL_SD with useSD (the group's standard deviation is reduced over A N k^2 values in another order), wiener_tol(N, useSD) for
groups on clusters; normalised estimates within EST_ABS; complete runs within PSNR_DB of the oracle's LF_denoised."""
import os
import subprocess

import numpy as np
import pytest

import lfdata

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "lfbm5d_b200", "_lib")

STEP2_REL = 2e-5        # step-2 num / den, relative to the largest |value| of the pass
STEP2_REL_SD = 1e-4     # the same with useSD
EST_ABS = 1e-3          # num / den after normalisation, absolute in [0, 255]
PSNR_DB = 0.01          # LF_denoised of a complete run against the oracle's


def wiener_tol(N, useSD):
    """Relative tolerance of a step-2 pass. Like the reference, the oracle adds the N * 9 * 256 Wiener coefficients of a group
    (and useSD's sums) one by one in float; the error of such a sum of n non-negative terms is bounded by (n - 1) * 2^-24 of the
    sum, which grows with the group and is far above STEP2_REL at these N. Measured on one B200 on the inputs of
    test_large_groups_gpu.py: switching the oracle's weight sum to double moves the oracle by up to 2.1e-4 at N = 32 (5e-5 already
    at N = 8 on the one-CTA k_groups), while the GPU, which sums in blocks and then in rank order, stays within 3e-6 of the double
    sum. A wrong patch, coefficient or weight gives errors of order 1e-1 and more."""
    return max(STEP2_REL_SD if useSD else STEP2_REL, N * 9 * 256 * 2.0 ** -24)


@pytest.fixture(scope="module")
def eng():
    import lfbm5d_b200 as L
    e = L.LFBM5D(0)
    yield e
    e.close()


def estimate(num, den, sub):
    return np.where(den != 0, num / np.where(den != 0, den, 1), sub).astype(np.float32)


def psnr_on(clean, m):
    """PSNR against `clean` over the SAIs of mask m."""
    c1 = clean[m == 1]
    return lambda x: 10.0 * np.log10(255.0 ** 2 / np.mean((x[m == 1] - c1) ** 2))


# -- inputs ------------------------------------------------------------------------------------------------------------------

def channel0_planes(oracle, H, W, sigma, nsai, n=24, quantise=False):
    """Padded channel-0 (OPP) planes of `nsai` views with 1 px/view disparity. quantise: coarse grey levels and a constant
    rectangle, so that exact distance ties occur (mirror axes, flat regions)."""
    clean = lfdata.synth_lf(nsai, 1, H, W)
    if quantise:
        clean = np.round(clean / 24.0) * 24.0
        clean[:, :, H // 4:H // 4 + 120, W // 3:W // 3 + 200] = 72.0
    y = oracle.add_noise(clean, sigma) if sigma > 0 else clean.copy()
    for st in range(nsai):
        oracle.lib().orc_color_space_transform(oracle.fp(y[st]), oracle.OPP, W, H, 3, 1)
    return np.stack([oracle.symetrize(y[st][:1], n)[0] for st in range(nsai)])


def pad_inputs5(oracle, H, W, sigma, n=24, C=3):
    """Noisy padded SAIs of a 5x5 light field (OPP when C == 3)."""
    clean = lfdata.synth_lf(5, 5, H, W)[:, :C]
    noisy = oracle.add_noise(np.ascontiguousarray(clean), sigma)
    y = noisy.copy()
    if C == 3:
        for st in range(25):
            oracle.lib().orc_color_space_transform(oracle.fp(y[st]), oracle.OPP, W, H, 3, 1)
    return np.stack([oracle.symetrize(y[st], n) for st in range(25)])


# -- single passes ---------------------------------------------------------------------------------------------------------

def check_bm(eng, oracle, planes, step, k, N, tau, nDisp=6, self_too=True):
    """debug_block_matching on channel-0 planes padded by nSim + nDisp = 18 + nDisp (plane 0 = the reference SAI) against
    orc_bm_self / orc_bm_stereo. Returns (reference patches with matches, tied disparity minima the oracle saw)."""
    import lfbm5d_b200 as L
    n = 18 + nDisp
    H, W = planes.shape[1] - 2 * n, planes.shape[2] - 2 * n
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
    return int((cnt > 0).sum()), nties


def check_pass(eng, oracle, step, sym, basic, num0, den0, mask, proc, k, N, t2, t4, t5, an=1, pst=None, cst=None, sigma=25.0, lam=2.7,
               nSim=18, nDisp=6, p=4, useSD=0, rel=None, est=True):
    """One window pass (debug_pass) against the oracle's on padded SAIs `sym` of a (2 an + 1)^2 window, reference SAI pst (default
    the centre one), cst = pst unless given. Match tables bit-exact; step 1 without useSD bit-identical; otherwise num / den within
    `rel` (default STEP2_REL, STEP2_REL_SD with useSD) of their largest value. est: the estimates within EST_ABS as well.
    Returns (on, od, gn, gd, gdbg)."""
    import lfbm5d_b200 as L
    A, C, hb, wb = sym.shape
    asw = 2 * an + 1
    pst = A // 2 if pst is None else pst
    H, W = hb - 2 * (nSim + nDisp), wb - 2 * (nSim + nDisp)
    oracle.lib().orc_set_use_sd(int(useSD))
    try:
        on, od, odbg = oracle.run_pass(step, sym, basic, num0, den0, mask, proc, pst, asw, sigma, lam, nSim, nDisp, k, N, p, t2, t4, t5,
                                       debug=True, cst=cst)
    finally:
        oracle.lib().orc_set_use_sd(0)
    prm = L.make_params(sigma, lam, asw, asw, an, W, H, C, N, nSim, nDisp, k, p, t2, t4, t5, useSD=int(useSD))
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
        if rel is None:
            rel = STEP2_REL_SD if useSD else STEP2_REL
        assert np.abs(gn - on).max() <= rel * np.abs(on).max() and np.abs(gd - od).max() <= rel * np.abs(od).max()
    if est:
        sub = sym if step == 1 else basic
        err = np.abs(estimate(on, od, sub) - estimate(gn, gd, sub)).max()
        assert err <= EST_ABS, err
    return on, od, gn, gd, gdbg


# -- complete runs -----------------------------------------------------------------------------------------------------------

def check_complete_run(eng, oracle, clean, m, p1, p2, calls_only=False):
    """Both steps on `clean` plus the oracle's noise through the host-buffer and the device-resident entry points, against the
    oracle with the same parameters, on the SAIs of mask m: the window schedules (calls_only: their length and core calls per
    window), the colour-round-tripped noisy light field and LF_basic bit-identical, LF_denoised within PSNR_DB. The light field
    travels in place through the device entry points: it comes back colour-round-tripped after step 1.
    Returns (noisy, sched, sched2, d, dd, od) with the step-1 / step-2 schedules and the denoised host, device and oracle results."""
    import torch
    import lfbm5d_b200 as L

    def same_schedule(sched):
        s = eng.schedule()
        if calls_only:
            return len(s) == len(sched) and np.array_equal(s[:, 3], sched[:, 3])
        return np.array_equal(s, sched)

    noisy = oracle.add_noise(clean, p1.sigma)
    args1 = (p1.sigma, p1.lambda_, p1.awidth, p1.aheight, p1.an, p1.N, p1.nSim, p1.nDisp, p1.k, p1.p, p1.tau_2D, p1.tau_4D, p1.tau_5D)
    args2 = (p2.sigma, p2.awidth, p2.aheight, p2.an, p2.N, p2.nSim, p2.nDisp, p2.k, p2.p, p2.tau_2D, p2.tau_4D, p2.tau_5D)
    b, nrt = eng.step1(p1, noisy, m)
    ob, onrt, sched = oracle.run_step1(noisy, m, *args1)
    assert same_schedule(sched)
    assert np.array_equal(nrt[m == 1], onrt[m == 1])
    assert np.array_equal(b[m == 1], ob[m == 1])                                 # step 1 is bit-identical
    d, _, _ = eng.step2(p2, nrt, b, m)
    # both sides start step 2 from the same colour-round-tripped noisy light field and the same basic estimate
    od, _, _, sched2 = oracle.run_step2(nrt, ob, m, *args2)
    assert same_schedule(sched2)
    psnr = psnr_on(clean, m)
    assert abs(psnr(d) - psnr(od)) <= PSNR_DB, (psnr(d), psnr(od))
    dev = torch.device("cuda", 0)
    w = torch.from_numpy(noisy.copy()).to(dev)
    bd, dd = torch.zeros_like(w), torch.zeros_like(w)
    eng.step1_device(p1, w.data_ptr(), m, bd.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(bd.cpu().numpy()[m == 1], ob[m == 1])
    eng.step2_device(p2, w.data_ptr(), bd.data_ptr(), m, dd.data_ptr())
    dd = dd.cpu().numpy()
    assert abs(psnr(dd) - psnr(od)) <= PSNR_DB, (psnr(dd), psnr(od))
    return noisy, sched, sched2, d, dd, od


# -- teams -------------------------------------------------------------------------------------------------------------------

def run_single(L, eng, torch, noisy, mask, p1, p2):
    w, b, o = noisy.clone(), torch.zeros_like(noisy), torch.zeros_like(noisy)
    eng.step1_device(p1, w.data_ptr(), mask, b.data_ptr())
    s1 = eng.schedule().copy()
    eng.step2_device(p2, w.data_ptr(), b.data_ptr(), mask, o.data_ptr())
    torch.cuda.synchronize()
    return w, b, o, s1


def run_team(L, torch, world, noisy, mask, p1, p2, gather, peer_view=True, lanes=1):
    team = L.Team.emulated(0, world)
    if lanes > 1:
        team.set_lanes(lanes)
    if not peer_view:
        team.disable_peer_view()
    ws = [noisy.clone() for _ in range(world)]
    bs = [torch.zeros_like(noisy) for _ in range(world)]
    outs = [torch.zeros_like(noisy) for _ in range(world)]
    team.step(1, p1, [t.data_ptr() for t in ws], None, mask, [t.data_ptr() for t in bs], gather=gather)
    bands1 = [team.band(g) for g in range(world)]
    team.step(2, p2, [t.data_ptr() for t in ws], [t.data_ptr() for t in bs], mask, [t.data_ptr() for t in outs], gather=gather)
    bands2 = [team.band(g) for g in range(world)]
    torch.cuda.synchronize()
    st = team.stats()
    team.close()
    return ws, bs, outs, bands1, bands2, st


def assert_team_matches_single(oracle, world, p1, p2):
    """An emulated team of `world` ranks (gathered results) against one context on a light field of p1's shape with sigma 15
    noise: LF_basic, LF_denoised and the colour-round-tripped input bit-identical on every rank, and the ranks exchanged rows."""
    import torch
    import lfbm5d_b200 as L
    dev = torch.device("cuda", 0)
    clean = lfdata.synth_lf(p1.awidth, p1.aheight, p1.height, p1.width)
    noisy = torch.from_numpy(oracle.add_noise(np.ascontiguousarray(clean), 15.0)).to(dev)
    mask = np.ones(p1.awidth * p1.aheight, np.uint32)
    e = L.LFBM5D(0)
    w0, b0, o0, _ = run_single(L, e, torch, noisy, mask, p1, p2)
    e.close()
    ws, bs, outs, _, _, st = run_team(L, torch, world, noisy, mask, p1, p2, gather=1)
    assert st["bytes_exchanged"] > 0
    for g in range(world):
        assert torch.equal(bs[g], b0) and torch.equal(outs[g], o0) and torch.equal(ws[g], w0)


# -- command lines -----------------------------------------------------------------------------------------------------------

def write_lf(tmp_path, clean, aw):
    """`clean` as 8-bit RGB PNGs SAI_<s>_<t>.png in tmp_path/sourceLF, and empty output directories beside it."""
    from PIL import Image
    src = tmp_path / "sourceLF"
    for dname in ("sourceLF", "noisyLF", "basicLF", "denoisedLF", "diffLF"):
        (tmp_path / dname).mkdir()
    for s in range(aw):
        for t in range(aw):
            img = np.clip(np.floor(clean[s * aw + t] + 0.5), 0, 255).astype(np.uint8).transpose(1, 2, 0)
            Image.fromarray(img).save(str(src / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))
    return src


def run_cli(args):
    """Runs a command-line driver with the reference's noise seed; it must succeed. Returns its output."""
    env = dict(os.environ, LFBM5D_SEED="20171016")
    p = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, timeout=300)
    out = p.stdout.decode()
    assert p.returncode == 0, out[-2000:]
    return out


def check_pngs(tmp_path, arrays, aw):
    """The PNGs in the directories named by `arrays` ((dirname, light field) pairs) are the light fields rounded floor(x + .5) and
    clamped, as the reference writes them."""
    from PIL import Image
    for s in range(aw):
        for t in range(aw):
            st = s * aw + t
            for dname, arr in arrays:
                img = np.asarray(Image.open(str(tmp_path / dname / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))).transpose(2, 0, 1)
                assert np.array_equal(img, np.clip(np.floor(arr[st] + np.float32(0.5)), 0, 255).astype(np.uint8)), (dname, st)


def assert_rejected(eng, calls):
    """Each (callable, match) pair raises a RuntimeError that matches, and none of them launches a kernel."""
    eng.reset_stats()
    for call, match in calls:
        with pytest.raises(RuntimeError, match=match):
            call()
    assert eng.stats().kernel_launches == 0
