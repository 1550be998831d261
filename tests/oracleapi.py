"""ctypes bindings for oracle/liblfbm5d_oracle.so (CPU restatement). TEST INFRASTRUCTURE ONLY."""
import contextlib
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
ORC_SO = os.path.join(ROOT, "oracle", "liblfbm5d_oracle.so")

YUV, YCBCR, OPP, RGB, ID, DCT, SADCT, BIOR, HADAMARD, HAAR, NONE, ROWMAJOR, COLMAJOR = range(13)

_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(ROOT, "oracle", "lfbm5d_oracle.c")
        if not os.path.exists(ORC_SO) or os.path.getmtime(ORC_SO) < os.path.getmtime(src):
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "oracle"], stdout=subprocess.DEVNULL)
        _lib = C.CDLL(ORC_SO)
        _lib.orc_LF_denoised_percent.restype = C.c_float
        _lib.orc_mt_res53.restype = C.c_double
        _lib.orc_ind_initialize.restype = C.c_uint
    return _lib


def fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def up(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_uint))


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def set_dct_mode(m):
    lib().orc_set_dct_mode(int(m))


@contextlib.contextmanager
def sum_mode(m):
    """Runs the block with orc_set_sum_mode(m) (1: the group's Wiener weight and useSD sums added in double and rounded to
    float once, 0: term by term in float as the reference does) and restores mode 0 however it ends."""
    lib().orc_set_sum_mode(int(m))
    try:
        yield
    finally:
        lib().orc_set_sum_mode(0)


def add_noise(clean, sigma, seed0=20171016):
    """clean [A, C, H, W] -> noisy, SAI st seeded with seed0 + st (serial, unclipped)."""
    out = np.empty_like(clean, dtype=np.float32)
    for st in range(clean.shape[0]):
        src = f32(clean[st])
        dst = np.empty_like(src)
        lib().orc_add_noise(fp(src), fp(dst), C.c_size_t(src.size), C.c_float(sigma), C.c_ulong(seed0 + st))
        out[st] = dst
    return out


def psnr(a, b):
    p, r = C.c_float(), C.c_float()
    a, b = f32(a), f32(b)
    lib().orc_psnr(fp(a), fp(b), C.c_size_t(a.size), C.byref(p), C.byref(r))
    return p.value, r.value


def symetrize(img, N):
    Cn, H, W = img.shape
    out = np.empty((Cn, H + 2 * N, W + 2 * N), np.float32)
    lib().orc_symetrize(fp(f32(img)), fp(out), W, H, Cn, N)
    return out


def bm_self(img, k, N, nHW, nSim, p, tau):
    h, w = img.shape
    cnt = np.zeros(h * w, np.uint32)
    idx = np.zeros((h * w, N + 1), np.uint32)
    lib().orc_bm_self(fp(f32(img)), w, h, k, N, nHW, nSim, p, C.c_float(tau), up(cnt), up(idx), N + 1)
    return cnt, idx


def bm_stereo(img1, img2, k, nHW, nDisp, tau):
    h, w = img1.shape
    first = np.zeros(h * w, np.uint32)
    shape = np.zeros(h * w, np.uint32)
    ties = np.zeros(h * w, np.uint32)
    lib().orc_bm_stereo(fp(f32(img1)), fp(f32(img2)), w, h, k, nHW, nDisp, C.c_float(tau), up(first), up(shape), up(ties))
    return first, shape, ties


def run_pass(step, noisy_sym, basic_sym, num_sym, den_sym, mask, proc, pst, asw, sigma, lam, nSim, nDisp, k, N, p,
             tau2, tau4, tau5, cs=OPP, debug=False, cst=None):
    A, Cn, hb, wb = noisy_sym.shape
    num = f32(num_sym).copy()
    den = f32(den_sym).copy()
    ns = f32(noisy_sym)
    bs = f32(basic_sym) if basic_sym is not None else ns
    dbg = [None] * 4
    if debug:
        dbg = [np.zeros(hb * wb, np.uint32), np.zeros((hb * wb, N + 1), np.uint32),
               np.zeros((A, hb * wb), np.uint32), np.zeros((A, hb * wb), np.uint32)]
    rc = lib().orc_pass_ex(step, C.c_float(sigma), C.c_float(lam), fp(ns), fp(bs), fp(num), fp(den), up(u32(mask)), up(u32(proc)),
                           pst if cst is None else cst, pst, asw, wb, hb, Cn, nSim, nDisp, k, N, p, cs, tau2, tau4, tau5, *[up(d) for d in dbg])
    assert rc == 0, rc
    return (num, den, dbg) if debug else (num, den)


def run_step1(noisy, mask, sigma, lam, aw, ah, an, N, nSim, nDisp, k, p, tau2, tau4, tau5, cs=OPP, ang_major=ROWMAJOR,
              max_passes=0):
    A, Cn, H, W = noisy.shape
    n = f32(noisy).copy()
    basic = np.zeros_like(n)
    sched = np.zeros((A + 1, 4), np.uint32)
    ns = C.c_uint(0)
    rc = lib().orc_run_step1(C.c_float(sigma), C.c_float(lam), fp(n), up(u32(mask)), fp(basic), ang_major, aw, ah, an, W, H, Cn,
                             N, nSim, nDisp, k, p, tau2, tau4, tau5, cs, up(sched), A + 1, C.byref(ns), max_passes)
    assert rc == 0, rc
    return basic, n, sched[:ns.value]


def run_step2(noisy, basic, mask, sigma, aw, ah, an, N, nSim, nDisp, k, p, tau2, tau4, tau5, cs=OPP, ang_major=ROWMAJOR,
              max_passes=0):
    A, Cn, H, W = noisy.shape
    n = f32(noisy).copy()
    b = f32(basic).copy()
    den = np.zeros_like(n)
    sched = np.zeros((A + 1, 4), np.uint32)
    ns = C.c_uint(0)
    rc = lib().orc_run_step2(C.c_float(sigma), fp(n), up(u32(mask)), fp(b), fp(den), ang_major, aw, ah, an, W, H, Cn,
                             N, nSim, nDisp, k, p, tau2, tau4, tau5, cs, up(sched), A + 1, C.byref(ns), max_passes)
    assert rc == 0, rc
    return den, b, n, sched[:ns.value]


def run_bm3d_lf(noisy, mask, sigma, nHard, nWien, kHard, kWien, NHard, NWien, pHard, pWien, tau2h, tau2w, lam, cs=OPP):
    A, Cn, H, W = noisy.shape
    n = f32(noisy).copy()
    basic = np.zeros_like(n)
    den = np.zeros_like(n)
    rc = lib().orc_run_bm3d_LF(C.c_float(sigma), fp(n), up(u32(mask)), fp(basic), fp(den), A, W, H, Cn, nHard, nWien, kHard, kWien,
                               NHard, NWien, pHard, pWien, tau2h, tau2w, C.c_float(lam), cs)
    assert rc == 0, rc
    return basic, den, n
