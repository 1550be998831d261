"""ctypes bindings for oracle/_ref/libref_lfbm5d.so (the unmodified reference + shims).

TEST INFRASTRUCTURE ONLY: used to pin the oracle and to generate golden fixtures in the
build container; it is not available where /root/reference was never mounted unless the
prebuilt .so travelled with the snapshot.
"""
import ctypes as C
import hashlib
import json
import os
import sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref_lfbm5d.so")
PINS = os.path.join(HERE, "golden", "ref_pins.json")

YUV, YCBCR, OPP, RGB, ID, DCT, SADCT, BIOR, HADAMARD, HAAR, NONE, ROWMAJOR, COLMAJOR = range(13)

_lib = None


def available():
    return os.path.exists(REF_SO)


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(REF_SO)
        _lib.ref_LF_denoised_percent.restype = C.c_float
        _lib.ref_mt_res53.restype = C.c_double
        _lib.ref_ind_initialize.restype = C.c_uint
    return _lib


def _values(x):
    return tuple(x) if isinstance(x, (tuple, list)) else (x,)


def digest(values):
    """SHA-256 over dtype, shape and bytes of each value: equal digests mean bit-identical values."""
    h = hashlib.sha256()
    for v in _values(values):
        a = np.ascontiguousarray(np.asarray(v))
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


class Pinned:
    """The reference's side of the oracle-vs-reference comparisons. Where oracle/_ref is built, `check` compares with the
    reference live. Elsewhere it compares the SHA-256 of the values under test with the digest stored in
    tests/golden/ref_pins.json, which holds the reference's values on the same seeded inputs. With LFBM5D_RECORD_REF_PINS=1
    the digests of the checked values are written back to that file: python -m pytest tests/test_oracle_vs_ref.py
    tests/test_host_io.py -k "not gpu"."""

    def __init__(self):
        self.live = available()
        self.record = os.environ.get("LFBM5D_RECORD_REF_PINS") == "1"
        self.pins = {}
        if os.path.exists(PINS):
            with open(PINS) as f:
                self.pins = json.load(f)

    def check(self, key, got, want):
        """got: the values under test (an array or a tuple of them); want(refapi): the same values computed by the reference."""
        if self.live:
            w = _values(want(sys.modules[__name__]))
            g = _values(got)
            assert len(g) == len(w) and all(np.array_equal(a, b) for a, b in zip(g, w)), key
        if self.record:
            self.pins[key] = digest(got)
        elif not self.live:
            assert key in self.pins, "no stored reference values for %s (tests/golden/ref_pins.json)" % key
            assert digest(got) == self.pins[key], key

    def save(self):
        with open(PINS, "w") as f:
            json.dump(self.pins, f, indent=0, sort_keys=True)
            f.write("\n")


def fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def up(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint))


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def run_step1(noisy, mask, sigma, lam, aw, ah, an, N, nSim, nDisp, k, p, tau2, tau4, tau5, cs=OPP,
              useSD=False, ang_major=ROWMAJOR, nb_threads=1):
    """noisy: [asize, C, H, W] float32 RGB. Returns (basic, noisy_roundtrip)."""
    A, Cn, H, W = noisy.shape
    n = f32(noisy).copy()
    basic = np.zeros_like(n)
    m = u32(mask)
    rc = lib().ref_run_bm5d_1st_step(C.c_float(sigma), C.c_float(lam), fp(n), up(m), fp(basic), ang_major, aw, ah, an,
                                     W, H, Cn, N, nSim, nDisp, k, p, int(useSD), tau2, tau4, tau5, cs, nb_threads)
    assert rc == 0
    return basic, n


def run_step2(noisy, basic, mask, sigma, aw, ah, an, N, nSim, nDisp, k, p, tau2, tau4, tau5, cs=OPP,
              useSD=False, ang_major=ROWMAJOR, nb_threads=1):
    A, Cn, H, W = noisy.shape
    n = f32(noisy).copy()
    b = f32(basic).copy()
    den = np.zeros_like(n)
    m = u32(mask)
    rc = lib().ref_run_bm5d_2nd_step(C.c_float(sigma), fp(n), up(m), fp(b), fp(den), ang_major, aw, ah, an,
                                     W, H, Cn, N, nSim, nDisp, k, p, int(useSD), tau2, tau4, tau5, cs, nb_threads)
    assert rc == 0
    return den, b, n


def pass_step1(noisy_sym, num_sym, den_sym, mask, proc, cst, pst, asw, sigma, lam, nSim, nDisp, k, N, p,
               tau2, tau4, tau5, cs=OPP, useSD=False):
    """One window pass on padded buffers [A, C, h_b, w_b]; returns updated (num, den)."""
    A, Cn, hb, wb = noisy_sym.shape
    num = f32(num_sym).copy()
    den = f32(den_sym).copy()
    lib().ref_bm5d_1st_step_pass(C.c_float(sigma), C.c_float(lam), fp(f32(noisy_sym)), fp(num), fp(den), up(u32(mask)),
                                 up(u32(proc)), cst, pst, asw, wb, hb, Cn, nSim, nDisp, k, N, p, int(useSD), cs,
                                 tau2, tau4, tau5)
    return num, den


def pass_step2(noisy_sym, basic_sym, num_sym, den_sym, mask, proc, cst, pst, asw, sigma, nSim, nDisp, k, N, p,
               tau2, tau4, tau5, cs=OPP, useSD=False):
    A, Cn, hb, wb = noisy_sym.shape
    num = f32(num_sym).copy()
    den = f32(den_sym).copy()
    lib().ref_bm5d_2nd_step_pass(C.c_float(sigma), fp(f32(noisy_sym)), fp(f32(basic_sym)), fp(num), fp(den),
                                 up(u32(mask)), up(u32(proc)), cst, pst, asw, wb, hb, Cn, nSim, nDisp, k, N, p,
                                 int(useSD), cs, tau2, tau4, tau5)
    return num, den


def precompute_bm(img, k, N, nHW, nSim, p, tau):
    h, w = img.shape
    cnt = np.zeros(h * w, np.uint32)
    idx = np.zeros((h * w, N + 1), np.uint32)
    lib().ref_precompute_BM(fp(f32(img)), w, h, k, N, nHW, nSim, p, C.c_float(tau), up(cnt), up(idx), N + 1)
    return cnt, idx


def precompute_bm_stereo(img1, img2, k, nHW, nDisp, tau, want_all=False):
    h, w = img1.shape
    first = np.zeros(h * w, np.uint32)
    shape = np.zeros(h * w, np.uint32)
    Ns2 = (2 * nDisp + 1) ** 2
    allv = np.zeros((h * w, Ns2), np.uint32) if want_all else None
    rc = lib().ref_precompute_BM_stereo(fp(f32(img1)), fp(f32(img2)), w, h, k, nHW, nDisp, 1, C.c_float(tau), up(first),
                                        up(shape), up(allv) if want_all else None)
    assert rc == 0
    return first, shape, allv


def run_bm3d_lf(noisy, mask, sigma, nHard, nWien, kHard, kWien, NHard, NWien, pHard, pWien, tau2h, tau2w, lam, cs=OPP, nb_threads=1):
    A, Cn, H, W = noisy.shape
    n = f32(noisy).copy()
    basic = np.zeros_like(n)
    den = np.zeros_like(n)
    rc = lib().ref_run_bm3d_LF(C.c_float(sigma), fp(n), up(u32(mask)), fp(basic), fp(den), A, W, H, Cn, nHard, nWien, kHard, kWien,
                               NHard, NWien, pHard, pWien, 0, 0, tau2h, tau2w, C.c_float(lam), cs, nb_threads)
    assert rc == 0
    return basic, den, n
