"""lfbm5d_b200 — B200-native (sm_100a CUDA) LFBM5D light-field denoising hot path.

This package is a thin ctypes view of the C ABI in include/lfbm5d_cuda.h (the drop-in boundary);
the C++ adapters with the reference's own signatures live in csrc/lfbm5d_host.{h,cpp}.
There is no CPU fallback: if the CUDA library is missing or no GPU is present, calls raise.

Reference interface mirrored (V-Sense/LFBM5D): run_bm5d_1st_step / run_bm5d_2nd_step (bm5d.h:11-62),
run_bm3d_LF (bm3d_LF.h:10-35); enum values are the reference's #defines (main.cpp:20-32).
"""
import ctypes as C
import os

import numpy as np

YUV, YCBCR, OPP, RGB, ID, DCT, SADCT, BIOR, HADAMARD, HAAR, NONE, ROWMAJOR, COLMAJOR = range(13)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "liblfbm5d_cuda.so")


class Params(C.Structure):
    """POD mirror of lfbm5d_params (include/lfbm5d_cuda.h)."""
    _fields_ = [("sigma", C.c_float), ("lambda_", C.c_float), ("ang_major", C.c_uint), ("awidth", C.c_uint),
                ("aheight", C.c_uint), ("an", C.c_uint), ("width", C.c_uint), ("height", C.c_uint), ("chnls", C.c_uint),
                ("N", C.c_uint), ("nSim", C.c_uint), ("nDisp", C.c_uint), ("k", C.c_uint), ("p", C.c_uint),
                ("useSD", C.c_uint), ("tau_2D", C.c_uint), ("tau_4D", C.c_uint), ("tau_5D", C.c_uint),
                ("color_space", C.c_uint), ("nb_threads", C.c_uint)]


class Params3D(C.Structure):
    """POD mirror of lfbm3d_params (include/lfbm5d_cuda.h)."""
    _fields_ = [("sigma", C.c_float), ("asize", C.c_uint), ("width", C.c_uint), ("height", C.c_uint), ("chnls", C.c_uint),
                ("nHard", C.c_uint), ("nWien", C.c_uint), ("kHard", C.c_uint), ("kWien", C.c_uint), ("NHard", C.c_uint),
                ("NWien", C.c_uint), ("pHard", C.c_uint), ("pWien", C.c_uint), ("useSD_h", C.c_uint), ("useSD_w", C.c_uint),
                ("tau_2D_hard", C.c_uint), ("tau_2D_wien", C.c_uint), ("lambdaHard3D", C.c_float), ("color_space", C.c_uint),
                ("nb_threads", C.c_uint)]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_ulonglong), ("window_passes", C.c_uint), ("ms_block_matching", C.c_float),
                ("ms_groups", C.c_float), ("ms_aggregate", C.c_float), ("ms_other", C.c_float), ("ms_sat", C.c_float)]


EXPORTS = ["lfbm5d_create", "lfbm5d_destroy", "lfbm5d_last_error", "lfbm5d_reset_stats", "lfbm5d_get_stats",
           "lfbm5d_enable_timing", "lfbm5d_stream", "lfbm5d_step1", "lfbm5d_step2", "lfbm3d_run", "lfbm5d_step1_device",
           "lfbm5d_step2_device", "lfbm3d_run_device", "lfbm5d_set_max_passes", "lfbm5d_group_cluster", "lfbm5d_group_kernel", "lfbm5d_debug_pass", "lfbm5d_debug_pass_ex",
           "lfbm5d_debug_schedule", "lfbm5d_step_plan", "lfbm5d_debug_block_matching", "lfbm5d_team_create_emulated", "lfbm5d_team_unique_id",
           "lfbm5d_team_create_nccl", "lfbm5d_team_destroy", "lfbm5d_team_local_ranks", "lfbm5d_team_step", "lfbm5d_team_band",
           "lfbm5d_team_stats", "lfbm5d_team_disable_peer_view", "lfbm5d_team_timing", "lfbm5d_team_plan_band", "lfbm5d_copy_rows", "lfbm5d_sync", "lfbm5d_team_use_peer_exchange", "lfbm5d_team_set_lanes", "lfbm5d_team_launches"]

HOST_LIB_PATH = os.path.join(_HERE, "_lib", "liblfbm5d_host.so")
HOST_EXPORTS = ["lfio_add_noise", "lfio_psnr", "lfio_png_read", "lfio_png_write", "lfio_psnr_LF", "lfio_diff_LF", "lfio_write_psnr_LF", "lfio_load_LF", "lfio_save_LF"]      # include/lfbm5d_host_c.h

_lib = None
_host = None


def load_host_library():
    """liblfbm5d_host.so: C++ adapters with the reference's signatures + the C exports of include/lfbm5d_host_c.h."""
    global _host
    if _host is None:
        load_library()
        if not os.path.exists(HOST_LIB_PATH):
            raise RuntimeError("%s not found: run __graft_entry__.build()" % HOST_LIB_PATH)
        _host = C.CDLL(HOST_LIB_PATH)
    return _host


def add_noise(clean, sigma, seed0=20171016, threads=None):
    """The reference's host noise (utilities.cpp:154-185, mt19937ar + Box-Muller): SAI st uses its own generator seeded
    seed0 + st; unclipped float32. clean [asize, C, H, W]. SAIs are independent, so they are generated on `threads` host threads."""
    from concurrent.futures import ThreadPoolExecutor
    h = load_host_library()
    src = np.ascontiguousarray(clean, np.float32)
    out = np.empty_like(src)

    def one(st):
        h.lfio_add_noise(_fp(src[st]), _fp(out[st]), C.c_size_t(src[st].size), C.c_float(sigma), C.c_ulong(seed0 + st))
    with ThreadPoolExecutor(max_workers=threads or min(32, os.cpu_count() or 1)) as ex:
        list(ex.map(one, range(src.shape[0])))
    return out


def psnr(a, b):
    """compute_psnr (utilities.cpp:412-435) of two images -> (psnr, rmse)."""
    h = load_host_library()
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    p, r = C.c_float(), C.c_float()
    h.lfio_psnr(_fp(a), _fp(b), C.c_size_t(a.size), C.byref(p), C.byref(r))
    return p.value, r.value


def psnr_lf(a, b):
    """Mean over the SAIs of the per-SAI PSNR (compute_psnr_LF, utilities_LF.cpp:639-700)."""
    return float(np.mean([psnr(a[st], b[st])[0] for st in range(a.shape[0])]))


def load_library():
    """Load the CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)" % LIB_PATH)
        _lib = C.CDLL(LIB_PATH)
        _lib.lfbm5d_last_error.restype = C.c_char_p
        _lib.lfbm5d_stream.restype = C.c_void_p
        _lib.lfbm5d_debug_schedule.restype = C.c_uint
    return _lib


def make_params(sigma, lam, aw, ah, an, width, height, chnls, N, nSim, nDisp, k, p, tau_2D, tau_4D, tau_5D,
                color_space=OPP, ang_major=ROWMAJOR, useSD=0, nb_threads=1):
    return Params(sigma, lam, ang_major, aw, ah, an, width, height, chnls, N, nSim, nDisp, k, p, useSD, tau_2D, tau_4D,
                  tau_5D, color_space, nb_threads)


def make_params3d(sigma, asize, width, height, chnls, nHard, nWien, kHard, kWien, NHard, NWien, pHard, pWien, tau_2D_hard,
                  tau_2D_wien, lambdaHard3D=2.7, color_space=OPP, nb_threads=1):
    return Params3D(sigma, asize, width, height, chnls, nHard, nWien, kHard, kWien, NHard, NWien, pHard, pWien, 0, 0, tau_2D_hard,
                    tau_2D_wien, lambdaHard3D, color_space, nb_threads)


def step_plan(prm, mask):
    """Static window schedule of a step: rows (ps, pt, min_s, min_t, level, sadct); windows of one level share no SAI."""
    lib = load_library()
    m = np.ascontiguousarray(mask, np.uint32)
    out = np.zeros((int(prm.awidth * prm.aheight) + 1, 6), np.uint32)
    lib.lfbm5d_step_plan.restype = C.c_uint
    n = lib.lfbm5d_step_plan(C.byref(prm), m.ctypes.data_as(C.POINTER(C.c_uint)), out.ctypes.data_as(C.POINTER(C.c_uint)), out.shape[0])
    return out[:n]


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _up(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_uint))


class LFBM5D(object):
    """One context per GPU. Host-array methods copy in and out (the reference-facing path)."""

    def __init__(self, device=0):
        self.lib = load_library()
        self.ctx = C.c_void_p()
        if self.lib.lfbm5d_create(C.byref(self.ctx), int(device)) != 0:
            raise RuntimeError("lfbm5d_create: " + self.error())

    def error(self):
        return self.lib.lfbm5d_last_error().decode()

    def close(self):
        if self.ctx:
            self.lib.lfbm5d_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- bookkeeping --------------------------------------------------------------------------
    def reset_stats(self):
        self.lib.lfbm5d_reset_stats(self.ctx)

    def stats(self):
        s = Stats()
        self.lib.lfbm5d_get_stats(self.ctx, C.byref(s))
        return s

    def enable_timing(self, on=True):
        self.lib.lfbm5d_enable_timing(self.ctx, int(on))

    def set_max_passes(self, n):
        self.lib.lfbm5d_set_max_passes(self.ctx, int(n))

    def stream(self):
        return self.lib.lfbm5d_stream(self.ctx)

    def group_cluster(self, step, prm):
        """(cluster size, cudaOccupancyMaxActiveClusters) of the group kernel of `step` with these parameters: (1, 0) when one
        CTA holds a group."""
        cl, occ = C.c_int(0), C.c_int(0)
        if self.lib.lfbm5d_group_cluster(self.ctx, int(step), C.byref(prm), C.byref(cl), C.byref(occ)) != 0:
            raise RuntimeError(self.error())
        return cl.value, occ.value

    def group_kernel(self, step, prm):
        """Name of the group kernel a window pass of `step` launches with these parameters, e.g. "k_groups_w8<3>" (debug)."""
        buf = C.create_string_buffer(64)
        if self.lib.lfbm5d_group_kernel(self.ctx, int(step), C.byref(prm), buf, len(buf)) != 0:
            raise RuntimeError(self.error())
        return buf.value.decode()

    def schedule(self, max_entries=4096):
        out = np.zeros((max_entries, 4), np.uint32)
        n = self.lib.lfbm5d_debug_schedule(self.ctx, _up(out), max_entries)
        return out[:n]

    # -- host-buffer entry points (like run_bm5d_1st_step / run_bm5d_2nd_step) --------------------
    @staticmethod
    def _ptrs(arr):
        n = arr.shape[0]
        return (C.POINTER(C.c_float) * n)(*[_fp(arr[i]) for i in range(n)])

    def step1(self, prm, noisy, mask):
        """noisy [asize, C, H, W] float32 RGB -> (basic, noisy round-tripped through the colour space)."""
        n = np.ascontiguousarray(noisy, np.float32).copy()
        basic = np.zeros_like(n)
        m = np.ascontiguousarray(mask, np.uint32)
        if self.lib.lfbm5d_step1(self.ctx, C.byref(prm), self._ptrs(n), _up(m), self._ptrs(basic)) != 0:
            raise RuntimeError("lfbm5d_step1: " + self.error())
        return basic, n

    def step2(self, prm, noisy, basic, mask):
        n = np.ascontiguousarray(noisy, np.float32).copy()
        b = np.ascontiguousarray(basic, np.float32).copy()
        out = np.zeros_like(n)
        m = np.ascontiguousarray(mask, np.uint32)
        if self.lib.lfbm5d_step2(self.ctx, C.byref(prm), self._ptrs(n), self._ptrs(b), _up(m), self._ptrs(out)) != 0:
            raise RuntimeError("lfbm5d_step2: " + self.error())
        return out, b, n

    def bm3d(self, prm3, noisy, mask):
        """run_bm3d_LF on host arrays [asize, C, H, W] -> (basic, denoised, noisy round-tripped)."""
        n = np.ascontiguousarray(noisy, np.float32).copy()
        basic, out = np.zeros_like(n), np.zeros_like(n)
        m = np.ascontiguousarray(mask, np.uint32)
        if self.lib.lfbm3d_run(self.ctx, C.byref(prm3), self._ptrs(n), _up(m), self._ptrs(basic), self._ptrs(out)) != 0:
            raise RuntimeError("lfbm3d_run: " + self.error())
        return basic, out, n

    def bm3d_device(self, prm3, d_noisy, mask, d_basic, d_out):
        m = np.ascontiguousarray(mask, np.uint32)
        if self.lib.lfbm3d_run_device(self.ctx, C.byref(prm3), C.c_void_p(d_noisy), _up(m), C.c_void_p(d_basic), C.c_void_p(d_out)) != 0:
            raise RuntimeError("lfbm3d_run_device: " + self.error())

    # -- device-resident entry points (raw device pointers, e.g. torch tensors' data_ptr()) -------
    def step1_device(self, prm, d_noisy, mask, d_basic):
        m = np.ascontiguousarray(mask, np.uint32)
        if self.lib.lfbm5d_step1_device(self.ctx, C.byref(prm), C.c_void_p(d_noisy), _up(m), C.c_void_p(d_basic)) != 0:
            raise RuntimeError("lfbm5d_step1_device: " + self.error())

    def step2_device(self, prm, d_noisy, d_basic, mask, d_out):
        m = np.ascontiguousarray(mask, np.uint32)
        if self.lib.lfbm5d_step2_device(self.ctx, C.byref(prm), C.c_void_p(d_noisy), C.c_void_p(d_basic), _up(m),
                                        C.c_void_p(d_out)) != 0:
            raise RuntimeError("lfbm5d_step2_device: " + self.error())

    def copy_rows(self, host_ptrs, d_lf, mask, asize, chnls, width, height, row_lo, row_hi, to_device):
        """Rows [row_lo, row_hi) of every plane between host arrays (ctypes array of asize float pointers) and a device light field;
        asynchronous on the engine's stream (sync() waits)."""
        m = np.ascontiguousarray(mask, np.uint32)
        if self.lib.lfbm5d_copy_rows(self.ctx, host_ptrs, C.c_void_p(d_lf), _up(m), int(asize), int(chnls), int(width), int(height),
                                     int(row_lo), int(row_hi), int(to_device)) != 0:
            raise RuntimeError("lfbm5d_copy_rows: " + self.error())

    def sync(self):
        if self.lib.lfbm5d_sync(self.ctx) != 0:
            raise RuntimeError("lfbm5d_sync: " + self.error())

    def debug_block_matching(self, step, prm, planes):
        """planes [nplanes, hb, wb] channel-0 estimates (plane 0 = reference SAI) -> (count, idx, first, shape)."""
        pl = np.ascontiguousarray(planes, np.float32)
        npl, hb, wb = pl.shape
        cnt, idx = np.zeros(hb * wb, np.uint32), np.zeros((hb * wb, prm.N + 1), np.uint32)
        first, shape = np.zeros((npl, hb * wb), np.uint32), np.zeros((npl, hb * wb), np.uint32)
        if self.lib.lfbm5d_debug_block_matching(self.ctx, int(step), C.byref(prm), _fp(pl), npl, _up(cnt), _up(idx), _up(first), _up(shape)) != 0:
            raise RuntimeError("lfbm5d_debug_block_matching: " + self.error())
        return cnt, idx, first, shape

    # -- parity/debug: one window pass on padded host buffers --------------------------------------
    def debug_pass(self, step, prm, noisy_sym, basic_sym, num_sym, den_sym, mask, proc, pst, debug=False, cst=None):
        A, Cn, hb, wb = noisy_sym.shape
        ns = np.ascontiguousarray(noisy_sym, np.float32)
        bs = None if basic_sym is None else np.ascontiguousarray(basic_sym, np.float32)
        num = np.ascontiguousarray(num_sym, np.float32).copy()
        den = np.ascontiguousarray(den_sym, np.float32).copy()
        dbg = [None] * 4
        if debug:
            dbg = [np.zeros(hb * wb, np.uint32), np.zeros((hb * wb, prm.N + 1), np.uint32),
                   np.zeros((A, hb * wb), np.uint32), np.zeros((A, hb * wb), np.uint32)]
        rc = self.lib.lfbm5d_debug_pass_ex(self.ctx, int(step), C.byref(prm), _fp(ns), None if bs is None else _fp(bs),
                                           _fp(num), _fp(den), _up(np.ascontiguousarray(mask, np.uint32)),
                                           _up(np.ascontiguousarray(proc, np.uint32)), int(pst if cst is None else cst), int(pst),
                                           *[_up(d) for d in dbg])
        if rc != 0:
            raise RuntimeError("lfbm5d_debug_pass: " + self.error())
        return (num, den, dbg) if debug else (num, den)


def plan_band(world, rank, step, prm):
    """(row_lo, row_hi, keep_hi) of rank `rank` in a team of `world` ranks for a step with parameters prm (before it runs)."""
    lib = load_library()
    lo, hi, keep = C.c_int(), C.c_int(), C.c_int()
    if lib.lfbm5d_team_plan_band(int(world), int(rank), int(step), C.byref(prm), C.byref(lo), C.byref(hi), C.byref(keep)) != 0:
        raise RuntimeError("lfbm5d_team_plan_band: " + lib.lfbm5d_last_error().decode())
    return lo.value, hi.value, keep.value


class Team(object):
    """One light field on several GPUs: the ranks of a team split every window pass (include/lfbm5d_cuda.h, csrc/team.cuh).
    Team.nccl: one process per GPU (this process is rank `rank`); Team.emulated: `world` ranks on ONE device (tests)."""

    def __init__(self, handle, engine=None):
        self.lib = load_library()
        self.handle = handle
        self.engine = engine          # keeps the context of an NCCL team alive

    @classmethod
    def emulated(cls, device, world):
        lib = load_library()
        h = C.c_void_p()
        if lib.lfbm5d_team_create_emulated(C.byref(h), int(device), int(world)) != 0:
            raise RuntimeError("lfbm5d_team_create_emulated: " + lib.lfbm5d_last_error().decode())
        return cls(h)

    @staticmethod
    def unique_id():
        lib = load_library()
        buf = C.create_string_buffer(128)
        if lib.lfbm5d_team_unique_id(buf) != 0:
            raise RuntimeError("lfbm5d_team_unique_id: " + lib.lfbm5d_last_error().decode())
        return buf.raw

    @classmethod
    def nccl(cls, engine, rank, world, unique_id):
        lib = load_library()
        h = C.c_void_p()
        if lib.lfbm5d_team_create_nccl(C.byref(h), engine.ctx, int(rank), int(world), C.c_char_p(bytes(unique_id))) != 0:
            raise RuntimeError("lfbm5d_team_create_nccl: " + lib.lfbm5d_last_error().decode())
        return cls(h, engine)

    def close(self):
        if self.handle:
            self.lib.lfbm5d_team_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def local_ranks(self):
        return int(self.lib.lfbm5d_team_local_ranks(self.handle))

    def step(self, step, prm, d_noisy, d_basic, mask, d_out, gather=0):
        """d_noisy / d_basic / d_out: lists of device pointers, one per local rank (d_basic ignored for step 1)."""
        n = self.local_ranks()
        arr = lambda ptrs: (C.c_void_p * n)(*[C.c_void_p(int(x)) for x in ptrs])
        m = np.ascontiguousarray(mask, np.uint32)
        rc = self.lib.lfbm5d_team_step(self.handle, int(step), C.byref(prm), arr(d_noisy), arr(d_basic) if int(step) == 2 else None, _up(m),
                                       arr(d_out), int(gather))
        if rc != 0:
            raise RuntimeError("lfbm5d_team_step: " + self.lib.lfbm5d_last_error().decode())

    def band(self, rank):
        """(row_lo, row_hi, keep_hi): rank owns the interior rows [row_lo, row_hi) and holds valid results on [row_lo, keep_hi)."""
        lo, hi, keep = C.c_int(), C.c_int(), C.c_int()
        if self.lib.lfbm5d_team_band(self.handle, int(rank), C.byref(lo), C.byref(hi), C.byref(keep)) != 0:
            raise RuntimeError("lfbm5d_team_band: " + self.lib.lfbm5d_last_error().decode())
        return lo.value, hi.value, keep.value

    def stats(self):
        b, r, t, pv = C.c_ulonglong(), C.c_uint(), C.c_ulonglong(), C.c_int()
        self.lib.lfbm5d_team_stats(self.handle, C.byref(b), C.byref(r), C.byref(t), C.byref(pv))
        return {"bytes_exchanged": int(b.value), "passes_redone": int(r.value), "tie_patches": int(t.value), "peer_view": bool(pv.value)}

    def timing(self, on=True):
        """Switch the per-phase timing on / off; returns the ms accumulated so far for (pad, est0 exchange, block matching, match
        exchange, selection + groups + aggregation 1, border exchange, aggregation 2, border + counter exchange; inside block matching:
        self planes, partial selection, disparity planes, disparity argmin)."""
        out = (C.c_float * 12)()
        self.lib.lfbm5d_team_timing(self.handle, int(on), out)
        return [float(x) for x in out]

    def set_lanes(self, n):
        """n windows of a plan level run concurrently (each lane: own pass buffers); results do not change."""
        if self.lib.lfbm5d_team_set_lanes(self.handle, int(n)) != 0:
            raise RuntimeError("lfbm5d_team_set_lanes: " + self.lib.lfbm5d_last_error().decode())

    def launches(self):
        self.lib.lfbm5d_team_launches.restype = C.c_ulonglong
        return int(self.lib.lfbm5d_team_launches(self.handle))

    def use_peer_exchange(self, on=True):
        self.lib.lfbm5d_team_use_peer_exchange(self.handle, int(on))

    def disable_peer_view(self):
        self.lib.lfbm5d_team_disable_peer_view(self.handle)
