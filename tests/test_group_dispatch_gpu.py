"""Every branch of the group-kernel dispatch against the CPU oracle. launch_groups picks one of the group kernels from (step, k, an,
N, C, tau_2D, tau_5D, useSD); each row here first asserts which kernel its parameters select (eng.group_kernel), so that a moved
dispatch condition fails the row instead of quietly testing another kernel, and then runs one window pass through gpucheck.check_pass
on 40 x 48 inputs with a flat region (groups of N patches) and a region of strong noise (groups of 2): RGB, or its channel 0 where
C = 1. Match tables bit-exact, step 1 bit-identical, step 2 within STEP2_REL and useSD within STEP2_REL_SD of the exact-sum oracle.

The an = 0 rows (a window of one SAI, k_groups<S,1>) are checked against the oracle only: its angular code is generic in the window
size but pinned against the reference at asw = 3, and the reference is not part of this tree."""
import numpy as np
import pytest

import lfdata
from gpucheck import check_complete_run, check_pass, eng, estimate, psnr_on, spread_inputs  # noqa: F401 (eng is the engine fixture)

pytestmark = pytest.mark.gpu

T = {"id": 4, "dct": 5, "sadct": 6, "bior": 7, "hw": 8, "haar": 9}      # tau values of include/lfbm5d_cuda.h (= oracleapi's)


def _rows():
    """(step, k, an, N, C, tau_2D, tau_4D, tau_5D, useSD, expected kernel)"""
    r = []
    for N in (1, 2, 4):                                                  # id16 with nSx = 1 and small groups
        r.append((1, 16, 1, N, 3, "id", "sadct", "haar", 0, "k_groups_id16<3>"))
    for t4 in ("id", "dct", "sadct"):
        for t5 in ("haar", "hw"):
            r.append((1, 16, 1, 8, 3, "id", t4, t5, 0, "k_groups_id16<3>"))
    r.append((1, 16, 1, 8, 1, "id", "sadct", "haar", 0, "k_groups_id16<1>"))
    for t2 in ("id", "dct", "bior"):
        r.append((1, 16, 1, 16, 3, t2, "sadct", "haar", 0, "k_groups<1,3>"))      # first N past id16; 156,672 B with dct / bior
        r.append((1, 8, 1, 32, 3, t2, "sadct", "haar", 0, "k_groups<1,3>"))
    r.append((2, 8, 1, 1, 3, "dct", "sadct", "haar", 0, "k_groups_w8<3>"))         # w8 with nSx = 1
    r.append((2, 8, 1, 16, 1, "dct", "sadct", "haar", 0, "k_groups_w8<1>"))
    r.append((2, 8, 1, 32, 3, "dct", "sadct", "haar", 0, "k_groups<2,3>"))         # first N past w8: 165,888 B
    for t2 in ("id", "bior"):
        r.append((2, 8, 1, 16, 3, t2, "sadct", "haar", 0, "k_groups<2,3>"))       # tau_2D excludes w8
    for N in (1, 2, 4, 8):
        for t2 in ("id", "dct", "bior"):
            r.append((2, 16, 1, N, 3, t2, "sadct", "haar", 0, "k_groups<2,3>"))
    for t4 in ("id", "dct", "sadct"):
        for t5 in ("haar", "hw", "dct"):
            if (t4, t5) != ("sadct", "haar"):
                r.append((2, 16, 1, 8, 3, "dct", t4, t5, 0, "k_groups<2,3>"))     # 156,672 B
    r.append((2, 16, 1, 8, 1, "dct", "sadct", "haar", 0, "k_groups<2,3>"))
    # useSD on the largest groups one CTA holds
    r.append((1, 16, 1, 8, 3, "id", "sadct", "haar", 1, "k_groups<1,3>"))
    r.append((1, 16, 1, 16, 3, "bior", "sadct", "haar", 1, "k_groups<1,3>"))
    r.append((2, 8, 1, 32, 3, "dct", "sadct", "haar", 1, "k_groups<2,3>"))
    r.append((2, 16, 1, 8, 3, "dct", "sadct", "haar", 1, "k_groups<2,3>"))
    for step in (1, 2):                                                  # an = 0: one SAI per window
        for k in (8, 16):
            for N in (1, 8, 32):
                for C in (3, 1):
                    for t2 in ("id", "dct", "bior"):
                        r.append((step, k, 0, N, C, t2, "sadct", "haar", 0, "k_groups<%d,1>" % step))
    return r


ROWS = _rows()


def _row_id(r):
    return "s%d-k%d-an%d-N%d-C%d-%s-%s-%s%s" % (r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], "-sd" if r[8] else "")


@pytest.fixture(scope="module")
def inputs(oracle):
    """The padded 3x3 light field and a basic estimate for step 2: the oracle's step-1 pass at the README's step-1 parameters."""
    sym = spread_inputs()
    z = np.zeros_like(sym)
    on, od = oracle.run_pass(1, sym, None, z, z, np.ones(9, np.uint32), np.zeros(9, np.uint32), 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4,
                             oracle.ID, oracle.SADCT, oracle.HAAR)
    return sym, estimate(on, od, sym)


@pytest.mark.parametrize("row", ROWS, ids=[_row_id(r) for r in ROWS])
def test_group_kernel_pass(eng, oracle, inputs, row):
    import lfbm5d_b200 as L
    step, k, an, N, C, t2, t4, t5, useSD, kernel = row
    sym, basic = inputs
    sais = slice(None) if an == 1 else slice(4, 5)                      # an = 0: the centre SAI alone
    sym, basic = np.ascontiguousarray(sym[sais, :C]), np.ascontiguousarray(basic[sais, :C])
    A, _, hb, wb = sym.shape
    lam = 2.7 if step == 1 else 0.0
    prm = L.make_params(25.0, lam, 2 * an + 1, 2 * an + 1, an, wb - 48, hb - 48, C, N, 18, 6, k, 4, T[t2], T[t4], T[t5], useSD=useSD)
    assert eng.group_kernel(step, prm) == kernel
    z = np.zeros_like(sym)
    gdbg = check_pass(eng, oracle, step, sym, basic if step == 2 else None, z, z, np.ones(A, np.uint32), np.zeros(A, np.uint32), k, N,
                      T[t2], T[t4], T[t5], an=an, lam=lam, useSD=useSD)[4]
    assert (gdbg[0] == N).any()                                          # some groups are full


def test_quantised_ties_k16_step2(eng, oracle):
    """k = 16 step 2 at N = 8 on one CTA on coarse grey levels: exact distance ties, groups of N patches."""
    import golden_inputs as gi
    import lfbm5d_b200 as L
    _, _, sym = gi.pad_inputs(40, 48, 25.0)
    q = (np.round(sym / 64.0) * 64.0).astype(np.float32)
    z = np.zeros_like(q)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    prm = L.make_params(25.0, 0.0, 3, 3, 1, 48, 40, 3, 8, 18, 6, 16, 4, L.DCT, L.SADCT, L.HAAR)
    assert eng.group_kernel(2, prm) == "k_groups<2,3>"
    on, od, _, _, _ = check_pass(eng, oracle, 1, q, None, z, z, mask, proc, 16, 8, oracle.ID, oracle.SADCT, oracle.HAAR)
    gdbg = check_pass(eng, oracle, 2, q, estimate(on, od, q), z, z, mask, proc, 16, 8, oracle.DCT, oracle.SADCT, oracle.HAAR, lam=0.0)[4]
    cnt = gdbg[0][gdbg[0] > 0]
    assert (cnt == 8).all(), np.unique(cnt, return_counts=True)


@pytest.mark.parametrize("C,masked", [(3, False), (1, True)])
def test_complete_runs_an0(eng, oracle, C, masked):
    """Both steps at an = 0 (`8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar`) through the host-buffer and the
    device-resident entry points, against the oracle; grayscale with an empty centre SAI."""
    import lfbm5d_b200 as L
    H, W = 32, 36
    clean = np.ascontiguousarray(lfdata.synth_lf(3, 3, H, W)[:, :C])
    m = np.ones(9, np.uint32)
    if masked:
        m[4] = 0
    p1 = L.make_params(25.0, 2.7, 3, 3, 0, W, H, C, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, 3, 3, 0, W, H, C, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    assert eng.group_kernel(1, p1) == "k_groups<1,1>" and eng.group_kernel(2, p2) == "k_groups<2,1>"
    noisy, _, _, d, _, _ = check_complete_run(eng, oracle, clean, m, p1, p2)
    psnr = psnr_on(clean, m)
    assert psnr(d) > psnr(noisy) + 3.0


# One parameter set per group kernel the dispatch can select: (step, k, an, N, C, tau_2D, tau_5D, useSD) -> kernel
KERNELS = [
    ((1, 16, 1, 8, 3, "id", "haar", 0), "k_groups_id16<3>"),
    ((1, 16, 1, 8, 1, "id", "haar", 0), "k_groups_id16<1>"),
    ((2, 8, 1, 16, 3, "dct", "haar", 0), "k_groups_w8<3>"),
    ((2, 8, 1, 16, 1, "dct", "haar", 0), "k_groups_w8<1>"),
    ((1, 16, 1, 16, 3, "dct", "haar", 0), "k_groups<1,3>"),
    ((2, 8, 1, 32, 3, "dct", "haar", 0), "k_groups<2,3>"),
    ((1, 16, 0, 8, 3, "id", "haar", 0), "k_groups<1,1>"),
    ((2, 8, 0, 16, 3, "dct", "haar", 0), "k_groups<2,1>"),
    ((1, 12, 1, 16, 3, "id", "haar", 0), "k_groups12<1,3>"),
    ((2, 12, 1, 16, 3, "dct", "haar", 0), "k_groups12<2,3>"),
    ((1, 12, 0, 16, 3, "id", "haar", 0), "k_groups12<1,1>"),
    ((2, 12, 0, 16, 3, "dct", "haar", 0), "k_groups12<2,1>"),
    ((1, 16, 2, 8, 3, "id", "haar", 0), "k_groups25<1>"),
    ((2, 8, 2, 16, 3, "dct", "haar", 0), "k_groups25<2>"),
    ((1, 16, 1, 32, 3, "id", "haar", 0), "k_groups_cl<1,2>"),
    ((2, 16, 1, 16, 3, "dct", "haar", 0), "k_groups_cl<2,2>"),
    ((2, 16, 1, 32, 3, "dct", "haar", 0), "k_groups_cl<2,4>"),
]


def test_every_group_kernel_has_a_row(eng):
    """The names the dispatch returns for KERNELS are exactly the kernels it can select. k_groups_cl<1,4> is compiled but not among
    them: a step-1 group (N <= 32) needs at most 2 CTAs. A kernel the dispatch gains without a row here fails this test."""
    import lfbm5d_b200 as L
    got = []
    for (step, k, an, N, C, t2, t5, useSD), want in KERNELS:
        aw = 5 if an == 2 else 3
        prm = L.make_params(25.0, 2.7 if step == 1 else 0.0, aw, aw, an, 64, 64, C, N, 18, 6, k, 4, T[t2], T["sadct"], T[t5], useSD=useSD)
        got.append(eng.group_kernel(step, prm))
        assert got[-1] == want, (step, k, an, N, C, t2, t5, got[-1])
    assert len(set(got)) == len(KERNELS) == 17
    # ROWS cover the kernels of k = 8 and 16 at an <= 1 on one CTA; test_patch12_gpu, test_angular_window_gpu and
    # test_large_groups_gpu run the others
    elsewhere = ("k_groups12<", "k_groups25<", "k_groups_cl<")
    assert {r[-1] for r in ROWS} == {name for _, name in KERNELS if not name.startswith(elsewhere)}
