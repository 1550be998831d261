"""12 x 12 patches (k = 12) on the host side: parameter validation (plan_band runs validate() without a device) and known answers
of the CPU oracle at k = 12, the only check of the GPU path at this size (there is no reference pin at k = 12). No GPU needed."""
import numpy as np
import pytest

# the reference's 12 x 12 Kaiser window, top-left 6 x 6 quadrant (bm3d.cpp:1101-1169)
K12_QUADRANT = np.array([
    0.1924, 0.2615, 0.3251, 0.3782, 0.4163, 0.4362, 0.2615, 0.3554, 0.4419, 0.5139, 0.5657, 0.5927,
    0.3251, 0.4419, 0.5494, 0.6390, 0.7033, 0.7369, 0.3782, 0.5139, 0.6390, 0.7433, 0.8181, 0.8572,
    0.4163, 0.5657, 0.7033, 0.8181, 0.9005, 0.9435, 0.4362, 0.5927, 0.7369, 0.8572, 0.9435, 0.9885], np.float32).reshape(6, 6)


def params(L, step, k=12, an=1, N=None, nDisp=6, t2=None, aw=3, H=200, W=64, C=3):
    if N is None:
        N = 16 if step == 1 else 32
    if t2 is None:
        t2 = L.ID if step == 1 else L.DCT
    return L.make_params(15.0, 2.7 if step == 1 else 0.0, aw, aw, an, W, H, C, N, 18, nDisp, k, 4, t2, L.SADCT, L.HAAR)


@pytest.mark.parametrize("an", [0, 1])
@pytest.mark.parametrize("nDisp", [6, 16])
def test_plan_band_accepts_k12(an, nDisp):
    import lfbm5d_b200 as L
    for step, N, t2 in ((1, 16, L.ID), (1, 32, L.DCT), (2, 16, L.DCT), (2, 8, L.ID)):
        assert L.plan_band(1, 0, step, params(L, step, an=an, N=N, nDisp=nDisp, t2=t2)) == (0, 200, 200)


def test_plan_band_team_bands_at_k12():
    import lfbm5d_b200 as L
    for world in (2, 3):
        for step in (1, 2):
            b = [L.plan_band(world, g, step, params(L, step, N=16)) for g in range(world)]
            assert b[0][0] == 0 and b[-1][1] == 200
            assert all(b[g][1] == b[g + 1][0] for g in range(world - 1))


def test_plan_band_rejects_k12_limits():
    import lfbm5d_b200 as L
    for step in (1, 2):
        with pytest.raises(RuntimeError, match="tau_2D = bior needs a power-of-two patch size"):
            L.plan_band(1, 0, step, params(L, step, N=8, t2=L.BIOR))
        with pytest.raises(RuntimeError, match="an = 2 is not supported at k = 12"):
            L.plan_band(1, 0, step, params(L, step, an=2, aw=5, N=2))
    # one channel of a step-2 group at an = 1, N = 32: 2 * 32 * 9 * 12 * 13 * 4 B = 351 KB of shared memory; N = 16 fits
    with pytest.raises(RuntimeError, match=r"k = 12 needs N \* A \* k \* \(k \+ 1\) \* 4 B"):
        L.plan_band(1, 0, 2, params(L, 2, N=32))
    assert L.plan_band(1, 0, 2, params(L, 2, N=16)) == (0, 200, 200)
    assert L.plan_band(1, 0, 1, params(L, 1, N=32)) == (0, 200, 200)
    # an = 0: the group holds one SAI, N = 32 fits in both steps
    assert L.plan_band(1, 0, 2, params(L, 2, an=0, N=32)) == (0, 200, 200)
    for k in (10, 4, 32):
        with pytest.raises(RuntimeError, match="patch size must be 8, 12 or 16"):
            L.plan_band(1, 0, 1, params(L, 1, k=k))


def test_oracle_dct_2d_round_trip_k12(oracle):
    rng = np.random.RandomState(12)
    p = (rng.rand(144) * 255.0).astype(np.float32)
    fwd = []
    try:
        for mode in (0, 1):
            oracle.set_dct_mode(mode)
            b = np.zeros_like(p)
            oracle.lib().orc_dct_2d_forward(oracle.fp(p), oracle.fp(b), 12)
            fwd.append(b.copy())
            oracle.lib().orc_dct_2d_inverse(oracle.fp(b), 12)
            assert np.abs(b - p).max() < 1e-2                    # inverse(forward(x)) == x
    finally:
        oracle.set_dct_mode(0)
    assert np.abs(fwd[0] - fwd[1]).max() <= 1e-4 * np.abs(fwd[0]).max()      # both DCT modes give the same coefficients
    # a constant patch has only a DC coefficient
    c = np.full(144, 10.0, np.float32)
    b = np.zeros_like(c)
    oracle.lib().orc_dct_2d_forward(oracle.fp(c), oracle.fp(b), 12)
    assert abs(b[0]) > 1.0 and np.abs(b[1:]).max() < 1e-4 * abs(b[0])


def test_oracle_kaiser_window_k12(oracle):
    kai, cn, cni = (np.zeros(144, np.float32) for _ in range(3))
    oracle.lib().orc_preProcess(oracle.fp(kai), oracle.fp(cn), oracle.fp(cni), 12)
    kai = kai.reshape(12, 12)
    assert np.array_equal(kai, kai.T) and np.array_equal(kai, kai[::-1, :]) and np.array_equal(kai, kai[:, ::-1])
    assert np.array_equal(kai[:6, :6], K12_QUADRANT)
    # the table is the outer product of a Kaiser window of length 12 and beta 2, rounded to four decimals
    w = np.kaiser(12, 2.0)
    assert np.abs(kai - np.outer(w, w)).max() < 1e-4
    cn = cn.reshape(12, 12)
    assert cn[0, 0] == np.float32(0.5 * 0.5 / 12) and cn[3, 5] == np.float32(0.5 / 12)
