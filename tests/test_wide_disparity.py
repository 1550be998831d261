"""Disparity search windows up to nDisp = 16 on the host side: parameter validation (plan_band runs validate() without a device)
and the team's row bands at a wide disparity window. No GPU needed."""
import pytest


def params(L, nDisp, step=1, H=620, W=48):
    if step == 1:
        return L.make_params(15.0, 2.7, 3, 3, 1, W, H, 3, 8, 18, nDisp, 16, 4, L.ID, L.SADCT, L.HAAR)
    return L.make_params(15.0, 0.0, 3, 3, 1, W, H, 3, 16, 18, nDisp, 8, 4, L.DCT, L.SADCT, L.HAAR)


@pytest.mark.parametrize("nDisp", [0, 6, 7, 10, 12, 16])
def test_plan_band_accepts_ndisp_up_to_16(nDisp):
    import lfbm5d_b200 as L
    for step in (1, 2):
        assert L.plan_band(1, 0, step, params(L, nDisp, step)) == (0, 620, 620)


def test_plan_band_rejects_ndisp_17():
    import lfbm5d_b200 as L
    for step in (1, 2):
        with pytest.raises(RuntimeError, match="nDisp > 16 is not supported by this build"):
            L.plan_band(1, 0, step, params(L, 17, step))
    # the padding check stays: 30 rows < nSim + nDisp = 18 + 16
    with pytest.raises(RuntimeError, match="image smaller than the padding nSim \\+ nDisp"):
        L.plan_band(1, 0, 1, params(L, 16, H=30))


@pytest.mark.parametrize("world", range(1, 9))
def test_team_bands_tile_rows_at_ndisp_12(world):
    import lfbm5d_b200 as L
    H = 620
    for step in (1, 2):
        b = [L.plan_band(world, g, step, params(L, 12, step, H=H)) for g in range(world)]
        assert b[0][0] == 0 and b[-1][1] == H
        assert all(b[g][1] == b[g + 1][0] for g in range(world - 1))
        assert all(b[g][0] <= b[g][1] <= b[g][2] <= H for g in range(world))
