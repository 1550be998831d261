"""Re-creates the inputs the golden vectors (tests/make_golden.py) were generated from."""
import os

import numpy as np

import lfdata
import oracleapi as O

FIXTURE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sourceLF")


def config1_fixture():
    """The reference's fixture `testing/sourceLF` (3x3 SAIs 256x256 RGB) as [9, 3, 256, 256] uint8, row-major SAI order, read
    from its lossless copy tests/golden/sourceLF/SAI_<s>_<t>.png (s, t from 1)."""
    from PIL import Image
    return np.stack([np.asarray(Image.open(os.path.join(FIXTURE_DIR, "SAI_%02d_%02d.png" % (s + 1, t + 1))).convert("RGB")).transpose(2, 0, 1)
                     for s in range(3) for t in range(3)])


def pad_inputs(H, W, sigma, n=24):
    clean = lfdata.synth_lf(3, 3, H, W)
    noisy = O.add_noise(clean, sigma)
    y = noisy.copy()
    for st in range(9):
        O.lib().orc_color_space_transform(O.fp(y[st]), O.OPP, W, H, 3, 1)
    return clean, noisy, np.stack([O.symetrize(y[st], n) for st in range(9)])


def run_inputs(tag):
    aw, H, W = {"3x3": (3, 32, 40), "5x5": (5, 24, 28)}[tag]
    clean = lfdata.synth_lf(aw, aw, H, W)
    return aw, clean, O.add_noise(clean, 25.0)


def partial_holes(num, den):
    """Accumulators of a first core call with the weights of SAI 1 and 6 removed in places (tests/make_golden.py)."""
    num, den = num.copy(), den.copy()
    num[1][:, 30:52, 28:70] = 0; den[1][:, 30:52, 28:70] = 0
    num[1][:, 60:, :40] = 0; den[1][:, 60:, :40] = 0
    num[6][:, :, 60:] = 0; den[6][:, :, 60:] = 0
    return num, den
