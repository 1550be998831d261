"""Generates tests/golden/config1.npz: BASELINE.json configs[0] — the reference's own fixture `testing/sourceLF`
(3x3 SAIs 256x256 RGB, README.md:50: sigma 25, `8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar`, opp) — run through
the UNMODIFIED reference (oracle/_ref, nb_threads = 1).

Stored: the fixture's pixels as 8-bit RGB PNGs under tests/golden/sourceLF (lossless; the tests read them with
tests/golden_inputs.config1_fixture), the PSNRs of the reference's basic / denoised estimates (utilities.cpp:412-435 via the
oracle's restatement), cropped tiles of both estimates, and the same PSNRs with the FFTW stand-in accumulating in double
(DCT mode 1): the reference's own sensitivity to the unpinned FFTW arithmetic (SURVEY A11).
The noisy input is re-created anywhere by tests/oracleapi.add_noise (mt19937ar, seed 20171016 + st, utilities.cpp:154-185).

Run:  python tests/make_golden_config1.py <reference checkout>     (needs oracle/_ref built and PIL)"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import golden_inputs as gi  # noqa: E402
import oracleapi as O  # noqa: E402
import refapi as R  # noqa: E402

GOLD = os.path.join(HERE, "golden")
SAIS = [0, 4, 8]          # tiles are stored for these SAIs (corner, centre, corner of the angular window)
TILES = {"centre": (slice(96, 160), slice(96, 160)), "corner": (slice(0, 40), slice(0, 40)), "edge": (slice(216, 256), slice(100, 164))}


def store_fixture(src):
    """<reference>/testing/sourceLF -> tests/golden/sourceLF, re-encoded by Pillow (same pixels, smaller files)."""
    from PIL import Image
    os.makedirs(gi.FIXTURE_DIR, exist_ok=True)
    for s in range(3):
        for t in range(3):      # utilities_LF.cpp:105-112: <dir>/<name><sep>%02d<sep>%02d.png with s + s_start, t + t_start (both 1)
            name = "SAI_%02d_%02d.png" % (s + 1, t + 1)
            Image.open(os.path.join(src, name)).convert("RGB").save(os.path.join(gi.FIXTURE_DIR, name), optimize=True)


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/make_golden_config1.py <reference checkout>")
    store_fixture(os.path.join(sys.argv[1], "testing", "sourceLF"))
    clean = gi.config1_fixture().astype(np.float32)
    noisy = O.add_noise(clean, 25.0)
    mask = np.ones(9)
    out = {}
    for mode in (0, 1):
        R.lib().ref_set_dct_mode(mode)
        b, nrt = R.run_step1(noisy, mask, 25.0, 2.7, 3, 3, 1, 8, 18, 6, 16, 4, R.ID, R.SADCT, R.HAAR)
        d, b2, _ = R.run_step2(nrt, b, mask, 25.0, 3, 3, 1, 16, 18, 6, 8, 4, R.DCT, R.SADCT, R.HAAR)
        tag = "" if mode == 0 else "_f64dct"
        out["psnr_basic" + tag] = np.float64(O.psnr(b, clean)[0])
        out["psnr_denoised" + tag] = np.float64(O.psnr(d, clean)[0])
        if mode == 0:
            for name, (ys, xs) in TILES.items():
                out["basic_" + name] = b[SAIS][:, :, ys, xs]
                out["denoised_" + name] = d[SAIS][:, :, ys, xs]
            out["noisy_rt_centre"] = nrt[SAIS][:, :, TILES["centre"][0], TILES["centre"][1]]
    R.lib().ref_set_dct_mode(0)
    np.savez_compressed(os.path.join(GOLD, "config1.npz"), **out)
    print({k: (float(v) if v.shape == () else v.shape) for k, v in out.items()})
    print("config1.npz", os.path.getsize(os.path.join(GOLD, "config1.npz")))


if __name__ == "__main__":
    main()
