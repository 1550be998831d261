"""`sigma = auto` on the command lines without a GPU: with a ground-truth light field it has no meaning (noise of the given sigma is
added to it), so both drivers refuse it before they read a file or touch the GPU."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("driver", ["LFBM5Ddenoising", "LFBM3Ddenoising"])
def test_sigma_auto_needs_no_ground_truth(tmp_path, driver):
    import subprocess
    from PIL import Image
    src = tmp_path / "sourceLF"
    src.mkdir()
    img = np.random.default_rng(3).integers(0, 256, size=(24, 32, 3)).astype(np.uint8)
    for s in range(3):
        for t in range(3):
            Image.fromarray(img).save(str(src / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))
    outs = [tmp_path / d for d in ("noisyLF", "basicLF", "denoisedLF", "diffLF")]
    for d in outs:
        d.mkdir()
    report = tmp_path / "report.txt"
    args = [os.path.join(ROOT, "lfbm5d_b200", "_lib", driver), str(src), "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "auto", "2.7"]
    args += [str(d) for d in outs]
    if driver == "LFBM5Ddenoising":
        args += ["8", "18", "6", "16", "4", "id", "sadct", "haar", "0", "16", "18", "6", "8", "4", "dct", "sadct", "haar", "0"]
    else:
        args += ["16", "16", "8", "3", "bior", "0", "32", "16", "8", "3", "dct", "0"]
    args += ["opp", "0", str(report)]
    p = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=120)
    txt = p.stdout.decode()
    assert p.returncode == 1, txt
    assert "sigma = auto needs LF_dir = none" in txt
    assert "Read input image" not in txt            # refused before the light field is read
    assert all(os.listdir(str(d)) == [] for d in outs) and not report.exists()
