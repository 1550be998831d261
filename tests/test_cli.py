"""The LFBM5Ddenoising command line (same 37 positional arguments as the reference, README.md:50) end to end on the GPU:
PNG in, PNG out, report file in the reference's format; and the C++ adapters with the reference's signatures."""
import os
import re
import subprocess

import numpy as np
import pytest

import lfdata
from gpucheck import LIBDIR, check_pngs, run_cli, write_lf


def test_cli_binary_and_host_library_exist():
    """CPU-side check: the drivers are built and link against the C-ABI library only."""
    for f in ("LFBM5Ddenoising", "liblfbm5d_host.so"):
        assert os.path.exists(os.path.join(LIBDIR, f)), f
    out = subprocess.check_output(["nm", "-D", "--defined-only", "-C", os.path.join(LIBDIR, "liblfbm5d_host.so")]).decode()
    for sym in ("run_bm5d_1st_step", "run_bm5d_2nd_step", "run_bm3d_LF"):
        assert sym + "(" in out
    p = subprocess.run([os.path.join(LIBDIR, "LFBM5Ddenoising")], stdout=subprocess.PIPE)
    assert p.returncode == 1 and b"usage: LFBM5Ddenoising LF_dir SAI_name" in p.stdout


@pytest.mark.gpu
def test_cli_readme_command(tmp_path):
    from PIL import Image
    clean = lfdata.synth_lf(3, 3, 64, 72)
    src = write_lf(tmp_path, clean, 3)
    report = tmp_path / "objectiveResults.txt"
    # README.md:50 command line
    args = [os.path.join(LIBDIR, "LFBM5Ddenoising"), str(src), "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "25", "2.7",
            str(tmp_path / "noisyLF"), str(tmp_path / "basicLF"), str(tmp_path / "denoisedLF"), str(tmp_path / "diffLF"),
            "8", "18", "6", "16", "4", "id", "sadct", "haar", "0", "16", "18", "6", "8", "4", "dct", "sadct", "haar", "0",
            "opp", "0", str(report)]
    out = run_cli(args)
    assert "Step 1 done in" in out and "Step 2 done in" in out and "THIS IS THE END" in out
    for d in ("noisyLF", "basicLF", "denoisedLF", "diffLF"):
        assert len(os.listdir(str(tmp_path / d))) == 9
    txt = report.read_text()
    vals = [float(x) for x in re.findall(r"-> Average PSNR \w+ = ([0-9.]+)", txt)]
    assert len(vals) == 3 and vals[0] < vals[1] < vals[2] and vals[2] - vals[0] > 5.0
    den = np.asarray(Image.open(str(tmp_path / "denoisedLF" / "SAI_02_02.png")), dtype=np.float32).transpose(2, 0, 1)
    assert np.sqrt(np.mean((den - clean[4]) ** 2)) < 8.0
    # The files and the report are exactly what the library's entry points give on the same input, written in the reference's
    # formats: noise = mt19937ar seeded LFBM5D_SEED + st on the 8-bit source (utilities.cpp:154-185), images rounded floor(x + .5)
    # and clamped (io_png.c:648-650), PSNR / RMSE of the unrounded floats with the reference's accumulation (utilities.cpp:412-435).
    import lfbm5d_b200 as L
    src8 = np.clip(np.floor(clean + 0.5), 0, 255).astype(np.float32)
    noisy = L.add_noise(src8, 25.0, seed0=20171016)
    mask = np.ones(9, np.uint32)
    eng = L.LFBM5D(0)
    p1 = L.make_params(25.0, 2.7, 3, 3, 1, 72, 64, 3, 8, 18, 6, 16, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(25.0, 0.0, 3, 3, 1, 72, 64, 3, 16, 18, 6, 8, 4, L.DCT, L.SADCT, L.HAAR)
    basic, n1 = eng.step1(p1, noisy, mask)
    out, b2, n2 = eng.step2(p2, n1, basic, mask)
    eng.close()
    check_pngs(tmp_path, (("noisyLF", noisy), ("basicLF", basic), ("denoisedLF", out)), 3)      # basic is saved before step 2 round-trips it
    blocks = re.findall(r"-> Average PSNR (\w+) = ([0-9.]+)\n-> Standard deviation PSNR \w+ = ([0-9.e+-]+)\nPSNR for all \w+ SAIs:\n((?:[0-9. ]+\n){3})", txt)
    assert [b[0] for b in blocks] == ["noisy", "basic", "denoised"]
    for (name, avg, std, rows), arr in zip(blocks, (noisy, basic, out)):
        want = [L.psnr(src8[st], arr[st])[0] for st in range(9)]
        got = [float(v) for v in rows.split()]
        assert np.allclose(got, want, rtol=0, atol=1e-4) and abs(float(avg) - np.mean(want)) < 2e-4, (name, got, want)   # 6 significant digits printed
    # second mode: no ground truth, noisy light field read back from disk (utilities_LF.cpp:1187)
    args[1] = "none"
    assert "Loading noisy LF elapsed time" in run_cli(args)


@pytest.mark.gpu
def test_cli_grayscale_and_lfbm3d(tmp_path):
    """Grayscale PNGs through LFBM5Ddenoising (every window takes several core calls: the partial-window branch) and the
    LFBM3Ddenoising driver (31 positional arguments of main_bm3d_LF.cpp, README.md:62 parameters) on RGB PNGs."""
    from PIL import Image
    clean = lfdata.synth_lf(3, 3, 48, 56)
    env = dict(os.environ, LFBM5D_SEED="7")
    for tag in ("gray", "rgb"):
        base = tmp_path / tag
        base.mkdir()
        for d in ("sourceLF", "noisyLF", "basicLF", "denoisedLF", "diffLF"):
            (base / d).mkdir()
        for s in range(3):
            for t in range(3):
                img = np.clip(np.floor(clean[s * 3 + t] + 0.5), 0, 255).astype(np.uint8)
                im = Image.fromarray(img[0]) if tag == "gray" else Image.fromarray(img.transpose(1, 2, 0))
                im.save(str(base / "sourceLF" / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))
        report = base / "results.txt"
        dirs = [str(base / d) for d in ("noisyLF", "basicLF", "denoisedLF", "diffLF")]
        if tag == "gray":
            args = [os.path.join(LIBDIR, "LFBM5Ddenoising"), str(base / "sourceLF"), "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "20", "2.7"] + dirs + \
                   ["8", "18", "6", "16", "4", "id", "sadct", "haar", "0", "16", "18", "6", "8", "4", "dct", "sadct", "haar", "0", "opp", "0", str(report)]
        else:
            args = [os.path.join(LIBDIR, "LFBM3Ddenoising"), str(base / "sourceLF"), "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "20", "2.7"] + dirs + \
                   ["16", "16", "8", "3", "bior", "0", "32", "16", "8", "3", "dct", "0", "opp", "0", str(report)]
        p = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, timeout=300)
        out = p.stdout.decode()
        assert p.returncode == 0, out[-2000:]
        assert len(os.listdir(dirs[2])) == 9
        vals = [float(x) for x in re.findall(r"-> Average PSNR \w+ = ([0-9.]+)", report.read_text())]
        assert len(vals) == 3 and vals[2] - vals[0] > 4.0, vals
        den = np.asarray(Image.open(os.path.join(dirs[2], "SAI_02_02.png")), dtype=np.float32)
        assert den.shape == ((48, 56) if tag == "gray" else (48, 56, 3))
