"""Host glue of the command lines (SURVEY.md 8(f) rank 1-2), CPU only: the PNG codec of lfbm5d_b200/csrc/lf_io.h against an
independent decoder (Pillow) — every colour type, bit depth and interlace method read_png_f32 accepts (io_png.c:116-260), the
writer's rounding (io_png.c:648-650) — and the metrics / difference images / PSNR report against the UNMODIFIED reference
functions (compute_psnr_LF, compute_diff_LF, write_psnr_LF; utilities_LF.cpp:639-869): live where oracle/_ref is built, else
against the stored digests of their results (tests/golden/ref_pins.json)."""
import ctypes as C
import os
import struct
import zlib

import numpy as np
import pytest

import lfbm5d_b200 as L


def host():
    h = L.load_host_library()
    h.lfio_png_read.argtypes = [C.c_char_p, C.POINTER(C.c_float), C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    h.lfio_png_write.argtypes = [C.c_char_p, C.POINTER(C.c_float), C.c_size_t, C.c_size_t, C.c_size_t]
    return h


def png_read(path):
    h = host()
    w, hh, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
    if h.lfio_png_read(str(path).encode(), None, 0, C.byref(w), C.byref(hh), C.byref(c)) != 0:
        return None
    out = np.zeros((c.value, hh.value, w.value), np.float32)
    assert h.lfio_png_read(str(path).encode(), out.ctypes.data_as(C.POINTER(C.c_float)), out.size, C.byref(w), C.byref(hh), C.byref(c)) == 0
    return out


def _chunk(t, d):
    return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xffffffff)


def encode_png(samples, depth, ctype, interlace, filters=(0, 1, 2, 3, 4), idat_split=0):
    """Minimal PNG encoder for the tests: samples [h, w, nch] (integers < 2**depth), any filter type per scanline (cycled),
    non-interlaced or Adam7, optionally several IDAT chunks. Follows the PNG specification (sections 7-9)."""
    h, w, nch = samples.shape
    fb = max(1, nch * depth // 8)

    def pack_rows(sub):
        ph, pw, _ = sub.shape
        rows = []
        prev = None
        for y in range(ph):
            flat = sub[y].reshape(-1).astype(np.int64)
            if depth == 8:
                line = flat.astype(np.uint8)
            elif depth == 16:
                line = np.stack([flat >> 8, flat & 255], axis=1).reshape(-1).astype(np.uint8)
            else:
                per = 8 // depth
                pad = (-len(flat)) % per
                f2 = np.concatenate([flat, np.zeros(pad, np.int64)]).reshape(-1, per)
                line = np.zeros(len(f2), np.int64)
                for i in range(per):
                    line = (line << depth) | f2[:, i]
                line = line.astype(np.uint8)
            ft = filters[y % len(filters)]
            cur = line.astype(np.int64)
            a = np.concatenate([np.zeros(fb, np.int64), cur[:-fb]]) if len(cur) > fb else np.zeros(len(cur), np.int64)
            if len(cur) <= fb:
                a = np.zeros(len(cur), np.int64)
            b = prev if prev is not None else np.zeros(len(cur), np.int64)
            c = np.concatenate([np.zeros(fb, np.int64), b[:-fb]]) if len(cur) > fb else np.zeros(len(cur), np.int64)
            if ft == 0:
                enc = cur
            elif ft == 1:
                enc = cur - a
            elif ft == 2:
                enc = cur - b
            elif ft == 3:
                enc = cur - (a + b) // 2
            else:
                p = a + b - c
                pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
                pred = np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))
                enc = cur - pred
            rows.append(bytes([ft]) + (enc & 255).astype(np.uint8).tobytes())
            prev = cur
        return b"".join(rows)

    if interlace:
        raw = b""
        for x0, y0, dx, dy in ((0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)):
            sub = samples[y0::dy, x0::dx]
            if sub.shape[0] and sub.shape[1]:
                raw += pack_rows(sub)
    else:
        raw = pack_rows(samples)
    z = zlib.compress(raw, 6)
    png = b"\x89PNG\r\n\x1a\n" + _chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, 1 if interlace else 0))
    if ctype == 3:
        png += _chunk(b"PLTE", bytes(range(256)) * 3)
    if idat_split:
        for i in range(0, len(z), idat_split):
            png += _chunk(b"IDAT", z[i:i + idat_split])
    else:
        png += _chunk(b"IDAT", z)
    return png + _chunk(b"IEND", b"")


CASES = [(0, 1), (0, 2), (0, 4), (0, 8), (0, 16), (2, 8), (2, 16), (3, 1), (3, 2), (3, 4), (3, 8), (4, 8), (4, 16), (6, 8), (6, 16)]


@pytest.mark.parametrize("interlace", [0, 1])
@pytest.mark.parametrize("ctype,depth", CASES)
def test_png_reader_every_format(tmp_path, ctype, depth, interlace):
    """Own encoder -> lf_io reader, checked sample by sample, and against Pillow where Pillow decodes the format without converting
    it. Sizes around the Adam7 8 x 8 cell (empty passes, partial bytes of the packed depths), all five filter types."""
    from PIL import Image
    nch = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}[ctype]
    rng = np.random.default_rng(100 * ctype + depth + interlace)
    for (h, w) in ((1, 1), (2, 3), (5, 7), (8, 8), (9, 17), (33, 41)):
        samples = rng.integers(0, 2 ** depth, size=(h, w, nch))
        path = tmp_path / ("t_%d_%d_%d_%dx%d.png" % (ctype, depth, interlace, h, w))
        path.write_bytes(encode_png(samples, depth, ctype, interlace, idat_split=37 if (h * w) % 2 else 0))
        got = png_read(path)
        assert got is not None, path
        want = (samples >> 8) if depth == 16 else samples           # PNG_TRANSFORM_STRIP_16; smaller depths unpacked, not scaled
        assert got.shape == (nch, h, w)
        assert np.array_equal(got, want.transpose(2, 0, 1).astype(np.float32)), (ctype, depth, interlace, h, w)
        if depth == 8 and ctype in (0, 2, 4, 6):                  # independent decoder on the same file
            pil = np.asarray(Image.open(str(path)))
            pil = pil.reshape(h, w, nch)
            assert np.array_equal(pil.transpose(2, 0, 1).astype(np.float32), got)


def test_png_reader_on_the_reference_fixture():
    """The nine SAIs of the reference's fixture `testing/sourceLF` (config 1), stored losslessly as 8-bit RGB PNGs under
    tests/golden/sourceLF: same pixels as Pillow."""
    from PIL import Image
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sourceLF")
    names = sorted(f for f in os.listdir(d) if f.endswith(".png"))
    assert len(names) == 9
    for f in names:
        got = png_read(os.path.join(d, f))
        pil = np.asarray(Image.open(os.path.join(d, f)).convert("RGB"), dtype=np.float32).transpose(2, 0, 1)
        assert got is not None and np.array_equal(got[:3], pil)


def test_png_reader_rejects_broken_files(tmp_path):
    good = encode_png(np.arange(48).reshape(4, 4, 3) % 256, 8, 2, 0)
    for name, data in (("trunc.png", good[:40]), ("sig.png", b"\x89PNX" + good[4:]), ("empty.png", b""),
                       ("depth.png", good[:24] + b"\x03" + good[25:]), ("short.png", good[:-20])):
        (tmp_path / name).write_bytes(data)
        assert png_read(tmp_path / name) is None, name
    assert png_read(tmp_path / "missing.png") is None


@pytest.mark.parametrize("c", [1, 3])
def test_png_writer_rounding_and_round_trip(tmp_path, c):
    """write_png_f32 (io_png.c:560-700): 8 bits, floor(x + .5), clamped to [0, 255]; gray or RGB; Pillow reads the same pixels."""
    from PIL import Image
    h = host()
    rng = np.random.default_rng(5)
    img = (rng.random((c, 13, 21)) * 300.0 - 20.0).astype(np.float32)
    img[0, 0, :6] = [0.5, 1.4999, 254.5, 255.49, -0.5, 1e9]
    path = tmp_path / "w.png"
    assert h.lfio_png_write(str(path).encode(), img.ctypes.data_as(C.POINTER(C.c_float)), 21, 13, c) == 0
    want = np.clip(np.floor(img + np.float32(0.5)), 0, 255).astype(np.uint8)
    pil = np.asarray(Image.open(str(path)))
    pil = pil[None] if c == 1 else pil.transpose(2, 0, 1)
    assert np.array_equal(pil, want)
    assert np.array_equal(png_read(path), want.astype(np.float32))


@pytest.mark.parametrize("major", ["row", "col"])
def test_metrics_and_report_equal_the_reference(tmp_path, ref, major):
    """PSNR / RMSE per SAI with their averages and standard deviations, difference images, and the report file, byte for byte."""
    h = host()
    aw, ah, each = 4, 3, 3 * 20 * 24
    asize = aw * ah
    rng = np.random.default_rng(11)
    a = (rng.random((asize, each)) * 255).astype(np.float32)
    b = (a + rng.normal(0, 9, a.shape)).astype(np.float32)
    mask = np.ones(asize, np.uint32)
    mask[5] = 0
    fp, up = (lambda x: x.ctypes.data_as(C.POINTER(C.c_float))), (lambda x: x.ctypes.data_as(C.POINTER(C.c_uint)))

    def metrics(lib, pre):
        ps, rm, st = np.zeros(asize, np.float32), np.zeros(asize, np.float32), np.zeros(4, np.float32)
        f = getattr(lib, pre + "psnr_LF")
        f.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_uint), C.c_uint, C.c_size_t, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]
        assert f(fp(a), fp(b), up(mask), asize, each, fp(ps), fp(rm), fp(st)) == 0
        d = np.zeros_like(a)
        g = getattr(lib, pre + "diff_LF")
        g.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_uint), C.c_uint, C.c_size_t, C.c_float, C.POINTER(C.c_float)]
        assert g(fp(a), fp(b), up(mask), asize, each, 10.0, fp(d)) == 0
        return ps, rm, st, d
    ours = metrics(h, "lfio_")
    ref.check("metrics_LF", ours, lambda R: metrics(R.lib(), "ref_compute_"))
    ps, rm, st, _ = ours

    def report(f, name):
        f.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(C.c_uint), C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_float), C.c_float, C.c_float,
                      C.POINTER(C.c_float), C.c_float, C.c_float]
        path = tmp_path / (name + ".txt")
        for label in (b"noisy", b"denoised"):          # the report is appended to
            assert f(str(path).encode(), label, up(mask), L.ROWMAJOR if major == "row" else L.COLMAJOR, aw, ah, fp(ps), float(st[0]), float(st[1]),
                     fp(rm), float(st[2]), float(st[3])) == 0
        return np.frombuffer(path.read_bytes(), np.uint8)
    text = report(h.lfio_write_psnr_LF, "ours")
    ref.check("write_psnr_LF_" + major, text, lambda R: report(R.lib().ref_write_psnr_LF, "ref"))
    assert b"No SAI" in text.tobytes()


def _write_lf(tmp_path, arr, s_start=1, t_start=1, gray=False):
    """arr [ah, aw, C, H, W] uint8 -> <tmp>/SAI_%02d_%02d.png"""
    from PIL import Image
    ah, aw = arr.shape[:2]
    for s in range(ah):
        for t in range(aw):
            a = arr[s, t]
            im = Image.fromarray(a[0]) if gray else Image.fromarray(a.transpose(1, 2, 0))
            im.save(str(tmp_path / ("SAI_%02d_%02d.png" % (s + s_start, t + t_start))))


def _load_lf(d, aw, ah, major, s_start=1, t_start=1):
    h = host()
    h.lfio_load_LF.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_float), C.c_size_t,
                               C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
    w, hh, c = C.c_uint(), C.c_uint(), C.c_uint()
    mask = np.zeros(aw * ah, np.uint32)
    mp = mask.ctypes.data_as(C.POINTER(C.c_uint))
    if h.lfio_load_LF(str(d).encode(), b"SAI", b"_", major, aw, ah, s_start, t_start, None, 0, mp, C.byref(w), C.byref(hh), C.byref(c)) != 0:
        return None
    out = np.zeros((aw * ah, c.value, hh.value, w.value), np.float32)
    assert h.lfio_load_LF(str(d).encode(), b"SAI", b"_", major, aw, ah, s_start, t_start, out.ctypes.data_as(C.POINTER(C.c_float)), out.size, mp,
                          C.byref(w), C.byref(hh), C.byref(c)) == 0
    return out, mask


@pytest.mark.parametrize("threads", ["1", "5"])
def test_load_and_save_light_field(tmp_path, monkeypatch, threads):
    """load_LF / save_LF (utilities_LF.cpp:72-231): file naming with start indices, row / column major ordering, the mask of empty SAIs
    (:149-154), a gray image stored as RGB counting one channel (:123-130), masked SAIs not written; same result on one thread and
    on several (the files are decoded / encoded on the host cores)."""
    from PIL import Image
    monkeypatch.setenv("LFBM5D_IO_THREADS", threads)
    rng = np.random.default_rng(3)
    aw, ah, H, W = 3, 2, 11, 14
    arr = rng.integers(1, 256, size=(ah, aw, 3, H, W)).astype(np.uint8)
    arr[1, 0] = 0                                        # an empty SAI
    src = tmp_path / "src"
    src.mkdir()
    _write_lf(src, arr, s_start=2, t_start=5)
    for major, order in ((L.ROWMAJOR, lambda s, t: s * aw + t), (L.COLMAJOR, lambda s, t: s + t * ah)):
        lf, mask = _load_lf(src, aw, ah, major, 2, 5)
        assert lf.shape == (6, 3, H, W)
        for s in range(ah):
            for t in range(aw):
                assert np.array_equal(lf[order(s, t)], arr[s, t].astype(np.float32))
                assert mask[order(s, t)] == (0 if (s, t) == (1, 0) else 1)
    assert _load_lf(src, aw + 1, ah, L.ROWMAJOR, 2, 5) is None          # SAI_02_08.png does not exist
    # gray stored as RGB -> one channel
    g = tmp_path / "gray"
    g.mkdir()
    garr = np.repeat(rng.integers(1, 256, size=(1, 2, 1, H, W)).astype(np.uint8), 3, axis=2)
    _write_lf(g, garr)
    lf, mask = _load_lf(g, 2, 1, L.ROWMAJOR)
    assert lf.shape == (2, 1, H, W) and np.array_equal(lf[1, 0], garr[0, 1, 0].astype(np.float32))
    # save: rounded floor(x + .5), clamped; the masked SAI gets no file
    h = host()
    h.lfio_save_LF.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_float), C.POINTER(C.c_uint), C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_uint,
                               C.c_uint, C.c_uint, C.c_uint]
    out = tmp_path / "out"
    out.mkdir()
    lf, mask = _load_lf(src, aw, ah, L.COLMAJOR, 2, 5)
    lf = (lf + rng.normal(0, 30, lf.shape)).astype(np.float32)
    assert h.lfio_save_LF(str(out).encode(), b"SAI", b"_", lf.ctypes.data_as(C.POINTER(C.c_float)), mask.ctypes.data_as(C.POINTER(C.c_uint)), L.COLMAJOR,
                          aw, ah, 1, 1, W, H, 3) == 0
    assert sorted(os.listdir(str(out))) == ["SAI_%02d_%02d.png" % (s + 1, t + 1) for s in range(ah) for t in range(aw) if (s, t) != (1, 0)]
    for s in range(ah):
        for t in range(aw):
            if (s, t) == (1, 0):
                continue
            img = np.asarray(Image.open(str(out / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))).transpose(2, 0, 1)
            assert np.array_equal(img, np.clip(np.floor(lf[s + t * ah] + np.float32(0.5)), 0, 255).astype(np.uint8))


@pytest.mark.parametrize("driver", ["LFBM5Ddenoising", "LFBM3Ddenoising"])
def test_cli_front_half_without_a_gpu(tmp_path, driver):
    """Both command lines up to the first GPU call, wherever it runs: PNGs read, noise added with LFBM5D_SEED, noisy light field and the
    first report block written — identical on one I/O thread and on several, and equal to the library's own noise — and, on a machine
    without a CUDA device, a clean failure instead of a CPU fallback."""
    import re
    import subprocess
    from PIL import Image
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(ROOT, "lfbm5d_b200", "_lib", driver)
    rng = np.random.default_rng(9)
    arr = rng.integers(0, 256, size=(3, 3, 3, 40, 48)).astype(np.uint8)
    src = tmp_path / "sourceLF"
    src.mkdir()
    _write_lf(src, arr)
    outs = {}
    for threads in ("1", "6"):
        base = tmp_path / ("run" + threads)
        base.mkdir()
        for d in ("noisyLF", "basicLF", "denoisedLF", "diffLF"):
            (base / d).mkdir()
        args = [exe, str(src), "SAI", "_", "3", "3", "1", "1", "1", "1", "row", "25", "2.7", str(base / "noisyLF"), str(base / "basicLF"),
                str(base / "denoisedLF"), str(base / "diffLF")]
        if driver == "LFBM5Ddenoising":      # README.md:50
            args += ["8", "18", "6", "16", "4", "id", "sadct", "haar", "0", "16", "18", "6", "8", "4", "dct", "sadct", "haar", "0", "opp", "0"]
        else:                                # README.md:62 (main_bm3d_LF.cpp)
            args += ["16", "16", "8", "3", "bior", "0", "32", "16", "8", "3", "dct", "0", "opp", "0"]
        args.append(str(base / "report.txt"))
        env = dict(os.environ, LFBM5D_SEED="77", LFBM5D_IO_THREADS=threads)
        p = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, timeout=600)
        txt = p.stdout.decode()
        assert " - nb of channels = 3" in txt and " - width          = 48" in txt
        import torch
        if not torch.cuda.is_available():
            assert p.returncode == 1 and "THIS IS THE END" not in txt          # no CPU fallback
        noisy = np.stack([np.asarray(Image.open(str(base / "noisyLF" / ("SAI_%02d_%02d.png" % (s + 1, t + 1))))).transpose(2, 0, 1)
                          for s in range(3) for t in range(3)])
        outs[threads] = (noisy, (base / "report.txt").read_text().split("-> Average RMSE")[0])
    assert np.array_equal(outs["1"][0], outs["6"][0]) and outs["1"][1] == outs["6"][1]
    want = L.add_noise(arr.reshape(9, 3, 40, 48).astype(np.float32), 25.0, seed0=77)
    assert np.array_equal(outs["1"][0], np.clip(np.floor(want + np.float32(0.5)), 0, 255).astype(np.uint8))
    assert re.search(r"-> Average PSNR noisy = [0-9.]+", outs["1"][1])
