"""Diagnostic: BASELINE config-2 parameters (bior / N = 1 / nDisp = 3 / p = 3) through emulated teams vs one context."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import lfbm5d_b200 as L
import lfdata
import gpucheck as T

dev = torch.device("cuda", 0)
def psnr(a, b): return float(10 * torch.log10(255.0 ** 2 / torch.mean((a - b) ** 2)))
cases = [("cfg2", 4, 3, 217, 157, dict(s1=(1, 18, 3, 16, 3, L.BIOR), s2=(8, 18, 3, 8, 3, L.DCT))),
         ("cfg2-N8", 4, 3, 217, 157, dict(s1=(8, 18, 3, 16, 3, L.BIOR), s2=(8, 18, 3, 8, 3, L.DCT))),
         ("cfg2-id", 4, 3, 217, 157, dict(s1=(1, 18, 3, 16, 3, L.ID), s2=(8, 18, 3, 8, 3, L.DCT))),
         ("cfg3-nd3", 4, 3, 217, 157, dict(s1=(8, 18, 3, 16, 4, L.ID), s2=(16, 18, 3, 8, 4, L.DCT))),
         ("cfg2-full", 15, 15, 434, 625, dict(s1=(1, 18, 3, 16, 3, L.BIOR), s2=(8, 18, 3, 8, 3, L.DCT))),
         ("cfg2-tall", 3, 3, 434, 157, dict(s1=(1, 18, 3, 16, 3, L.BIOR), s2=(8, 18, 3, 8, 3, L.DCT))),
         ("cfg3-p3", 4, 3, 217, 157, dict(s1=(8, 18, 6, 16, 3, L.ID), s2=(16, 18, 6, 8, 3, L.DCT)))]
which = sys.argv[1:] or [c[0] for c in cases]
worlds = [int(x) for x in os.environ.get('WORLDS', '2,3,8').split(',')]
for name, aw, ah, H, W, pr in cases:
    if name not in which: continue
    clean = lfdata.synth_lf(aw, ah, H, W)
    noisy = torch.from_numpy(L.add_noise(clean, 10.0)).to(dev)
    cl = torch.from_numpy(clean).to(dev)
    mask = np.ones(aw * ah, np.uint32)
    N1, ns1, nd1, k1, p1_, t1 = pr["s1"]; N2, ns2, nd2, k2, p2_, t2 = pr["s2"]
    p1 = L.make_params(10.0, 2.7, aw, ah, 1, W, H, 3, N1, ns1, nd1, k1, p1_, t1, L.SADCT, L.HAAR)
    p2 = L.make_params(10.0, 0.0, aw, ah, 1, W, H, 3, N2, ns2, nd2, k2, p2_, t2, L.SADCT, L.HAAR)
    eng = L.LFBM5D(0)
    w0, b0, o0, s0 = T.run_single(L, eng, torch, noisy, mask, p1, p2)
    eng.close()
    print(name, "single: psnr noisy %.2f basic %.2f denoised %.2f" % (psnr(noisy, cl), psnr(b0, cl), psnr(o0, cl)), flush=True)
    for world in worlds:
        try:
            ws, bs, outs, bands1, bands2, st = T.run_team(L, torch, world, noisy, mask, p1, p2, gather=1)
        except Exception as e:
            print(name, "world", world, "FAILED:", str(e)[:300], flush=True); continue
        eqb = [bool(torch.equal(bs[g], b0)) for g in range(world)]
        eqo = [bool(torch.equal(outs[g], o0)) for g in range(world)]
        db = max(float((bs[g] - b0).abs().max()) for g in range(world))
        do = max(float((outs[g] - o0).abs().max()) for g in range(world))
        print(name, "world", world, "basic equal", all(eqb), "max|d| %.4g" % db, "| denoised equal", all(eqo), "max|d| %.4g" % do,
              "psnr %.2f" % psnr(outs[0], cl), "ties", st["tie_patches"], "redone", st["passes_redone"], "bands", bands1[:3], flush=True)
        if not all(eqb):
            d = (bs[0] - b0).abs().amax(dim=(1, 3))      # [sai][row]
            rows = torch.nonzero(d.amax(dim=0) > 0).flatten().tolist()
            print("   basic differs on rank 0 in rows", rows[:6], "...", rows[-6:], "SAIs", torch.nonzero(d.amax(dim=1) > 0).flatten().tolist(), flush=True)
