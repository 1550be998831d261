"""Diagnostic: a team with idle ranks (more ranks than row bands) running the two steps TWICE on the same team object
(stale buffers of the first repetition), config-2 parameters, emulated on one GPU."""
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
for name, aw, ah, H, W, s1, s2 in [("cfg2", 4, 3, 217, 157, (1, 18, 3, 16, 3, L.BIOR), (8, 18, 3, 8, 3, L.DCT)),
                                    ("cfg3", 4, 3, 217, 157, (8, 18, 6, 16, 4, L.ID), (16, 18, 6, 8, 4, L.DCT))]:
    clean = lfdata.synth_lf(aw, ah, H, W)
    noisy = torch.from_numpy(L.add_noise(clean, 10.0)).to(dev)
    cl = torch.from_numpy(clean).to(dev)
    mask = np.ones(aw * ah, np.uint32)
    p1 = L.make_params(10.0, 2.7, aw, ah, 1, W, H, 3, *s1[:5], s1[5], L.SADCT, L.HAAR)
    p2 = L.make_params(10.0, 0.0, aw, ah, 1, W, H, 3, *s2[:5], s2[5], L.SADCT, L.HAAR)
    eng = L.LFBM5D(0)
    w0, b0, o0, _ = T.run_single(L, eng, torch, noisy, mask, p1, p2)
    eng.close()
    for world in (4, 8):
        team = L.Team.emulated(0, world)
        for rep in range(3):
            ws = [noisy.clone() for _ in range(world)]
            bs = [torch.zeros_like(noisy) for _ in range(world)]
            outs = [torch.zeros_like(noisy) for _ in range(world)]
            team.step(1, p1, [t.data_ptr() for t in ws], None, mask, [t.data_ptr() for t in bs], gather=0)
            team.step(2, p2, [t.data_ptr() for t in ws], [t.data_ptr() for t in bs], mask, [t.data_ptr() for t in outs], gather=1)
            torch.cuda.synchronize()
            st = team.stats()
            print(name, "world", world, "rep", rep, "denoised equal", all(bool(torch.equal(outs[g], o0)) for g in range(world)),
                  "psnr %.2f (single %.2f)" % (psnr(outs[0], cl), psnr(o0, cl)), "ties", st["tie_patches"], "redone", st["passes_redone"], flush=True)
        team.close()
