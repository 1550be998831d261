"""bench_large_groups.py — k = 16 groups too large for the shared memory of one CTA, which run on 2- and 4-CTA clusters
(k_groups_cl), against the README parameters; one process, one GPU, device-resident, on the synthetic 17x17x1024^2 RGB light field
of bench_angular.py (opp, an = 1):

  readme        8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar      (every group on one CTA: the reference point)
  n16_k16       8 18 6 16 4 id sadct haar / 16 18 6 16 4 dct sadct haar     (step 2 on 2-CTA clusters)
  n32_k16       32 18 6 16 4 id sadct haar / 32 18 6 16 4 dct sadct haar    (step 1 on 2-CTA clusters, step 2 on 4-CTA clusters)

Prints one JSON line: per case LF Mpix/s of both steps (CUDA events), core calls, kernel launches, the per-phase ms of
lfbm5d_get_stats (a further run with the library's per-pass timing on), the group kernel's ms per core call, peak device memory,
the cluster size and cudaOccupancyMaxActiveClusters of each step's group kernel, and the PSNR against the clean light field at
sigma = 25 (timed) and sigma = 50 (information only: mean over the SAIs of the per-SAI PSNR of the final estimate); GPU name and
power limit, read in the same run. The sigma = 50 run comes first and is the warm-up (module loads, buffers, plane tables).

    python tools/bench_large_groups.py [--cases a,b,...] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_angular import AW, AH, H, W, C, gpu_info  # noqa: E402
from bench_patch12 import psnr_lf  # noqa: E402

AN = 1
CASES = {"readme": (8, 16, 16, 8), "n16_k16": (8, 16, 16, 16), "n32_k16": (32, 16, 32, 16)}     # N1, k1, N2, k2


def params(L, sigma, case):
    N1, k1, N2, k2 = CASES[case]
    p1 = L.make_params(sigma, 2.7, AW, AH, AN, W, H, C, N1, 18, 6, k1, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(sigma, 0.0, AW, AH, AN, W, H, C, N2, 18, 6, k2, 4, L.DCT, L.SADCT, L.HAAR)
    return p1, p2


def run_case(L, torch, case, noisy, clean, mask):
    dev = noisy[25].device
    free0, total = torch.cuda.mem_get_info(dev)
    used = [total - free0]
    eng = L.LFBM5D(0)

    def once(sigma, timing):
        w = noisy[sigma].clone()
        b, o = torch.zeros_like(w), torch.zeros_like(w)
        eng.enable_timing(timing)
        p1, p2 = params(L, sigma, case)
        res = {}
        for step in (1, 2):
            eng.reset_stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            if step == 1:
                eng.step1_device(p1, w.data_ptr(), mask, b.data_ptr())
            else:
                eng.step2_device(p2, w.data_ptr(), b.data_ptr(), mask, o.data_ptr())
            e1.record()
            torch.cuda.synchronize()
            s = eng.stats()
            res[step] = dict(ms=e0.elapsed_time(e1), core_calls=int(s.window_passes), kernel_launches=int(s.kernel_launches),
                             ms_block_matching=s.ms_block_matching, ms_sat=s.ms_sat, ms_groups=s.ms_groups,
                             ms_aggregate=s.ms_aggregate, ms_other=s.ms_other)
        used.append(total - torch.cuda.mem_get_info(dev)[0])
        res["psnr"] = psnr_lf(torch, o, clean)
        del w, b, o
        return res

    psnr50 = once(50, False)["psnr"]          # also the warm-up
    t = once(25, False)
    ph = once(25, True)
    out = {}
    p1, p2 = params(L, 25, case)
    for step, prm in ((1, p1), (2, p2)):
        cl, occ = eng.group_cluster(step, prm)
        out["step%d" % step] = {
            "ms": t[step]["ms"], "core_calls": t[step]["core_calls"], "kernel_launches": t[step]["kernel_launches"],
            "group_cluster_ctas": cl, "max_active_clusters": occ if cl > 1 else None,
            "phases_ms_timed_run": {k: ph[step][k] for k in ("ms_block_matching", "ms_sat", "ms_groups", "ms_aggregate", "ms_other")},
            "groups_ms_per_core_call_timed_run": ph[step]["ms_groups"] / max(1, ph[step]["core_calls"]),
        }
    ms = t[1]["ms"] + t[2]["ms"]
    out["lf_mpix_s"] = AW * AH * H * W / (ms * 1e-3) / 1e6
    out["ms_both_steps"] = ms
    out["psnr_sigma25_db"] = t["psnr"]
    out["psnr_sigma50_db"] = psnr50
    out["peak_device_memory_gb"] = max(used) / 1e9
    out["device_memory_before_gb"] = used[0] / 1e9
    eng.close()
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default=",".join(CASES), help="comma-separated cases: " + ", ".join(CASES))
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    import torch
    import lfbm5d_b200 as L
    import lfdata
    if not torch.cuda.is_available():
        raise SystemExit("bench_large_groups.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    clean = torch.from_numpy(lfdata.synth_lf(AW, AH, H, W, C, seed=12345)).to(dev)
    noisy = {}
    for sigma in (25, 50):
        g = torch.Generator(device=dev)
        g.manual_seed(20171016)
        noisy[sigma] = (clean + float(sigma) * torch.randn(clean.shape, generator=g, device=dev)).contiguous()
    mask = np.ones(AW * AH, np.uint32)
    name, pl = gpu_info()
    line = {"tool": "bench_large_groups", "workload": "synthetic LF %dx%d SAIs %dx%d RGB, an %d, opp, device-resident, noise: torch normal "
                    "(seed 20171016), sigma 25 (timed) and 50 (warm-up, PSNR only)" % (AW, AH, W, H, AN),
            "gpu": name or torch.cuda.get_device_name(dev), "power_limit_w": pl,
            "timing": "CUDA events around each step after a warm-up run; phases from a further run with per-pass timing on (adds syncs)",
            "cases": {"readme": "8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar",
                      "n16_k16": "8 18 6 16 4 id sadct haar / 16 18 6 16 4 dct sadct haar",
                      "n32_k16": "32 18 6 16 4 id sadct haar / 32 18 6 16 4 dct sadct haar"}}
    for case in args.cases.split(","):
        line[case] = run_case(L, torch, case, noisy, clean, mask)
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
