"""bench_patch12.py — 12 x 12 patches against the README patch sizes, one process, one GPU, device-resident, on the synthetic
17x17x1024^2 RGB light field of bench_angular.py / bench_disparity.py (opp, an = 1):

  lfbm5d_k16_k8  README parameters: 8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar
  lfbm5d_k12     k = 12 in both steps: 8 18 6 12 4 id sadct haar / 16 18 6 12 4 dct sadct haar
  lfbm5d_k16_k8_cp_async  the README parameters with the TMA source-row loads of the summed-area planes switched off
                 (LFBM5D_NO_TMA): k = 12 always takes the cp.async variant, so this is the cost of that choice at k = 8 / 16
  lfbm3d_k8      config 4 parameters: 16 16 8 3 bior / 32 16 8 3 dct
  lfbm3d_k12     12 x 12 patches, dct in both steps: 16 16 12 3 dct / 32 16 12 3 dct

Prints one JSON line: per case LF Mpix/s of both steps (CUDA events, after a warm-up run), kernel launches, the per-phase ms of
lfbm5d_get_stats (LFBM5D: a further run with the library's per-pass timing on), peak device memory, and the PSNR against the clean
light field at sigma = 10 and sigma = 50 (for information: mean over the SAIs of the per-SAI PSNR of the final estimate); GPU name
and power limit, read in the same run.

    python tools/bench_patch12.py [--cases a,b,...] [--out FILE]
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

AN = 1
CASES = ["lfbm5d_k16_k8", "lfbm5d_k12", "lfbm5d_k16_k8_cp_async", "lfbm3d_k8", "lfbm3d_k12"]


def params5(L, sigma, case):
    k1, k2 = (12, 12) if case == "lfbm5d_k12" else (16, 8)
    p1 = L.make_params(sigma, 2.7, AW, AH, AN, W, H, C, 8, 18, 6, k1, 4, L.ID, L.SADCT, L.HAAR)
    p2 = L.make_params(sigma, 0.0, AW, AH, AN, W, H, C, 16, 18, 6, k2, 4, L.DCT, L.SADCT, L.HAAR)
    return p1, p2


def params3(L, sigma, case):
    if case == "lfbm3d_k12":
        return L.make_params3d(sigma, AW * AH, W, H, C, 16, 16, 12, 12, 16, 32, 3, 3, L.DCT, L.DCT, 2.7)
    return L.make_params3d(sigma, AW * AH, W, H, C, 16, 16, 8, 8, 16, 32, 3, 3, L.BIOR, L.DCT, 2.7)


def psnr_lf(torch, out, clean):
    mse = ((out.double() - clean.double()) ** 2).flatten(1).mean(1)
    return float((10.0 * torch.log10(255.0 ** 2 / mse)).mean())


def run_case(L, torch, case, noisy, clean, mask):
    dev = noisy[10].device
    free0, total = torch.cuda.mem_get_info(dev)
    used = [total - free0]
    eng = L.LFBM5D(0)
    bm3d = case.startswith("lfbm3d")

    def once(sigma, timing):
        w = noisy[sigma].clone()
        b, o = torch.zeros_like(w), torch.zeros_like(w)
        eng.enable_timing(timing)
        res = {}
        if bm3d:
            eng.reset_stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            eng.bm3d_device(params3(L, sigma, case), w.data_ptr(), mask, b.data_ptr(), o.data_ptr())
            e1.record()
            torch.cuda.synchronize()
            s = eng.stats()
            res["both"] = dict(ms=e0.elapsed_time(e1), kernel_launches=int(s.kernel_launches))
        else:
            p1, p2 = params5(L, sigma, case)
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

    once(10, False)                      # warm-up: module loads, buffers, plane tables
    t = once(10, False)
    out = {}
    if bm3d:
        ms = t["both"]["ms"]
        out["kernel_launches"] = t["both"]["kernel_launches"]
    else:
        ph = once(10, True)
        ms = t[1]["ms"] + t[2]["ms"]
        for step in (1, 2):
            out["step%d" % step] = {
                "ms": t[step]["ms"], "core_calls": t[step]["core_calls"], "kernel_launches": t[step]["kernel_launches"],
                "phases_ms_timed_run": {k: ph[step][k] for k in ("ms_block_matching", "ms_sat", "ms_groups", "ms_aggregate", "ms_other")},
            }
    out["lf_mpix_s"] = AW * AH * H * W / (ms * 1e-3) / 1e6
    out["ms_both_steps"] = ms
    out["psnr_sigma10_db"] = t["psnr"]
    out["psnr_sigma50_db"] = once(50, False)["psnr"]
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
        raise SystemExit("bench_patch12.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    clean = torch.from_numpy(lfdata.synth_lf(AW, AH, H, W, C, seed=12345)).to(dev)
    noisy = {}
    for sigma in (10, 50):
        g = torch.Generator(device=dev)
        g.manual_seed(20171016)
        noisy[sigma] = (clean + float(sigma) * torch.randn(clean.shape, generator=g, device=dev)).contiguous()
    mask = np.ones(AW * AH, np.uint32)
    name, pl = gpu_info()
    line = {"tool": "bench_patch12", "workload": "synthetic LF %dx%d SAIs %dx%d RGB, an %d, opp, device-resident, noise: torch normal "
                    "(seed 20171016), sigma 10 (timed) and 50 (PSNR only)" % (AW, AH, W, H, AN),
            "gpu": name or torch.cuda.get_device_name(dev), "power_limit_w": pl,
            "timing": "CUDA events around each step (LFBM3D: around both steps) after one warm-up run; LFBM5D phases from a further "
                      "run with per-pass timing on (adds syncs)",
            "cases": {"lfbm5d_k16_k8": "8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar",
                      "lfbm5d_k12": "8 18 6 12 4 id sadct haar / 16 18 6 12 4 dct sadct haar",
                      "lfbm5d_k16_k8_cp_async": "README parameters, LFBM5D_NO_TMA=1 (cp.async source rows, as k = 12 always uses)",
                      "lfbm3d_k8": "16 16 8 3 bior / 32 16 8 3 dct", "lfbm3d_k12": "16 16 12 3 dct / 32 16 12 3 dct"}}
    for case in args.cases.split(","):
        if case.endswith("_cp_async"):
            os.environ["LFBM5D_NO_TMA"] = "1"
        line[case] = run_case(L, torch, case, noisy, clean, mask)
        os.environ.pop("LFBM5D_NO_TMA", None)
    if "lfbm5d_k16_k8" in line and "lfbm5d_k12" in line:
        line["lfbm5d_time_k12_over_k16_k8"] = line["lfbm5d_k16_k8"]["lf_mpix_s"] / line["lfbm5d_k12"]["lf_mpix_s"]
    if "lfbm3d_k8" in line and "lfbm3d_k12" in line:
        line["lfbm3d_time_k12_over_k8"] = line["lfbm3d_k8"]["lf_mpix_s"] / line["lfbm3d_k12"]["lf_mpix_s"]
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
