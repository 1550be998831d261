"""bench_disparity.py — both LFBM5D steps at disparity half windows nDisp = 6, 8, 12, 16 on the same synthetic 17x17x1024^2 RGB
light field, README parameters otherwise (8 18 nDisp 16 4 id sadct haar / 16 18 nDisp 8 4 dct sadct haar, sigma 10, opp, an = 1),
one GPU, device-resident. Prints one JSON line: per nDisp, LF Mpix/s of both steps (CUDA events), core calls per step, the per-phase
ms of lfbm5d_get_stats (a second run with the library's per-pass timing on), the stereo slots the disparity sums buffer holds and
peak device memory; GPU name and power limit, read in the same run.

    python tools/bench_disparity.py [--ndisp 6,8,12,16] [--out FILE]
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

from bench_angular import AW, AH, H, W, C, SIGMA, gpu_info  # noqa: E402

AN = 1


def params(L, step, nDisp):
    if step == 1:
        return L.make_params(SIGMA, 2.7, AW, AH, AN, W, H, C, 8, 18, nDisp, 16, 4, L.ID, L.SADCT, L.HAAR)
    return L.make_params(SIGMA, 0.0, AW, AH, AN, W, H, C, 16, 18, nDisp, 8, 4, L.DCT, L.SADCT, L.HAAR)


def buffer_slots(nDisp):
    """Stereo slots of the disparity sums buffer (stereo_buffer_slots in csrc/lfbm5d_cuda.cu)."""
    a1 = (2 * AN + 1) ** 2 - 1
    return min(a1, max(1, a1 * 169 // (2 * nDisp + 1) ** 2))


def run(L, torch, eng, noisy0, mask, nDisp):
    p1, p2 = params(L, 1, nDisp), params(L, 2, nDisp)
    dev = noisy0.device
    free0, total = torch.cuda.mem_get_info(dev)
    used = [total - free0]

    def both(timing):
        w = noisy0.clone()
        b, o = torch.zeros_like(w), torch.zeros_like(w)
        eng.enable_timing(timing)
        out = {}
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
            used.append(total - torch.cuda.mem_get_info(dev)[0])
            s = eng.stats()
            out[step] = dict(ms=e0.elapsed_time(e1), core_calls=int(s.window_passes), kernel_launches=int(s.kernel_launches),
                             ms_block_matching=s.ms_block_matching, ms_sat=s.ms_sat, ms_groups=s.ms_groups, ms_aggregate=s.ms_aggregate,
                             ms_other=s.ms_other)
        del w, b, o
        return out

    both(False)                          # warm-up: module loads, buffers, plane tables
    t = both(False)
    ph = both(True)
    ms = t[1]["ms"] + t[2]["ms"]
    res = {"nDisp": nDisp, "disparity_planes": (2 * nDisp + 1) ** 2, "sums_buffer_slots": buffer_slots(nDisp),
           "lf_mpix_s": AW * AH * H * W / (ms * 1e-3) / 1e6, "ms_both_steps": ms}
    for step in (1, 2):
        res["step%d" % step] = {
            "ms": t[step]["ms"], "core_calls": t[step]["core_calls"], "kernel_launches": t[step]["kernel_launches"],
            "phases_ms_timed_run": {k: ph[step][k] for k in ("ms_block_matching", "ms_sat", "ms_groups", "ms_aggregate", "ms_other")},
        }
    res["peak_device_memory_gb"] = max(used) / 1e9
    res["device_memory_before_gb"] = used[0] / 1e9
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ndisp", default="6,8,12,16", help="comma-separated disparity half windows")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    import torch
    import lfbm5d_b200 as L
    import lfdata
    if not torch.cuda.is_available():
        raise SystemExit("bench_disparity.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    clean = torch.from_numpy(lfdata.synth_lf(AW, AH, H, W, C, seed=12345)).to(dev)
    g = torch.Generator(device=dev)
    g.manual_seed(20171016)
    noisy = (clean + SIGMA * torch.randn(clean.shape, generator=g, device=dev)).contiguous()
    del clean
    mask = np.ones(AW * AH, np.uint32)
    name, pl = gpu_info()
    line = {"tool": "bench_disparity", "workload": "synthetic LF %dx%d SAIs %dx%d RGB, sigma %g, an %d, 8 18 nDisp 16 4 id sadct haar / "
                    "16 18 nDisp 8 4 dct sadct haar, opp, device-resident, noise: torch normal (seed 20171016)" % (AW, AH, W, H, SIGMA, AN),
            "gpu": name or torch.cuda.get_device_name(dev), "power_limit_w": pl,
            "timing": "CUDA events around each step after one warm-up run; phases from a further run with per-pass timing on (adds syncs)"}
    rates = {}
    for nd in [int(x) for x in args.ndisp.split(",")]:
        eng = L.LFBM5D(0)
        line["ndisp%d" % nd] = run(L, torch, eng, noisy, mask, nd)
        rates[nd] = line["ndisp%d" % nd]["lf_mpix_s"]
        eng.close()
        torch.cuda.synchronize()
    if 6 in rates:
        line["time_over_ndisp6"] = {str(nd): rates[6] / r for nd, r in rates.items()}
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
