"""bench_angular.py — both LFBM5D steps at angular half-windows an = 1 (3x3 SAIs per group) and an = 2 (5x5) on the same synthetic
17x17x1024^2 RGB light field, README parameters (8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar, sigma 10, opp), one GPU,
device-resident. Prints one JSON line: per an, LF Mpix/s of both steps (CUDA events), window passes per step, the per-phase ms of
lfbm5d_get_stats (a second run with the library's per-pass timing on), the group kernel's time with its algorithmic bytes per launch
(G * 4 B written, G = R * N * A * C * k^2, DESIGN.md 4.3) over that time, and peak device memory; GPU name and power limit.
G counts every reference patch of the grid; core calls of the partial-window branch process fewer, so with such calls in a step
(an = 2) the bytes-per-second figure is an upper bound.

    python tools/bench_angular.py [--an 1,2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

AW = AH = 17
H = W = 1024
C = 3
SIGMA = 10.0
STEPS = {1: dict(lam=2.7, N=8, nSim=18, nDisp=6, k=16, p=4, tau2="id"), 2: dict(lam=0.0, N=16, nSim=18, nDisp=6, k=8, p=4, tau2="dct")}


def params(L, step, an):
    s = STEPS[step]
    tau2 = {"id": L.ID, "dct": L.DCT}[s["tau2"]]
    return L.make_params(SIGMA, s["lam"], AW, AH, an, W, H, C, s["N"], s["nSim"], s["nDisp"], s["k"], s["p"], tau2, L.SADCT, L.HAAR)


def grid_refs(step):
    """Reference patches per pass: ind_initialize over the padded image (utilities.cpp:697-712)."""
    s = STEPS[step]
    n = s["nSim"] + s["nDisp"]

    def cnt(dim):
        m = dim + 2 * n - s["k"] + 1
        idx = list(range(n, m - n, s["p"]))
        if idx[-1] < m - n - 1:
            idx.append(m - n - 1)
        return len(idx)
    return cnt(H) * cnt(W)


def group_bytes(step, an):
    """Algorithmic bytes of one group-kernel launch: the G filtered coefficients it writes, G = R * N * A * C * k^2, 4 B each."""
    s = STEPS[step]
    A = (2 * an + 1) ** 2
    return grid_refs(step) * s["N"] * A * C * s["k"] ** 2 * 4.0


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                                      timeout=20).decode().strip().splitlines()[0]
        name, pl = [x.strip() for x in out.split(",")]
        return name, float(pl)
    except Exception:
        return None, None


def run(L, torch, eng, noisy0, mask, an):
    p1, p2 = params(L, 1, an), params(L, 2, an)
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
            out[step] = dict(ms=e0.elapsed_time(e1), passes=int(s.window_passes), ms_block_matching=s.ms_block_matching, ms_sat=s.ms_sat,
                             ms_groups=s.ms_groups, ms_aggregate=s.ms_aggregate)
        del w, b, o
        return out

    both(False)                          # warm-up: module loads, buffers, plane tables
    t = both(False)
    ph = both(True)
    ms = t[1]["ms"] + t[2]["ms"]
    res = {"an": an, "lf_mpix_s": AW * AH * H * W / (ms * 1e-3) / 1e6, "ms_both_steps": ms}
    for step in (1, 2):
        g = group_bytes(step, an)
        res["step%d" % step] = {
            "ms": t[step]["ms"], "passes": t[step]["passes"],
            "phases_ms_timed_run": {k: ph[step][k] for k in ("ms_block_matching", "ms_sat", "ms_groups", "ms_aggregate")},
            "group_kernel": {"kernel": "k_groups25<%d>" % step if an == 2 else "3x3 group kernel", "ms_total": ph[step]["ms_groups"],
                             "ms_per_launch": ph[step]["ms_groups"] / max(1, ph[step]["passes"]), "bytes_per_launch": g,
                             "gb_s": g * ph[step]["passes"] / (ph[step]["ms_groups"] * 1e-3) / 1e9 if ph[step]["ms_groups"] > 0 else None},
        }
    res["peak_device_memory_gb"] = max(used) / 1e9
    res["device_memory_before_gb"] = used[0] / 1e9
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--an", default="1,2", help="comma-separated angular half-windows")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    import torch
    import lfbm5d_b200 as L
    import lfdata
    if not torch.cuda.is_available():
        raise SystemExit("bench_angular.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    clean = torch.from_numpy(lfdata.synth_lf(AW, AH, H, W, C, seed=12345)).to(dev)
    g = torch.Generator(device=dev)
    g.manual_seed(20171016)
    noisy = (clean + SIGMA * torch.randn(clean.shape, generator=g, device=dev)).contiguous()
    del clean
    mask = np.ones(AW * AH, np.uint32)
    name, pl = gpu_info()
    line = {"tool": "bench_angular", "workload": "synthetic LF %dx%d SAIs %dx%d RGB, sigma %g, 8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct "
                    "haar, opp, device-resident, noise: torch normal (seed 20171016)" % (AW, AH, W, H, SIGMA),
            "gpu": name or torch.cuda.get_device_name(dev), "power_limit_w": pl,
            "timing": "CUDA events around each step after one warm-up run; phases from a further run with per-pass timing on (adds syncs)"}
    for an in [int(x) for x in args.an.split(",")]:
        eng = L.LFBM5D(0)
        line["an%d" % an] = run(L, torch, eng, noisy, mask, an)
        eng.close()
        torch.cuda.synchronize()
    if "an1" in line and "an2" in line:
        line["rate_an2_over_an1"] = line["an2"]["lf_mpix_s"] / line["an1"]["lf_mpix_s"]
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
