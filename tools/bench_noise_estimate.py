"""bench_noise_estimate.py — the noise-level estimate (lfbm5d_estimate_sigma) on the synthetic 17x17x1024^2 RGB light field of
bench_angular.py with the reference's noise (lfbm5d_b200.add_noise, sigma 10), one GPU.

  device entry  lfbm5d_estimate_sigma_device on a device-resident light field: one warm-up call, then --calls calls timed with CUDA
                events on the engine's stream; ms per call, and the bytes the three passes read (3 x the light field, computed here)
                over that time as GB/s and as a fraction of the B200's 7.7 TB/s. That fraction is against the read bound: every pass
                reads the whole light field once and nothing else of size.
  host entry    lfbm5d_estimate_sigma on host arrays (upload of every SAI included): wall clock around each synchronous call.

Prints one JSON line with the GPU name and power limit read in the same run.

    python tools/bench_noise_estimate.py [--calls N] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_angular import AW, AH, H, W, C, gpu_info  # noqa: E402

SIGMA = 10.0
PEAK_BYTES_S = 7.7e12          # HBM3e bandwidth of one B200 (NVIDIA data sheet)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20, help="timed calls of the device entry (>= 20)")
    ap.add_argument("--host-calls", type=int, default=3, help="timed calls of the host entry")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    import torch
    import lfbm5d_b200 as L
    import lfdata
    if not torch.cuda.is_available():
        raise SystemExit("bench_noise_estimate.py needs a CUDA device")
    calls = max(20, args.calls)
    asize = AW * AH
    noisy = L.add_noise(lfdata.synth_lf(AW, AH, H, W, C), SIGMA)
    mask = np.ones(asize, np.uint32)
    eng = L.LFBM5D(0)
    dev = torch.device("cuda", 0)
    d = torch.from_numpy(noisy).to(dev)
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)

    res = eng.estimate_sigma_device(d.data_ptr(), mask, asize, C, W, H)      # warm-up: module load, buffers
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.reset_stats()
    e0.record(stream)
    for _ in range(calls):
        res = eng.estimate_sigma_device(d.data_ptr(), mask, asize, C, W, H)
    e1.record(stream)
    e1.synchronize()
    ms = e0.elapsed_time(e1) / calls
    launches = int(eng.stats().kernel_launches) // calls
    lf_bytes = asize * C * (H // 2 * 2) * (W // 2 * 2) * 4
    read = 3 * lf_bytes

    host_s = []
    for _ in range(args.host_calls):
        t0 = time.perf_counter()
        hres = eng.estimate_sigma(noisy, mask)
        host_s.append(time.perf_counter() - t0)
    assert hres[0] == res[0] and np.array_equal(hres[2], res[2]), "host and device entry points disagree"
    eng.close()

    name, pl = gpu_info()
    line = {"tool": "bench_noise_estimate",
            "workload": "synthetic LF %dx%d SAIs %dx%d RGB, reference noise (add_noise, seed 20171016 + st), sigma %g" % (AW, AH, W, H, SIGMA),
            "gpu": name or torch.cuda.get_device_name(dev), "power_limit_w": pl,
            "device_entry": {"calls_timed": calls, "ms_per_call": ms, "kernel_launches_per_call": launches,
                             "bytes_read_per_call": read, "gb_s": read / (ms * 1e-3) / 1e9,
                             "fraction_of_7.7TB_s_read_bound": read / (ms * 1e-3) / PEAK_BYTES_S,
                             "timing": "CUDA events on the engine's stream around %d back-to-back calls (each ends with a stream "
                                       "synchronise and a 1.2 KB copy of the result); light field %.2f GB, larger than L2" % (calls, lf_bytes / 1e9)},
            "host_entry": {"s_per_call": host_s, "upload_gb": lf_bytes / 1e9,
                           "timing": "wall clock around the synchronous call (pageable host arrays, upload included)"},
            "sigma_true": SIGMA, "sigma": res[0], "sigma_chnl": [float(x) for x in res[1]],
            "sigma_sai_min_max": [float(res[2].min()), float(res[2].max())]}
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
