#!/usr/bin/env python
"""bench.py — LF Mpix/s of both LFBM5D steps on a synthetic 17x17x1024^2 RGB light field (BASELINE.json configs[2]).

  python bench.py --gpus N --steps K --warmup W           # this framework, one rank per GPU
  python bench.py --impl reference --gpus N ...            # the reference's own CPU code on the host cores
  python bench.py ... --dump-outputs DIR                   # also write a fixed sample of the last timed step's outputs

A "step" is one full denoising of the light field: hard-threshold step then Wiener step. The noisy input is produced on the
host by the reference's generator (mt19937ar + Box-Muller, utilities.cpp:154-185; the product's own restatement in
lfbm5d_b200/csrc/lf_io.h, SAI st seeded 20171016 + st).
  N = 1: `value` is measured with the light field resident in HBM (device pointers into the C ABI); `e2e` goes through the
         host-buffer C ABI calls a drop-in user makes (pinned host arrays, H2D / D2H inside the timed region).
  N > 1: ONE light field on all N GPUs ("scaling": "strong"): every window pass is split inside the window over the ranks of a
         team (lfbm5d_b200/csrc/team.cuh: plane-parallel block matching, row-band groups / aggregation, NCCL send/recv for the
         halo rows, the border sums and the match tables); results are bit-identical to one GPU. `e2e`: every rank uploads the
         rows of its band from pinned host memory and downloads its band of the result.
Rank 0 prints ONE JSON line."""
import argparse
import ctypes as Cc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")      # team lanes: concurrent streams must not share a hardware queue

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# BASELINE.json configs[2] / SURVEY.md 8(d) "Config 3": README.md:61 parameters
CFG = dict(aw=17, ah=17, H=1024, W=1024, C=3, sigma=10.0, lam=2.7, an=1,
           s1=dict(N=8, nSim=18, nDisp=6, k=16, p=4, tau2="id"), s2=dict(N=16, nSim=18, nDisp=6, k=8, p=4, tau2="dct"))
WORKLOAD = "configs[2]: Stanford-shaped synthetic LF 17x17 SAIs 1024x1024 RGB, sigma 10, 8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar, opp"
METRIC = "LF Mpix/s (both steps) 17x17x1024^2 RGB"
N_PASSES = 64            # window passes per step at 17x17 with an = 1 (SURVEY.md A1)
SEED0 = 20171016
DUMP_SAMPLES = 1 << 22   # elements kept per dumped output: 16 MB of float32 each, three outputs at most


def config_dict(world):
    """Identical for both arms (the reference arm times a bounded sample of this same workload; see its cpu_baseline.sample)."""
    return {"workload": WORKLOAD,
            "partition": "one light field on one GPU" if world == 1 else
                         "one light field on %d GPUs: every window pass split inside the window (offset planes of the block matching dealt out whole, "
                         "reference rows and the pixel rows they aggregate into in bands, halo = search radius + patch size)" % world,
            "l2": "inputs (3.6 GB per buffer) larger than L2", "passes_per_step": N_PASSES,
            "noise": "host mt19937ar + Box-Muller (utilities.cpp:154-185), seed 20171016 + st"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.check_output(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                               "--format=csv,noheader,nounits"], timeout=5).decode().strip()
                self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def params(L, which, aw=None, ah=None, H=None, W=None, sigma=None):
    s = CFG[which]
    tau2 = {"id": L.ID, "dct": L.DCT, "bior": L.BIOR}[s["tau2"]]
    return L.make_params(sigma or CFG["sigma"], CFG["lam"] if which == "s1" else 0.0, aw or CFG["aw"], ah or CFG["ah"], CFG["an"], W or CFG["W"],
                         H or CFG["H"], CFG["C"], s["N"], s["nSim"], s["nDisp"], s["k"], s["p"], tau2, L.SADCT, L.HAAR)


def grid_counts(which):
    s = CFG[which]
    n = s["nSim"] + s["nDisp"]

    def cnt(dim):
        m = dim + 2 * n - s["k"] + 1
        idx = list(range(n, m - n, s["p"]))
        if idx[-1] < m - n - 1:
            idx.append(m - n - 1)
        return len(idx)
    return cnt(CFG["H"]) * cnt(CFG["W"])


def algorithmic_bytes_groups(which):
    """SURVEY.md 8(d): unfused two-kernel model, 2*G*4 B per window pass, G = R*N*A*C*k^2 coefficients."""
    s = CFG[which]
    G = grid_counts(which) * s["N"] * 9 * CFG["C"] * s["k"] ** 2
    return 2.0 * G * 4.0


def algorithmic_flops_bm(which):
    """SURVEY.md 8(d): direct-SSD count, 3 flop per pixel pair: self R*(2nSim+1)^2*k^2*3 + stereo (A-1)*min(P,R*N)*(2nDisp+1)^2*k^2*3."""
    s = CFG[which]
    n = s["nSim"] + s["nDisp"]
    R = grid_counts(which)
    P = (CFG["H"] + 2 * n - s["k"] + 1 - 2 * s["nDisp"]) * (CFG["W"] + 2 * n - s["k"] + 1 - 2 * s["nDisp"])
    return R * (2 * s["nSim"] + 1) ** 2 * s["k"] ** 2 * 3.0 + 8 * min(P, R * s["N"]) * (2 * s["nDisp"] + 1) ** 2 * s["k"] ** 2 * 3.0


def executed_flops_bm(which):
    """What the summed-area kernels execute per pass: 14 flop per (pixel, offset plane), (nSim+1)(2nSim+1) self and 8 (2nDisp+1)^2 disparity planes."""
    s = CFG[which]
    n = s["nSim"] + s["nDisp"]
    planes = (s["nSim"] + 1) * (2 * s["nSim"] + 1) + 8 * (2 * s["nDisp"] + 1) ** 2
    return planes * float(CFG["H"] + n) * float(CFG["W"] + n) * 14.0


def clean_lf(aw, ah, H, W, C, seed=12345):
    """Deterministic synthetic clean light field: procedural texture cropped at 1 px / view disparity (tests/lfdata.py)."""
    import lfdata
    return lfdata.synth_lf(aw, ah, H, W, C, seed=seed)


def sample_outputs(torch, arrays):
    """Host copies of the same fixed DUMP_SAMPLES flat positions (drawn without replacement from seed 0, ascending) of each
    equally shaped device array, so that the outputs of two builds can be compared element for element."""
    n = next(iter(arrays.values())).numel()
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SAMPLES), replace=False, shuffle=False))
    idx = torch.from_numpy(idx).to(next(iter(arrays.values())).device)
    return {name: t.reshape(-1)[idx].cpu().numpy() for name, t in arrays.items()}


def host_ptrs(t, asize):
    each = t[0].numel()
    return (Cc.POINTER(Cc.c_float) * asize)(*[Cc.cast(t.data_ptr() + 4 * each * i, Cc.POINTER(Cc.c_float)) for i in range(asize)])


def run_ours(args):
    import torch
    import lfbm5d_b200 as L

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng = L.LFBM5D(local)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    asize, H, W, C = CFG["aw"] * CFG["ah"], CFG["H"], CFG["W"], CFG["C"]
    lf_pix = asize * H * W
    # ---- inputs: rank 0 builds the clean LF and the reference's host noise; the others receive the noisy LF ----
    noisy0 = torch.empty((asize, C, H, W), device=dev)
    clean = None
    if rank == 0:
        clean_h = clean_lf(CFG["aw"], CFG["ah"], H, W, C)
        noisy_h = L.add_noise(clean_h, CFG["sigma"], SEED0)
        noisy0.copy_(torch.from_numpy(noisy_h))
        clean = torch.from_numpy(clean_h).to(dev)
        del noisy_h
    if world > 1:
        dist.broadcast(noisy0, src=0)
    work, basic, out = torch.empty_like(noisy0), torch.empty_like(noisy0), torch.empty_like(noisy0)
    mask = np.ones(asize, np.uint32)
    p1, p2 = params(L, "s1"), params(L, "s2")
    if args.passes:
        eng.set_max_passes(args.passes)
    team = None
    if world > 1:
        from lfbm5d_b200 import dist as D
        team = D.make_team(eng, dist, dev)
        if args.lanes > 1:
            team.set_lanes(args.lanes)
    torch.cuda.synchronize()

    def one_step():
        with torch.cuda.stream(stream):
            work.copy_(noisy0, non_blocking=True)
        if team is None:
            eng.step1_device(p1, work.data_ptr(), mask, basic.data_ptr())
            eng.step2_device(p2, work.data_ptr(), basic.data_ptr(), mask, out.data_ptr())
        else:       # the basic estimate stays band-resident between the steps; the result is gathered: every rank ends with all of it
            team.step(1, p1, [work.data_ptr()], None, mask, [basic.data_ptr()], gather=0)
            team.step(2, p2, [work.data_ptr()], [basic.data_ptr()], mask, [out.data_ptr()], gather=1)

    for _ in range(args.warmup):
        one_step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    eng.reset_stats()
    bytes0 = team.stats()["bytes_exchanged"] if team else 0
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        one_step()
    e1.record(stream)
    e1.synchronize()
    barrier()
    # what a caller of the timed path holds after its last step, taken before the profile run below overwrites it. The team
    # path leaves basic and the round-tripped noisy LF band-resident; only the gathered result is complete on a rank.
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = sample_outputs(torch, {"denoised": out, "basic": basic, "noisy_roundtrip": work} if team is None else {"denoised": out})
    ms = e0.elapsed_time(e1)
    st = eng.stats()
    launches = int(st.kernel_launches)
    sampler.stop_flag = True
    tmax = torch.tensor([ms, float(launches)], device=dev, dtype=torch.float64)
    if world > 1:
        tm = tmax.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = tmax.clone()
        dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        ms = float(tm[0].item())
        tl = torch.tensor([float(team.launches())], device=dev, dtype=torch.float64)
        dist.all_reduce(tl, op=dist.ReduceOp.SUM)
        launches = int(tl.item())
    ms_per_step = ms / args.steps
    frac_passes = 1.0 if not args.passes else args.passes / float(N_PASSES)
    value = lf_pix * frac_passes / (ms_per_step * 1e-3) / 1e6
    team_info = None
    if team is not None:
        tst = team.stats()
        team_info = {"lanes": args.lanes, "nvlink_bytes_sent_per_rank_per_step": (tst["bytes_exchanged"] - bytes0) / args.steps, "peer_view": tst["peer_view"],
                     "passes_redone": tst["passes_redone"], "band_rows_rank0": team.band(0)}

    # quality of the timed output: PSNR against the clean LF (utilities.cpp:412-435, mean over the SAIs)
    psnr = None
    if rank == 0 and not args.passes:
        oh, nh, ch = out.cpu().numpy(), noisy0.cpu().numpy(), clean.cpu().numpy()
        psnr = {"noisy": L.psnr_lf(nh, ch), "denoised": L.psnr_lf(oh, ch)}
        del oh, nh, ch

    # ---- e2e: host buffers, copies inside the timed region ----
    e2e = measure_e2e(args, L, torch, dist, eng, team, dev, rank, world, noisy0, mask, p1, p2, lf_pix, frac_passes, barrier) if not args.no_e2e else None

    # ---- per-kernel timing for the roofline (separate short run with per-phase CUDA events on the library's stream) ----
    roof, roof_other, roof_bm, phases, team_phases = None, None, None, None, None
    if world > 1 and args.profile_passes > 0:
        eng.set_max_passes(args.profile_passes)
        team.timing(True)
        work.copy_(noisy0)
        torch.cuda.synchronize()
        team.step(1, p1, [work.data_ptr()], None, mask, [basic.data_ptr()], gather=0)
        t1 = team.timing(False)
        team.timing(True)
        team.step(2, p2, [work.data_ptr()], [basic.data_ptr()], mask, [out.data_ptr()], gather=0)
        t2 = team.timing(False)
        eng.set_max_passes(args.passes or 0)
        names = ["pad", "x_est0", "block_matching", "x_match_tables", "selection_groups_aggregate1", "x_border_rows", "aggregate2", "x_border_rows_back_counters",
                 "bm_self_planes", "bm_partial_selection", "bm_disparity_planes", "bm_disparity_argmin"]
        team_phases = {"rank0_ms_per_pass": {"step1": {k: v / args.profile_passes for k, v in zip(names, t1)},
                                             "step2": {k: v / args.profile_passes for k, v in zip(names, t2)}}}
    if rank == 0 and world == 1 and args.profile_passes > 0:
        eng.enable_timing(True)
        eng.set_max_passes(args.profile_passes)
        eng.reset_stats()
        work.copy_(noisy0)
        eng.step1_device(p1, work.data_ptr(), mask, basic.data_ptr())
        s1 = eng.stats()
        eng.reset_stats()
        eng.step2_device(p2, work.data_ptr(), basic.data_ptr(), mask, out.data_ptr())
        s2 = eng.stats()
        eng.enable_timing(False)
        eng.set_max_passes(args.passes or 0)
        hbm, how = peaks()
        n1, n2 = max(1, s1.window_passes), max(1, s2.window_passes)
        g_ms = (s1.ms_groups / n1, s2.ms_groups / n2)
        a_ms = (s1.ms_aggregate / n1, s2.ms_aggregate / n2)
        sat_ms = (s1.ms_sat / n1, s2.ms_sat / n2)
        # SURVEY 8(d) two-kernel model: the transform kernel writes G*4 B of filtered coefficients (and reads the 9 padded
        # SAIs once), the aggregation kernel reads G*4 B and writes num/den once
        half = (algorithmic_bytes_groups("s1") / 2.0, algorithmic_bytes_groups("s2") / 2.0)
        wb = (CFG["W"] + 48) * (CFG["H"] + 48) * 9 * CFG["C"] * 4.0
        bytes_t = (half[0] + wb, half[1] + 2 * wb)
        bytes_a = (half[0] + 2 * wb, half[1] + 2 * wb)
        traffic = ncu_traffic()

        def entry(kernel, ncu_name, nbytes, ms_, model):
            t = traffic.get(ncu_name)
            ach = nbytes / (ms_ * 1e-3) / 1e9
            return {"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                    "traffic": None if t is None else t["dram_gb_per_launch"] * 1e9, "traffic_source": None if t is None else traffic["_file"],
                    "algorithmic_bytes": nbytes, "ms_per_launch": ms_, "peak_source": how, "model": model}

        m_t = "algorithmic bytes per launch = G*4 B written + padded window read once (SURVEY 8(d)), G=R*N*A*C*k^2"
        m_a = "algorithmic bytes per launch = G*4 B read + num/den read and written once (SURVEY 8(d))"
        kernels = [entry("k_groups_id16<3> (step 1)", "k_groups_id16<3>", bytes_t[0], g_ms[0], m_t),
                   entry("k_groups_w8<3> (step 2)", "k_groups_w8<3>", bytes_t[1], g_ms[1], m_t),
                   entry("k_aggregate<16, 3> (step 1)", "k_aggregate<16, 3>", bytes_a[0], a_ms[0], m_a),
                   entry("k_aggregate<8, 3> (step 2)", "k_aggregate<8, 3>", bytes_a[1], a_ms[1], m_a)]
        kernels[1]["note"] = "issue-limited, not bandwidth-limited: ~100 flop per coefficient (2-D + angular DCT, Haar, Wiener, inverses)"
        kernels.sort(key=lambda e: -e["ms_per_launch"])
        roof, roof_other = kernels[0], kernels[1:]
        fl = (algorithmic_flops_bm("s1"), algorithmic_flops_bm("s2"))
        ach_bm = (fl[0] + fl[1]) / ((sat_ms[0] + sat_ms[1]) * 1e-3) / 1e12
        fp32 = fp32_peak()
        ex = (executed_flops_bm("s1"), executed_flops_bm("s2"))
        ex_bm = (ex[0] + ex[1]) / ((sat_ms[0] + sat_ms[1]) * 1e-3) / 1e12
        roof_bm = {"kernel": "k_sat_edges + k_sat2 (summed-area planes of a pass, both streams; source rows by TMA)", "bound": "fp32", "achieved": ex_bm, "peak": fp32["tflops"],
                   "unit": "TFLOP/s", "frac": ex_bm / fp32["tflops"], "peak_source": fp32["source"],
                   "model": "EXECUTED flops: 14 per (pixel, offset plane) of the reference's float32 summed-area recurrence (4 differences, 4 squares, 6 additions; "
                            "703 self + 8 x 169 disparity planes of ~(H + n) x (W + n) sums). The recurrence is issue / latency bound (shared-memory operands, one "
                            "shuffle and a dependent chain of 6 additions per step), not FMA bound: see the issue and FMA-pipe columns of profiles/*_kernels.md",
                   "direct_ssd_equivalent": {"tflops": ach_bm, "of_fp32_peak": ach_bm / fp32["tflops"],
                                             "model": "SURVEY 8(d): the flops a direct block matching (3 per pixel pair) would execute for the same match lists; "
                                                      "an equivalence, not a pipe utilisation (it exceeds 1 because the summed areas share work between patches)"},
                   "ms_per_pass": {"step1": sat_ms[0], "step2": sat_ms[1]}}
        phases = {"step1_ms_per_pass": {"block_matching": s1.ms_block_matching / n1, "groups": g_ms[0], "aggregate": a_ms[0]},
                  "step2_ms_per_pass": {"block_matching": s2.ms_block_matching / n2, "groups": g_ms[1], "aggregate": a_ms[1]}}

    # ---- CPU baseline on the host cores (bounded sample) and the parity block: rank 0 at N = 1 only ----
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_sample(size=int(os.environ.get("LFBM5D_CPU_SAMPLE", "512")))
        parity = parity_block(L, eng)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "LF Mpix/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config_dict(world),
                "e2e": e2e, "gpu_launches": launches, "clocks": sampler.summary(), "roofline": roof, "roofline_other": roof_other, "roofline_bm": roof_bm,
                "phases": phases, "team": team_info, "team_phases": team_phases, "cpu_baseline": cpu, "parity": parity, "psnr": psnr}
        print(json.dumps(line))
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if team is not None:
        team.close()
    if world > 1:
        dist.destroy_process_group()


def measure_e2e(args, L, torch, dist, eng, team, dev, rank, world, noisy0, mask, p1, p2, lf_pix, frac_passes, barrier):
    asize = noisy0.shape[0]
    H, W, C = CFG["H"], CFG["W"], CFG["C"]
    ok = 1
    try:
        h_noisy0 = torch.empty(noisy0.shape, pin_memory=True)
        h_noisy0.copy_(noisy0)
        h_out = torch.empty(noisy0.shape, pin_memory=True)
        if world == 1:
            h_noisy = torch.empty(noisy0.shape, pin_memory=True)
            h_basic = torch.empty(noisy0.shape, pin_memory=True)
    except RuntimeError:
        ok = 0
    if world > 1:
        f = torch.tensor([ok], device=dev)
        dist.all_reduce(f, op=dist.ReduceOp.MIN)
        ok = int(f.item())
    if not ok:
        return {"value": None, "unit": "LF Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": "pinned host allocation failed"}
    m = mask.ctypes.data_as(Cc.POINTER(Cc.c_uint))
    nbytes = noisy0.numel() * 4
    if world == 1:
        def e2e_step():
            h_noisy.copy_(h_noisy0)      # untimed: the call overwrites its input with the colour-round-tripped copy (the reference's side effect)
            t0 = time.perf_counter()
            if eng.lib.lfbm5d_step1(eng.ctx, Cc.byref(p1), host_ptrs(h_noisy, asize), m, host_ptrs(h_basic, asize)) != 0:
                raise RuntimeError(eng.error())
            if eng.lib.lfbm5d_step2(eng.ctx, Cc.byref(p2), host_ptrs(h_noisy, asize), host_ptrs(h_basic, asize), m, host_ptrs(h_out, asize)) != 0:
                raise RuntimeError(eng.error())
            _ = float(h_out[0, 0, 0, 0])      # the result is read on the host
            return time.perf_counter() - t0
        h2d, d2h = 3 * nbytes, 5 * nbytes
        note = "host-buffer C ABI (lfbm5d_step1 / lfbm5d_step2): noisy up, basic + colour-round-tripped noisy down, both up again, denoised + round-tripped inputs down"
    else:
        # every rank uploads the rows of the noisy LF its band reads (union of both steps' bands) and downloads its band of the result
        b1, b2 = L.plan_band(world, rank, 1, p1), L.plan_band(world, rank, 2, p2)
        up_lo, up_hi = min(b1[0], b2[0]), max(b1[2], b2[2])
        d_work, d_basic, d_out = torch.empty_like(noisy0), torch.empty_like(noisy0), torch.empty_like(noisy0)
        hp_in, hp_out = host_ptrs(h_noisy0, asize), host_ptrs(h_out, asize)

        def e2e_step():
            eng.copy_rows(hp_in, d_work.data_ptr(), mask, asize, C, W, H, up_lo, up_hi, 1)
            team.step(1, p1, [d_work.data_ptr()], None, mask, [d_basic.data_ptr()], gather=0)
            team.step(2, p2, [d_work.data_ptr()], [d_basic.data_ptr()], mask, [d_out.data_ptr()], gather=0)
            lo, hi, _ = team.band(rank)
            eng.copy_rows(hp_out, d_out.data_ptr(), mask, asize, C, W, H, lo, hi, 0)
            eng.sync()
            _ = float(h_out[0, 0, lo, 0]) if hi > lo else 0.0
            return None
        rows = torch.tensor([float(up_hi - up_lo), float(b2[1] - b2[0])], device=dev, dtype=torch.float64)
        dist.all_reduce(rows, op=dist.ReduceOp.SUM)
        h2d, d2h = int(rows[0].item()) * asize * C * W * 4, int(rows[1].item()) * asize * C * W * 4
        note = "every rank uploads the rows its band reads (own band + halo) from pinned host memory and downloads its band of the denoised LF; bytes summed over the ranks"
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    inner = 0.0
    for _ in range(args.steps):
        dt = e2e_step()
        inner += dt if dt is not None else 0.0
    torch.cuda.synchronize()
    # N = 1: the synchronous host-buffer calls are timed one by one (the refresh of the input array between them is not part of
    # the path); N > 1: wall clock around the whole loop
    t_e2e = torch.tensor([inner if world == 1 else time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    return {"value": lf_pix * frac_passes / (float(t_e2e.item()) / args.steps) / 1e6, "unit": "LF Mpix/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "timer": "host wall clock around the (synchronous) calls, max over ranks", "path": note}


def fp32_peak():
    """FP32 FMA peak from the microbenchmark tools/fp32_peak (profiles/*fp32_peak.json), else the nominal figure."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*fp32_peak.json")))
    if files:
        d = json.load(open(files[-1]))
        return {"tflops": float(d["fp32_fma_tflops"]), "source": "measured FFMA microbenchmark, profiles/" + os.path.basename(files[-1])}
    return {"tflops": 74.4, "source": "nominal 148 SM x 128 lanes x 2 x 1.965 GHz (no measured FP32 peak)"}


def ncu_traffic():
    """DRAM bytes per launch of the main kernels from the newest committed ncu capture (profiles/*_traffic.json, written by
    tools/ncu_kernel_table.py from an `ncu --set full` run of this same workload)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files:
        return {}
    d = json.load(open(files[-1]))
    d["_file"] = "profiles/" + os.path.basename(files[-1])
    return d


def sample_inputs(size, sigma):
    """One 3x3 angular window of size x size SAIs of the synthetic light field, with the reference's host noise."""
    import oracleapi as O
    clean = clean_lf(3, 3, size, size, CFG["C"])
    return clean, O.add_noise(clean, sigma, SEED0)


def cpu_sample(size=512, threads=None, mode="all"):
    """The reference's own CPU code (oracle/_ref = the unmodified sources; the oracle port if it is not built) on ONE window pass per
    step (3x3 SAIs of size^2), on the host cores; extrapolated to the light field by pixels x passes (every `pst == cst` pass costs
    the same, SURVEY 8(d)). mode "all": nb_threads = host cores rounded down to a power of two (main.cpp:96-105: the reference's
    tiled multi-thread path, a different (lossy) algorithm, SURVEY A9); mode "one": nb_threads = 1, the semantics the GPU path has."""
    import oracleapi as O
    cores = threads or os.cpu_count() or 1
    clean, noisy = sample_inputs(size, CFG["sigma"])
    mask = np.ones(9, np.uint32)
    use_ref = False
    try:
        import refapi as R
        use_ref = R.available()
    except Exception:
        use_ref = False
    s1, s2 = CFG["s1"], CFG["s2"]
    t0 = time.perf_counter()
    if use_ref:
        nb = 1
        if mode == "all":
            while nb * 2 <= cores:
                nb *= 2
        os.environ["LFBM5D_REF_OMP_THREADS"] = str(cores if mode == "all" else 1)
        b, n = R.run_step1(noisy, mask, CFG["sigma"], CFG["lam"], 3, 3, 1, s1["N"], s1["nSim"], s1["nDisp"], s1["k"], s1["p"], R.ID, R.SADCT, R.HAAR, nb_threads=nb)
        d, _, _ = R.run_step2(n, b, mask, CFG["sigma"], 3, 3, 1, s2["N"], s2["nSim"], s2["nDisp"], s2["k"], s2["p"], R.DCT, R.SADCT, R.HAAR, nb_threads=nb)
        kind, used = "reference", nb
    else:
        O.lib().orc_set_threads(cores)
        b, n, _ = O.run_step1(noisy, mask, CFG["sigma"], CFG["lam"], 3, 3, 1, s1["N"], s1["nSim"], s1["nDisp"], s1["k"], s1["p"], O.ID, O.SADCT, O.HAAR)
        d, _, _, _ = O.run_step2(n, b, mask, CFG["sigma"], 3, 3, 1, s2["N"], s2["nSim"], s2["nDisp"], s2["k"], s2["p"], O.DCT, O.SADCT, O.HAAR)
        kind, used = "port", cores
    dt = time.perf_counter() - t0
    # one window pass over 9 SAIs of size^2; the full LF needs 64 passes over 9 SAIs of 1024^2 per step
    scale = N_PASSES * (CFG["H"] * CFG["W"]) / float(size * size)
    lf_pix = CFG["aw"] * CFG["ah"] * CFG["H"] * CFG["W"]
    return {"value": lf_pix / (dt * scale) / 1e6, "unit": "LF Mpix/s", "cores": used, "kind": kind, "seconds": dt, "extrapolated_s_per_lf": dt * scale,
            "psnr_sample": {"noisy": float(O.psnr(noisy, clean)[0]), "denoised": float(O.psnr(d, clean)[0])},
            "sample": "one window pass per step (3x3 SAIs of %dx%d, both steps), nb_threads = %d%s, extrapolated x%g to 64 passes of 1024^2 SAIs; "
                      "DCTs via the O(N^2) FFTW stand-in (oracle/shim)" % (size, size, used, " (the reference's tiled multi-thread algorithm)" if used > 1 else "", scale)}


def parity_block(L, eng):
    """GPU against the CPU oracle (bit-pinned to the unmodified reference, tests/test_oracle_vs_ref.py) on a config-1-shaped
    synthetic light field (3x3 SAIs of 256^2, sigma 25, README.md:50 parameters) with the reference's host noise: complete run
    through the host-buffer C ABI (max |diff|, p99.99, fraction > 1e-3, dPSNR) and the match tables of one teacher-forced pass."""
    import oracleapi as O
    size, sigma = 256, 25.0
    clean, noisy = sample_inputs(size, sigma)
    mask = np.ones(9, np.uint32)
    q1, q2 = params(L, "s1", 3, 3, size, size, sigma), params(L, "s2", 3, 3, size, size, sigma)
    s1, s2 = CFG["s1"], CFG["s2"]
    gb, gn = eng.step1(q1, noisy, mask)
    gd, _, _ = eng.step2(q2, gn, gb, mask)
    ob, on, _ = O.run_step1(noisy, mask, sigma, CFG["lam"], 3, 3, 1, s1["N"], s1["nSim"], s1["nDisp"], s1["k"], s1["p"], O.ID, O.SADCT, O.HAAR)
    od, _, _, _ = O.run_step2(on, ob, mask, sigma, 3, 3, 1, s2["N"], s2["nSim"], s2["nDisp"], s2["k"], s2["p"], O.DCT, O.SADCT, O.HAAR)
    out = {"config": "configs[0]-shaped: 3x3 SAIs 256x256 RGB, sigma 25, 8 18 6 16 4 id sadct haar / 16 18 6 8 4 dct sadct haar, opp; noise mt19937ar seed 20171016 + st",
           "oracle": "oracle/lfbm5d_oracle.c (bit-identical to the unmodified reference on complete runs, tests/test_oracle_vs_ref.py, tests/test_golden.py)"}
    for name, g, o in (("basic", gb, ob), ("denoised", gd, od)):
        diff = np.abs(g - o).ravel()
        out[name] = {"max_abs": float(diff.max()), "p9999": float(np.quantile(diff, 0.9999)), "frac_gt_1e-3": float((diff > 1e-3).mean()),
                     "dpsnr": float(O.psnr(g, clean)[0] - O.psnr(o, clean)[0])}
    # match tables of one teacher-forced step-1 pass (self-match lists, disparity argmin, shape flags)
    y = noisy.copy()
    for st in range(9):
        O.lib().orc_color_space_transform(O.fp(y[st]), O.OPP, size, size, 3, 1)
    sym = np.stack([O.symetrize(y[st], 24) for st in range(9)])
    z = np.zeros_like(sym)
    proc = np.zeros(9, np.uint32)
    _, _, odbg = O.run_pass(1, sym, None, z, z, mask, proc, 4, 3, sigma, CFG["lam"], 18, 6, 16, 8, 4, O.ID, O.SADCT, O.HAAR, debug=True)
    _, _, gdbg = eng.debug_pass(1, q1, sym, None, z, z, mask, proc, 4, debug=True)
    refs = odbg[0] > 0
    mm = np.arange(9)[None, :] < odbg[0][:, None]
    lists_equal = np.all((odbg[1] * mm) == (gdbg[1] * mm), axis=1) & (odbg[0] == gdbg[0])
    out["match_list_equal_rate"] = float(lists_equal[refs].mean())
    grid = odbg[2] != 0xFFFFFFFF
    out["disparity_argmin_equal_rate"] = float((odbg[2] == gdbg[2])[grid].mean())
    out["shape_flag_equal_rate"] = float((odbg[3] == gdbg[3])[grid].mean())
    return out


def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path on the host cores, all the threads it can use, on a
    bounded sample of this arm's workload per step (one 3x3 window pass per LFBM5D step on SAIs of S^2; S = the largest of 1024 /
    512 / 256 for which `steps` samples fit LFBM5D_REF_BUDGET_S, default 240 s)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    budget = float(os.environ.get("LFBM5D_REF_BUDGET_S", "240"))
    probe = cpu_sample(size=256)
    size = 256
    for s in (1024, 512):
        if args.steps * probe["seconds"] * (s / 256.0) ** 2 <= budget:
            size = s
            break
    for _ in range(max(0, args.warmup - 1)):
        cpu_sample(size=128)
    t0 = time.perf_counter()
    vals = [cpu_sample(size=size) for _ in range(args.steps)]
    dt = time.perf_counter() - t0
    v = float(np.mean([x["value"] for x in vals]))
    cpu = dict(vals[-1])
    cpu["value"] = v
    # nb_threads = 1 is the algorithm the GPU path implements (the multi-thread path tiles the SAIs and drops halo contributions,
    # SURVEY A9): its rate and its PSNR beside the tiled run's on the SAME small sample (128^2 SAIs keep a single thread within the
    # time budget; the 24-pixel padding weighs more on them than on 1024^2 SAIs, so both rates of this pair are pessimistic)
    one = None
    if os.environ.get("LFBM5D_REF_ONE_THREAD", "1") != "0":
        s_one, s_all = cpu_sample(size=128, mode="one"), cpu_sample(size=128, mode="all")
        one = {"nb_threads_1": {k: s_one[k] for k in ("value", "unit", "cores", "seconds", "psnr_sample", "sample")},
               "all_cores_same_sample": {k: s_all[k] for k in ("value", "unit", "cores", "seconds", "psnr_sample")},
               "tiling_costs_db": s_one["psnr_sample"]["denoised"] - s_all["psnr_sample"]["denoised"]}
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "LF Mpix/s",
                      "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
                      "ms_per_step_is": "wall time of one bounded sample (cpu_baseline.sample); value = light-field pixels / (sample time x cpu_baseline extrapolation factor)",
                      "extrapolated_ms_per_light_field": 1e3 * float(np.mean([x["extrapolated_s_per_lf"] for x in vals])),
                      "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": config_dict(world), "cpu_baseline": cpu, "exact_algorithm_sample": one,
                      "e2e": {"value": v, "unit": "LF Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--passes", type=int, default=0, help="debug: stop each step after this many window passes (value is scaled)")
    ap.add_argument("--profile-passes", type=int, default=4)
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("LFBM5D_LANES", "3")),
                    help="N > 1: independent windows of a plan level run concurrently, one per lane (own pass buffers, ~22 GB each)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed, seeded sample (%d elements each) of the outputs of the last timed step as DIR/<name>.npy, float32; "
                         "--impl ours only (the reference arm times a smaller CPU sample, not this workload)" % DUMP_SAMPLES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        # the reference arm times a bounded, extrapolated CPU sample of another size, not the 17x17x1024^2 light field
        ap.error("--dump-outputs writes the outputs of the 17x17x1024^2 workload, which only --impl ours computes")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
