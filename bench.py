#!/usr/bin/env python
"""bench.py -- headline benchmark of coslam_b200 (contract: see DESIGN.md "Measurement").

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle) timed
                                                           # on the host cores, rank 0 only
  --dump-outputs DIR: the c3 feature tables of the last timed step as DIR/klt_*.npy, so that two
  builds run with the same arguments can be compared output for output.

Primary line  : KLT features/s on BASELINE config c3 (4 cameras 1280x720, 2000 feature slots per
                camera, CoSLAM's live tracker settings: 3x3 gain tracker, levels 5/3/1 x 12
                iterations, re-detection every frame).  One step = GPUKLT::next for all 4 cameras.
                N GPUs = N independent replicas (the path does not shard, SURVEY.md 8e) -> "weak".
Nested "ba"   : BA LM-iterations/s on BASELINE config c4 (4 cams x 200 key frames x 50 k points),
                points sharded over the N GPUs, one NCCL all-reduce of the reduced camera system
                per LM trial -> "strong".
One JSON line on stdout (rank 0)."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KLT_W, KLT_H, KLT_C, KLT_FW, KLT_FH, KLT_L = 1280, 720, 4, 50, 40, 6
KLT_FRAMES = 8
BA_CAMS, BA_KF, BA_PTS = 4, 200, 50000
FP64_NOMINAL_TFLOPS = 40.0  # fallback only: the measured figure is in profiles/r2_peaks.json


def pipe_peaks():
    """fp64 / fp32 peaks of this pool's B200s measured with tools/peaks.cu (register-only FMA and
    DMMA chains on all SMs); MEASURED_PEAKS.json only holds HBM and bf16 tensor figures."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_peaks.json")))
        return {"fp64": float(d["fp64_fma_tflops"]), "fp64_dmma": float(d["fp64_dmma_tflops"]),
                "fp32": float(d["fp32_fma_tflops"]), "source": "measured (tools/peaks.cu, profiles/r2_peaks.json)"}
    except Exception:
        return {"fp64": FP64_NOMINAL_TFLOPS, "fp64_dmma": FP64_NOMINAL_TFLOPS, "fp32": 74.4, "source": "nominal"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML from a polling thread
    (about 1 kHz), nvidia-smi one-shot queries if NVML is not importable."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.sm, self.mx, self.reasons = gpu_index, [], [], set()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if gpu_index < len(ids) and ids[gpu_index].isdigit():
                    phys = int(ids[gpu_index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def start(self):
        self.stop_flag = False
        self.t = threading.Thread(target=self._poll_nvml if self.nvml else self._poll_smi, daemon=True)
        self.t.start()

    def _poll_nvml(self):
        n = self.nvml
        bits = {"hw_slowdown": getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        try:
            self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)))
        except Exception:
            pass
        while not self.stop_flag:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for nm, b in bits.items():
                    if r & b:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.001)

    def _poll_smi(self):
        cmd = ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
               str(self.gpu)]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    r = line.strip().split(", ")
                    self.sm.append(float(r[1]))
                    self.mx.append(float(r[2]))
                    for k, nm in enumerate(names):
                        if r[5 + k].strip().lower().startswith("active"):
                            self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.05)

    def stop(self):
        self.stop_flag = True
        self.t.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": float(max(self.mx)) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self.nvml else "nvidia-smi"}


# dominant kernel of every timed class, and its DRAM bytes per launch from the committed ncu capture
KERNEL_OF_CLASS = {"klt_track": "klt_gain_fused", "klt_pyramid": "klt_front",
                   "ba_solve": "ba_tile_solve", "ba_schur": "ba_schur_pairs"}


def ncu_traffic(kernel):
    try:
        t = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles",
                                        "traffic.json")))
        return float(t[kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def make_sequences(rank):
    from coslam_b200 import synth
    return [synth.ImageSequence(KLT_H, KLT_W, synth.BASE_SEED + 2 + 17 * rank + c,
                                n_frames=KLT_FRAMES) for c in range(KLT_C)]


def klt_cfg():
    from coslam_b200.ctypes_defs import KltConfig
    return KltConfig.coslam_live(with_gain=True)


def dump_outputs(out_dir, feats, counts):
    """--dump-outputs: the c3 feature tables (cameras x slots) and per-camera counts of the last
    timed step, field by field as DIR/klt_<field>.npy.  Integer fields are stored as float32, which
    holds them exactly."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {f"klt_{name}": feats[name] for name in feats.dtype.names}
    arrays["klt_counts"] = counts
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float32))


# =================================================================== reference arm (CPU oracle)
def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return
    from coslam_b200 import synth
    from coslam_b200.ctypes_defs import BaOptions
    from oracle import orc
    cores = orc.max_threads()
    orc.set_threads(cores)
    cfg = klt_cfg()
    seqs = make_sequences(0)
    trk = [orc.OracleKlt(cfg, KLT_W, KLT_H, KLT_L, KLT_FW, KLT_FH) for _ in range(KLT_C)]
    for c in range(KLT_C):
        trk[c].first(seqs[c].frame(0))
    steps = max(1, args.steps)  # one step = one 4-camera frame (~50 ms of CPU): no cap
    warm = max(1, args.warmup)
    i = 1
    for _ in range(warm):
        for c in range(KLT_C):
            trk[c].next(seqs[c].frame(i))
        i += 1
    t0 = time.perf_counter()
    for _ in range(steps):
        last = [trk[c].next(seqs[c].frame(i)) for c in range(KLT_C)]
        i += 1
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.stack([f for f, _ in last]), np.array([n for _, n in last]))
    val = KLT_C * KLT_FW * KLT_FH * steps / dt
    # BA c4 on the host cores: a bounded number of LM trials
    prob, _ = synth.make_ba_scene(BA_CAMS, BA_KF, BA_PTS, KLT_W, KLT_H, seed=synth.BASE_SEED + 4,
                                  m_con=BA_CAMS, n_con=0)
    opt = BaOptions.defaults()
    ntr = 3
    p = prob.copy()
    tb = time.perf_counter()
    info = orc.ba_run_fixed(p, opt, ntr)
    ba_dt = time.perf_counter() - tb
    ba_val = info[9] / info[11] if info[11] > 0 else 0.0
    sample = f"{steps} frames x {KLT_C} cameras of the c3 sequence"
    line = {
        "impl": "reference", "metric": "klt_features_per_s", "value": val, "unit": "features/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "c3: 4 cams 1280x720, 2000 feature slots/cam, KLT next() "
                               "(pyramid + 3x3 gain LK levels 5/3/1 x 12 it + re-detect)"},
        "cpu_baseline": {"value": val, "unit": "features/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": val, "unit": "features/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "ba": {"metric": "ba_lm_iters_per_s", "value": ba_val, "unit": "LM-iter/s",
               "config": {"workload": f"c4: {prob.m} poses, {prob.n} points, {prob.nobs} obs"},
               "cpu_baseline": {"value": ba_val, "unit": "LM-iter/s", "cores": cores,
                                "kind": "port", "sample": f"{int(info[9])} LM trials, "
                                f"{ba_dt:.1f} s incl. setup"},
               "e2e": {"value": info[9] / ba_dt, "unit": "LM-iter/s", "h2d_bytes_per_step": 0,
                       "d2h_bytes_per_step": 0}},
    }
    emit(line)


# =================================================================== CUDA arm
def run_cuda(args):
    import torch
    rank, world, local = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from coslam_b200 import api, synth
    from coslam_b200.ctypes_defs import BaOptions

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    hbm_peak, peak_src = peaks()
    cfg = klt_cfg()
    F = KLT_FW * KLT_FH
    # ------------------------------------------------------------------ KLT (c3), one replica/rank
    seqs = make_sequences(rank)
    grp = api.KltGroup(cfg, KLT_C, KLT_W, KLT_H, KLT_L, KLT_FW, KLT_FH, device=local)
    stream = torch.cuda.ExternalStream(grp.stream(), device=local)
    host = [[torch.from_numpy(seqs[c].frames[k]).pin_memory() for c in range(KLT_C)]
            for k in range(KLT_FRAMES)]
    dev = [[h.cuda() for h in row] for row in host]
    torch.cuda.synchronize()

    def fidx(i):
        return seqs[0].frame_index(i)

    feats, n0 = grp.first([host[0][c].numpy() for c in range(KLT_C)])
    n_detected = [int(v) for v in n0]
    K, Wm = args.steps, max(3, args.warmup)
    i = 1
    for _ in range(Wm):
        grp.next_dev([t.data_ptr() for t in dev[fidx(i)]], KLT_W)
        i += 1
    grp.sync()
    # ---- value: frames resident in HBM, no host transfer, device-timed on the launching stream
    clocks = ClockSampler(local)
    clocks.start()
    barrier()
    launches0 = api.kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(K):
        grp.next_dev([t.data_ptr() for t in dev[fidx(i)]], KLT_W)
        i += 1
    e1.record(stream)
    grp.sync()
    barrier()
    gpu_launches = api.kernel_launch_count() - launches0
    ms_val = max_over_ranks(e0.elapsed_time(e1))
    feats, cnt = grp.fetch()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, feats, cnt)
    tracked_frac = float(np.mean([(feats[c]["status"] == 0).mean() for c in range(KLT_C)]))
    # ---- roofline: second pass of the same region with per-kernel-class CUDA events
    grp.profile_enable(True)
    for _ in range(K):
        grp.next_dev([t.data_ptr() for t in dev[fidx(i)]], KLT_W)
        i += 1
    grp.sync()
    prof = grp.profile()
    grp.profile_enable(False)
    px = KLT_C * KLT_W * KLT_H
    alg = {"klt_pyramid": 17.0 * px, "klt_track": 4640.0 * KLT_C * F,
           "klt_detect": 8.0 * px + 48.0 * KLT_C * F, "klt_select": 48.0 * KLT_C * F}
    top = max(prof, key=lambda k: prof[k][0])
    top_ms = prof[top][0] / max(1, prof[top][1])
    achieved = alg[top] / (top_ms * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
            "frac": achieved / hbm_peak, "traffic": ncu_traffic(KERNEL_OF_CLASS.get(top)),
            "peak_source": peak_src,
            "algorithmic_bytes_per_step": alg[top], "avg_ms_per_step": top_ms,
            "share_of_step": {k: v[0] / max(1e-9, sum(x[0] for x in prof.values()))
                              for k, v in prof.items()},
            "frame_total": {"algorithmic_bytes": grp.algorithmic_bytes(),
                            "achieved": grp.algorithmic_bytes() / (ms_val / K * 1e-3) / 1e9,
                            "frac": grp.algorithmic_bytes() / (ms_val / K * 1e-3) / 1e9 / hbm_peak}}
    # SURVEY 8(d) lists the LK solve as FP32-SIMT co-bound: 123 kflop per feature (70 w^2 flops per
    # window evaluation, 36 evaluations); denominator = the fp32 FMA peak measured by tools/peaks.cu.
    if top == "klt_track":
        lk_flops = 123.0e3 * KLT_C * F
        pp = pipe_peaks()
        roof["fp32_co_bound"] = {"algorithmic_flops_per_step": lk_flops,
                                 "achieved_tflops": lk_flops / (top_ms * 1e-3) / 1e12,
                                 "peak_tflops": pp["fp32"], "peak_source": pp["source"],
                                 "frac": lk_flops / (top_ms * 1e-3) / 1e12 / pp["fp32"]}
    # ---- e2e: host buffers through the public C-ABI call, H2D + D2H inside the timed region
    host_np = [[h.numpy() for h in row] for row in host]
    host_args = [grp.host_ptrs(row) for row in host_np]  # pointer arrays built once per frame
    for _ in range(3):
        grp.next_raw(host_args[fidx(i)])
        i += 1
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall = time.perf_counter()
    e2.record(stream)
    for _ in range(K):
        grp.next_raw(host_args[fidx(i)])
        i += 1
    e3.record(stream)
    grp.sync()
    wall = time.perf_counter() - t_wall
    ms_e2e = max_over_ranks(max(e2.elapsed_time(e3), wall * 1e3))
    # the real caller's frames (SingleSLAM::m_img) are pageable: same call from ordinary numpy arrays
    e2e_pageable = None
    if rank == 0:
        pag = [[np.array(h.numpy(), copy=True) for h in row] for row in host]
        pag_args = [grp.host_ptrs(row) for row in pag]
        for _ in range(3):
            grp.next_raw(pag_args[fidx(i)])
            i += 1
        tpg = time.perf_counter()
        for _ in range(K):
            grp.next_raw(pag_args[fidx(i)])
            i += 1
        grp.sync()
        mspg = 1e3 * (time.perf_counter() - tpg)
        e2e_pageable = {"value": KLT_C * F * K / (mspg * 1e-3), "unit": "features/s", "ms_per_step": mspg / K,
                        "note": "pageable host frames (plain numpy), rank 0 only"}
    # frame-pipelined ingest (cosl_klt_group_submit / _collect): frame n+1 is submitted before frame n
    # is collected, so its upload runs under frame n's kernels; every frame's result is still read back
    e2e_pipelined = None
    if rank == 0:
        grp.submit_raw(host_args[fidx(i)])
        i += 1
        for _ in range(3):
            grp.submit_raw(host_args[fidx(i)])
            grp.collect()
            i += 1
        tpl = time.perf_counter()
        for _ in range(K):
            grp.submit_raw(host_args[fidx(i)])
            grp.collect()
            i += 1
        mspl = 1e3 * (time.perf_counter() - tpl)
        grp.collect()
        e2e_pipelined = {"value": KLT_C * F * K / (mspl * 1e-3), "unit": "features/s", "ms_per_step": mspl / K,
                         "note": "pinned host frames, cosl_klt_group_submit(n+1) before _collect(n): one frame of "
                                 "latency, same bytes per step; rank 0 only"}
    clk = clocks.stop()  # sampled across the device-resident, profiled and end-to-end regions
    barrier()
    klt_value = world * KLT_C * F * K / (ms_val * 1e-3)
    # ---- the same frame with the plain 2x2 tracker (north_star's kernel; CoSLAM's live default is
    # the 3x3 gain tracker measured above): device-resident frames, value only
    klt2 = None
    if rank == 0:
        from coslam_b200.ctypes_defs import KltConfig
        g2 = api.KltGroup(KltConfig.coslam_live(with_gain=False), KLT_C, KLT_W, KLT_H, KLT_L, KLT_FW,
                          KLT_FH, device=local)
        s2 = torch.cuda.ExternalStream(g2.stream(), device=local)
        g2.first([host[0][c].numpy() for c in range(KLT_C)])
        j = 1
        for _ in range(Wm):
            g2.next_dev([t.data_ptr() for t in dev[fidx(j)]], KLT_W)
            j += 1
        g2.sync()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(s2)
        for _ in range(K):
            g2.next_dev([t.data_ptr() for t in dev[fidx(j)]], KLT_W)
            j += 1
        a1.record(s2)
        g2.sync()
        ms2 = a0.elapsed_time(a1)
        f2, _ = g2.fetch()
        klt2 = {"metric": "klt_features_per_s", "value": KLT_C * F * K / (ms2 * 1e-3),
                "unit": "features/s", "ms_per_step": ms2 / K,
                "tracked_fraction": float(np.mean([(f2[c]["status"] == 0).mean() for c in range(KLT_C)])),
                "config": {"workload": "c3 with trackWithGain = false (2x2 LK, levels 5/3/1 x 5 iterations: the "
                                       "reference build always runs 5, v3d_gpuklt.cpp quirk kept), frames resident in HBM"}}
        g2.close()
    klt_e2e = world * KLT_C * F * K / (ms_e2e * 1e-3)

    # ------------------------------------------------------------------ pose (latency, rank 0)
    # The GPU legs of pose and BA run before anything imports the CPU oracle: its OpenMP / OpenBLAS
    # worker threads compete with the host-side work of the calls for the container's CPU quota.
    pose = None
    if rank == 0:
        cases = [synth.make_pose_case(192, KLT_W, KLT_H, seed=100 + c) for c in range(KLT_C)]
        pa = ([c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases],
              [c[3] for c in cases], [c[4] for c in cases], 10.0)
        for _ in range(3):
            api.pose_intracam_batch(*pa, device=local)
        nrep = 40
        t0 = time.perf_counter()
        for _ in range(nrep):
            api.pose_intracam_batch(*pa, device=local)
        us = (time.perf_counter() - t0) / nrep * 1e6
        pose = {"metric": "pose_batch_latency", "value": us, "unit": "us per call", "higher_is_better": False,
                "config": {"workload": "intraCamEstimate for 4 cameras x 192 points in one launch, "
                                       "host arrays in/out (cosl_pose_intracam_batch)"}}

    # ------------------------------------------------------------------ BA (c4), sharded
    ba = run_ba(args, api, synth, BaOptions, torch, dist, rank, world, local, barrier,
                max_over_ranks)

    if pose is not None:
        if world == 1 and not args.no_cpu:
            from oracle import orc as _orc
            t0 = time.perf_counter()
            for _ in range(10):
                for c in cases:
                    _orc.pose_intracam(c[0], c[1], c[2], c[3], c[4], 10.0)
            pose["cpu_baseline"] = {"value": (time.perf_counter() - t0) / 10 * 1e6, "unit": "us per 4 cameras",
                                    "cores": 1, "kind": "port", "sample": "10 repetitions"}


    # ------------------------------------------------------------------ the other BASELINE configs
    extra = {}
    if rank == 0 and world == 1 and not args.quick:
        # c3: local BA per key frame (20 poses / 20 k points) and the 30 fps pipeline target
        lb3, prob3 = run_local_ba(api, synth, BaOptions, torch, local, "c3", 4, 20000, KLT_W, KLT_H, args.no_cpu)
        extra["c3_local_ba"] = lb3
        extra["pipeline"] = run_pipeline(api, synth, BaOptions, torch, local, grp, seqs, host_args, prob3)
        # c2: 2 cameras 640x480, 1 k features/camera, 5 k-point local BA
        k2, g2c, _, _ = run_klt_leg(api, synth, torch, local, "c2", 2, 640, 480, 40, 25, min(K, 50), synth.BASE_SEED + 200)
        g2c.close()
        lb2, _ = run_local_ba(api, synth, BaOptions, torch, local, "c2", 2, 5000, 640, 480, args.no_cpu)
        extra["c2"] = {"klt": k2, "local_ba": lb2}
        extra["posegraph"] = run_posegraph(api, synth, local, args.no_cpu)
    if not args.quick:
        # c5: 8 cameras 1920x1080, 4 k features/camera; camera c -> GPU c mod N (replicas only)
        ncam5 = max(1, 8 // world)
        k5, g5, _, _ = run_klt_leg(api, synth, torch, local, "c5", ncam5, 1920, 1080, 80, 50, min(K, 30),
                                   synth.BASE_SEED + 300 + 16 * rank, frames=3)
        g5.close()
        ms5 = max_over_ranks(k5["e2e"]["ms_per_step"])
        if rank == 0:
            k5["config"]["workload"] += f"; 8 cameras over {world} GPU(s), {ncam5} per GPU"
            k5["fps_8cam_e2e"] = 1e3 / ms5
            k5["meets_30fps"] = bool(1e3 / ms5 >= 30.0)
            extra["c5"] = k5
    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1)
    cpu = None
    klt_parity = None
    if rank == 0 and not args.no_cpu:
        # oracle parity of the LK solve + slot logic on the benchmark's own sequence (camera 0,
        # first + 2 x next): max |dpos| in pixels and status flips
        from oracle import orc as _o
        _o.set_threads(_o.max_threads())
        gk = api.KltTracker(cfg, KLT_W, KLT_H, KLT_L, KLT_FW, KLT_FH, device=local)
        ok = _o.OracleKlt(cfg, KLT_W, KLT_H, KLT_L, KLT_FW, KLT_FH)
        fg, _ = gk.first(seqs[0].frames[0])
        fo, _ = ok.first(seqs[0].frames[0])
        worst, flips = 0.0, 0
        for kk in (1, 2):
            fg, _ = gk.next(seqs[0].frames[kk])
            fo, _ = ok.next(seqs[0].frames[kk])
            same = fg["status"] == fo["status"]
            flips += int((~same).sum())
            live = same & (fo["status"] >= 0)
            if live.any():
                worst = max(worst, float((np.abs(fg["pos"][live] - fo["pos"][live]) * [KLT_W, KLT_H]).max()))
        klt_parity = {"parity_max_dpos_px": worst, "status_flips": flips, "slots": KLT_FW * KLT_FH,
                      "sample": "camera 0 of the bench sequence, first() + 2 x next() vs the CPU oracle"}
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline_klt(cfg, seqs)
    if rank == 0:
        line = {
            "metric": "klt_features_per_s", "value": klt_value, "unit": "features/s",
            "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms_val / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "c3: 4 cams 1280x720, 2000 feature slots/cam, KLT next() "
                                   "(pyramid + 3x3 gain LK levels 5/3/1 x 12 it + re-detect)",
                       "replicas": world, "frames": f"{KLT_FRAMES}-frame ping-pong sequence/cam",
                       "l2": "working set (2 pyramids + cornerness + images, ~190 MB/replica) "
                             "exceeds the 126 MB L2; no explicit flush",
                       "detected_at_frame0": n_detected, "tracked_fraction": tracked_frac},
            "e2e": {"value": klt_e2e, "unit": "features/s",
                    "h2d_bytes_per_step": KLT_C * KLT_W * KLT_H,
                    "d2h_bytes_per_step": KLT_C * F * 20 + KLT_C * 32,
                    "ms_per_step": ms_e2e / K},
            "gpu_launches": int(gpu_launches),
            "clocks": clk, "roofline": roof,
            "fps_4cam": K / (ms_e2e * 1e-3),
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if klt2 is not None:
            line["klt_2x2"] = klt2
        if ba is not None:
            line["ba"] = ba
        if pose is not None:
            line["pose"] = pose
        if klt_parity is not None:
            line["klt_parity"] = klt_parity
        if e2e_pageable is not None:
            line["e2e"]["pageable"] = e2e_pageable
        if e2e_pipelined is not None:
            line["e2e"]["pipelined"] = e2e_pipelined
        line.update(extra)
        line["peaks"] = {"hbm_gbs": hbm_peak, "hbm_source": peak_src, **pipe_peaks()}
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline_klt(cfg, seqs):
    from oracle import orc
    cores = orc.max_threads()
    orc.set_threads(cores)
    trk = [orc.OracleKlt(cfg, KLT_W, KLT_H, KLT_L, KLT_FW, KLT_FH) for _ in range(KLT_C)]
    for c in range(KLT_C):
        trk[c].first(seqs[c].frame(0))
    nfr = 16  # ~1 s of wall time on 16 threads (~15 core-seconds)
    t0 = time.perf_counter()
    for k in range(1, 1 + nfr):
        for c in range(KLT_C):
            trk[c].next(seqs[c].frame(k))
    dt = time.perf_counter() - t0
    return {"value": KLT_C * KLT_FW * KLT_FH * nfr / dt, "unit": "features/s", "cores": cores,
            "kind": "port", "sample": f"{nfr} frames x {KLT_C} cameras of the same c3 sequence",
            "ms_per_step": 1e3 * dt / nfr}


def ba_roofline(tm, trials, prob, st, world, solver):
    """Roofline of the dominant kernel class of an LM trial (per-class CUDA events)."""
    tot = sum(v[0] for v in tm.values())
    top = max(tm, key=lambda k: tm[k][0])
    top_ms = tm[top][0] / max(1, trials)
    ns = 6 * (prob.m - prob.m_con)
    pp = pipe_peaks()
    if top == "ba_solve":
        # multiply-adds the tile Cholesky + substitutions really perform (ba_plan.h counts them on
        # the used rows: nested dissection adds fill but cuts the dependency chain); the kernel is
        # bound by that chain, not by the fp64 pipe -- the fraction says how far
        flops = 2.0 * st["factor_flops"]
        roof = {"bound": "tensor", "kernel": "ba_tile_solve (persistent dataflow tile Cholesky, fp64 DMMA)",
                "achieved": flops / (top_ms * 1e-3) / 1e12, "peak": pp["fp64_dmma"], "unit": "TFLOP/s",
                "frac": flops / (top_ms * 1e-3) / 1e12 / pp["fp64_dmma"],
                "traffic": ncu_traffic("ba_tile_solve"), "peak_source": pp["source"],
                "algorithmic_flops_per_trial": flops, "dense_flops_per_trial": 2.0 * ns ** 3 / 3.0,
                "plan": solver.plan_info()}
    else:
        hbm_peak, src = peaks()
        byts = {"ba_schur": 8.0 * st["reduce_doubles"] + 144.0 * prob.nobs + 48.0 * prob.n,
                "ba_linearize": 24.0 * prob.nobs + 24.0 * prob.n + 144.0 * prob.nobs,
                "ba_backsub": 8.0 * prob.nobs + 48.0 * prob.n, "ba_cost": 24.0 * prob.nobs,
                "ba_allreduce": 8.0 * st["reduce_doubles"] * world}.get(top, 0.0) / world
        roof = {"bound": "hbm", "kernel": top, "achieved": byts / (top_ms * 1e-3) / 1e9,
                "peak": hbm_peak, "unit": "GB/s", "frac": byts / (top_ms * 1e-3) / 1e9 / hbm_peak,
                "traffic": ncu_traffic(KERNEL_OF_CLASS.get(top)), "peak_source": src,
                "algorithmic_bytes_per_trial": byts}
    roof["share_of_trial"] = {k: v[0] / max(tot, 1e-9) for k, v in tm.items()}
    roof["ms_per_trial_by_class"] = {k: v[0] / max(1, trials) for k, v in tm.items()}
    roof["avg_ms_per_trial"] = top_ms
    return roof


def run_ba(args, api, synth, BaOptions, torch, dist, rank, world, local, barrier, max_over_ranks):
    prob, truth = synth.make_ba_scene(BA_CAMS, BA_KF, BA_PTS, KLT_W, KLT_H,
                                      seed=synth.BASE_SEED + 4, m_con=BA_CAMS, n_con=0,
                                      sort_by_home=os.environ.get("COSL_BENCH_BA_SORTED", "0") == "1")
    opt = BaOptions.defaults()
    opt.device = local
    comm = None
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.from_numpy(api.nccl_unique_id()))
        dist.broadcast(uid, 0)
        comm = api.BaComm(uid.cpu().numpy(), rank, world, local)
        shard, (lo, hi) = prob.shard(rank, world)
    else:
        shard = prob
    t_setup = time.perf_counter()
    solver = api.BaSolver(shard, opt, comm)
    setup_s = time.perf_counter() - t_setup
    stream = torch.cuda.ExternalStream(solver.stream(), device=local)
    K = max(4, min(args.steps, 20))
    Wm = 3
    solver.run_fixed(Wm)
    solver.reset()
    barrier()
    launches0 = api.kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t0 = time.perf_counter()
    info = solver.run_fixed(K)
    e1.record(stream)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = max_over_ranks(max(e0.elapsed_time(e1), wall * 1e3))
    launches = api.kernel_launch_count() - launches0
    trials = int(info[9])
    # per-kernel-class shares and the roofline of the dominant one
    solver.reset()
    solver.profile_enable(True)
    solver.run_fixed(K)
    tm = solver.timers()
    solver.profile_enable(False)
    kk = np.diff(prob.ptr).astype(np.float64)
    st = solver.stats()
    roof = ba_roofline(tm, trials, prob, st, world, solver)
    ns = 6 * (prob.m - prob.m_con)
    # parity at full size at EVERY N: the same 3 LM trials -> the same cost as the CPU oracle
    solver.reset()
    ig = solver.run_fixed(3)
    # e2e: the drop-in call with host buffers (upload + index build + solve + download)
    e2e = None
    if world == 1:
        o2 = BaOptions.defaults()
        o2.device = local
        o2.max_err, o2.outer_iters, o2.inner_iters = 6.0, 1, 10
        api.ba_solve(prob.copy(), o2)  # warm-up call: the device memory pool grows once
        reps, dt = 3, 0.0
        for _ in range(reps):
            p2 = prob.copy()
            t0 = time.perf_counter()
            inf2 = api.ba_solve(p2, o2)
            dt += time.perf_counter() - t0
        dt /= reps
        h2d = prob.nobs * (8 * 2 + 4 + 4) + prob.n * 24 + prob.m * 8 * 21
        e2e = {"value": inf2[9] / dt, "unit": "LM-iter/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(prob.n * 24 + prob.m * 48 + prob.nobs),
               "call": "cosl_ba_solve (1 robust round x 10 LM iterations, host arrays in/out); "
                       "mean of 3 calls after 1 warm-up call",
               "seconds": dt, "lm_trials": int(inf2[9]), "rms_after": p2.rms(~truth["is_outlier"])}
    out = {"metric": "ba_lm_iters_per_s", "value": trials / (ms * 1e-3), "unit": "LM-iter/s",
           "scaling": "strong", "ms_per_trial": ms / max(1, trials), "lm_trials": trials,
           "gpu_launches": int(launches), "setup_s": setup_s,
           "config": {"workload": f"c4: {prob.m} poses ({prob.m_con} fixed), {prob.n} points, "
                                  f"{prob.nobs} obs, reduced system {ns}x{ns} fp64",
                      "sum_k2": float((kk * kk).sum()), "shards": world},
           "roofline": roof}
    if e2e is not None:
        out["e2e"] = e2e
    if rank == 0 and not args.no_cpu:
        from oracle import orc
        cores = orc.max_threads()
        orc.set_threads(cores)
        p3 = prob.copy()
        i3 = orc.ba_run_fixed(p3, opt, 3)
        if world == 1:
            out["cpu_baseline"] = {"value": i3[9] / i3[11], "unit": "LM-iter/s", "cores": cores,
                                   "kind": "port", "sample": f"{int(i3[9])} LM trials of the same c4 "
                                   "problem (OpenMP + OpenBLAS dpotrf)"}
        out["parity_rel_cost_diff_3_trials"] = abs(ig[1] - i3[1]) / i3[1]
    solver.close()
    if comm is not None:
        comm.close()
    return out


def run_local_ba(api, synth, BaOptions, torch, local, name, n_cams, n_pts, W, H, no_cpu):
    """Local BA of BASELINE c2 / c3: 5 key frames x n_cams poses, the oldest two key frames fixed
    (nCamsCon = 2 C, app/SL_CoSLAM.cpp:1769), 2 fixed points: LM trials/s with the solver resident
    + the drop-in call, against the HBM contract of SURVEY.md 8(d) (one pass over the observations
    and points per LM iteration)."""
    prob, truth = synth.make_ba_scene(n_cams, 5, n_pts, W, H, seed=synth.BASE_SEED + (3 if n_cams == 4 else 2),
                                      m_con=2 * n_cams, n_con=2)
    opt = BaOptions.defaults()
    opt.device = local
    solver = api.BaSolver(prob, opt)
    stream = torch.cuda.ExternalStream(solver.stream(), device=local)
    solver.run_fixed(5)
    solver.reset()
    K = 40
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = api.kernel_launch_count()
    e0.record(stream)
    info = solver.run_fixed(K)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = api.kernel_launch_count() - l0
    trials = int(info[9])
    solver.reset()
    solver.profile_enable(True)
    solver.run_fixed(K)
    tm = solver.timers()
    solver.profile_enable(False)
    hbm_peak, src = peaks()
    byts = 32.0 * prob.nobs + 72.0 * prob.n  # SURVEY 8(d) "Local BA LM-iteration" contract
    out = {"metric": "ba_lm_iters_per_s", "value": trials / (ms * 1e-3), "unit": "LM-iter/s",
           "us_per_trial": 1e3 * ms / max(1, trials), "lm_trials": trials, "gpu_launches": int(launches),
           "config": {"workload": f"{name} local BA: {prob.m} poses ({prob.m_con} fixed), {prob.n} points, "
                                  f"{prob.nobs} obs, reduced system {6 * (prob.m - prob.m_con)}^2"},
           "roofline": {"bound": "hbm", "kernel": "whole LM trial", "achieved": byts / (ms / max(1, trials) * 1e-3) / 1e9,
                        "peak": hbm_peak, "unit": "GB/s", "peak_source": src,
                        "frac": byts / (ms / max(1, trials) * 1e-3) / 1e9 / hbm_peak,
                        "algorithmic_bytes_per_trial": byts,
                        "us_per_trial_by_class": {k: 1e3 * v[0] / max(1, trials) for k, v in tm.items()}}}
    # drop-in call (robust loop with the live parameters: 5 rounds x 10 iterations, host arrays)
    o2 = BaOptions.defaults()
    o2.device = local
    api.ba_solve(prob.copy(), o2)
    reps, dt = 3, 0.0
    for _ in range(reps):
        p2 = prob.copy()
        t0 = time.perf_counter()
        inf2 = api.ba_solve(p2, o2)
        dt += time.perf_counter() - t0
    dt /= reps
    out["e2e"] = {"value": inf2[10] / dt, "unit": "LM-iter/s", "ms_per_call": 1e3 * dt, "lm_trials": int(inf2[10]),
                  "h2d_bytes_per_step": int(prob.nobs * 24 + prob.n * 24 + prob.m * 168),
                  "d2h_bytes_per_step": int(prob.n * 24 + prob.m * 96 + prob.nobs),
                  "call": "bundleAdjustRobust drop-in (cosl_ba_solve, maxErr 6, 5 rounds x 10 LM iterations)",
                  "rms_after": p2.rms(~truth["is_outlier"])}
    if not no_cpu:
        from oracle import orc
        po = prob.copy()
        t0 = time.perf_counter()
        io = orc.ba_solve(po, o2)
        dto = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": io[10] / dto, "unit": "LM-iter/s", "cores": orc.max_threads(), "kind": "port",
                               "sample": "one bundleAdjustRobust call of the same problem", "ms_per_call": 1e3 * dto}
        out["parity_rel_rms_diff"] = abs(p2.rms() - po.rms()) / po.rms()
    solver.close()
    return out, prob


def run_klt_leg(api, synth, torch, local, name, C, W, H, fw, fh, K, seed0, frames=4):
    """KLT next() for C cameras of W x H with fw x fh slots: device-resident value + host-buffer e2e."""
    cfg = klt_cfg()
    seqs = [synth.ImageSequence(H, W, seed0 + c, n_frames=frames) for c in range(C)]
    grp = api.KltGroup(cfg, C, W, H, KLT_L, fw, fh, device=local)
    stream = torch.cuda.ExternalStream(grp.stream(), device=local)
    host = [[torch.from_numpy(seqs[c].frames[k]).pin_memory() for c in range(C)] for k in range(frames)]
    dev = [[h.cuda() for h in row] for row in host]
    torch.cuda.synchronize()
    grp.first([host[0][c].numpy() for c in range(C)])
    fidx = seqs[0].frame_index
    i = 1
    for _ in range(3):
        grp.next_dev([t.data_ptr() for t in dev[fidx(i)]], W)
        i += 1
    grp.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(K):
        grp.next_dev([t.data_ptr() for t in dev[fidx(i)]], W)
        i += 1
    e1.record(stream)
    grp.sync()
    ms = e0.elapsed_time(e1)
    feats, _ = grp.fetch()
    tracked = float(np.mean([(feats[c]["status"] == 0).mean() for c in range(C)]))
    host_args = [grp.host_ptrs([h.numpy() for h in row]) for row in host]
    for _ in range(3):
        grp.next_raw(host_args[fidx(i)])
        i += 1
    t0 = time.perf_counter()
    for _ in range(K):
        grp.next_raw(host_args[fidx(i)])
        i += 1
    grp.sync()
    ms_e2e = 1e3 * (time.perf_counter() - t0)
    hbm_peak, src = peaks()
    out = {"metric": "klt_features_per_s", "value": C * fw * fh * K / (ms * 1e-3), "unit": "features/s",
           "ms_per_step": ms / K, "fps": K / (ms_e2e * 1e-3), "tracked_fraction": tracked,
           "config": {"workload": f"{name}: {C} cams {W}x{H}, {fw * fh} slots/cam, KLT next()"},
           "e2e": {"value": C * fw * fh * K / (ms_e2e * 1e-3), "unit": "features/s", "ms_per_step": ms_e2e / K,
                   "h2d_bytes_per_step": C * W * H, "d2h_bytes_per_step": C * fw * fh * 20 + C * 32},
           "roofline": {"bound": "hbm", "kernel": "whole frame", "achieved": grp.algorithmic_bytes() / (ms / K * 1e-3) / 1e9,
                        "peak": hbm_peak, "unit": "GB/s", "peak_source": src,
                        "frac": grp.algorithmic_bytes() / (ms / K * 1e-3) / 1e9 / hbm_peak}}
    return out, grp, seqs, host_args


def run_posegraph(api, synth, local, no_cpu, n_cams=8, n_frames=4000, key_every=20, reps=20):
    """Post-BA pose-graph spreading (SURVEY.md 8f-2): all cameras' chains in ONE cosl_posegraph_spread_chains
    call with host arrays (H2D + kernel + D2H inside the timed region).  Parity of the same call on a
    smaller graph against the oracle (pinned to the compiled reference) is reported beside it."""
    g = synth.make_pose_chains([n_frames] * n_cams, key_every=key_every, seed=77, shift=0.05)
    args = (g["chain_off"], g["fixed"], g["R"], g["t"], g["eR"], g["et"])
    for _ in range(3):
        api.posegraph_spread_chains(*args, device=local)
    t0 = time.perf_counter()
    for _ in range(reps):
        api.posegraph_spread_chains(*args, device=local)
    ms = 1e3 * (time.perf_counter() - t0) / reps
    N = n_cams * n_frames
    out = {"metric": "posegraph_nodes_per_s", "value": N / (ms * 1e-3), "unit": "nodes/s", "ms_per_call": ms,
           "config": {"workload": f"{n_cams} camera chains x {n_frames} frames, key frame every {key_every}, "
                                  "host arrays through cosl_posegraph_spread_chains"},
           "h2d_bytes_per_call": N * (72 + 24 + 72 + 24 + 1), "d2h_bytes_per_call": N * 96}
    if not no_cpu:
        from oracle import orc as _orc
        gs = synth.make_pose_chains([200], key_every=key_every, seed=78, shift=0.05)
        t0 = time.perf_counter()
        oR, ot = _orc.posegraph_spread(gs["fixed"], gs["R"], gs["t"], gs["id1"], gs["id2"], gs["eR_list"], gs["et_list"])
        cpu_ms = 1e3 * (time.perf_counter() - t0)
        nR, nt = api.posegraph_spread_chains(gs["chain_off"], gs["fixed"], gs["R"], gs["t"], gs["eR"], gs["et"],
                                             device=local)
        out["parity_max_abs_diff_vs_oracle"] = float(max(np.abs(nR - oR).max(), np.abs(nt - ot).max()))
        out["cpu_baseline"] = {"value": 200 / (cpu_ms * 1e-3), "unit": "nodes/s", "cores": 1, "kind": "port",
                               "sample": "one 200-node chain; the port solves DENSE least squares (the reference's "
                                         "sparse solver is in the absent LibVisualSLAM), so this is not a "
                                         "like-for-like speed baseline"}
    return out


def run_pipeline(api, synth, BaOptions, torch, local, grp, seqs, host_args, ba_prob, n_frames=60, kf_every=10):
    """north_star target: >= 30 fps end to end on 4 synthetic 1280x720 streams at 2k features/cam
    WITH per-key-frame local BA on one B200.  Per frame: cosl_klt_group_next (host frames in,
    features out) + cosl_pose_intracam_batch (4 cameras x 192 points, host arrays); every
    `kf_every`-th frame a key frame: the bundleAdjustRobust drop-in on the c3 local-BA problem (20
    poses / 20 k points, host arrays), run synchronously (the reference runs it on a second thread)."""
    cases = [synth.make_pose_case(192, KLT_W, KLT_H, seed=200 + c) for c in range(len(seqs))]
    pa = ([c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases],
          [c[3] for c in cases], [c[4] for c in cases], 10.0)
    o2 = BaOptions.defaults()
    o2.device = local
    fidx = seqs[0].frame_index
    i = 1
    for _ in range(3):
        grp.next_raw(host_args[fidx(i)])
        api.pose_intracam_batch(*pa, device=local)
        i += 1
    api.ba_solve(ba_prob.copy(), o2)
    t_klt = t_pose = t_ba = 0.0
    nkf = 0
    t0 = time.perf_counter()
    for f in range(n_frames):
        a = time.perf_counter()
        grp.next_raw(host_args[fidx(i)])
        grp.sync()
        b = time.perf_counter()
        api.pose_intracam_batch(*pa, device=local)
        c = time.perf_counter()
        if f % kf_every == kf_every - 1:
            api.ba_solve(ba_prob.copy(), o2)
            nkf += 1
        d = time.perf_counter()
        t_klt += b - a
        t_pose += c - b
        t_ba += d - c
        i += 1
    dt = time.perf_counter() - t0
    # the same loop with the frame-pipelined ingest: frame f+1 is submitted as soon as frame f's features are
    # collected, so its upload and kernels run under the pose solve / local BA of frame f
    grp.submit_raw(host_args[fidx(i)])
    i += 1
    t1 = time.perf_counter()
    for f in range(n_frames):
        grp.collect()
        grp.submit_raw(host_args[fidx(i)])
        api.pose_intracam_batch(*pa, device=local)
        if f % kf_every == kf_every - 1:
            api.ba_solve(ba_prob.copy(), o2)
        i += 1
    dtp = time.perf_counter() - t1
    grp.collect()
    return {"metric": "fps_pipeline", "value": n_frames / dt, "unit": "frames/s (4 cameras each)",
            "pipelined_ingest_fps": n_frames / dtp,
            "target": 30.0, "meets_target": bool(n_frames / dt >= 30.0),
            "config": {"workload": f"c3 pipeline: KLT next (4 x 1280x720, 2000 slots) + batched pose (4 x 192 pts) every "
                                   f"frame, local BA (20 poses / 20 k points, 5 x 10 LM iterations) every {kf_every}th frame, "
                                   "all through the C-ABI with host buffers, single thread"},
            "frames": n_frames, "key_frames": nkf,
            "ms_per_frame": {"klt": 1e3 * t_klt / n_frames, "pose": 1e3 * t_pose / n_frames,
                             "local_ba_amortised": 1e3 * t_ba / n_frames,
                             "local_ba_per_key_frame": 1e3 * t_ba / max(1, nkf)}}


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, C-level prints of
    libraries) was redirected to stderr at start-up."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # fd 1 -> stderr for the rest of the process
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--quick", action="store_true", help="headline KLT c3 + BA c4 only (skip c2 / c3 local BA / "
                    "pipeline / c5 legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the c3 feature tables of the last timed step "
                    "as DIR/klt_*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
