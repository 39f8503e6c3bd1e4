#!/usr/bin/env python
"""Throughput of the stage-1 neural-atlas loop (BASELINE.json metric: atlas iters/sec, 80 frames
768x432, 10 000 points per iteration) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--precision tc|fp32]
                    [--workload atlas|raft|stage2|seg] [--dump-outputs DIR]

One "step" = one loop trip of src/stage1_neural_atlas.py:151-231 (sampling, 7 mapping + 3 atlas
evaluations, 4 losses, backward, Adam).  Prints ONE JSON line on rank 0.  Keys beyond the driver's
contract:
  roofline      every tagged launch site of the step is timed live with CUDA events (a second captured
                graph that carries the event records, so the headline region is not perturbed); the site
                with the largest time is reported as `kernel`, its algorithmic FLOPs come from SURVEY.md
                §8(d) with R_map = (7|5)B + n_f + n_b (valid flow rows only); `kernels` lists all sites;
                `hbm` is the HBM side of the weight-gradient kernel (image bytes it must read / time)
  cpu_baseline  the oracle on this box's host cores, bounded sample
  ref_gpu       the oracle's torch ops on cuda:0 with the video tensors on the host, as the reference
                keeps them (the "R-GPU" row the >= 10x target of BASELINE.md is defined against)
  e2e           same metric through AtlasTrainer.step_host: pinned H2D of the index batch + D2H of
                the loss vector + sync every step
  pretrain_steps_per_s, render_s   the two other loops of a stage-1 run (pre_train_mapping, full render)
`--workload raft|stage2` times BASELINE.json configs[3]/[4] (1080p) with the same line format; `--workload seg` the
segmentation variant of the stage-1 loop (SURVEY §8 f3) at the headline geometry.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "all-in-one-deflicker_b200"))

H, W, T, BATCH = 432, 768, 80, 10000          # BASELINE.json configs[1]
MAC_MAP, MAC_ATLAS = 263424, 414584           # SURVEY.md §8: MACs per row
CPU_THREADS = 32      # the oracle gets SLOWER beyond this on the B200 hosts (128 threads: 0.03-0.08 it/s, measured)
TAGS = {1: "map_fwd", 2: "map_bwd", 3: "atlas_fwd", 4: "atlas_bwd", 5: "wgrad", 6: "adam"}


def r_map(with_global: bool, n_f: float, n_b: float) -> float:
    return (7 if with_global else 5) * BATCH + n_f + n_b


def algorithmic_flop(with_global: bool, n_f: float, n_b: float) -> float:
    """6 x (R_map x 263 424 + R_atlas x 414 584), SURVEY.md §8(d)."""
    return 6.0 * (r_map(with_global, n_f, n_b) * MAC_MAP + 3 * BATCH * MAC_ATLAS)


def site_flop(site: str, rm: float) -> float:
    """Algorithmic FLOPs of one tagged site: 2 FLOP/MAC x rows x MACs/row; forward, dgrad and wgrad each count
    the full per-row MAC figure of SURVEY.md §8(d)."""
    ra = 3.0 * BATCH
    return {"map_fwd": 2 * rm * MAC_MAP, "map_bwd": 2 * rm * MAC_MAP, "atlas_fwd": 2 * ra * MAC_ATLAS,
            "atlas_bwd": 2 * ra * MAC_ATLAS, "wgrad": 2 * (rm * MAC_MAP + ra * MAC_ATLAS), "adam": 0.0}[site]


def wgrad_image_bytes(rm: float) -> float:
    """Bytes the weight-gradient kernel must read: for every GEMM dW = dZ^T H both operand images, two fp16
    terms each (DESIGN.md §2).  mapping: 4 x (256+256) + (64+256) columns, atlas: 6 x 512 + 2 x 320 + 320 + 128."""
    return rm * (4 * 512 + 320) * 4.0 + 3.0 * BATCH * (6 * 512 + 2 * 320 + 320 + 128) * 4.0


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled through NVML every ~2 ms for the whole life of the benchmark
    (warm-up, timed region, end-to-end region); `summary(t0, t1)` reports the samples inside the timed region,
    widening to every sample taken while the GPU was busy when the region was too short to catch >= 3."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.stop_flag, self.h, self.max_mhz, self.how = [], False, None, None, "unavailable"
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.how = "nvml"
        except Exception:
            self.h = None
        self.index = index

    def _one(self):
        if self.h is not None:
            nv = self.nv
            sm = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            return sm, rs
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm,"
                              "clocks_event_reasons.active", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip().split(",")
        self.max_mhz = int(float(out[1]))
        self.how = "nvidia-smi"
        return int(float(out[0])), int(out[2].strip(), 16)

    def run(self):
        while not self.stop_flag:
            try:
                sm, rs = self._one()
                self.samples.append((time.perf_counter(), sm, rs))
            except Exception:
                pass
            time.sleep(0.002 if self.h is not None else 0.1)

    def summary(self, t0, t1):
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        scope = "timed region"
        if len(inside) < 3:
            inside, scope = list(self.samples), "whole benchmark (timed region shorter than 3 samples)"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"], "source": self.how}
        sm = sorted(s[1] for s in inside)
        bits = 0
        for s in inside:
            bits |= s[2]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": [n for b, n in self.REASONS.items() if bits & b], "samples": len(sm), "scope": scope,
                "source": self.how}


def run_oracle_steps(data, steps, warmup, threads=None, budget_s=None, fraction=1.0, device="cpu"):
    """The restatement of the reference loop (oracle = test/baseline code) on the host cores, or with its networks
    on `device` and the video on the host as the reference keeps it.  Returns (seconds, steps timed).
    `fraction` < 1 times a sub-batch of the 10 000 samples per step (bounded sample); `budget_s` stops early once
    that much time has been spent (>= 3 steps)."""
    from oracle import atlas_oracle as O
    if threads:
        torch.set_num_threads(threads)
    video = O.Video(**{k: v for k, v in data.items() if k != "clean"})
    torch.manual_seed(0)
    mp = [p.to(device).requires_grad_(True) for p in O.init_mlp(O.MAPPING_SPEC)]
    ap = [p.to(device).requires_grad_(True) for p in O.init_mlp(O.ATLAS_SPEC)]
    opt = O.make_optimizer(mp, ap)
    npix = video.H * video.W * video.T
    g = torch.Generator().manual_seed(1)
    batch = max(64, int(BATCH * fraction))
    total, done = 0.0, 0
    sync = (lambda: torch.cuda.synchronize()) if device != "cpu" else (lambda: None)
    for i in range(warmup + steps):
        it = 0 if i < warmup + (steps + 1) // 2 else 6000           # half with / half without global rigidity
        inds = torch.randint(npix, (batch, 1), generator=g)
        sync()
        t0 = time.perf_counter()
        O.train_iteration(video, mp, ap, opt, inds, it, device=device)
        sync()
        if i >= warmup:
            total += time.perf_counter() - t0
            done += 1
            if budget_s is not None and done >= 3 and total >= budget_s:
                break
    return float(total), done


ATLAS_CONFIG = {"workload": "stage-1 atlas loop, 80 frames 768x432, 10000 samples/iter, config_flow_100.json "
                            "coefficients, no segmentation (BASELINE.json configs[1])",
                "frames": T, "height": H, "width": W, "samples_batch": BATCH,
                "regime": "first half of the timed steps with the global rigidity term (i<=5000), second half without",
                "l2": "per-step working set (~1 GB of activation images + random gathers from 1.7 GB of pixel "
                      "records) exceeds the 126 MB L2; no explicit flush"}


def reference_arm(args, rank):
    """--impl reference: the CPU oracle port on the host cores, same metric / config."""
    if rank != 0:
        return
    from b200 import synth
    K = args.steps
    data = synth.throughput_set(H, W, T, seed=0)
    cores = os.cpu_count() or 1
    threads = min(cores, CPU_THREADS)
    # calibrate one full iteration, then size the per-step sample so that K steps take ~150 s
    t_full, _ = run_oracle_steps(data, 1, 1, threads=threads)
    fraction = min(1.0, 150.0 / max(K * t_full, 1e-9))
    secs, done = run_oracle_steps(data, K, 1, threads=threads, fraction=fraction)
    batch = max(64, int(BATCH * fraction))
    val = done * (batch / BATCH) / secs          # full-iteration equivalents per second
    line = {"impl": "reference", "metric": "atlas_iters_per_sec", "value": val, "unit": "it/s", "n_gpus": args.gpus,
            "steps": K, "warmup": 1, "ms_per_step": 1000.0 * secs / done, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "config": ATLAS_CONFIG,
            "cpu_baseline": {"value": val, "unit": "it/s", "cores": threads, "kind": "port",
                             "sample": f"{done} steps of {batch} samples each ({batch / BATCH:.3f} of an iteration; "
                                       f"cost is linear in the samples) of the oracle restatement of "
                                       f"src/stage1_neural_atlas.py:151-231, torch CPU fp32, {threads} threads of "
                                       f"{cores} cores"},
            "e2e": {"value": val, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def C_void(ev):
    import ctypes
    return ctypes.c_void_p(ev.cuda_event)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="atlas", choices=["atlas", "raft", "stage2", "seg"])
    ap.add_argument("--precision", default=os.environ.get("B200_PRECISION", "auto"), choices=["auto", "tc", "fp32"])
    ap.add_argument("--cpu-sample-steps", type=int, default=12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the pre-training / render side measurements")
    ap.add_argument("--emulate-world", type=int, default=0,
                    help="profiling aid: ONE process does the work of rank 0 of an N-GPU run (frame shard 0, no "
                         "collective), so that ncu can list the per-rank kernels of the sharded step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (the loss vector and the "
                         "updated parameters, float32) as DIR/losses.npy and DIR/params.npy; the inputs depend only "
                         "on the arguments, so two builds can be compared output for output (the step sums with fp32 "
                         "atomics: two runs of one build agree to summation order, not bit for bit)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "atlas" or args.impl != "b200"):
        ap.error("--dump-outputs is implemented for --workload atlas --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload != "atlas":
        import bench_aux
        return bench_aux.driver_line(args, rank, world, local)
    if args.impl == "reference":
        return reference_arm(args, rank)
    K, Wm = args.steps, max(args.warmup, 3)
    from b200 import synth

    # ------------------------------------------------------------------ B200 arm
    import torch.distributed as dist
    from b200 import _native as N
    from b200 import atlas as A
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        # NCCL_DEBUG is left to the caller (the driver reads the rank count from NCCL's INFO log)
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    lib = N.lib()
    prec = args.precision
    if prec == "auto":
        prec = "tc" if lib.b200_device_supports_tc() else "fp32"
    precision = N.PREC_TC if prec == "tc" else N.PREC_FP32
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()

    data = synth.throughput_set(H, W, T, seed=0)
    t0, t1 = A.frame_range(rank, world, T)
    if args.emulate_world > 1:
        assert world == 1
        t0, t1 = A.frame_range(0, args.emulate_world, T)
    video = A.DeviceVideo.from_reference_layout(data, dev, t0, t1)
    trainer = A.AtlasTrainer(video, {"samples_batch": BATCH}, precision=precision, device=dev, process_group=pg)
    torch.manual_seed(0)
    trainer.init_like_reference()
    if world > 1:
        dist.broadcast(trainer.params, 0)
    npix = H * W * T
    gen = torch.Generator().manual_seed(1)            # same stream on every rank -> identical index batches
    total = Wm + K
    inds_cpu = torch.randint(npix, (total, BATCH), generator=gen)
    inds_dev = inds_cpu.to(dev)
    if rank != 0 or (args.no_cpu_baseline and args.no_ref_gpu):
        del data
    half = Wm + (K + 1) // 2
    it_of = lambda i: 0 if i < half else 6000

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lib.b200_set_kernel_timer(None, None, 0)
    # both graphs are captured during warm-up (no event records inside them)
    launches0 = lib.b200_launch_count()
    trainer.indices.copy_(inds_dev[0]); trainer.step(0)
    n_g = lib.b200_launch_count() - launches0
    launches0 = lib.b200_launch_count()
    trainer.indices.copy_(inds_dev[0]); trainer.step(6000)
    n_ng = lib.b200_launch_count() - launches0
    per_step = {True: n_g // 2, False: n_ng // 2}      # each first call = 1 eager warm-up + 1 capture
    for i in range(Wm):
        trainer.indices.copy_(inds_dev[i]); trainer.step(it_of(i))
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    mid = torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(Wm, total):
        if i == half:
            mid.record()                  # regime switch (i > stop_global_rigidity): an event record, no extra work
        trainer.indices.copy_(inds_dev[i]); trainer.step(it_of(i))
    stop.record()
    barrier()
    wall1 = time.perf_counter()
    ms = start.elapsed_time(stop)
    n_with = max(0, min(total, half) - Wm)
    regimes = None
    if 0 < n_with < K:
        regimes = {"with_global_rigidity (i <= 5000)": {"steps": n_with, "it_per_s": n_with / (start.elapsed_time(mid) / 1000.0)},
                   "without (i > 5000)": {"steps": K - n_with, "it_per_s": (K - n_with) / (mid.elapsed_time(stop) / 1000.0)},
                   "note": "this rank's device time; the headline value is all K steps"}
    losses_last = trainer.losses.cpu().numpy().copy()
    params_last = trainer.params.cpu().numpy().copy() if args.dump_outputs else None
    if world > 1:
        tms = torch.tensor([ms], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms)
    value = K / (ms / 1000.0)

    # ---- e2e: host index batches in, loss vector out, every step
    k_e2e = max(10, K // 2)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for j in range(k_e2e):
        i = Wm + (j * 2) % K
        trainer.step_host(inds_cpu[i], it_of(i))
    e1.record()
    barrier()
    ems = e0.elapsed_time(e1)
    if world > 1:
        tms = torch.tensor([ems], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ems = float(tms)
    e2e_val = k_e2e / (ems / 1000.0)

    # ---- per-site kernel times: second pair of graphs that carry event records around every tagged launch
    events = {t: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for t in TAGS}
    for t, (a, b) in events.items():
        a.record(); b.record()
        lib.b200_set_kernel_timer(C_void(a), C_void(b), t)
    trainer._graphs.clear()
    site_ms = {True: {n: [] for n in TAGS.values()}, False: {n: [] for n in TAGS.values()}}
    for wg, it in ((True, 0), (False, 6000)):
        for j in range(12):
            trainer.indices.copy_(inds_dev[Wm + j % K]); trainer.step(it)
            torch.cuda.synchronize()
            if j >= 2:
                for t, (a, b) in events.items():
                    site_ms[wg][TAGS[t]].append(a.elapsed_time(b))
    lib.b200_set_kernel_timer(None, None, 0)
    trainer._graphs.clear()
    site_med = {wg: {n: float(np.median(v)) for n, v in d.items() if v} for wg, d in site_ms.items()}
    if world > 1:      # max over ranks, per site
        keys = [(wg, n) for wg in (True, False) for n in TAGS.values()]
        tv = torch.tensor([site_med[wg].get(n, 0.0) for wg, n in keys], device=dev)
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        for (wg, n), v in zip(keys, tv.tolist()):
            site_med[wg][n] = v

    extras = {}
    if rank == 0 and not args.no_extras and world == 1:
        extras = side_measurements(trainer, A, N, dev)

    if rank == 0:
        if sampler:
            sampler.stop_flag = True
        peaks, how = measured_peaks()
        n_f = float(losses_last[6]) / world  # every rank writes the GLOBAL count (whole-video bitmaps are replicated);
        n_b = float(losses_last[7]) / world  # the all-reduce of the loss vector sums them
        flop_step = 0.5 * (algorithmic_flop(True, n_f, n_b) + algorithmic_flop(False, n_f, n_b))
        peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
        hbm_gbs = float(peaks.get("hbm_gbs"))
        kernels = {}
        for n in TAGS.values():
            tw, tn = site_med[True].get(n), site_med[False].get(n)
            if not tw or not tn:
                continue
            fw = site_flop(n, r_map(True, n_f, n_b)) / world
            fn = site_flop(n, r_map(False, n_f, n_b)) / world
            kernels[n] = {"ms_with_global": tw, "ms_without": tn,
                          "tflops": 0.5 * (fw / tw + fn / tn) / 1e9 if fw else None}
        dom = max(kernels, key=lambda n: kernels[n]["ms_with_global"] + kernels[n]["ms_without"]) if kernels else None
        names = {"map_fwd": "tc_fwd_kernel<mapping>", "map_bwd": "tc_bwd_kernel<mapping>",
                 "atlas_fwd": "tc_fwd_kernel<atlas>", "atlas_bwd": "tc_bwd_kernel<atlas>",
                 "wgrad": "tc_wgrad_kernel", "adam": "adam_kernel"}
        roof = {"bound": "tensor", "kernel": None, "achieved": None, "peak": peak_tf, "unit": "TFLOP/s", "frac": None,
                "peak_source": f"{how} bf16_tflops_sustained (fp32-grade products cost 3 MMAs: attainable ceiling = peak/3)"}
        if dom:
            roof.update(kernel=names[dom] if precision == N.PREC_TC else dom + " (fp32 CUDA-core path)",
                        achieved=kernels[dom]["tflops"], frac=kernels[dom]["tflops"] / peak_tf if kernels[dom]["tflops"] else None,
                        kernel_ms=0.5 * (kernels[dom]["ms_with_global"] + kernels[dom]["ms_without"]))
        if "wgrad" in kernels and precision == N.PREC_TC:
            bw = 0.5 * (wgrad_image_bytes(r_map(True, n_f, n_b)) / world / kernels["wgrad"]["ms_with_global"] +
                        wgrad_image_bytes(r_map(False, n_f, n_b)) / world / kernels["wgrad"]["ms_without"]) / 1e6
            roof["hbm"] = {"kernel": "tc_wgrad_kernel", "achieved": bw, "peak": hbm_gbs, "unit": "GB/s",
                           "frac": bw / hbm_gbs, "bytes": "algorithmic: both fp16-term images of every dW = dZ^T H operand"}
        traffic_path = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
        roof["traffic"] = None
        if os.path.exists(traffic_path) and dom:
            with open(traffic_path) as f:
                tr = json.load(f)
            roof["traffic"] = tr.get(names[dom])           # dram read+write bytes per launch from the committed ncu capture
            roof["traffic_source"] = "profiles/r2_ncu_traffic.json (ncu --set full, with-global regime)"
        roof.update(kernels=kernels, step_algorithmic_gflop=flop_step / 1e9, step_tflops=flop_step * value / 1e12,
                    step_frac=flop_step * value / 1e12 / peak_tf, rows={"n_f": n_f, "n_b": n_b})
        line = {"metric": "atlas_iters_per_sec", "value": value, "unit": "it/s", "n_gpus": world, "steps": K,
                "warmup": Wm, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None,
                "dtype": "fp32" if precision == N.PREC_FP32 else "fp32 (2-term fp16 split on tcgen05, fp32 accumulate)",
                "data": "synthetic", "config": dict(ATLAS_CONFIG, parallelism=f"frame-sharded dp{world}" if args.emulate_world < 2
                                                    else f"PROFILING AID: rank 0 of an emulated dp{args.emulate_world} run, no collective",
                                                    precision=prec, cuda_graph=True),
                "e2e": {"value": e2e_val, "unit": "it/s", "h2d_bytes_per_step": BATCH * 8,
                        "d2h_bytes_per_step": N.LOSS_FLOATS * 4, "steps": k_e2e},
                "gpu_launches": int(sum(per_step[it_of(i) == 0] for i in range(Wm, total))),
                "launches_per_step": {"with_global": per_step[True], "without": per_step[False]},
                "roofline": roof,
                "clocks": sampler.summary(wall0, wall1) if sampler else None,
                "losses_last": [float(x) for x in losses_last[:6]]}
        if regimes:
            line["regimes"] = regimes
        line.update(extras)
        cores = os.cpu_count() or 1
        threads = min(cores, CPU_THREADS)
        if not args.no_cpu_baseline and world == 1:
            secs, done = run_oracle_steps(data, args.cpu_sample_steps, 1, threads=threads, budget_s=20.0)
            line["cpu_baseline"] = {"value": done / secs, "unit": "it/s", "cores": threads, "kind": "port",
                                    "sample": f"{done} full iterations of the oracle (torch CPU fp32 restatement of "
                                              f"src/stage1_neural_atlas.py:151-231) on the same synthetic video, "
                                              f"{threads} threads of {cores} cores"}
        if not args.no_ref_gpu and world == 1:
            del trainer, video, inds_dev
            torch.cuda.empty_cache()
            secs, done = run_oracle_steps(data, 24, 4, threads=threads, budget_s=15.0, device=str(dev))
            line["ref_gpu"] = {"value": done / secs, "unit": "it/s", "iters": done,
                               "kind": "oracle port (the reference's torch ops) with the networks on this GPU and "
                                       "the video tensors on the host, as src/stage1_neural_atlas.py keeps them",
                               "speedup_e2e": e2e_val / (done / secs)}
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "losses.npy"), losses_last.astype(np.float32))
            np.save(os.path.join(args.dump_outputs, "params.npy"), params_last.astype(np.float32))
        print(json.dumps(line), flush=True)
    if world > 1:
        # orderly teardown: every rank is past its last collective; drop the captured graphs (they hold NCCL
        # work) before the communicator, and never block the launcher on a straggling destructor
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def side_measurements(trainer, A, N, dev):
    """pre_train_mapping steps/s (unwrap_utils.py:176-198) and the full-video render (evaluate.py:640-708) at the
    benchmark geometry, through the same public methods the stage-1 script calls."""
    out = {}
    snap = trainer.params.clone()
    try:
        g = torch.Generator().manual_seed(3)
        trainer.pretrain(8, H, W, 1, generator=g)                  # warm-up (graph capture when available)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sweeps = 5
        trainer.pretrain(T, H, W, sweeps, generator=g)
        torch.cuda.synchronize()
        out["pretrain_steps_per_s"] = sweeps * T / (time.perf_counter() - t0)
    except Exception as e:                                          # never lose the headline line to a side number
        out["pretrain_steps_per_s"] = None
        out["pretrain_error"] = repr(e)[:200]
    trainer.params.copy_(snap)
    try:
        trainer.render_frame(0, H, W, T, want_u8=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for f in range(T):
            trainer.render_frame(f, H, W, T, want_u8=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out["render_s"] = dt
        out["render_tflops"] = 2.0 * H * W * T * (MAC_MAP + MAC_ATLAS) / dt / 1e12
    except Exception as e:
        out["render_s"] = None
        out["render_error"] = repr(e)[:200]
    return out


if __name__ == "__main__":
    main()
