#!/usr/bin/env python
"""Secondary benchmarks of BASELINE.json configs[3] and configs[4] (not the headline metric; bench.py is):

  config 4  RAFT at 1080p (H/8 x W/8 = 135 x 240): all-pairs correlation volume + pyramid, windowed lookup,
            one update-block iteration, and a whole frame pair (20 iterations, both kernels + encoders)
  config 5  stage 2 at 1088 x 1920: UNet neural filter and TransformNet local refinement, frames/s

Each number is CUDA-event time of OUR kernels through the C ABI.  With --with-eager the same operators are also
timed as plain torch ops (cuBLAS/cuDNN) on the same GPU for orientation: that leg runs the oracle restatement
and therefore lives under tests/ (tests/perf/eager_aux.py).  One JSON line.
    python bench_aux.py [--small] [--conv tc|fp32] [--with-eager]
"""
import argparse
import json
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "all-in-one-deflicker_b200"))


def timed(fn, iters=3, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--small", action="store_true", help="quarter resolution (quick check)")
    ap.add_argument("--conv", choices=["fp32", "tc"], default="tc", help="convolution arithmetic (b200.nn)")
    ap.add_argument("--with-eager", action="store_true", help="also time torch-eager restatements (tests/perf/eager_aux.py)")
    args = ap.parse_args()
    from b200 import nn as K
    K.set_conv_precision(args.conv)
    eager = None
    if args.with_eager:
        sys.path.insert(0, os.path.join(ROOT, "tests", "perf"))
        import eager_aux as eager
    from src.models.network_filter import UNet
    from src.models.network_local import TransformNet
    from src.models.stage_1.core.raft import RAFT
    from src.models.stage_1.core.update import BasicUpdateBlock
    dev = "cuda"
    H, W = (272, 480) if args.small else (1080, 1920)
    h8, w8 = (H + 7) // 8, (W + 7) // 8
    out = {"config": {"raft_frame": [H, W], "h8_w8": [h8, w8], "conv": args.conv}}
    g = torch.Generator(device="cpu").manual_seed(0)
    # ---------------- RAFT correlation
    f1 = torch.randn(1, 256, h8, w8, generator=g).to(dev)
    f2 = torch.randn(1, 256, h8, w8, generator=g).to(dev)
    hw = h8 * w8
    pyr = [None]
    def build():
        pyr[0] = None                      # release the previous 5.6 GB pyramid first: no allocator growth in the timed region
        pyr[0] = K.corr_build(f1, f2)
    ms = timed(build, iters=2)
    vol_bytes = 4.0 * hw * hw * (1 + 0.25 + 0.0625 + 0.015625)
    out["corr_build"] = {"ms": ms, "tflops": 2.0 * hw * hw * 256 / ms / 1e9, "gb_written": vol_bytes / 1e9,
                         "gbs": vol_bytes / ms / 1e6}
    ys, xs = torch.meshgrid(torch.arange(h8).float(), torch.arange(w8).float(), indexing="ij")
    coords = (torch.stack([xs, ys])[None] + torch.randn(1, 2, h8, w8, generator=g)).to(dev)
    ms = timed(lambda: K.corr_lookup(pyr[0], coords), iters=5)
    out["corr_lookup"] = {"ms": ms, "taps_per_s": hw * 324 * 4 / ms * 1e3}
    if eager:
        out["torch_eager_corr"] = eager.corr(timed, f1, f2, coords)
    # ---------------- update block, one iteration
    ub = BasicUpdateBlock(types.SimpleNamespace(corr_levels=4, corr_radius=4), hidden_dim=128).to(dev)
    net = torch.tanh(torch.randn(1, 128, h8, w8, generator=g)).to(dev)
    inp = torch.relu(torch.randn(1, 128, h8, w8, generator=g)).to(dev)
    flow = torch.randn(1, 2, h8, w8, generator=g).to(dev)
    corr = K.corr_lookup(pyr[0], coords)
    ms = timed(lambda: ub(net, inp, corr, flow), iters=3)
    out["update_block_iter"] = {"ms": ms, "tflops": 2 * 3.118e6 * hw / ms / 1e9}
    if eager:
        out["torch_eager_update_block_iter_ms"] = eager.update_block(timed, ub, net, inp, corr, flow)
    del pyr, corr
    torch.cuda.empty_cache()
    # ---------------- whole pair
    import argparse as ap2
    raft = RAFT(ap2.Namespace(small=False, mixed_precision=True)).to(dev).eval()
    im1 = (torch.rand(1, 3, H // 8 * 8, W // 8 * 8, generator=g) * 255).to(dev)
    im2 = (torch.rand(1, 3, H // 8 * 8, W // 8 * 8, generator=g) * 255).to(dev)
    ms = timed(lambda: raft(im1, im2, iters=20, test_mode=True), iters=1, warm=1)
    out["raft_pair_20iters"] = {"ms": ms, "pairs_per_s_both_directions": 1000.0 / (2 * ms)}
    del raft
    torch.cuda.empty_cache()
    # ---------------- stage 2
    Hp, Wp = (288, 480) if args.small else (1088, 1920)
    unet = UNet(6, 3, 32).to(dev).eval()
    tn = TransformNet(types.SimpleNamespace(nf=32, norm="IN", model="TransformNet", blocks=5), 12, 3).to(dev).eval()
    x6 = torch.rand(1, 6, Hp, Wp, generator=g).to(dev)
    x12 = torch.rand(1, 12, Hp, Wp, generator=g).to(dev)
    ms_u = timed(lambda: unet(x6), iters=2)
    ms_t = timed(lambda: tn(x12, None), iters=2)
    out["stage2"] = {"unet_ms": ms_u, "transformnet_ms": ms_t, "frames_per_s": 1000.0 / (ms_u + ms_t),
                     "unet_tflops": 2 * 524e9 * (Hp * Wp) / (1088 * 1920) / ms_u / 1e9,
                     "transformnet_tflops": 2 * 559e9 * (Hp * Wp) / (1088 * 1920) / ms_t / 1e9}
    if eager:
        out["torch_eager_stage2"] = eager.stage2(timed, unet, tn, x6, x12)
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------------
# driver-format lines for `bench.py --workload raft|stage2` (BASELINE.json configs[3] / configs[4])
# ------------------------------------------------------------------------------------------------------
def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return json.load(open(path)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def _event_ms(fn, iters, warm, world=1, dev=None):
    import torch.distributed as dist
    for _ in range(warm):
        fn()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    return ms / iters


def _reference_line(args):
    """--impl reference for the two secondary workloads: the oracle restatements (plain torch ops) on the host
    cores, bounded sample."""
    import time
    from oracle import flow_oracle as FO, stage2_oracle as SO
    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    if args.workload == "stage2":
        from src.models.network_filter import UNet
        from src.models.network_local import TransformNet
        Hp, Wp = 1088, 1920
        sd_u = UNet(6, 3, 32).state_dict()
        sd_t = TransformNet(types.SimpleNamespace(nf=32, norm="IN", model="TransformNet", blocks=5), 12, 3).state_dict()
        x6, x12 = torch.rand(1, 6, Hp, Wp, generator=g), torch.rand(1, 12, Hp, Wp, generator=g)
        with torch.no_grad():
            t0 = time.perf_counter(); SO.unet_forward(sd_u, x6); SO.transformnet_forward(sd_t, x12)
            dt = time.perf_counter() - t0
        val, unit, metric = 1.0 / dt, "frames/s", "stage2_frames_per_sec"
        sample = f"1 frame at 1088x1920 through the oracle UNet + TransformNet (torch CPU fp32), {threads} threads of {cores}"
    else:
        h8, w8 = 135, 240
        f1, f2 = torch.randn(1, 256, h8, w8, generator=g), torch.randn(1, 256, h8, w8, generator=g)
        ub_sd = {}
        from src.models.stage_1.core.update import BasicUpdateBlock
        ub_sd = BasicUpdateBlock(types.SimpleNamespace(corr_levels=4, corr_radius=4), hidden_dim=128).state_dict()
        ys, xs = torch.meshgrid(torch.arange(h8).float(), torch.arange(w8).float(), indexing="ij")
        coords = torch.stack([xs, ys])[None]
        net, inp, flow = torch.randn(1, 128, h8, w8), torch.randn(1, 128, h8, w8), torch.zeros(1, 2, h8, w8)
        with torch.no_grad():
            t0 = time.perf_counter(); pyr = FO.corr_pyramid(f1, f2); t_c = time.perf_counter() - t0
            t0 = time.perf_counter(); c = FO.corr_lookup(pyr, coords); FO.update_block(ub_sd, net, inp, c, flow)
            t_i = time.perf_counter() - t0
        dt = 2 * (t_c + 20 * t_i)
        val, unit, metric = 1.0 / dt, "pairs/s", "raft_pairs_per_sec"
        sample = (f"one direction: correlation pyramid ({t_c:.2f} s) + 1 of 20 lookup+update iterations ({t_i:.2f} s), "
                  f"extrapolated to 2 directions x 20 iterations, encoders and upsampling NOT counted (favours the CPU); "
                  f"oracle torch CPU fp32, {threads} threads of {cores}")
    print(json.dumps({"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus,
                      "steps": 1, "warmup": 0, "ms_per_step": 1000.0 / val, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
                      "config": {"workload": args.workload},
                      "cpu_baseline": {"value": val, "unit": unit, "cores": threads, "kind": "port", "sample": sample},
                      "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def seg_line(args, rank, world, local):
    """`bench.py --workload seg`: the segmentation variant of the stage-1 loop (SURVEY §8 f3) at the headline geometry
    (80 x 432 x 768, 10 000 samples per iteration, config_flow_100.json), one GPU.  A step = one loop trip
    (b200_seg_loss_grad + b200_adam_step).  `--impl reference` / cpu_baseline: oracle/seg_oracle.py on the host cores,
    a bounded sample of whole iterations."""
    import time
    from b200 import synth
    T, H, W, B = 80, 432, 768, 10000
    config = {"workload": "stage-1 atlas loop, segmentation variant (two mappings + alpha + atlas), 80 frames 768x432, "
                          "10000 samples/iter, config_flow_100.json coefficients", "frames": T, "height": H, "width": W,
              "samples_batch": B, "regime": "first half of the timed steps with the global rigidity terms, second half without",
              "l2": "per-step working set (~2 GB of activations) exceeds the 126 MB L2"}
    metric, unit = "seg_iterations_per_sec", "it/s"
    data = synth.throughput_set(H, W, T, seed=0)
    gm = torch.Generator().manual_seed(2)
    masks = (torch.rand(H, W, T, generator=gm) < 0.4).float()

    def cpu_leg(n_steps, threads):
        from oracle import atlas_oracle as O, seg_oracle as S
        torch.set_num_threads(threads)
        video = O.Video(**data)
        torch.manual_seed(0)
        nets = {k: [p.requires_grad_(True) for p in v] for k, v in S.init_nets().items()}
        opt = S.make_optimizer(nets)
        g = torch.Generator().manual_seed(1)
        total = 0.0
        for i in range(1 + n_steps):
            inds = torch.randint(H * W * T, (B, 1), generator=g)
            t0 = time.perf_counter()
            terms = S.seg_iteration_losses(video, masks, nets, inds, 0 if i <= n_steps // 2 else 6000)
            opt.zero_grad(); terms["total"].backward(); opt.step()
            if i >= 1:
                total += time.perf_counter() - t0
        return n_steps / total

    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    if args.impl == "reference":
        if rank == 0:
            n = max(2, min(args.steps, 4))
            v = cpu_leg(n, threads)
            print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": n,
                              "warmup": 1, "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "strong",
                              "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "config": config,
                              "cpu_baseline": {"value": v, "unit": unit, "cores": threads, "kind": "port",
                                               "sample": f"{n} whole iterations of oracle/seg_oracle.py, {threads} threads"},
                              "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    assert world == 1, "the segmentation variant is single-GPU (whole video resident)"
    from b200 import _native as N, atlas as A, seg as SG
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    vid = A.DeviceVideo.from_reference_layout(data, dev)
    prec = N.PREC_TC if (args.precision != "fp32" and N.lib().b200_device_supports_tc()) else N.PREC_FP32
    tr = SG.SegTrainer(vid, SG.pack_mask_frames(masks, dev), None, precision=prec, device=dev)
    torch.manual_seed(0)
    tr.init_like_reference()
    steps, warm = args.steps, max(3, args.warmup)
    g = torch.Generator().manual_seed(1)
    inds_d = [torch.randint(H * W * T, (B,), generator=g).to(dev) for _ in range(8)]
    inds_h = [torch.randint(H * W * T, (B, 1), generator=g) for _ in range(8)]
    k = [0]

    def step():
        i = k[0]; k[0] += 1
        tr.indices.copy_(inds_d[i % 8])
        tr.step(0 if (i % steps) < steps // 2 else 6000)
    tr.indices.copy_(inds_d[0])
    l0 = N.lib().b200_launch_count()
    tr.step(0, use_graph=False)                       # kernels of one trip, counted on an eager (un-captured) trip
    n_launch = float(N.lib().b200_launch_count() - l0)
    ms = _event_ms(step, steps, warm)
    k[0] = 0
    ems = _event_ms(lambda: (tr.step_host(inds_h[k[0] % 8], 0 if k[0] % steps < steps // 2 else 6000), k.__setitem__(0, k[0] + 1)),
                    steps, 2)
    out = {"metric": metric, "value": 1000.0 / ms, "unit": unit, "n_gpus": 1, "steps": steps, "warmup": warm,
           "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": ("mapping1 + atlas: 2-term fp16 split operands / fp32 accumulate (tcgen05); mapping2 + alpha: fp32 CUDA cores"
                     if prec == N.PREC_TC else "fp32"), "data": "synthetic", "config": config,
           "e2e": {"value": 1000.0 / ems, "unit": unit, "h2d_bytes_per_step": B * 8, "d2h_bytes_per_step": N.SEG_LOSS_FLOATS * 4},
           "gpu_launches": int(round(n_launch * steps)), "launches_per_step": n_launch,
           "cuda_graph": "one replayed graph per regime (global rigidity on / off)", "losses_last": tr.loss_dict()}
    if not args.no_cpu_baseline:
        v = cpu_leg(2, threads)
        out["cpu_baseline"] = {"value": v, "unit": unit, "cores": threads, "kind": "port",
                               "sample": f"2 whole iterations of oracle/seg_oracle.py, {threads} threads"}
    print(json.dumps(out), flush=True)


def driver_line(args, rank, world, local):
    """`bench.py --workload raft|stage2`: a step = one 1080p frame pair (both flow directions, 20 refinement
    iterations) / one 1088x1920 frame through UNet + TransformNet.  Pairs and neural-filter frames are independent
    units: with N GPUs every rank runs its own (weak scaling, no collective)."""
    if args.workload == "seg":
        return seg_line(args, rank, world, local)
    if args.impl == "reference":
        if rank == 0:
            _reference_line(args)
        return
    import argparse as ap2
    import torch.distributed as dist
    from b200 import nn as K
    from b200 import _native as N
    assert torch.cuda.is_available()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K.set_conv_precision("tc")
    steps, warm = args.steps, max(1, min(args.warmup, 3))
    g = torch.Generator().manual_seed(rank)
    peaks, how = _peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    launches0 = N.lib().b200_launch_count()
    if args.workload == "raft":
        from src.models.stage_1.core.raft import RAFT
        from src.models.stage_1.core.update import BasicUpdateBlock
        Hh, Ww = 1080, 1920
        h8, w8 = Hh // 8, Ww // 8
        hw = h8 * w8
        raft = RAFT(ap2.Namespace(small=False, mixed_precision=True)).to(dev).eval()
        im1_h = (torch.rand(1, 3, Hh, Ww, generator=g) * 255).pin_memory()
        im2_h = (torch.rand(1, 3, Hh, Ww, generator=g) * 255).pin_memory()
        im1, im2 = im1_h.to(dev), im2_h.to(dev)
        with torch.no_grad():
            ms = _event_ms(lambda: raft.forward_both(im1, im2, iters=20), steps, warm, world, dev)
            n_launch = (N.lib().b200_launch_count() - launches0) // (steps + warm)
            res = {}
            def e2e():
                a, b = im1_h.to(dev, non_blocking=True), im2_h.to(dev, non_blocking=True)
                (_, u12), (_, u21) = raft.forward_both(a, b, iters=20)
                res["f"] = (u12[0].permute(1, 2, 0).cpu(), u21[0].permute(1, 2, 0).cpu())
            ems = _event_ms(e2e, max(1, steps // 2), 1, world, dev)
            # dominant component: the update block (20 x 2 calls per pair), timed alone
            ub = raft.update_block
            net = torch.tanh(torch.randn(1, 128, h8, w8, generator=g)).to(dev)
            inp = torch.relu(torch.randn(1, 128, h8, w8, generator=g)).to(dev)
            flow = torch.randn(1, 2, h8, w8, generator=g).to(dev)
            corr = torch.randn(1, 324, h8, w8, generator=g).to(dev)
            ub_ms = _event_ms(lambda: ub(net, inp, corr, flow), 10, 2)
            f1 = torch.randn(1, 256, h8, w8, generator=g).to(dev)
            pyr = [None]
            def build():
                pyr[0] = None
                pyr[0] = K.corr_build(f1, f1)
            cb_ms = _event_ms(build, 3, 1)
        value, unit, metric = world * 1000.0 / ms, "pairs/s", "raft_pairs_per_sec"
        e2e_v = world * 1000.0 / ems
        h2d, d2h = 2 * 3 * Hh * Ww * 4, 2 * Hh * Ww * 2 * 4
        ub_tf = 2 * 3.118e6 * hw / ub_ms / 1e9
        vol = 4.0 * hw * hw * (1 + 0.25 + 0.0625 + 0.015625)
        roof = {"bound": "tensor", "kernel": "conv2d_tma_kernel (BasicUpdateBlock, one refinement iteration)",
                "achieved": ub_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ub_tf / peak_tf, "kernel_ms": ub_ms,
                "share_of_step": 40 * ub_ms / ms, "traffic": None, "peak_source": how,
                "hbm": {"kernel": "corr_build (conv2d_tma_kernel, split operands: level 0 + three pooled-feature GEMMs)", "achieved": vol / cb_ms / 1e6,
                        "peak": float(peaks["hbm_gbs"]), "unit": "GB/s", "frac": vol / cb_ms / 1e6 / float(peaks["hbm_gbs"]),
                        "kernel_ms": cb_ms, "share_of_step": 2 * cb_ms / ms}}
        config = {"workload": "RAFT flow pre-pass, 1080x1920 synthetic frame pair, both directions, 20 refinement "
                              "iterations, random-init RAFT-things weights (BASELINE.json configs[3])",
                  "l2": "4.2 GB correlation volume per direction exceeds L2"}
        dtype = "fp16 operands / fp32 accumulate convolutions (the reference's autocast), fp32-grade correlation"
    else:
        from src.models.network_filter import UNet
        from src.models.network_local import TransformNet
        Hp, Wp = 1088, 1920
        unet = UNet(6, 3, 32).to(dev).eval()
        tn = TransformNet(types.SimpleNamespace(nf=32, norm="IN", model="TransformNet", blocks=5), 12, 3).to(dev).eval()
        c_h = torch.rand(1, 3, Hp, Wp, generator=g).pin_memory()
        s_h = torch.rand(1, 3, Hp, Wp, generator=g).pin_memory()
        content, style = c_h.to(dev), s_h.to(dev)
        state = {"o1": torch.rand(1, 3, Hp, Wp, generator=g).to(dev), "p1": torch.rand(1, 3, Hp, Wp, generator=g).to(dev)}
        def frame(c, s):
            pred = unet(torch.cat([c, s], dim=1))
            out, _ = tn(torch.cat((pred, state["o1"], pred, state["p1"]), dim=1), None)
            o2 = pred + out
            state["p1"], state["o1"] = pred, o2
            return o2
        with torch.no_grad():
            ms = _event_ms(lambda: frame(content, style), steps, warm, world, dev)
            n_launch = (N.lib().b200_launch_count() - launches0) // (steps + warm)
            res = {}
            def e2e():
                o = frame(c_h.to(dev, non_blocking=True), s_h.to(dev, non_blocking=True))
                res["o"] = o.cpu()
            ems = _event_ms(e2e, max(1, steps // 2), 1, world, dev)
            x6 = torch.rand(1, 6, Hp, Wp, generator=g).to(dev)
            x12 = torch.rand(1, 12, Hp, Wp, generator=g).to(dev)
            u_ms = _event_ms(lambda: unet(x6), 4, 1)
            t_ms = _event_ms(lambda: tn(x12, None), 4, 1)
        value, unit, metric = world * 1000.0 / ms, "frames/s", "stage2_frames_per_sec"
        e2e_v = world * 1000.0 / ems
        h2d, d2h = 2 * 3 * Hp * Wp * 4, 3 * Hp * Wp * 4
        t_tf = 2 * 559e9 / t_ms / 1e9
        roof = {"bound": "tensor", "kernel": "conv2d_tma_kernel (TransformNet forward)", "achieved": t_tf,
                "peak": peak_tf, "unit": "TFLOP/s", "frac": t_tf / peak_tf, "kernel_ms": t_ms, "traffic": None,
                "peak_source": how, "unet": {"ms": u_ms, "tflops": 2 * 524e9 / u_ms / 1e9}}
        config = {"workload": "stage 2: UNet neural filter + TransformNet local refinement on 1088x1920 frames "
                              "(1080p padded to /32), random-init weights (BASELINE.json configs[4])",
                  "note": "the refinement chain is sequential over frames; with N GPUs each rank filters its own video "
                          "(replicas)", "l2": "per-layer activations (up to 267 MB) exceed L2"}
        dtype = "fp16 operands / fp32 accumulate (tcgen05), the operand width of the reference's TF32 cuDNN convolutions"
    if rank == 0:
        print(json.dumps({"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": steps, "warmup": warm,
                          "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": dtype, "data": "synthetic", "config": config,
                          "e2e": {"value": e2e_v, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                          "gpu_launches": int(n_launch * steps), "roofline": roof}), flush=True)
    if world > 1:
        torch.cuda.synchronize(); dist.barrier()
        sys.stdout.flush(); os._exit(0)


if __name__ == "__main__":
    main()
