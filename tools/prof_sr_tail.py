#!/usr/bin/env python
"""Measure the uint8 reconstruction tail on the GPU and write one JSON file.

    python tools/prof_sr_tail.py --out DIR [--rounds 5]          -> DIR/sr_tail.json
    python tools/prof_sr_tail.py --out DIR --yuv [--rounds 5]    -> DIR/sr_tail_yuv.json
    python tools/prof_sr_tail.py --out DIR --hbd [--rounds 5]    -> DIR/sr_tail_hbd.json
    python tools/prof_sr_tail.py --out DIR --psnr [--rounds 5]   -> DIR/sr_tail_psnr.json

(a) The tail of one frame at the benchmark's operating point: 8 images of 64 x 1088 x 1920 bf16 features (2.1 GB,
    far more than L2) -> 8 frames of 1080 x 1920 x 3 uint8.  The fused kernel (`ops.sr_tail_u8`) against the
    composition it replaces in `EAVSRP.forward` + the reference's visuals: cuDNN conv_last + F.interpolate + add +
    crop + clamp * 255 + round + uint8.  Each arm is one CUDA graph; CUDA events time `--reps` replays; the arms
    alternate `--rounds` times after a warm-up.  The HBM floor counts 128 B/px of features read, 3 B/px written and
    12 B per LR pixel, at the data-sheet 7.7 TB/s.
(b) End to end, host to host, 8 clips of 30 x 270 x 480 per step, seeded weights, both arms graph-captured and
    alternated: the benchmark's recipe (pinned fp32 clip -> H2D -> forward -> crop -> visuals -> D2H uint8) and
    `forward_uint8` (pinned uint8 (n, t, h, w, 3) -> H2D -> forward_uint8 -> D2H).  Also reports how many output
    values differ between the two arms (the benchmark's path rounds conv_last's output to bf16).
With --yuv, the Y'CbCr 4:2:0 variant instead:
(a) the tail at the same operating point, 8 frames of 1080 x 1920 written as BT.709 I420 planes: the 4:2:0 kernel
    (`ops.sr_tail_yuv420`), the RGB kernel (`ops.sr_tail_u8`) and the PyTorch composition (cuDNN conv_last +
    F.interpolate + add + crop + `yuv.rgb_to_yuv420`), alternated.  The 4:2:0 HBM floor counts 1.5 B/px written.
(b) host to host, 8 clips of 30 x 270 x 480: `forward_yuv420` (pinned I420 planes -> H2D -> graph -> D2H) against
    `forward_uint8` (pinned RGB frames), both graph-captured and alternated.  Also the device time of the PyTorch
    ingest of one step (`pad_clip(yuv420_to_rgb(...))`, captured, CUDA events) next to forward_uint8's ingest, and the
    host CPU time of converting forward_uint8's output to I420 with torch on the CPU, timed on one clip of 30 frames
    and scaled to the 8 clips of a step.
With --hbd, the high-bit-depth variants:
(a) the tail at the same operating point: 16-bit RGB (`ops.sr_tail_u16`) and 10-bit BT.709 4:2:0 written as P010
    (`ops.sr_tail_yuv420_u16`, shift 6, chroma interleaved) against the 8-bit RGB and I420 kernels, alternated.  The
    HBM floors count 6 and 3 B/px written.
(b) host to host, 8 clips of 30 x 270 x 480: `forward_yuv420_u16` on P010 (pinned Y and interleaved UV planes -> H2D
    -> graph -> D2H) against `forward_yuv420` on I420, both graph-captured and alternated.
With --psnr, the squared error against ground-truth frames:
(a) the tail at the same operating point with 8 ground-truth frames of 1080 x 1920 x 3 uint8: the RGB kernel
    (`ops.sr_tail_u8`), the squared-error kernel without and with the store (`ops.sr_tail_u8_sse`), and the
    composition it replaces (`ops.sr_tail_u8`, then the int64 SSE of that frame in PyTorch), alternated.  The HBM
    floors count 3 B/px read for the ground truth, and 3 more written with the store.
(b) host to host, 8 clips of 30 x 270 x 480 and their 8 x 30 ground-truth frames of 1080 x 1920 per step:
    `psnr_uint8` (pinned LR and ground-truth frames -> H2D -> graph -> D2H of the (n, t) PSNR and SSE) against
    `forward_uint8` + the int64 SSE in PyTorch on the device + D2H of the frames and the SSE, both graph-captured and
    alternated.
The GPU name, power limit and maximum SM clock are read with nvidia-smi in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from eavsr_b200 import ops  # noqa: E402
from eavsr_b200.model import EAVSRP, pad_clip  # noqa: E402
from eavsr_b200.synthetic import clip_inputs, gen, seeded_parameters  # noqa: E402
from eavsr_b200.yuv import MATRICES, rgb_to_yuv420, yuv420_to_rgb  # noqa: E402

HBM_BPS = 7.7e12


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True, check=True)
    keys = [k.strip() for k in r.stdout.splitlines()[0].split(",")]
    vals = [v.strip() for v in r.stdout.splitlines()[1].split(",")]
    return dict(zip(keys, vals))


def capture(fn, pool=None):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()                                   # warm-up outside capture: cuDNN algorithm choice, packed weights
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, pool=pool):
        out = fn()
    return g, out


def time_replays(g, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / reps   # us per replay


def _tail_operands(dev):
    n, h, w, s, oh, ow = 8, 1088, 1920, 4, 1080, 1920
    g = gen(0)
    conv = torch.nn.Conv2d(64, 3, 3, 1, 1)
    with torch.no_grad():
        conv.weight.copy_((torch.rand(conv.weight.shape, generator=g) * 2 - 1) / 24)
        conv.bias.copy_((torch.rand(3, generator=g) * 2 - 1) * 0.05)
    conv = conv.to(dev, torch.bfloat16).eval()
    x = torch.empty((n, 64, h, w), dtype=torch.bfloat16, device=dev, memory_format=torch.channels_last)
    x.normal_().relu_()                                   # LeakyReLU-like features
    lr = torch.rand(n, 3, h // s, w // s, device=dev)
    return conv, x, lr, (n, h, w, s, oh, ow)


def tail(dev, rounds, reps):
    conv, x, lr, (n, h, w, s, oh, ow) = _tail_operands(dev)
    out = torch.empty((n, oh, ow, 3), dtype=torch.uint8, device=dev)

    def fused():
        return ops.sr_tail_u8(conv, x, lr, s, out, oh, ow)

    def composed():
        sr = conv(x).float() + F.interpolate(lr, scale_factor=s, mode="bilinear", align_corners=False)
        return torch.clamp(sr[..., :oh, :ow] * 255, 0, 255).round().to(torch.uint8)

    with torch.no_grad():
        assert ops.sr_tail_u8_eligible(conv, x)
        ga, oa = capture(fused)
        gb, ob = capture(composed)
        t = {"fused": [], "composed": []}
        time_replays(ga, 3)
        time_replays(gb, 3)
        for _ in range(rounds):
            t["fused"].append(time_replays(ga, reps))
            t["composed"].append(time_replays(gb, reps))
        diff = (oa.permute(0, 3, 1, 2).int() - ob.int()).abs()
    nbytes = n * (h * w * 128 + oh * ow * 3 + (h // s) * (w // s) * 12)
    floor_us = nbytes / HBM_BPS * 1e6
    fa, fb = statistics.median(t["fused"]), statistics.median(t["composed"])
    return {
        "shape": {"images": n, "features": [64, h, w], "out": [oh, ow, 3], "scale": s},
        "us_per_frame": {"fused": fa, "composed": fb}, "us_per_image": {"fused": fa / n, "composed": fb / n},
        "rounds_us_per_frame": t, "replays_per_round": reps,
        "hbm_bytes": nbytes, "hbm_floor_us_at_7.7TBps": floor_us, "fused_fraction_of_hbm_floor": floor_us / fa,
        "speedup": fb / fa, "max_level_diff_vs_composed": diff.max().item(),
        "fraction_differing_vs_composed": (diff > 0).double().mean().item(),
    }


def e2e(dev, rounds, steps):
    clips, t, h, w = 8, 30, 270, 480
    net = EAVSRP(4).eval()
    seeded_parameters(net)
    net = net.to(dev).prepare(torch.bfloat16)
    f32 = torch.cat([clip_inputs(1, t, h, w, seed=1234 + i) for i in range(clips)])
    u8 = (f32 * 255).round().to(torch.uint8)
    host_f32 = (u8.float() / 255).pin_memory()                     # the same frames in both arms
    host_u8 = u8.permute(0, 1, 3, 4, 2).contiguous().pin_memory()
    out_bench = torch.empty((clips, t, 3, 4 * h, 4 * w), dtype=torch.uint8).pin_memory()
    out_u8 = torch.empty((clips, t, 4 * h, 4 * w, 3), dtype=torch.uint8).pin_memory()
    static_f32 = pad_clip(host_f32.to(dev))
    static_u8 = host_u8.to(dev)

    def bench_dev():
        sr = net(static_f32)[..., :4 * h, :4 * w]
        return torch.clamp(sr.float() * 255, 0, 255).round().to(torch.uint8)

    with torch.no_grad():
        ga, va = capture(bench_dev)
        # one memory pool for both graphs: they never run concurrently and their outputs stay referenced
        gb, vb = capture(lambda: net.forward_uint8(static_u8), pool=ga.pool())

    def step_bench():
        static_f32.copy_(pad_clip(host_f32.to(dev, non_blocking=True)))
        ga.replay()
        out_bench.copy_(va, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def step_u8():
        static_u8.copy_(host_u8, non_blocking=True)
        gb.replay()
        out_u8.copy_(vb, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    res = {"bench_recipe": [], "forward_uint8": []}
    step_bench()
    step_u8()
    for _ in range(rounds):
        for name, fn in (("bench_recipe", step_bench), ("forward_uint8", step_u8)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            res[name].append(clips * t * steps / (time.perf_counter() - t0))
    ndiff, maxdiff = 0, 0
    for i in range(clips):                              # clip by clip: the whole batch is 1.5 G values
        d = (vb[i].permute(0, 3, 1, 2).int() - va[i].int()).abs()
        ndiff, maxdiff = ndiff + int((d > 0).sum()), max(maxdiff, d.max().item())
    return {
        "clips": clips, "frames_per_clip": t, "lr": [h, w], "out": [4 * h, 4 * w, 3], "steps_per_round": steps,
        "frames_per_s": {k: statistics.median(v) for k, v in res.items()}, "rounds_frames_per_s": res,
        "h2d_bytes": {"bench_recipe": host_f32.numel() * 4, "forward_uint8": host_u8.numel()},
        "d2h_bytes": {"bench_recipe": out_bench.numel(), "forward_uint8": out_u8.numel()},
        "max_level_diff": maxdiff, "fraction_differing": ndiff / va.numel(),
    }


def tail_yuv(dev, rounds, reps):
    conv, x, lr, (n, h, w, s, oh, ow) = _tail_operands(dev)
    kr, kb = MATRICES["bt709"]
    rgb = torch.empty((n, oh, ow, 3), dtype=torch.uint8, device=dev)
    planes = (torch.empty((n, oh, ow), dtype=torch.uint8, device=dev),
              torch.empty((n, oh // 2, ow // 2), dtype=torch.uint8, device=dev),
              torch.empty((n, oh // 2, ow // 2), dtype=torch.uint8, device=dev))

    arms = {
        "yuv420_kernel": lambda: ops.sr_tail_yuv420(conv, x, lr, s, *planes, oh, ow, kr, kb),
        "rgb_kernel": lambda: ops.sr_tail_u8(conv, x, lr, s, rgb, oh, ow),
        "composed_yuv420": lambda: rgb_to_yuv420(
            (conv(x).float() + F.interpolate(lr, scale_factor=s, mode="bilinear", align_corners=False))[..., :oh, :ow],
            kr, kb),
    }
    with torch.no_grad():
        assert ops.sr_tail_u8_eligible(conv, x)
        graphs = {k: capture(fn) for k, fn in arms.items()}
        t = {k: [] for k in arms}
        for g, _ in graphs.values():
            time_replays(g, 3)
        for _ in range(rounds):
            for k, (g, _) in graphs.items():
                t[k].append(time_replays(g, reps))
        diffs = [(a.int() - b.int()).abs() for a, b in zip(graphs["yuv420_kernel"][1], graphs["composed_yuv420"][1])]
    lr_bytes = (h // s) * (w // s) * 12
    nbytes = {"yuv420": n * (h * w * 128 + oh * ow * 3 // 2 + lr_bytes), "rgb": n * (h * w * 128 + oh * ow * 3 + lr_bytes)}
    med = {k: statistics.median(v) for k, v in t.items()}
    floor = {k: v / HBM_BPS * 1e6 for k, v in nbytes.items()}
    return {
        "shape": {"images": n, "features": [64, h, w], "out": [oh, ow], "scale": s, "matrix": "bt709"},
        "us_per_frame": med, "us_per_image": {k: v / n for k, v in med.items()},
        "rounds_us_per_frame": t, "replays_per_round": reps,
        "hbm_bytes": nbytes, "hbm_floor_us_at_7.7TBps": floor,
        "fraction_of_hbm_floor": {"yuv420_kernel": floor["yuv420"] / med["yuv420_kernel"],
                                  "rgb_kernel": floor["rgb"] / med["rgb_kernel"],
                                  "composed_yuv420": floor["yuv420"] / med["composed_yuv420"]},
        "yuv420_kernel_over_rgb_kernel": med["yuv420_kernel"] / med["rgb_kernel"],
        "composed_over_yuv420_kernel": med["composed_yuv420"] / med["yuv420_kernel"],
        "max_level_diff_vs_composed": {p: d.max().item() for p, d in zip("YUV", diffs)},
        "fraction_differing_vs_composed": {p: (d > 0).double().mean().item() for p, d in zip("YUV", diffs)},
    }


def e2e_yuv(dev, rounds, steps):
    clips, t, h, w = 8, 30, 270, 480
    kr, kb = MATRICES["bt709"]
    net = EAVSRP(4).eval()
    seeded_parameters(net)
    net = net.to(dev).prepare(torch.bfloat16)
    f32 = torch.cat([clip_inputs(1, t, h, w, seed=1234 + i) for i in range(clips)])
    host_u8 = (f32 * 255).round().to(torch.uint8).permute(0, 1, 3, 4, 2).contiguous().pin_memory()
    host_yuv = [p.contiguous().pin_memory() for p in rgb_to_yuv420(f32, kr, kb)]
    out_u8 = torch.empty((clips, t, 4 * h, 4 * w, 3), dtype=torch.uint8).pin_memory()
    out_yuv = [torch.empty((clips, t, 4 * h, 4 * w), dtype=torch.uint8).pin_memory()] + [
        torch.empty((clips, t, 2 * h, 2 * w), dtype=torch.uint8).pin_memory() for _ in range(2)]
    static_u8 = host_u8.to(dev)
    static_yuv = [p.to(dev) for p in host_yuv]

    with torch.no_grad():
        ga, va = capture(lambda: net.forward_uint8(static_u8))
        gb, vb = capture(lambda: net.forward_yuv420(*static_yuv), pool=ga.pool())
        # the ingest of each arm alone, as the graphs run it
        gi_yuv, _ = capture(lambda: pad_clip(yuv420_to_rgb(*static_yuv, kr, kb)))
        gi_u8, _ = capture(lambda: pad_clip(static_u8.permute(0, 1, 4, 2, 3).float().div(255).contiguous()))

    def step_u8():
        static_u8.copy_(host_u8, non_blocking=True)
        ga.replay()
        out_u8.copy_(va, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def step_yuv():
        for d, hst in zip(static_yuv, host_yuv):
            d.copy_(hst, non_blocking=True)
        gb.replay()
        for hst, d in zip(out_yuv, vb):
            hst.copy_(d, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    res = {"forward_uint8": [], "forward_yuv420": []}
    ingest = {"yuv420_to_rgb": [], "uint8_rgb": []}
    step_u8()
    step_yuv()
    time_replays(gi_yuv, 3)
    time_replays(gi_u8, 3)
    for _ in range(rounds):
        for name, fn in (("forward_uint8", step_u8), ("forward_yuv420", step_yuv)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            res[name].append(clips * t * steps / (time.perf_counter() - t0))
        ingest["yuv420_to_rgb"].append(time_replays(gi_yuv, 10))
        ingest["uint8_rgb"].append(time_replays(gi_u8, 10))
    fps = {k: statistics.median(v) for k, v in res.items()}
    ing = {k: statistics.median(v) for k, v in ingest.items()}

    # what a user of forward_uint8 otherwise spends on the host: its RGB output of one clip -> I420 with torch on
    # the CPU (timed on clip 0, scaled to the step's 8 clips)
    cpu_s = []
    for _ in range(3):
        t0 = time.perf_counter()
        rgb_to_yuv420(out_u8[0].permute(0, 3, 1, 2).float().div(255), kr, kb)
        cpu_s.append(time.perf_counter() - t0)
    return {
        "clips": clips, "frames_per_clip": t, "lr": [h, w], "out": [4 * h, 4 * w], "steps_per_round": steps,
        "matrix": "bt709", "frames_per_s": fps, "rounds_frames_per_s": res,
        "h2d_bytes": {"forward_uint8": host_u8.numel(), "forward_yuv420": sum(p.numel() for p in host_yuv)},
        "d2h_bytes": {"forward_uint8": out_u8.numel(), "forward_yuv420": sum(p.numel() for p in out_yuv)},
        "ingest_device_us_per_step": ing, "rounds_ingest_device_us_per_step": ingest,
        "ingest_share_of_yuv_step": ing["yuv420_to_rgb"] * 1e-6 / (clips * t / fps["forward_yuv420"]),
        "host_cpu_i420_conversion": {
            "torch_threads": torch.get_num_threads(), "frames_timed": t, "s_per_clip_runs": cpu_s,
            "s_per_step_scaled_from_one_clip": statistics.median(cpu_s) * clips},
    }


def tail_hbd(dev, rounds, reps):
    conv, x, lr, (n, h, w, s, oh, ow) = _tail_operands(dev)
    kr, kb = MATRICES["bt709"]
    u8 = lambda *shape: torch.empty(shape, dtype=torch.uint8, device=dev)      # noqa: E731
    u16 = lambda *shape: torch.empty(shape, dtype=torch.uint16, device=dev)    # noqa: E731
    rgb8, rgb16 = u8(n, oh, ow, 3), u16(n, oh, ow, 3)
    i420 = (u8(n, oh, ow), u8(n, oh // 2, ow // 2), u8(n, oh // 2, ow // 2))
    y10, uv10 = u16(n, oh, ow), u16(n, oh // 2, ow)
    arms = {
        "rgb16_kernel": lambda: ops.sr_tail_u16(conv, x, lr, s, rgb16, oh, ow, 16),
        "p010_kernel": lambda: ops.sr_tail_yuv420_u16(conv, x, lr, s, y10, uv10[..., 0::2], uv10[..., 1::2], oh, ow,
                                                      kr, kb, 10, 6),
        "rgb_kernel": lambda: ops.sr_tail_u8(conv, x, lr, s, rgb8, oh, ow),
        "yuv420_kernel": lambda: ops.sr_tail_yuv420(conv, x, lr, s, *i420, oh, ow, kr, kb),
    }
    with torch.no_grad():
        assert ops.sr_tail_u8_eligible(conv, x)
        graphs = {k: capture(fn) for k, fn in arms.items()}
        t = {k: [] for k in arms}
        for g, _ in graphs.values():
            time_replays(g, 3)
        for _ in range(rounds):
            for k, (g, _) in graphs.items():
                t[k].append(time_replays(g, reps))
        # the 16-bit codes against the 8-bit kernels' outputs, rescaled: at most half an 8-bit level apart
        d_rgb = (rgb16.int().double() * (255 / 65535) - rgb8.int().double()).abs().max().item()
        d_y = ((y10.int() >> 6).double() / 4 - i420[0].int().double()).abs().max().item()
    lr_bytes = (h // s) * (w // s) * 12
    written = {"rgb16_kernel": 6, "p010_kernel": 3, "rgb_kernel": 3, "yuv420_kernel": 1.5}
    nbytes = {k: n * (h * w * 128 + int(oh * ow * b) + lr_bytes) for k, b in written.items()}
    med = {k: statistics.median(v) for k, v in t.items()}
    floor = {k: v / HBM_BPS * 1e6 for k, v in nbytes.items()}
    return {
        "shape": {"images": n, "features": [64, h, w], "out": [oh, ow], "scale": s, "matrix": "bt709"},
        "us_per_frame": med, "us_per_image": {k: v / n for k, v in med.items()},
        "rounds_us_per_frame": t, "replays_per_round": reps, "bytes_written_per_px": written,
        "hbm_bytes": nbytes, "hbm_floor_us_at_7.7TBps": floor,
        "fraction_of_hbm_floor": {k: floor[k] / med[k] for k in med},
        "rgb16_over_rgb8": med["rgb16_kernel"] / med["rgb_kernel"],
        "p010_over_yuv420_8bit": med["p010_kernel"] / med["yuv420_kernel"],
        "max_abs_diff_in_8bit_levels": {"rgb16_vs_rgb8": d_rgb, "y10_vs_y8": d_y},
    }


def e2e_hbd(dev, rounds, steps):
    clips, t, h, w = 8, 30, 270, 480
    kr, kb = MATRICES["bt709"]
    net = EAVSRP(4).eval()
    seeded_parameters(net)
    net = net.to(dev).prepare(torch.bfloat16)
    f32 = torch.cat([clip_inputs(1, t, h, w, seed=1234 + i) for i in range(clips)])
    host_i420 = [p.contiguous().pin_memory() for p in rgb_to_yuv420(f32, kr, kb)]
    y, u, v = rgb_to_yuv420(f32, kr, kb, bits=10, shift=6)
    host_p010 = [y.contiguous().pin_memory(),
                 torch.stack([u.int(), v.int()], -1).to(torch.uint16).view(clips, t, h // 2, w).pin_memory()]
    out_i420 = [torch.empty((clips, t, 4 * h, 4 * w), dtype=torch.uint8).pin_memory()] + [
        torch.empty((clips, t, 2 * h, 2 * w), dtype=torch.uint8).pin_memory() for _ in range(2)]
    out_p010 = [torch.empty((clips, t, 4 * h, 4 * w), dtype=torch.uint16).pin_memory(),
                torch.empty((clips, t, 2 * h, 4 * w), dtype=torch.uint16).pin_memory()]
    static_i420 = [p.to(dev) for p in host_i420]
    static_p010 = [p.to(dev) for p in host_p010]
    dev_p010 = [torch.empty(p.shape, dtype=torch.uint16, device=dev) for p in out_p010]
    out_views = (dev_p010[0], dev_p010[1][..., 0::2], dev_p010[1][..., 1::2])

    with torch.no_grad():
        ga, va = capture(lambda: net.forward_yuv420(*static_i420))
        gb, _ = capture(lambda: net.forward_yuv420_u16(static_p010[0], static_p010[1][..., 0::2],
                                                       static_p010[1][..., 1::2], bits=10, shift=6, out=out_views),
                        pool=ga.pool())

    def step_i420():
        for d, hst in zip(static_i420, host_i420):
            d.copy_(hst, non_blocking=True)
        ga.replay()
        for hst, d in zip(out_i420, va):
            hst.copy_(d, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def step_p010():
        for d, hst in zip(static_p010, host_p010):
            d.copy_(hst, non_blocking=True)
        gb.replay()
        for hst, d in zip(out_p010, dev_p010):
            hst.copy_(d, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    res = {"forward_yuv420": [], "forward_yuv420_u16_p010": []}
    step_i420()
    step_p010()
    for _ in range(rounds):
        for name, fn in (("forward_yuv420", step_i420), ("forward_yuv420_u16_p010", step_p010)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            res[name].append(clips * t * steps / (time.perf_counter() - t0))
    # the P010 luma against the 8-bit luma of the same clips, rescaled (codes, in 8-bit levels), clip 0
    d_y = ((out_p010[0][0].int() >> 6).double() / 4 - out_i420[0][0].int().double()).abs()
    return {
        "clips": clips, "frames_per_clip": t, "lr": [h, w], "out": [4 * h, 4 * w], "steps_per_round": steps,
        "matrix": "bt709", "frames_per_s": {k: statistics.median(v) for k, v in res.items()},
        "rounds_frames_per_s": res,
        "h2d_bytes": {"forward_yuv420": sum(p.numel() for p in host_i420),
                      "forward_yuv420_u16_p010": sum(p.numel() * 2 for p in host_p010)},
        "d2h_bytes": {"forward_yuv420": sum(p.numel() for p in out_i420),
                      "forward_yuv420_u16_p010": sum(p.numel() * 2 for p in out_p010)},
        "luma_p010_vs_i420_clip0_8bit_levels": {"max": d_y.max().item(), "mean": d_y.mean().item()},
    }


def tail_psnr(dev, rounds, reps):
    conv, x, lr, (n, h, w, s, oh, ow) = _tail_operands(dev)
    hr = torch.randint(0, 256, (n, oh, ow, 3), dtype=torch.uint8, device=dev)
    rgb, rgb2 = (torch.empty((n, oh, ow, 3), dtype=torch.uint8, device=dev) for _ in range(2))
    sums, sums2 = (torch.zeros(n, dtype=torch.int64, device=dev) for _ in range(2))

    def composed():
        ops.sr_tail_u8(conv, x, lr, s, rgb, oh, ow)
        d = rgb.int() - hr.int()
        return (d * d).sum((1, 2, 3), dtype=torch.int64)

    arms = {
        "rgb_kernel": lambda: ops.sr_tail_u8(conv, x, lr, s, rgb, oh, ow),
        # the sums grow over the replays; the caller's zeroing (one memset per clip) is not part of the kernel
        "sse_kernel": lambda: ops.sr_tail_u8_sse(conv, x, lr, s, hr, sums, oh, ow),
        "sse_store_kernel": lambda: ops.sr_tail_u8_sse(conv, x, lr, s, hr, sums2, oh, ow, out=rgb2),
        "composed_sse": composed,
    }
    with torch.no_grad():
        assert ops.sr_tail_u8_eligible(conv, x)
        graphs = {k: capture(fn) for k, fn in arms.items()}
        t = {k: [] for k in arms}
        for g, _ in graphs.values():
            time_replays(g, 3)
        for _ in range(rounds):
            for k, (g, _) in graphs.items():
                t[k].append(time_replays(g, reps))
        # one more call of each on zeroed sums, against the composition's result
        sums.zero_()
        sums2.zero_()
        ops.sr_tail_u8_sse(conv, x, lr, s, hr, sums, oh, ow)
        ops.sr_tail_u8_sse(conv, x, lr, s, hr, sums2, oh, ow, out=rgb2)
        want = composed()
        exact = {"sse_kernel": torch.equal(sums, want), "sse_store_kernel": torch.equal(sums2, want),
                 "stored_frames_equal_rgb_kernel": torch.equal(rgb2, rgb)}
    lr_bytes = (h // s) * (w // s) * 12
    # per output pixel: ground truth read + frame written (the composition adds its int64 reduction's traffic on top)
    moved = {"rgb_kernel": 3, "sse_kernel": 3, "sse_store_kernel": 6, "composed_sse": 6}
    nbytes = {k: n * (h * w * 128 + oh * ow * b + lr_bytes) for k, b in moved.items()}
    med = {k: statistics.median(v) for k, v in t.items()}
    floor = {k: v / HBM_BPS * 1e6 for k, v in nbytes.items()}
    return {
        "shape": {"images": n, "features": [64, h, w], "out": [oh, ow, 3], "scale": s},
        "us_per_frame": med, "us_per_image": {k: v / n for k, v in med.items()},
        "rounds_us_per_frame": t, "replays_per_round": reps, "frame_bytes_per_px": moved,
        "hbm_bytes": nbytes, "hbm_floor_us_at_7.7TBps": floor,
        "fraction_of_hbm_floor": {k: floor[k] / med[k] for k in med},
        "over_rgb_kernel": {k: med[k] / med["rgb_kernel"] for k in med},
        "sse_equal_to_composed": exact, "sse_per_image": want.tolist(),
    }


def e2e_psnr(dev, rounds, steps):
    clips, t, h, w = 8, 30, 270, 480
    net = EAVSRP(4).eval()
    seeded_parameters(net)
    net = net.to(dev).prepare(torch.bfloat16)
    # the LR clips of the other arms; as ground truth, their bicubic x4 upsampling (the throughput does not depend on
    # what the frames show)
    f32 = torch.cat([clip_inputs(1, t, h, w, seed=1234 + i) for i in range(clips)])
    host_u8 = (f32 * 255).round().to(torch.uint8).permute(0, 1, 3, 4, 2).contiguous().pin_memory()
    host_hr = torch.empty((clips, t, 4 * h, 4 * w, 3), dtype=torch.uint8).pin_memory()
    for i in range(clips):
        up = F.interpolate(f32[i].to(dev), scale_factor=4, mode="bicubic", align_corners=False)
        host_hr[i] = (up.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).cpu()
    out_u8 = torch.empty((clips, t, 4 * h, 4 * w, 3), dtype=torch.uint8).pin_memory()
    out_sse = [torch.empty((clips, t), dtype=torch.int64).pin_memory() for _ in range(2)]
    out_psnr = torch.empty((clips, t), dtype=torch.float64).pin_memory()
    static_u8, static_hr = host_u8.to(dev), host_hr.to(dev)

    def forward_and_sse():
        sr = net.forward_uint8(static_u8)
        return sr, (sr.int() - static_hr.int()).pow(2).sum((2, 3, 4), dtype=torch.int64)

    with torch.no_grad():
        ga, (pa, sa) = capture(lambda: net.psnr_uint8(static_u8, static_hr))
        gb, (vb, sb) = capture(forward_and_sse, pool=ga.pool())

    def step_psnr():
        static_u8.copy_(host_u8, non_blocking=True)
        static_hr.copy_(host_hr, non_blocking=True)
        ga.replay()
        out_psnr.copy_(pa, non_blocking=True)
        out_sse[0].copy_(sa, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def step_forward():
        static_u8.copy_(host_u8, non_blocking=True)
        static_hr.copy_(host_hr, non_blocking=True)
        gb.replay()
        out_u8.copy_(vb, non_blocking=True)
        out_sse[1].copy_(sb, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    res = {"psnr_uint8": [], "forward_uint8_torch_sse": []}
    step_psnr()
    step_forward()
    for _ in range(rounds):
        for name, fn in (("psnr_uint8", step_psnr), ("forward_uint8_torch_sse", step_forward)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            res[name].append(clips * t * steps / (time.perf_counter() - t0))
    # two runs of the trunk agree to rounding only (float atomics, DESIGN.md 4): the sums of the two arms differ by
    # the few codes that moved by one level
    rel = ((out_sse[0] - out_sse[1]).abs().double() / out_sse[1].double()).max().item()
    return {
        "clips": clips, "frames_per_clip": t, "lr": [h, w], "out": [4 * h, 4 * w, 3], "steps_per_round": steps,
        "frames_per_s": {k: statistics.median(v) for k, v in res.items()}, "rounds_frames_per_s": res,
        "h2d_bytes": {k: host_u8.numel() + host_hr.numel() for k in res},
        "d2h_bytes": {"psnr_uint8": out_psnr.numel() * 8 + out_sse[0].numel() * 8,
                      "forward_uint8_torch_sse": out_u8.numel() + out_sse[1].numel() * 8},
        "mean_psnr_db": out_psnr.mean().item(), "max_relative_sse_difference_between_arms": rel,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--yuv", action="store_true", help="measure the Y'CbCr 4:2:0 tail instead (sr_tail_yuv.json)")
    ap.add_argument("--hbd", action="store_true", help="measure the 16-bit RGB and P010 tails (sr_tail_hbd.json)")
    ap.add_argument("--psnr", action="store_true", help="measure the squared-error tail and psnr_uint8 (sr_tail_psnr.json)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_sr_tail.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.benchmark = False
    result = {"gpu": gpu_info(), "torch": torch.__version__}
    if args.yuv or args.hbd or args.psnr:
        name, tail_fn, e2e_fn = (("sr_tail_psnr", tail_psnr, e2e_psnr) if args.psnr else
                                 ("sr_tail_hbd", tail_hbd, e2e_hbd) if args.hbd else ("sr_tail_yuv", tail_yuv, e2e_yuv))
        result["tail"] = tail_fn(dev, args.rounds, args.reps)
        print(json.dumps(result["tail"], indent=1), flush=True)
        torch.cuda.empty_cache()
        result["e2e"] = e2e_fn(dev, args.rounds, args.steps)
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, name + ".json"), "w") as f:
            json.dump(result, f, indent=1)
        print(json.dumps(result, indent=1))
        return
    result["tail"] = tail(dev, args.rounds, args.reps)
    print(json.dumps(result["tail"], indent=1), flush=True)
    torch.cuda.empty_cache()
    result["e2e"] = e2e(dev, args.rounds, args.steps)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "sr_tail.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
