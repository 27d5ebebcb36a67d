#!/usr/bin/env python
"""Measure the uint8 reconstruction tail on the GPU and write one JSON file.

    python tools/prof_sr_tail.py --out DIR [--rounds 5]

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


def tail(dev, rounds, reps):
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_sr_tail.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.benchmark = False
    result = {"gpu": gpu_info(), "torch": torch.__version__}
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
