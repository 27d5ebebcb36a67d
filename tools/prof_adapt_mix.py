#!/usr/bin/env python
"""Time `ops.adapt_mix` at the three resolutions the benchmark runs it at and write one JSON file.

    python tools/prof_adapt_mix.py --out DIR [--dtype bf16|f32] [--label NAME]   -> DIR/adapt_mix[_NAME].json
    python tools/prof_adapt_mix.py --dump DIR       (seeded outputs at the timed and the test shapes, bf16 and fp32)
    python tools/prof_adapt_mix.py --compare DIR_A DIR_B                      (torch.equal of two dumps)

Shapes: 8 images of 64 x 272 x 480 (flow_l1 / adastn of MultiAdSTN at full resolution), 64 x 136 x 240 and
64 x 68 x 120 (the half- and quarter-resolution levels).  Each shape is one CUDA graph of `k` calls on `k` distinct
(a, b, out) sets, with k chosen so that the sets span more than 300 MB (L2 is 126 MB), so every call reads its inputs
from HBM.  CUDA events time `--reps` replays after a warm-up; the median of `--rounds` is reported as us per call.
Floors: the HBM floor counts a and b read once and out written once (3 x 64 channels per pixel, 384 B/px in bf16) at
7.7 TB/s; the FMA floor counts the 2 304 useful multiply-adds per output pixel (9 x 128 depthwise + 9 x 2 x 64
grouped) at 148 SMs x 128 lanes x the maximum SM clock.  The library comes from EAVSR_B200_LIB when it is set, so
two builds can be alternated in one session.  GPU name, power limit and maximum SM clock are read with nvidia-smi.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from eavsr_b200 import ops  # noqa: E402

HBM_BPS = 7.7e12
SHAPES = [(8, 272, 480), (8, 136, 240), (8, 68, 120)]
TEST_SHAPES = [(1, 17, 23), (2, 8, 16), (1, 67, 120), (1, 5, 3), (3, 1, 1), (2, 9, 33)]
FMA_PER_PX = 9 * 128 + 9 * 2 * 64
DTYPES = {"bf16": torch.bfloat16, "f32": torch.float32}


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True, check=True)
    keys = [k.strip() for k in r.stdout.splitlines()[0].split(",")]
    vals = [v.strip() for v in r.stdout.splitlines()[1].split(",")]
    return dict(zip(keys, vals))


def operands(n, h, w, dtype, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    mk = lambda *s: torch.randn(*s, generator=g, device=dev)                      # noqa: E731
    a = mk(n, 64, h, w).to(dtype).contiguous(memory_format=torch.channels_last)
    b = mk(n, 64, h, w).to(dtype).contiguous(memory_format=torch.channels_last)
    params = (mk(128, 1, 3, 3) * 0.3, mk(128) * 0.1, mk(64, 2, 3, 3) * 0.3, mk(64) * 0.1)
    return a, b, [p.to(dtype) for p in params]


def time_shape(n, h, w, dtype, reps, rounds, dev):
    es = torch.finfo(dtype).bits // 8
    per_call = 3 * n * 64 * h * w * es
    k = max(2, math.ceil(300e6 / per_call))
    sets = [operands(n, h, w, dtype, 100 + i, dev) for i in range(k)]
    outs = [None] * k

    def calls():
        for i, (a, b, p) in enumerate(sets):
            outs[i] = ops.adapt_mix(a, b, *p, 0.2)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        calls()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        calls()
    for _ in range(3):
        g.replay()
    times = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3 / (reps * k))
    return k, per_call, times


def dump(path, dev):
    os.makedirs(path, exist_ok=True)
    for name, dtype in DTYPES.items():
        for n, h, w in SHAPES + TEST_SHAPES:
            a, b, p = operands(n, h, w, dtype, 7, dev)
            torch.save(ops.adapt_mix(a, b, *p, 0.2).cpu(), os.path.join(path, f"{name}_{n}x{h}x{w}.pt"))


def compare(pa, pb):
    res = {}
    for f in sorted(os.listdir(pa)):
        x, y = torch.load(os.path.join(pa, f)), torch.load(os.path.join(pb, f))
        res[f] = {"equal": bool(torch.equal(x, y)), "differing": int((x != y).sum())}
    return {"all_equal": all(v["equal"] for v in res.values()), "tensors": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--label", default="")
    ap.add_argument("--dtype", default="bf16", choices=sorted(DTYPES))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--dump")
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        print(json.dumps(compare(*args.compare)))
        return
    if not torch.cuda.is_available():
        sys.exit("prof_adapt_mix: needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False
    if args.dump:
        with torch.no_grad():
            dump(args.dump, dev)
        return
    info = gpu_info()
    clk = float(info["clocks.max.sm [MHz]"].split()[0]) * 1e6
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    dtype = DTYPES[args.dtype]
    rows = []
    with torch.no_grad():
        for n, h, w in SHAPES:
            k, per_call, times = time_shape(n, h, w, dtype, args.reps, args.rounds, dev)
            us = statistics.median(times)
            hbm_us = per_call / HBM_BPS * 1e6
            fma_us = n * h * w * FMA_PER_PX / (sms * 128 * clk) * 1e6
            rows.append({"shape": [n, 64, h, w], "us_per_call": round(us, 2), "rounds_us": [round(t, 2) for t in times],
                         "sets_rotated": k, "hbm_floor_us": round(hbm_us, 2), "fma_floor_us": round(fma_us, 2),
                         "frac_hbm_floor": round(hbm_us / us, 3), "frac_fma_floor": round(fma_us / us, 3)})
    # a MultiAdSTN call runs two full-resolution calls, one half and one quarter; a 30-frame step of 8 clips runs
    # 4 x (2 * 30 - 3) = 228 of them on 8 images each
    per_stn = 2 * rows[0]["us_per_call"] + rows[1]["us_per_call"] + rows[2]["us_per_call"]
    res = {"tool": "prof_adapt_mix", "label": args.label, "dtype": args.dtype, "gpu": info, "sms": sms,
           "lib": os.path.basename(os.environ.get("EAVSR_B200_LIB", "in-tree")), "shapes": rows,
           "us_per_multiadstn_8_images": round(per_stn, 1), "ms_per_30_frame_step_est": round(228 * per_stn / 1e3, 1)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        name = f"adapt_mix_{args.label}.json" if args.label else "adapt_mix.json"
        with open(os.path.join(args.out, name), "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
