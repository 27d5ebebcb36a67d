#!/usr/bin/env python
"""bench.py -- LR frames/s of EAVSR+ x4 on synthetic 270x480 clips (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload model|hotpath] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass over one synthetic 30-frame 270x480 LR clip per GPU:
  * workload "model"   : full EAVSR+ x4 forward (eavsr_b200.model.EAVSRP: SPyNet + encoder + 4
                         second-order propagation branches + upsampler) with the alignment hot path
                         (DCNv2 / flow_warp) on this repo's CUDA kernels, bf16 channels_last.
  * workload "hotpath" : only the alignment operators of that clip, in the model's call order and
                         shapes (228 DCNv2, 1140 64-ch warps, 112 2-ch warps, 12 border warps).
Clips are independent, so N GPUs run N clips per step with no collective (scaling = weak); the only
torch.distributed traffic is the timing barrier and the max-over-ranks of the elapsed time.

The JSON line carries `roofline` for the dominant hot-path kernel (tcgen05 DCNv2 forward), timed
live with CUDA events, `cpu_baseline` (the oracle port timed on the host cores on a bounded
sample) and `e2e` (host buffers in, host buffers out, copies inside the timed region).
`--impl reference` times the CPU oracle port of the same workload (the reference's own
`--gpu_ids -1` path needs the reference's source tree and mmcv, which this project does not ship).
`--dump-outputs DIR` (e.g. `bench_outputs`) writes what the last timed step returned as DIR/<name>.npy (see
`dump_outputs`), so that two builds of the project can be compared output for output on the same seeded inputs.
Compare with a tolerance: the channel-attention sums are accumulated with floating-point atomics, so two runs
of the same build agree to rounding, not bit for bit.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

T_FRAMES = 30
LR_H, LR_W = 270, 480
PAD_H = 272   # the reference's 3-level pyramid needs H, W % 4 == 0 (SURVEY.md F4): replicate-pad 270 -> 272
METRIC = "LR frames/s, EAVSR+ x4, 270x480"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.2] or [r for _, r in self.rows]
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
class HotpathWorkload:
    """The alignment operators of one 30-frame clip, in the model's order and shapes
    (SURVEY.md 3.2: 4 branches x (2T-3) MultiAdSTN calls = 5 warps + 1 DCN each; T-2 flow
    compositions per branch; 6-level SPyNet border warps for both directions)."""
    name = "eavsrp_x4_alignment_hotpath_30x272x480_bf16"
    # step() returns the last DCNv2 output of the clip, so --dump-outputs covers only that one call: the warps and
    # flow compositions of the step, and the other 227 DCNv2 calls, leave nothing that is compared
    output_name = "dcn_out"

    def __init__(self, device, dtype=torch.bfloat16, t=T_FRAMES, h=PAD_H, w=LR_W, dg=8):
        import eavsr_b200 as E
        self.E, self.t, self.h, self.w, self.dg, self.dtype = E, t, h, w, dg, dtype
        g = torch.Generator(device="cpu").manual_seed(1234)

        def feat(hh, ww, n=3):
            return [torch.randn(1, 64, hh, ww, generator=g).to(device, dtype).contiguous(
                memory_format=torch.channels_last) for _ in range(n)]

        def flow(hh, ww, n=3, sigma=2.0):
            return [(torch.randn(1, 2, hh, ww, generator=g) * sigma).to(device) for _ in range(n)]

        self.f1, self.f2, self.f4 = feat(h, w, 6), feat(h // 2, w // 2), feat(h // 4, w // 4)
        self.fl1, self.fl2, self.fl4 = flow(h, w), flow(h // 2, w // 2, sigma=1.0), flow(h // 4, w // 4, sigma=0.5)
        # offsets / masks pool larger than L2 (3 x 112 MB) so consecutive DCN calls stream from HBM
        self.off = [(torch.randn(1, dg * 18, h, w, generator=g) * 2).clamp(-12, 12).to(device) for _ in range(3)]
        self.msk = [torch.sigmoid(torch.randn(1, dg * 9, h, w, generator=g)).to(device) for _ in range(3)]
        self.weight = ((torch.rand(64, 64, 3, 3, generator=g) * 2 - 1) / 24).to(device, dtype)
        self.bias = torch.zeros(64, device=device, dtype=dtype)
        self.flow2 = [torch.randn(1, 2, h, w, generator=g).to(device) for _ in range(2)]
        self.flow2_nhw2 = [f.permute(0, 2, 3, 1).contiguous() for f in self.fl1]
        self.img = [torch.rand(t - 1, 3, 288 >> i, 480 >> i, generator=g).to(device) for i in range(6)]
        self.imgflow = [(torch.randn(t - 1, 288 >> i, 480 >> i, 2, generator=g)).to(device) for i in range(6)]
        self.frames_per_step = t
        self.h2d_bytes = self.d2h_bytes = 0
        self.launches_per_step = None

    def step(self):
        E, t = self.E, self.t
        k = 0
        out = None
        for _branch in range(4):
            for i in range(1, t):
                for order in (1, 2):
                    if order == 2 and i < 2:
                        continue
                    if order == 2:
                        E.flow_warp_nhw2(self.flow2[k % 2], self.flow2_nhw2[k % 3])
                    E.flow_warp(self.f4[k % 3], self.fl4[k % 3])
                    E.flow_warp(self.f2[k % 3], self.fl2[k % 3])
                    E.flow_warp(self.f1[k % 6], self.fl1[k % 3])
                    E.flow_warp(self.f1[(k + 1) % 6], self.fl1[(k + 1) % 3])
                    feat = E.flow_warp(self.f1[(k + 2) % 6], self.fl1[(k + 1) % 3])
                    out = E.modulated_deform_conv2d(feat, self.off[k % 3], self.msk[k % 3], self.weight, self.bias,
                                                    1, 1, 1, 1, self.dg)
                    k += 1
        for _direction in range(2):
            for lvl in range(6):
                E.flow_warp_nhw2(self.img[lvl], self.imgflow[lvl], padding_mode="border")
        return out

    def e2e_step(self):
        return None


NUM_CLIPS = 64      # BASELINE.json config 4: 64 synthetic 30-frame clips sharded over the GPUs


class ModelWorkload:
    """Full EAVSR+ x4 forward of one synthetic 30-frame 270x480 clip per step and GPU (BASELINE.json configs 3
    and 4).  The clip set is the 64 seeded clips of config 4 (`clip_inputs(seed=1234 + clip_id)`), sharded
    round-robin over the ranks by `eavsr_b200.clip_parallel.shard`; every step takes the next clip of this
    rank's shard (already resident in HBM for `step`, in pinned host memory for `e2e_step`).
    Seeded weights (all checkpoints are stripped from the reference), bf16 channels_last features,
    fp32 flows/offsets/masks; the clip is replicate-padded 270 -> 272 and the SR cropped back to
    1080x1920 (SURVEY.md F4).  The forward is captured once into a CUDA graph (the reference issues
    ~20k launches per clip from one Python thread) and replayed per step."""
    name = "eavsrp_x4_full_clip_30x270x480_bf16"
    output_name = "sr"              # step() returns the SR clips, (clips, 30, 3, 1080, 1920)

    def __init__(self, device, t=T_FRAMES, h=LR_H, w=LR_W, dtype=torch.bfloat16, graph=True, rank=0, world=1,
                 distinct=8, clips_per_step=1, streams=1, net=None):
        from eavsr_b200.clip_parallel import shard
        from eavsr_b200.model import EAVSRP, pad_clip
        from eavsr_b200.synthetic import clip_inputs, seeded_parameters
        self.device, self.t, self.h, self.w, self.cps = device, t, h, w, clips_per_step
        # `streams` > 1: the clips of a step run as independent forwards on that many CUDA streams (parallel branches
        # of the captured graph) instead of one batched forward: the tail of one clip's kernel overlaps the head of
        # the other's (every kernel here is a one-CTA-per-SM persistent grid of ~15 us)
        self.streams = max(1, min(streams, clips_per_step))
        assert clips_per_step % self.streams == 0
        if net is None:
            net = EAVSRP(4).eval()
            seeded_parameters(net)
            net = net.to(device).prepare(dtype)
        self.net = net
        if os.environ.get("EAVSR_BENCH_CHAIN", "1") != "1":     # A/B switch: one launch per convolution
            for m in self.net.modules():
                if hasattr(m, "chain"):
                    m.chain = False
        self.pad = lambda x: pad_clip(x, 4)
        # this rank's clips of the 64-clip set; `distinct` of them are materialised (47 MB each on the device)
        self.clip_ids = shard(NUM_CLIPS, rank, world)[:max(1, distinct) * clips_per_step]
        self.host_clips, self.dev_clips = [], []
        for j in range(0, len(self.clip_ids), clips_per_step):
            c = torch.cat([clip_inputs(1, t, h, w, seed=1234 + i) for i in self.clip_ids[j:j + clips_per_step]])
            self.host_clips.append(c.pin_memory())
            self.dev_clips.append(self.pad(c.to(device)))
        self.cursor = self.e2e_cursor = 0
        self.static_in = self.dev_clips[0].clone()
        self.frames_per_step = t * clips_per_step
        self.h2d_bytes = self.host_clips[0].numel() * 4
        self.host_out = torch.empty((clips_per_step, t, 3, 4 * h, 4 * w), dtype=torch.uint8).pin_memory()
        self.d2h_bytes = self.host_out.numel()
        self.graph = None
        self.launches_per_step = None
        self.use_graph = graph and os.environ.get("EAVSR_BENCH_GRAPH", "1") == "1"
        self.out = None
        self.last_clip = 0

    def _forward(self):
        if self.streams == 1:
            sr = self.net(self.static_in)
            return sr[..., : 4 * self.h, : 4 * self.w]
        cur = torch.cuda.current_stream()
        if not hasattr(self, "_side"):
            self._side = [torch.cuda.Stream() for _ in range(self.streams)]
        outs = []
        for st, part in zip(self._side, self.static_in.chunk(self.streams)):
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                outs.append(self.net(part)[..., : 4 * self.h, : 4 * self.w])
        for st in self._side:
            cur.wait_stream(st)
        return outs            # one SR tensor per stream (no concatenation copy inside the timed forward)

    def _replay(self):
        from eavsr_b200 import _lib
        if not self.use_graph:
            self.out = self._forward()
            return self.out
        if self.graph is None:
            torch.cuda.synchronize()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                l0 = _lib.launch_count()
                self._forward()                      # warm-up outside capture (cuDNN autotune, lazy init)
                self.launches_per_step = _lib.launch_count() - l0   # replayed as graph nodes every step
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.out = self._forward()
        self.graph.replay()
        return self.out

    def step(self):
        """Device-resident clip -> SR (device).  The 47 MB device-to-device copy into the graph's input
        buffer is part of the step."""
        self.last_clip = self.cursor % len(self.dev_clips)
        self.cursor += 1
        self.static_in.copy_(self.dev_clips[self.last_clip])
        return self._replay()

    def e2e_step(self):
        """Host clip in (pinned) -> H2D -> forward -> clamp*255 round (the reference's visuals,
        models/base_model.py:146-150) -> D2H uint8 frames."""
        self.last_clip = self.e2e_cursor % len(self.host_clips)
        self.e2e_cursor += 1
        self.static_in.copy_(self.pad(self.host_clips[self.last_clip].to(self.device, non_blocking=True)))
        sr = self._replay()
        parts = sr if isinstance(sr, list) else [sr]
        k = 0
        for part in parts:
            vis = torch.clamp(part.float() * 255, 0, 255).round().to(torch.uint8)
            self.host_out[k:k + vis.shape[0]].copy_(vis, non_blocking=True)
            k += vis.shape[0]
        torch.cuda.current_stream().synchronize()
        return self.host_out

    def parity(self):
        """What the timed path computes against the fp32 path of the same kernels (itself pinned to the
        reference's golden vectors at 64x64 and to the CPU oracle, tests/test_gpu_model.py), on the LAST
        TIMED CLIP, outside the timed region.  Errors are reported on the SR frames ([0,1] range; north_star
        bound 1e-2 for bf16), on the learned residual sr - bilinear(lr) -- the part the network actually
        computes -- and as the PSNR delta against the synthetic HR (bicubic x4 of the clip)."""
        import copy
        import torch.nn.functional as F
        self.static_in.copy_(self.dev_clips[self.last_clip])
        sr16 = self._replay()
        sr16 = (sr16[0] if isinstance(sr16, list) else sr16)[:1].float().clone()       # first clip of the step
        lr = self.dev_clips[self.last_clip][:1, ..., : self.h, : self.w]
        tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
        try:
            net32 = copy.deepcopy(self.net).float()
            net32.prepare(torch.float32)
            # the bf16 weights are the weights: the fp32 path runs on their exact values
            sr32 = net32(self.dev_clips[self.last_clip][:1])[..., : 4 * self.h, : 4 * self.w].float()
            del net32
        finally:
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
        n, t = lr.shape[:2]
        flat = lr.reshape(n * t, 3, self.h, self.w).float()
        base = F.interpolate(flat, scale_factor=4, mode="bilinear", align_corners=False).view_as(sr32)
        hr = F.interpolate(flat, scale_factor=4, mode="bicubic", align_corners=False).clamp(0, 1).view_as(sr32)
        r16, r32 = sr16 - base, sr32 - base
        vis = lambda x: torch.clamp(x * 255, 0, 255).round()                              # noqa: E731
        psnr = lambda a: (-10 * torch.log10(((vis(a) - vis(hr)) / 255).pow(2).mean())).item()   # noqa: E731
        rms32 = r32.pow(2).mean().sqrt().item()
        return {"against": "fp32 path of the same kernels on the timed clip (golden-pinned in tests/test_gpu_model.py)",
                "clip_id": int(self.clip_ids[self.last_clip * self.cps]),
                "sr_max_abs": round((sr16 - sr32).abs().max().item(), 6), "sr_max_abs_bound": 1e-2,
                "residual_rms": round(rms32, 6),
                "residual_rel_rms": round((r16 - r32).pow(2).mean().sqrt().item() / max(rms32, 1e-12), 5),
                "psnr_delta_db": round(abs(psnr(sr16) - psnr(sr32)), 5), "psnr_delta_bound_db": 0.01}


class TrainWorkload:
    """BASELINE config 5: one EAVSR+ x4 training step per step -- forward, L1 loss, backward through the DCNv2 /
    flow_warp kernels, Adam with the reference's two parameter groups (eavsr_b200.train.Trainer mirrors
    models/eavsrp_model.py:45-59,82-119) -- on 8 synthetic 15-frame 64x64 LR crops per GPU (train_x4.sh:17
    batch_size 8, patch_size 64), data-parallel over the ranks with NCCL DistributedDataParallel: the gradient
    all-reduce (12.28 M fp32 = 49.1 MB) is the collective.  bf16 = autocast with fp32 master weights."""
    name = "eavsrp_x4_train_step_8x15x64x64_bf16"
    output_name = "loss"            # step() returns the step's L1 loss

    def __init__(self, device, rank=0, world=1, batch=8, t=15, size=64, dtype=torch.bfloat16, distinct=4, pwc=False,
                 graph=False):
        import torch.nn.functional as F
        from eavsr_b200.model import EAVSRP
        from eavsr_b200.synthetic import clip_inputs, seeded_parameters
        from eavsr_b200.train import Trainer, trainable_bytes
        self.device, self.world, self.batch, self.t = device, world, batch, t
        net = EAVSRP(4)
        seeded_parameters(net)
        net = net.to(device).to(memory_format=torch.channels_last)
        pwcnet = None
        if pwc:
            from eavsr_b200.pwc import PWCNET
            pwcnet = PWCNET()
            seeded_parameters(pwcnet)
            pwcnet = pwcnet.to(device)
        self.graph = graph
        self.trainer = Trainer(net, lr=1e-4, dtype=dtype, ddp=world > 1, device_ids=[device.index], pwcnet=pwcnet,
                               npost=0 if pwc else 350, capturable=graph)
        self.grad_bytes = trainable_bytes(net)
        self.host, self.dev = [], []
        for k in range(distinct):
            lr = torch.cat([clip_inputs(1, t, size, size, seed=5000 + 1000 * rank + 10 * k + i) for i in range(batch)])
            hr = F.interpolate(lr.view(batch * t, 3, size, size), scale_factor=4, mode="bicubic",
                               align_corners=False).clamp(0, 1).view(batch, t, 3, 4 * size, 4 * size)
            self.host.append((lr.pin_memory(), hr.pin_memory()))
            self.dev.append((lr.to(device), hr.to(device)))
        self.cursor = 0
        self.frames_per_step = batch * t
        self.h2d_bytes = (self.host[0][0].numel() + self.host[0][1].numel()) * 4
        self.d2h_bytes = 4
        self.launches_per_step = None
        self.loss = None
        self.epoch = 0

    def _do(self, lr, hr, sync=True):
        with torch.enable_grad():
            if self.graph and sync:
                if self.trainer._graph is None:
                    self.trainer.capture(lr, hr, epoch=self.epoch)
                    self.launches_per_step = self.trainer.captured_launches
                return self.trainer.step_graphed(lr, hr)
            return self.trainer.step(lr, hr, epoch=self.epoch, sync=sync)

    def step(self, sync=True):
        lr, hr = self.dev[self.cursor % len(self.dev)]
        self.cursor += 1
        self.loss = self._do(lr, hr, sync)
        return self.loss

    def e2e_step(self):
        lr, hr = self.host[self.cursor % len(self.host)]
        self.cursor += 1
        loss = self._do(lr.to(self.device, non_blocking=True), hr.to(self.device, non_blocking=True))
        return loss.item()                      # D2H read of the step's result

    def collective(self, steps, time_steps):
        """What the gradient all-reduce costs: the same steps without it (DDP no_sync), the all-reduce alone on a
        flat buffer of the same size, and the part of it the backward pass does not hide."""
        import torch.distributed as dist
        if self.world == 1:
            return {"op": "none (1 GPU)", "bytes_per_step": self.grad_bytes}
        if self.graph:      # the all-reduce is inside the captured graph: only its stand-alone cost can be reported
            flat = torch.zeros(self.grad_bytes // 4, device=self.device)
            buckets = list(flat.split(25 * 1024 * 1024 // 4))
            t_alone = time_steps(lambda: [dist.all_reduce(b) for b in buckets], max(steps, 5))
            return {"op": "all_reduce (NCCL, DistributedDataParallel buckets of 25 MB, captured in the step's CUDA graph)",
                    "bytes_per_step": self.grad_bytes, "alone_ms": round(t_alone, 3),
                    "busbw_GBps_alone": round(2 * (self.world - 1) / self.world * self.grad_bytes / (t_alone / 1e3) / 1e9, 1)}
        t_sync = time_steps(lambda: self.step(True), steps)
        t_nosync = time_steps(lambda: self.step(False), steps)
        flat = torch.zeros(self.grad_bytes // 4, device=self.device)
        buckets = list(flat.split(25 * 1024 * 1024 // 4))
        t_alone = time_steps(lambda: [dist.all_reduce(b) for b in buckets], max(steps, 5))
        exposed = max(0.0, t_sync - t_nosync)
        return {"op": "all_reduce (NCCL, DistributedDataParallel buckets of 25 MB, gradient_as_bucket_view)",
                "bytes_per_step": self.grad_bytes, "alone_ms": round(t_alone, 3), "step_ms": round(t_sync, 3),
                "step_without_allreduce_ms": round(t_nosync, 3), "exposed_ms": round(exposed, 3),
                "overlap_frac": round(1.0 - min(1.0, exposed / max(t_alone, 1e-9)), 4),
                "busbw_GBps_alone": round(2 * (self.world - 1) / self.world * self.grad_bytes / (t_alone / 1e3) / 1e9, 1)}


def make_workload(name, device, rank=0, world=1, args=None):
    if name == "train":
        return TrainWorkload(device, rank, world, dtype=torch.float32 if (args and args.train_dtype == "f32") else torch.bfloat16,
                             pwc=bool(args and args.train_pwc), graph=bool(args and args.train_graph))
    if name == "hotpath":
        return HotpathWorkload(device, t=T_FRAMES)
    if name == "model":
        distinct = min(NUM_CLIPS // world, (args.steps + args.warmup) if args else 8, 16)
        return ModelWorkload(device, t=T_FRAMES, h=LR_H, w=LR_W, rank=rank, world=world, distinct=distinct,
                             clips_per_step=args.clips_per_step if args else 1, streams=args.streams if args else 1)
    raise SystemExit(f"unknown workload {name}")


DUMP_WHOLE = 8 << 20     # elements: an output up to this size is written whole (32 MiB in float32)
DUMP_SAMPLE = 4 << 20    # elements drawn from a larger one: 16 MiB of float32 values + 32 MiB of float64 indices
DUMP_LIMIT = 64 << 20    # bytes written in all


def dump_outputs(out_dir, name, out, seed=0):
    """Write `out`, what one step returned (a tensor, or a list of tensors that are the parts of one batch), as
    out_dir/<name>.npy in float32.  An output of more than DUMP_WHOLE elements is replaced by DUMP_SAMPLE of its
    elements, one drawn from each of DUMP_SAMPLE equal runs of its flat (row-major) index, at offsets that depend
    only on its size and `seed`; the increasing indices go to out_dir/<name>_index.npy as float64 (exact below
    2**53).  The sample is gathered from the output in place: no copy of the whole output is made.
    Returns {file name: bytes}."""
    import numpy as np
    parts = [p.detach() for p in out] if isinstance(out, (list, tuple)) else [out.detach()]
    shape = tuple(parts[0].shape)
    if len(parts) > 1:
        shape = (sum(p.shape[0] for p in parts),) + shape[1:]
    numel = math.prod(shape)
    arrays = {}
    if numel <= DUMP_WHOLE:
        arrays[name] = (parts[0] if len(parts) == 1 else torch.cat(parts)).float().cpu().numpy()
    else:
        g = torch.Generator().manual_seed(seed)
        k = torch.arange(DUMP_SAMPLE, dtype=torch.int64)
        lo, hi = k * numel // DUMP_SAMPLE, (k + 1) * numel // DUMP_SAMPLE
        idx = lo + (torch.rand(DUMP_SAMPLE, generator=g, dtype=torch.float64) * (hi - lo)).long()
        coords = torch.unravel_index(idx, shape)
        vals = torch.empty(DUMP_SAMPLE, dtype=torch.float32)
        first = 0
        for p in parts:                          # the parts are consecutive runs of dim 0
            sel = (coords[0] >= first) & (coords[0] < first + p.shape[0])
            at = (coords[0][sel] - first,) + tuple(c[sel] for c in coords[1:])
            vals[sel] = p[tuple(c.to(p.device) for c in at)].float().cpu()
            first += p.shape[0]
        arrays[name] = vals.numpy()
        arrays[name + "_index"] = idx.double().numpy()
    if sum(a.nbytes for a in arrays.values()) > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {name} exceeds {DUMP_LIMIT} bytes")
    os.makedirs(out_dir, exist_ok=True)
    for key, a in arrays.items():
        np.save(os.path.join(out_dir, key + ".npy"), a)
    return {key + ".npy": a.nbytes for key, a in arrays.items()}


# ------------------------------------------------------------------------------------------------
# roofline of the dominant kernel: tcgen05 DCNv2 forward, timed live with CUDA events
# ------------------------------------------------------------------------------------------------
def dcn_backward_us(device, dg, iters=5):
    """fwd+bwd of BASELINE config 2 (1x64x270x480): device time of one backward (all five gradients)
    through autograd, CUDA events, includes ~0.1 ms of host-side autograd glue per call."""
    import eavsr_b200 as E
    h, w = LR_H, LR_W
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 64, h, w, generator=g).to(device, torch.bfloat16).contiguous(memory_format=torch.channels_last)
    off = (torch.randn(1, dg * 18, h, w, generator=g) * 2).clamp(-12, 12).to(device)
    msk = torch.sigmoid(torch.randn(1, dg * 9, h, w, generator=g)).to(device)
    wgt = ((torch.rand(64, 64, 3, 3, generator=g) * 2 - 1) / 24).to(device, torch.bfloat16)
    bias = torch.zeros(64, device=device, dtype=torch.bfloat16)
    with torch.enable_grad():
        leaves = [t.requires_grad_() for t in (x, off, msk, wgt, bias)]
        out = E.modulated_deform_conv2d(*leaves, 1, 1, 1, 1, dg)
        go = torch.randn_like(out)
        for _ in range(2):
            torch.autograd.grad(out, leaves, go, retain_graph=True)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(iters):
            torch.autograd.grad(out, leaves, go, retain_graph=True)
        b.record()
        torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def dcn_affine_us(device, peaks, iters=40):
    """SURVEY.md 8 row f1, the kernel the model's inference path actually launches: DCNv2 with the offset
    expansion fused in (496 algorithmic B/px: x, the 120-channel bf16 affine block, out)."""
    from eavsr_b200 import ops
    h, w, D = LR_H, LR_W, 8
    g = torch.Generator().manual_seed(2)
    nbuf = 4
    xs = [torch.randn(1, 64, h, w, generator=g).to(device, torch.bfloat16).contiguous(
        memory_format=torch.channels_last) for _ in range(nbuf)]
    affs = []
    for _ in range(nbuf):
        a = torch.randn(1, 15 * D, h, w, generator=g)
        a[:, :4 * D] = a[:, :4 * D] * 0.2 + torch.tensor([1.0, 0.0, 0.0, 1.0]).repeat(D).view(1, -1, 1, 1)
        affs.append(a.to(device, torch.bfloat16).contiguous(memory_format=torch.channels_last))
    ab = (torch.randn(15 * D, generator=g) * 0.1).to(device, torch.bfloat16)
    wgt = ((torch.rand(64, 64, 3, 3, generator=g) * 2 - 1) / 24).to(device, torch.bfloat16)
    bias = torch.zeros(64, device=device, dtype=torch.bfloat16)

    def call(i):
        return ops.dcn_affine(xs[i % nbuf], affs[i % nbuf], ab, wgt, bias, D, static_weight=True)
    for i in range(4):
        call(i)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            keep = [call(i) for i in range(iters)]
        graph.replay()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        side.synchronize()
        a.record(side)
        graph.replay()
        b.record(side)
        side.synchronize()
    del keep
    sec = a.elapsed_time(b) / 1e3 / iters
    bytes_alg = h * w * (64 * 2 + 15 * D * 2 + 64 * 2)
    flops = 2.0 * h * w * 64 * 64 * 9
    return {"kernel": "win::dcn_fwd_win_kernel<dg=8,bf16,fused offsets>", "us_per_launch": round(sec * 1e6, 2),
            "algorithmic_bytes_per_launch": bytes_alg, "hbm_frac": round(bytes_alg / sec / 1e9 / peaks["hbm_gbs"], 4),
            "tensor_frac": round(flops / sec / 1e12 / peaks["bf16_tflops"], 4)}


DCN_WIN3_NCU_TRAFFIC = 138.66e6     # bytes per launch, profiles/r2_dcn_fwd_win3_ncu.txt


def dcn_roofline(device, peaks, dg=8, iters=60, nested=True):
    import eavsr_b200 as E
    h, w = LR_H, LR_W
    g = torch.Generator().manual_seed(0)
    nbuf = 4                                        # 4 x 145 MB of inputs: every launch streams from HBM (> L2)
    xs = [torch.randn(1, 64, h, w, generator=g).to(device, torch.bfloat16).contiguous(
        memory_format=torch.channels_last) for _ in range(nbuf)]
    offs = [(torch.randn(1, dg * 18, h, w, generator=g) * 2).clamp(-12, 12).to(device) for _ in range(nbuf)]
    msks = [torch.sigmoid(torch.randn(1, dg * 9, h, w, generator=g)).to(device) for _ in range(nbuf)]
    wgt = ((torch.rand(64, 64, 3, 3, generator=g) * 2 - 1) / 24).to(device, torch.bfloat16)
    bias = torch.zeros(64, device=device, dtype=torch.bfloat16)
    assert E.dcn_uses_tensor_cores(xs[0], wgt, 1, 1, 1, 1, dg)
    def call(i):
        return E.modulated_deform_conv2d(xs[i % nbuf], offs[i % nbuf], msks[i % nbuf], wgt, bias, 1, 1, 1, 1, dg,
                                         static_weight=True)   # constant weights, as in the model's inference path
    for i in range(4):
        call(i)
    torch.cuda.synchronize()
    # `iters` back-to-back launches of the kernel replayed as one CUDA graph on a side stream, timed with
    # events on that same stream: device time per launch without the ~25 us/call Python+ctypes host cost
    side = torch.cuda.Stream(device)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            keep = [call(i) for i in range(iters)]
        graph.replay()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        side.synchronize()
        a.record(side)
        graph.replay()
        b.record(side)
        side.synchronize()
    del keep
    sec = a.elapsed_time(b) / 1e3 / iters
    px = h * w
    bytes_alg = px * (64 * 2 + dg * 18 * 4 + dg * 9 * 4 + 64 * 2)       # SURVEY 8d: 1120 B/px at dg=8
    flops = 2.0 * px * 64 * 64 * 9
    ach = bytes_alg / sec / 1e9
    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this shape from the ncu --set full
    # capture summarised in profiles/r2_dcn_fwd_win3_ncu.txt (128.75 MB read + 9.91 MB written; the 16.6 MB
    # output is only partly evicted from L2 within the launch)
    traffic = DCN_WIN3_NCU_TRAFFIC if dg == 8 else None
    kname = "win3::dcn_fwd_win3_kernel<bf16> dg=8" if dg == 8 else "win::dcn_fwd_win_kernel<dg=%d,bf16>" % dg
    res = {"kernel": kname + " 1x64x270x480", "bound": "hbm", "achieved": round(ach, 1),
           "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(ach / peaks["hbm_gbs"], 4), "traffic": traffic,
           "peak_source": peaks["source"], "us_per_launch": round(sec * 1e6, 2),
           "algorithmic_bytes_per_launch": bytes_alg,
           "tensor": {"achieved_tflops": round(flops / sec / 1e12, 1), "peak_tflops": peaks["bf16_tflops"],
                      "frac": round(flops / sec / 1e12 / peaks["bf16_tflops"], 4)}}
    if nested:
        # BASELINE config 2 (the DCNv2 micro-bench the "DCN TC util" half of the metric is quoted on):
        # deform_groups = 16, forward + backward, same shape
        del xs, offs, msks
        torch.cuda.empty_cache()
        try:
            c2 = dcn_roofline(device, peaks, dg=16, iters=30, nested=False)
            bwd = dcn_backward_us(device, 16)
            res["config2_dg16"] = {"fwd_us": c2["us_per_launch"], "fwd_hbm_frac": c2["frac"],
                                   "fwd_tensor_frac": c2["tensor"]["frac"], "bwd_us": round(bwd, 1),
                                   "fwd_bwd_tensor_frac": round(3 * flops / ((c2["us_per_launch"] + bwd) * 1e-6) / 1e12
                                                                / peaks["bf16_tflops"], 4),
                                   "bwd_us_dg8": round(dcn_backward_us(device, 8), 1)}
        except Exception as exc:  # an extra, never a reason to lose the bench line
            res["config2_dg16"] = {"failed": repr(exc)}
        try:
            res["fused_offsets_dg8"] = dcn_affine_us(device, peaks)
        except Exception as exc:
            res["fused_offsets_dg8"] = {"failed": repr(exc)}
    return res


# ------------------------------------------------------------------------------------------------
# CPU baseline (oracle port on the host cores) -- also the `--impl reference` arm
# ------------------------------------------------------------------------------------------------
def cpu_hotpath_frames_per_s(budget_s=20.0):
    """Times the CPU path the reference would run for the same operators (torchvision's CPU DCNv2 --
    the mmcv stand-in -- and ATen grid_sample through the oracle's reference-faithful wrappers) on
    a bounded sample: whole MultiAdSTN-equivalents (5 warps + 1 DCN at 272x480) until the budget
    is spent, scaled to the 228 calls of a 30-frame clip."""
    from oracle import cpu_reference as R
    torch.set_num_threads(os.cpu_count() or 1)
    return R.time_hotpath_sample(PAD_H, LR_W, T_FRAMES, budget_s)


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU path for the same workload (oracle port: the reference is
    Python + mmcv + cupy, which this project does not ship) on all host threads, exactly `--steps` timed steps.
    model: a step = the complete x4 forward of a 6-frame clip at the stated 272x480 geometry (~70 s on 16 cores),
    after one untimed 3x64x64 clip that pays the lazy initialisations.  hotpath: a step = the 4 * (2T - 3) = 228
    MultiAdSTN-equivalents (5 warps + 1 DCNv2) of one 30-frame clip, after one untimed MultiAdSTN-equivalent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps = args.steps
    if args.workload == "model":
        from oracle import eavsrp_cpu as R
        sd = R._seeded_state_dict()
        t_s = 6
        R.time_clip_forward(3, 64, 64, sd)
        secs = [R.time_clip_forward(t_s, PAD_H, LR_W, sd, seed=1234 + i) for i in range(steps)]
        el = sum(secs) / len(secs)
        fps = t_s / el
        sample = (f"{steps} step(s); a step = full x4 forward of a {t_s}-frame {PAD_H}x{LR_W} clip ({el:.1f} s) on "
                  f"{torch.get_num_threads()} threads, fp32, ATen grid_sample + torchvision CPU DCNv2; no warm-up steps "
                  f"beyond a 3x64x64 clip; frames/s of the short clip (the 30-frame clip of the metric does 1.9 "
                  f"alignments per frame against {(2 * t_s - 3) / t_s:.1f} here: favours the CPU)")
        name, ms = ModelWorkload.name, el * 1e3
    else:
        from oracle import cpu_reference as R
        fps, sample = R.time_hotpath_sample(PAD_H, LR_W, T_FRAMES, clips=steps)
        name, ms = HotpathWorkload.name, T_FRAMES / fps * 1e3
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": steps, "steps_requested": args.steps, "warmup": 0, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(name, world, args.clips_per_step if args.workload == "model" else 1),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": sample},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def bench_config(workload, world, clips_per_gpu_step=1):
    """The `config` object of the JSON line -- identical for both arms (`--impl reference` times the same
    workload on the host cores)."""
    return {"workload": workload, "clip": f"{T_FRAMES}x3x{LR_H}x{LR_W}", "clips_per_step": world * clips_per_gpu_step,
            "clips_in_flight_per_gpu": clips_per_gpu_step,
            "parallelism": f"clip-parallel x{world} (no collective)",
            "l2": "working set per step >> 126 MB L2 (a different HBM-resident clip every step)"}


# ------------------------------------------------------------------------------------------------
def main():
    global T_FRAMES
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("EAVSR_BENCH_WORKLOAD", "model"))
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--frames", type=int, default=T_FRAMES, help="frames per clip (profiling runs only; default 30)")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--train-dtype", default="bf16", choices=["bf16", "f32"], help="--workload train: compute dtype")
    ap.add_argument("--train-eager", dest="train_graph", action="store_false",
                    help="--workload train: eager steps instead of ONE CUDA graph per step (forward, backward, all-reduce, "
                         "Adam).  The graph is 1.6x faster (the eager step is bound by ~45 k host launches); the eager mode "
                         "is what can report how much of the all-reduce the backward pass hides (`collective`).")
    ap.set_defaults(train_graph=True)
    ap.add_argument("--train-pwc", action="store_true",
                    help="--workload train: run the epoch >= npost branch too (PWC-Net cost volume + backwarp)")
    ap.add_argument("--streams", type=int, default=1,
                    help="run the clips of a step as this many concurrent forwards (CUDA streams) instead of one batch")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them returned as DIR/<name>.npy (rank 0)")
    ap.add_argument("--clips-per-step", type=int, default=8,
                    help="clips in flight per GPU and step (BASELINE config 4 gives every GPU 8 clips): clips-per-step / "
                         "streams are batched into one forward, the forwards run on `streams` CUDA streams; default: the 8 "
                         "clips of config 4 as ONE batch (+12 %% over one clip at a time, which is reported next to it as "
                         "`single_clip`: the per-layer barrier / set-up of the chained convolutions is amortised over 8 images)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; --impl reference does not run it")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch.distributed as dist
    from eavsr_b200 import _lib
    _lib.load()     # fail loudly if the CUDA library is missing
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner to STDOUT when the communicator is created (NCCL_DEBUG >= VERSION in
        # this image): send fd 1 to stderr until the first collective is through, so that stdout carries the
        # one JSON line and nothing else
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    peaks = load_peaks()
    T_FRAMES = args.frames
    wl = make_workload(args.workload, device, rank, world, args)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(args.warmup):
            wl.step()
        barrier()
        sampler = ClockSampler(local)
        sampler.start()
        time.sleep(0.3)
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.time()
        torch.cuda.profiler.start()          # no-op unless run under `ncu --profile-from-start off`
        e0.record()
        for _ in range(args.steps):
            out = wl.step()
        e1.record()
        barrier()
        torch.cuda.profiler.stop()
        t1 = time.time()
        launches = _lib.launch_count() - l0
        if getattr(wl, "launches_per_step", None):   # CUDA-graph replay: the counter only sees the capture
            launches = wl.launches_per_step * args.steps
        clocks = sampler.stop(t0, t1)
        ms = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([ms], device=device)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = tt.item()
        if args.dump_outputs and rank == 0:      # before the runs below overwrite the step's output buffers
            written = dump_outputs(args.dump_outputs, wl.output_name, out)
            print(f"bench.py: wrote {written} to {args.dump_outputs}", file=sys.stderr)

        # end to end: pinned host clip in, host result out, through the public API
        e2e = None
        if hasattr(wl, "e2e_step") and wl.h2d_bytes:
            for _ in range(2):
                wl.e2e_step()
            barrier()
            e0.record()
            for _ in range(args.steps):
                wl.e2e_step()
            e1.record()
            barrier()
            ems = e0.elapsed_time(e1)
            if world > 1:
                tt = torch.tensor([ems], device=device)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                ems = tt.item()
            e2e = {"value": round(world * wl.frames_per_step * args.steps / (ems / 1e3), 3), "unit": "frames/s",
                   "h2d_bytes_per_step": wl.h2d_bytes, "d2h_bytes_per_step": wl.d2h_bytes}

        collective = None
        if hasattr(wl, "collective"):          # every rank takes part
            def time_steps(fn, k):
                fn()
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(k):
                    fn()
                b.record()
                barrier()
                tt = torch.tensor([a.elapsed_time(b) / k], device=device)
                if world > 1:
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                return tt.item()
            collective = wl.collective(args.steps, time_steps)

        parity = None
        if rank == 0 and not args.no_parity and hasattr(wl, "parity"):
            try:
                parity = wl.parity()
            except Exception as exc:   # reported, never a reason to lose the bench line
                parity = {"failed": repr(exc)}
        single = None
        if rank == 0 and args.workload == "model" and getattr(wl, "cps", 1) > 1 and not args.no_parity:
            # BASELINE config 3 as literally written: ONE clip at a time (latency of a clip = this ms_per_clip)
            try:
                w1 = ModelWorkload(device, t=T_FRAMES, h=LR_H, w=LR_W, rank=rank, world=world, distinct=2,
                                   clips_per_step=1, streams=1, net=wl.net)
                for _ in range(3):
                    w1.step()
                torch.cuda.synchronize()
                a1, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                k1 = max(2, min(args.steps, 5))
                a1.record()
                for _ in range(k1):
                    w1.step()
                b1.record()
                torch.cuda.synchronize()
                ms1 = a1.elapsed_time(b1) / k1
                single = {"clips_in_flight": 1, "ms_per_clip": round(ms1, 3), "value": round(T_FRAMES / (ms1 / 1e3), 3),
                          "unit": "frames/s", "steps": k1}
                del w1
            except Exception as exc:
                single = {"failed": repr(exc)}
        roof = dcn_roofline(device, peaks) if (rank == 0 and not args.no_roofline and args.workload != "train") else None

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            if args.workload == "model":
                from oracle import eavsrp_cpu as R
                torch.set_num_threads(os.cpu_count() or 1)
                fps, sample, _, _ = R.time_model_sample(budget_s=40.0, h=PAD_H, w=LR_W, frames=(3,))
            elif args.workload == "train":
                from oracle import eavsrp_cpu as R
                torch.set_num_threads(os.cpu_count() or 1)
                fps, sample = R.time_train_sample()
            else:
                fps, sample = cpu_hotpath_frames_per_s(15.0)
            cpu = {"value": fps, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                   "sample": sample}
        except Exception as exc:  # the baseline is a reported number, never a reason to lose the bench line
            cpu = {"value": None, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
                   "sample": f"failed: {exc!r}"}

    if rank == 0 and args.workload == "train":
        value = world * wl.frames_per_step * args.steps / (ms / 1e3)
        line = {"metric": "LR frames/s, EAVSR+ x4 training step, 15-frame 64x64 LR crops", "value": round(value, 3),
                "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": args.train_dtype, "data": "synthetic",
                "config": {"workload": wl.name if args.train_dtype == "bf16" else wl.name.replace("bf16", "f32"),
                           "crops_per_gpu": wl.batch, "global_batch": wl.batch * world, "frames": wl.t,
                           "optimizer": "Adam, 2 groups (deform_align lr 1e-5)", "loss": "L1",
                           "npost_branch": bool(args.train_pwc), "cuda_graph": bool(args.train_graph),
                           "parallelism": f"ddp x{world} (NCCL all-reduce of {wl.grad_bytes / 1e6:.1f} MB gradients)",
                           "l2": "activations per step >> 126 MB L2"},
                "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e, "collective": collective,
                "loss": float(wl.loss), "cpu_baseline": cpu}
        print(json.dumps(line))
    elif rank == 0:
        value = world * wl.frames_per_step * args.steps / (ms / 1e3)
        line = {"metric": METRIC, "value": round(value, 3), "unit": "frames/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic",
                "config": bench_config(wl.name, world, getattr(wl, "cps", 1)),
                "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e, "roofline": roof,
                "cpu_baseline": cpu, "parity": parity, "single_clip": single,
                "clips": {"set": NUM_CLIPS, "seeds": "1234 + clip_id", "this_run_per_rank": len(getattr(wl, "dev_clips", [])),
                          "sharding": "clip i -> rank i mod N (eavsr_b200.clip_parallel.shard)"}}
        print(json.dumps(line))
    if world > 1:
        # A captured NCCL all-reduce (--train-graph) has been seen to hang the process-group teardown: drop the graph
        # first, and never let a stuck teardown hold the GPUs -- the JSON line is already out.
        sys.stdout.flush()
        watchdog = threading.Timer(30.0, lambda: os._exit(0))
        watchdog.daemon = True
        watchdog.start()
        if hasattr(wl, "trainer"):
            wl.trainer._graph = None
        torch.cuda.synchronize()
        dist.destroy_process_group()
        watchdog.cancel()


if __name__ == "__main__":
    main()
