"""CPU port of the reference's hot path, for the *reported* CPU baseline only.

TEST / BENCH INFRASTRUCTURE -- see oracle/__init__.py.  This is what `--gpu_ids -1` makes the
reference execute for the alignment operators, restated without importing /root/reference
(which does not exist on the GPU box):
  * flow_warp: host meshgrid + normalise + F.grid_sample(align_corners=True)
    (models/networks.py:699-739, models/eavsrp_model.py:587-626)
  * DCNv2: torchvision.ops.deform_conv2d CPU kernel, the stand-in for mmcv's CPU
    modulated_deform_conv (same MSRA algorithm; mmcv is not installable offline)
  * correlation: the reference has no CPU path (raises NotImplementedError,
    pwc/correlation/correlation.py:324-325); the oracle restatement is used.
"""
from __future__ import annotations

import time

import torch
import torch.nn.functional as F


def ref_flow_warp(x, flow_nhw2, padding_mode="zeros"):
    n, c, h, w = x.shape
    gy, gx = torch.meshgrid(torch.arange(0, h), torch.arange(0, w), indexing="ij")
    grid = torch.stack((gx, gy), 2).type_as(x)
    gf = grid + flow_nhw2
    gfx = 2.0 * gf[:, :, :, 0] / max(w - 1, 1) - 1.0
    gfy = 2.0 * gf[:, :, :, 1] / max(h - 1, 1) - 1.0
    return F.grid_sample(x, torch.stack((gfx, gfy), dim=3), mode="bilinear", padding_mode=padding_mode,
                         align_corners=True)


def ref_dcn(x, offset, mask, weight, bias, stride=1, padding=1, dilation=1):
    import torchvision
    return torchvision.ops.deform_conv2d(x, offset, weight, bias, stride=stride, padding=padding,
                                         dilation=dilation, mask=mask)


def time_hotpath_sample(h, w, t, budget_s=15.0, dg=8, clips=None):
    """Time whole MultiAdSTN-equivalents (quarter/half/3x full-res 64-ch warps + one DCNv2,
    models/networks.py:605-630) on the host until `budget_s` is spent, or, with `clips`, exactly the
    4*(2t-3) calls of that many t-frame clips; scale to the calls of one clip.
    Returns (LR frames/s, description of the sample)."""
    g = torch.Generator().manual_seed(0)
    f1 = torch.randn(1, 64, h, w, generator=g)
    f2 = torch.randn(1, 64, h // 2, w // 2, generator=g)
    f4 = torch.randn(1, 64, h // 4, w // 4, generator=g)
    fl1 = torch.randn(1, h, w, 2, generator=g) * 2
    fl2 = torch.randn(1, h // 2, w // 2, 2, generator=g)
    fl4 = torch.randn(1, h // 4, w // 4, 2, generator=g) * 0.5
    off = (torch.randn(1, dg * 18, h, w, generator=g) * 2).clamp(-12, 12)
    msk = torch.sigmoid(torch.randn(1, dg * 9, h, w, generator=g))
    wgt = (torch.rand(64, 64, 3, 3, generator=g) * 2 - 1) / 24
    bias = torch.zeros(64)

    def unit():
        ref_flow_warp(f4, fl4)
        ref_flow_warp(f2, fl2)
        ref_flow_warp(f1, fl1)
        ref_flow_warp(f1, fl1)
        feat = ref_flow_warp(f1, fl1)
        return ref_dcn(feat, off, msk, wgt, bias)

    units_per_clip = 4 * (2 * t - 3)
    with torch.no_grad():
        unit()                                    # warm-up (thread pool, allocator)
        n, t0 = 0, time.time()
        while True:
            unit()
            n += 1
            el = time.time() - t0
            if n >= clips * units_per_clip if clips else (el >= budget_s or n >= 64):
                break
    per_unit = el / n
    fps = t / (per_unit * units_per_clip)
    return fps, (f"{n} MultiAdSTN-equivalents (5 warps + 1 DCNv2 dg={dg}, fp32, {h}x{w}) in {el:.1f} s, "
                 f"scaled to {units_per_clip} per {t}-frame clip; torchvision CPU DCN + ATen grid_sample, "
                 f"{torch.get_num_threads()} threads")
