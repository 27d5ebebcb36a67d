"""8-bit limited-range ("TV") Y'CbCr 4:2:0 <-> RGB in [0, 1], stated once.

``EAVSRP.forward_yuv420`` converts its input with `yuv420_to_rgb` and defines its output as `rgb_to_yuv420` of the
SR frames; the fused tail kernel (``eavsr_sr_tail_yuv420_forward``) follows `rgb_to_yuv420`'s fp32 order of
operations.  A matrix is ``(Kr, Kb)`` with ``Kg = 1 - Kr - Kb``; Y' spans 16-235, Cb and Cr 16-240.

Chroma is centre-sited (JPEG / MPEG-1 siting): a chroma sample sits at the centre of its 2x2 block of luma samples.
Downsampling takes the mean of the block, upsampling is bilinear with ``align_corners=False``.
"""
from __future__ import annotations

import struct

import torch
import torch.nn.functional as F

__all__ = ["MATRICES", "coefficients", "yuv420_to_rgb", "rgb_to_yuv420"]

MATRICES = {"bt709": (0.2126, 0.0722), "bt601": (0.299, 0.114)}


def _f32(v: float) -> float:
    return struct.unpack("f", struct.pack("f", v))[0]


def coefficients(kr: float, kb: float):
    """``(kr, kg, kb, cu, cv)`` as fp32 values: ``kg = (1 - kr) - kb``, ``cu = 112 / (1 - kb)``,
    ``cv = 112 / (1 - kr)``, each operation rounded to fp32 as the kernel computes them."""
    kr, kb = _f32(kr), _f32(kb)
    return kr, _f32(_f32(1 - kr) - kb), kb, _f32(112 / _f32(1 - kb)), _f32(112 / _f32(1 - kr))


def yuv420_to_rgb(y, u, v, kr: float, kb: float):
    """``y`` (n, t, h, w) and ``u``, ``v`` (n, t, h/2, w/2) uint8 planes (any strides) -> (n, t, 3, h, w) fp32 RGB
    in [0, 1].  ``Yn = (Y - 16) / 219``, ``Pb = (U - 128) / 224``, ``Pr = (V - 128) / 224``; Pb and Pr are upsampled
    bilinearly (scale 2, ``align_corners=False``); ``R = Yn + 2(1 - Kr) Pr``, ``B = Yn + 2(1 - Kb) Pb``,
    ``G = (Yn - Kr R - Kb B) / Kg``, clamped to [0, 1]."""
    n, t, h, w = y.shape
    kg = 1 - kr - kb
    yn = (y.float() - 16) / 219
    pbr = (torch.stack([u, v], 2).float() - 128) / 224                      # (n, t, 2, h/2, w/2)
    pbr = F.interpolate(pbr.reshape(n * t, 2, h // 2, w // 2), scale_factor=2, mode="bilinear", align_corners=False)
    pb, pr = pbr.view(n, t, 2, h, w).unbind(2)
    r = yn + 2 * (1 - kr) * pr
    b = yn + 2 * (1 - kb) * pb
    g = (yn - kr * r - kb * b) / kg
    return torch.stack([r, g, b], 2).clamp_(0, 1)


def _luma(r, g, b, kr, kg, kb):
    return (kr * r + kg * g) + kb * b


def rgb_to_yuv420(rgb, kr: float, kb: float):
    """``rgb`` (..., 3, H, W) with even H, W -> uint8 planes ``Y`` (..., H, W), ``U`` and ``V`` (..., H/2, W/2).

    In fp32, in this order: ``p = clamp(rgb, 0, 1)``; ``Yc = (Kr r + Kg g) + Kb b``; ``Y = rint(16 + 219 Yc)``;
    the block mean ``m = ((p00 + p01) + (p10 + p11)) * 0.25``; ``U = rint(128 + (m_b - Yc(m)) * cu)`` and
    ``V = rint(128 + (m_r - Yc(m)) * cv)`` with the fp32 `coefficients`.  ``rint`` rounds half to even
    (``torch.round``)."""
    H, W = rgb.shape[-2:]
    if rgb.shape[-3] != 3 or H % 2 or W % 2:
        raise ValueError(f"rgb_to_yuv420 takes (..., 3, H, W) with even H and W, got {tuple(rgb.shape)}")
    kr, kg, kb, cu, cv = coefficients(kr, kb)
    p = rgb.float().clamp(0, 1)
    r, g, b = p.unbind(-3)
    y = torch.round(16 + 219 * _luma(r, g, b, kr, kg, kb))
    m = ((p[..., 0::2, 0::2] + p[..., 0::2, 1::2]) + (p[..., 1::2, 0::2] + p[..., 1::2, 1::2])) * 0.25
    mr, mg, mb = m.unbind(-3)
    ym = _luma(mr, mg, mb, kr, kg, kb)
    u = torch.round(128 + (mb - ym) * cu)
    v = torch.round(128 + (mr - ym) * cv)
    return y.to(torch.uint8), u.to(torch.uint8), v.to(torch.uint8)
