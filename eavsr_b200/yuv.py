"""Limited-range ("TV") Y'CbCr 4:2:0 <-> RGB in [0, 1] at 8, 10, 12 or 16 bits, stated once.

``EAVSRP.forward_yuv420`` and ``EAVSRP.forward_yuv420_u16`` convert their input with `yuv420_to_rgb` and define their
output as `rgb_to_yuv420` of the SR frames; the fused tail kernels (``eavsr_sr_tail_yuv420_forward``,
``eavsr_sr_tail_yuv420_u16_forward``) follow `rgb_to_yuv420`'s fp32 order of operations.  A matrix is ``(Kr, Kb)``
with ``Kg = 1 - Kr - Kb``.  At ``b`` bits, with ``k = 2**(b - 8)``, Y' spans 16k-235k and Cb, Cr 16k-240k (Rec. 709
and Rec. 2020 scale the 8-bit codes by ``k``).

Codes of more than 8 bits travel in uint16 samples moved up by ``shift`` bits: ``shift = 0`` keeps them in the low bits
(ffmpeg's ``yuv420p10le``), ``shift = 16 - b`` in the high bits (P010, P012).

Chroma is centre-sited (JPEG / MPEG-1 siting): a chroma sample sits at the centre of its 2x2 block of luma samples.
Downsampling takes the mean of the block, upsampling is bilinear with ``align_corners=False``.
"""
from __future__ import annotations

import struct

import torch
import torch.nn.functional as F

__all__ = ["MATRICES", "HBD_MATRICES", "coefficients", "yuv420_to_rgb", "rgb_to_yuv420", "check_bits"]

MATRICES = {"bt709": (0.2126, 0.0722), "bt601": (0.299, 0.114)}
# the high-bit-depth methods also take BT.2020 non-constant luminance (Rec. 2020 codes 10 and 12 bits only)
HBD_MATRICES = {**MATRICES, "bt2020": (0.2627, 0.0593)}


def _f32(v: float) -> float:
    return struct.unpack("f", struct.pack("f", v))[0]


def coefficients(kr: float, kb: float):
    """``(kr, kg, kb, cu, cv)`` as fp32 values: ``kg = (1 - kr) - kb``, ``cu = 112 / (1 - kb)``,
    ``cv = 112 / (1 - kr)``, each operation rounded to fp32 as the kernel computes them."""
    kr, kb = _f32(kr), _f32(kb)
    return kr, _f32(_f32(1 - kr) - kb), kb, _f32(112 / _f32(1 - kb)), _f32(112 / _f32(1 - kr))


def check_bits(who: str, bits: int, shift: int, allowed=(8, 10, 12, 16)) -> None:
    """ValueError unless ``bits`` is one of ``allowed`` and ``shift`` is 0 or ``16 - bits`` (0 at 8 bits)."""
    if bits not in allowed:
        raise ValueError(f"{who}: bits must be one of {list(allowed)}, got {bits!r}")
    if shift not in ((0,) if bits == 8 else (0, 16 - bits)):
        raise ValueError(f"{who}: shift must be 0 or 16 - bits = {16 - bits} at {bits} bits, got {shift!r}")


def _codes(p, shift: int):
    """uint8 / uint16 samples -> fp32 codes ``floor(p / 2**shift)`` (exact in fp32)."""
    return p.float() if shift == 0 else torch.floor(p.float() / 2 ** shift)


def yuv420_to_rgb(y, u, v, kr: float, kb: float, bits: int = 8, shift: int = 0):
    """``y`` (n, t, h, w) and ``u``, ``v`` (n, t, h/2, w/2) planes (any strides; uint8 at 8 bits, uint16 above) ->
    (n, t, 3, h, w) fp32 RGB in [0, 1].  With codes ``floor(sample / 2**shift)`` and ``k = 2**(bits - 8)``:
    ``Yn = (Y - 16k) / 219k``, ``Pb = (U - 128k) / 224k``, ``Pr = (V - 128k) / 224k``; Pb and Pr are upsampled
    bilinearly (scale 2, ``align_corners=False``); ``R = Yn + 2(1 - Kr) Pr``, ``B = Yn + 2(1 - Kb) Pb``,
    ``G = (Yn - Kr R - Kb B) / Kg``, clamped to [0, 1]."""
    check_bits("yuv420_to_rgb", bits, shift)
    n, t, h, w = y.shape
    k = 2 ** (bits - 8)
    kg = 1 - kr - kb
    yn = (_codes(y, shift) - 16 * k) / (219 * k)
    pbr = (torch.stack([_codes(u, shift), _codes(v, shift)], 2) - 128 * k) / (224 * k)      # (n, t, 2, h/2, w/2)
    pbr = F.interpolate(pbr.reshape(n * t, 2, h // 2, w // 2), scale_factor=2, mode="bilinear", align_corners=False)
    pb, pr = pbr.view(n, t, 2, h, w).unbind(2)
    r = yn + 2 * (1 - kr) * pr
    b = yn + 2 * (1 - kb) * pb
    g = (yn - kr * r - kb * b) / kg
    return torch.stack([r, g, b], 2).clamp_(0, 1)


def _luma(r, g, b, kr, kg, kb):
    return (kr * r + kg * g) + kb * b


def rgb_to_yuv420(rgb, kr: float, kb: float, bits: int = 8, shift: int = 0):
    """``rgb`` (..., 3, H, W) with even H, W -> planes ``Y`` (..., H, W), ``U`` and ``V`` (..., H/2, W/2): uint8 at
    8 bits, else uint16 holding the codes times ``2**shift``.

    In fp32, in this order, with ``k = 2**(bits - 8)``: ``p = clamp(rgb, 0, 1)``; ``Yc = (Kr r + Kg g) + Kb b``;
    ``Y = rint(16k + 219k Yc)``; the block mean ``m = ((p00 + p01) + (p10 + p11)) * 0.25``;
    ``U = rint(128k + (m_b - Yc(m)) * cu_b)`` and ``V = rint(128k + (m_r - Yc(m)) * cv_b)`` with the fp32
    `coefficients` ``cu_b = k cu``, ``cv_b = k cv`` (exact: k is a power of two, so the 8-bit codes are those of
    ``bits=8`` at any scale).  ``rint`` rounds half to even (``torch.round``)."""
    check_bits("rgb_to_yuv420", bits, shift)
    H, W = rgb.shape[-2:]
    if rgb.shape[-3] != 3 or H % 2 or W % 2:
        raise ValueError(f"rgb_to_yuv420 takes (..., 3, H, W) with even H and W, got {tuple(rgb.shape)}")
    k = 2 ** (bits - 8)
    kr, kg, kb, cu, cv = coefficients(kr, kb)
    p = rgb.float().clamp(0, 1)
    r, g, b = p.unbind(-3)
    y = torch.round(16 * k + 219 * k * _luma(r, g, b, kr, kg, kb))
    m = ((p[..., 0::2, 0::2] + p[..., 0::2, 1::2]) + (p[..., 1::2, 0::2] + p[..., 1::2, 1::2])) * 0.25
    mr, mg, mb = m.unbind(-3)
    ym = _luma(mr, mg, mb, kr, kg, kb)
    u = torch.round(128 * k + (mb - ym) * (cu * k))
    v = torch.round(128 * k + (mr - ym) * (cv * k))
    if bits == 8:
        return y.to(torch.uint8), u.to(torch.uint8), v.to(torch.uint8)
    return tuple((c * 2 ** shift).to(torch.uint16) for c in (y, u, v))
