"""Host-side mirror of the reference's alignment operators, bound to the CUDA library.

Same names, argument meaning and error behaviour as the symbols the reference resolves:

  * ``ModulatedDeformConv2d`` / ``modulated_deform_conv2d``  -- ``from mmcv.ops import ...`` at
    models/networks.py:573, subclassed at :575-583, called at :627-630
  * ``flow_warp`` (flow ``(n,2,h,w)``)      -- models/networks.py:699-739
  * ``flow_warp_nhw2`` (flow ``(n,h,w,2)``) -- models/eavsrp_model.py:587-626,
    models/eavsrpx2_model.py:588-627
  * ``FunctionCorrelation`` / ``ModuleCorrelation`` -- pwc/correlation/correlation.py:385-397

PyTorch is plumbing here (device memory, streams, autograd glue); every op runs in
libeavsr_b200.so.  CPU tensors raise NotImplementedError -- there is no fallback.

Precision policy: features/weights run in the dtype of ``x`` (fp32 or bf16, fp32 accumulate);
flow / offset / mask are always consumed as fp32 so sampling coordinates are never rounded.
Memory format: channels_last (NHWC) inputs take the vectorised / tensor-core paths with no
copies; 64-channel NCHW inputs to the DCN are converted once to channels_last.  Outputs of the
fast paths are channels_last.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple, Union

import threading
import weakref

import ctypes

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Function
from torch.autograd.function import once_differentiable
from torch.nn.modules.utils import _pair

from . import _lib as L
from .yuv import check_bits

__all__ = [
    "modulated_deform_conv2d", "ModulatedDeformConv2d", "dcn_affine", "dcn_affine_eligible", "flow_warp", "flow_warp_nhw2",
    "backwarp", "get_backwarp", "invalidate_caches", "flow_warp_pyramid", "flow_warp_pyramid_eligible",
    "spynet_level_input", "cat_channels", "grouped_conv3x3", "grouped_conv3x3_eligible", "conv2d_native_bias_grad", "channel_mean", "scale_residual",
    "FunctionCorrelation", "ModuleCorrelation", "dcn_uses_tensor_cores",
    "adapt_mix", "affine_offsets_mask", "ca_residual", "fused_inference_ok", "bias_act_", "conv2d_bias_act",
    "conv3x3_64", "conv3x3_64_ca", "conv3x3_64_eligible", "ca_scale", "conv2d_bias_act_shuffle",
    "conv3x3_chain_eligible", "rca_group_chain", "sr_tail_u8", "sr_tail_u8_eligible", "sr_tail_yuv420",
    "sr_tail_u16", "sr_tail_yuv420_u16", "sr_tail_u8_sse",
]

_DTYPES = {torch.float32: L.F32, torch.bfloat16: L.BF16}


def _require_cuda(name: str, *tensors: torch.Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise NotImplementedError(
                f"eavsr_b200.{name}: CUDA tensors only (the B200 library has no CPU fallback)")


def _dtype_code(name: str, t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"eavsr_b200.{name}: dtype {t.dtype} not supported (float32 / bfloat16)") from None


def _strides(t: Optional[torch.Tensor]):
    if t is None:
        return None
    s = list(t.stride())
    if t.dim() == 4 and t.shape[0] == 1:
        # the stride of a size-1 batch dimension is arbitrary in PyTorch (views such as `x.view(t, 1, ...).unbind(0)`
        # report 64 or t*C*H*W); the library checks `stride[0] >= extent of one image`, so hand it exactly that
        s[0] = max(t.shape[i] * s[i] for i in (1, 2, 3))       # also right for a channel slice of a wider buffer
    return L.Strides(*s)


# `isinstance(a, torch.Tensor)` costs ~0.1 us for a non-tensor, and most arguments are sizes: test those by type first
_PLAIN_ARGS = frozenset((int, float, type(None), L.Strides))


def _launch(entry: str, *args) -> None:
    """Call ``eavsr_<entry>(*args, stream)`` on the current stream of the first tensor argument's device, inside
    that device's guard.  Tensors are passed as their ``data_ptr()``; ``args`` keeps them alive until the call has
    been issued, so a converted temporary cannot be freed and its memory reused by a later argument."""
    cargs = [a if type(a) in _PLAIN_ARGS else a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args]
    dev = next(a for a in args if isinstance(a, torch.Tensor)).device
    fn = getattr(L.load(), "eavsr_" + entry)
    with torch.cuda.device(dev):
        # the handle of torch.cuda.current_stream(dev), without building a Stream object on every launch
        rc = fn(*cargs, torch._C._cuda_getCurrentRawStream(dev.index))
    L.check(rc, entry)


def _param(t: Optional[torch.Tensor], dtype) -> Optional[torch.Tensor]:
    """Detached contiguous ``dtype`` view / copy of a parameter (None stays None)."""
    return None if t is None else t.detach().to(dtype).contiguous()


def _grad(g: Optional[torch.Tensor], dtype) -> Optional[torch.Tensor]:
    """An fp32 gradient buffer cast to the dtype of its input (None stays None)."""
    return None if g is None else g.to(dtype)


def _is_channels_last(t: torch.Tensor) -> bool:
    return t.dim() == 4 and t.stride(1) == 1 and t.size(1) > 1


def _empty_like_layout(t: torch.Tensor, dtype=None, channels: Optional[int] = None,
                       hw: Optional[Tuple[int, int]] = None) -> torch.Tensor:
    """Dense tensor shaped like ``t`` (optionally other C/H/W), channels_last iff ``t`` is."""
    n, c, h, w = t.shape
    c = c if channels is None else channels
    h, w = (h, w) if hw is None else hw
    fmt = torch.channels_last if _is_channels_last(t) else torch.contiguous_format
    return torch.empty((n, c, h, w), dtype=dtype or t.dtype, device=t.device, memory_format=fmt)


def _dense(t: torch.Tensor) -> torch.Tensor:
    """Return ``t`` if it is dense NCHW or dense NHWC, else a dense copy in its nearest format."""
    if t.is_contiguous() or t.is_contiguous(memory_format=torch.channels_last):
        return t
    fmt = torch.channels_last if _is_channels_last(t) else torch.contiguous_format
    return t.contiguous(memory_format=fmt)


# ------------------------------------------------------------------------------------------
# flow_warp
# ------------------------------------------------------------------------------------------
class _FlowWarpFn(Function):
    @staticmethod
    def forward(ctx, x, flow, layout: int, pad: int):
        if (x.shape[1] * x.element_size()) % 16 == 0:
            xd = x.contiguous(memory_format=torch.channels_last)  # vectorised NHWC path
        else:
            xd = _dense(x)                                        # 2/3-channel maps: strided path
        flow32 = _param(flow, torch.float32)
        out = _empty_like_layout(xd)
        n, c, h, w = xd.shape
        _launch("flow_warp_forward", xd, _strides(xd), flow32, layout, out, _strides(out), n, c, h, w,
                _dtype_code("flow_warp", xd), pad)
        ctx.save_for_backward(xd, flow32)
        ctx.layout, ctx.pad, ctx.flow_dtype = layout, pad, flow.dtype
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        xd, flow32 = ctx.saved_tensors
        fmt = torch.channels_last if _is_channels_last(xd) else torch.contiguous_format
        g = gout.to(xd.dtype).contiguous(memory_format=fmt)
        gx32 = _empty_like_layout(xd, dtype=torch.float32) if ctx.needs_input_grad[0] else None
        gflow = torch.empty_like(flow32) if ctx.needs_input_grad[1] else None
        n, c, h, w = xd.shape
        _launch("flow_warp_backward", g, _strides(g), xd, _strides(xd), flow32, ctx.layout, gx32, _strides(gx32), gflow,
                n, c, h, w, _dtype_code("flow_warp", xd), ctx.pad)
        return _grad(gx32, xd.dtype), _grad(gflow, ctx.flow_dtype), None, None


def _flow_warp(name, x, flow, layout, interpolation, padding_mode, align_corners):
    hw = tuple(flow.shape[-2:]) if layout == L.FLOW_N2HW else tuple(flow.shape[1:3])
    if tuple(x.shape[-2:]) != hw:
        raise ValueError(f'The spatial sizes of input ({x.size()[-2:]}) and '
                         f'flow ({torch.Size(hw)}) are not the same.')
    if interpolation != 'bilinear' or not align_corners:
        raise NotImplementedError(
            f"eavsr_b200.{name}: only interpolation='bilinear', align_corners=True (what EAVSR uses)")
    if padding_mode not in ('zeros', 'border'):
        raise NotImplementedError(f"eavsr_b200.{name}: padding_mode {padding_mode!r} (zeros/border only)")
    _require_cuda(name, x, flow)
    if x.dim() != 4 or flow.dim() != 4 or flow.shape[0] != x.shape[0]:
        raise ValueError(f"eavsr_b200.{name}: expected x (n,c,h,w) and a matching flow, got "
                         f"{tuple(x.shape)} / {tuple(flow.shape)}")
    two = flow.shape[1] if layout == L.FLOW_N2HW else flow.shape[3]
    if two != 2:
        raise ValueError(f"eavsr_b200.{name}: flow must have 2 channels, got {tuple(flow.shape)}")
    return _FlowWarpFn.apply(x, flow, layout, L.PAD_ZEROS if padding_mode == 'zeros' else L.PAD_BORDER)


def flow_warp(x, flow, interpolation='bilinear', padding_mode='zeros', align_corners=True):
    """Drop-in for ``models.networks.flow_warp`` (models/networks.py:699-739): ``flow`` is
    ``(n, 2, h, w)``, channel 0 = x displacement, in pixels."""
    return _flow_warp("flow_warp", x, flow, L.FLOW_N2HW, interpolation, padding_mode, align_corners)


def flow_warp_nhw2(x, flow, interpolation='bilinear', padding_mode='zeros', align_corners=True):
    """Drop-in for ``models.eavsrp_model.flow_warp`` (models/eavsrp_model.py:587-626) and its
    eavsrpx2 twin: ``flow`` is ``(n, h, w, 2)``."""
    return _flow_warp("flow_warp", x, flow, L.FLOW_NHW2, interpolation, padding_mode, align_corners)


def flow_warp2(x1, x2, flow, padding_mode='zeros'):
    """``(flow_warp(x1, flow), flow_warp(x2, flow))`` in one launch when both are dense channels_last bf16
    64-channel maps and no gradient is needed (SURVEY.md section 8 row f2: ``nbr`` and ``feat_prop`` share
    one flow in MultiAdSTN.forward, models/networks.py:621-623); two ordinary calls otherwise."""
    ok = (fused_inference_ok(x1, x2, flow) and x1.dtype == torch.bfloat16 and x2.dtype == torch.bfloat16
          and x1.shape == x2.shape and x1.dim() == 4 and x1.shape[1] == 64
          and x1.is_contiguous(memory_format=torch.channels_last)
          and x2.is_contiguous(memory_format=torch.channels_last)
          and flow.dim() == 4 and flow.shape[1] == 2 and flow.shape[2:] == x1.shape[2:]
          and padding_mode in ('zeros', 'border'))
    if not ok:
        return flow_warp(x1, flow, padding_mode=padding_mode), flow_warp(x2, flow, padding_mode=padding_mode)
    n, c, h, w = x1.shape
    o1, o2 = torch.empty_like(x1), torch.empty_like(x2)
    _launch("flow_warp2_forward", x1, _strides(x1), x2, _strides(x2), _param(flow, torch.float32), L.FLOW_N2HW,
            o1, _strides(o1), o2, _strides(o2), n, c, h, w, L.BF16,
            L.PAD_ZEROS if padding_mode == 'zeros' else L.PAD_BORDER)
    return o1, o2


def flow_warp_pyramid_eligible(x, x2=None) -> bool:
    """True when `flow_warp_pyramid` can run: inference, dense channels_last 64-channel bf16 / fp32 maps."""
    ok = (fused_inference_ok(x, x2) and x.dim() == 4 and x.shape[1] == 64
          and x.is_contiguous(memory_format=torch.channels_last) and x.shape[2] * x.shape[3] * 64 < (1 << 31))
    if ok and x2 is not None:
        ok = (x2.shape == x.shape and x2.dtype == x.dtype == torch.bfloat16
              and x2.is_contiguous(memory_format=torch.channels_last))
    return ok


def flow_warp_pyramid(x, terms, x2=None, want_flow=False, keep=()):
    """``flow_warp(x, sum_i scale_i * F.interpolate(flow_i, size=x.shape[2:], mode='bilinear', align_corners=True))``
    with the resizes, scalings and the sum evaluated inside the warp kernel (SURVEY.md section 8 row f2: the
    interpolate -> scale -> add -> warp chains of MultiAdSTN.forward, models/networks.py:600-615,619).
    ``terms``: [(flow (n,2,hi,wi), scale), ...] (<= 4); ``x2``: a second map warped with the same flow (:621-623);
    ``want_flow``: also return the summed flow; ``keep``: indices of terms whose ``scale * resize(flow)`` is returned
    too.  Returns (out, [out2], [flow], [kept terms...]).  Inference only: check `flow_warp_pyramid_eligible`."""
    n, c, h, w = x.shape
    out = torch.empty_like(x)
    out2 = torch.empty_like(x2) if x2 is not None else None
    fl = torch.empty((n, 2, h, w), dtype=torch.float32, device=x.device) if want_flow else None
    arr = (L.FlowTerm * len(terms))()
    hold, kept = [], []             # `arr` holds raw addresses: the tensors behind them must outlive the launch
    for i, (a, (f, sc)) in enumerate(zip(arr, terms)):
        f32 = _param(f, torch.float32)
        hold.append(f32)
        a.flow, a.h, a.w, a.scale = f32.data_ptr(), f32.shape[2], f32.shape[3], float(sc)
        if i in keep:
            t = torch.empty((n, 2, h, w), dtype=torch.float32, device=x.device)
            kept.append(t)
            a.scaled_out = t.data_ptr()
    _launch("flow_warp_pyramid_forward", x, _strides(x), x2, _strides(x2), arr, len(terms), out, _strides(out),
            out2, _strides(out2), fl, n, c, h, w, _dtype_code("flow_warp_pyramid", x), L.PAD_ZEROS)
    res = [out]
    if out2 is not None:
        res.append(out2)
    if fl is not None:
        res.append(fl)
    return tuple(res + kept) if len(res) + len(kept) > 1 else out


def spynet_level_input(ref, supp, flow_prev=None):
    """``torch.cat([ref, flow_warp(supp, up.permute(0,2,3,1), padding_mode='border'), up], 1)`` with
    ``up = F.interpolate(flow_prev, scale_factor=2, mode='bilinear', align_corners=True) * 2`` (zero at the coarsest
    level, ``flow_prev=None``): the input of one SPyNet level (models/eavsrp_model.py:468-486) in one launch
    (SURVEY.md section 8 row f4).  NCHW fp32, inference only.  Returns (n, 8, h, w); channels 6:8 are ``up``."""
    _require_cuda("spynet_level_input", ref, supp, flow_prev)
    n, c, h, w = ref.shape
    if c != 3 or supp.shape != ref.shape or ref.dtype != torch.float32 or supp.dtype != torch.float32:
        raise ValueError(f"spynet_level_input: expected two (n,3,h,w) fp32 images, got {tuple(ref.shape)} / {tuple(supp.shape)}")
    fp = _param(flow_prev, torch.float32)
    out = torch.empty((n, 8, h, w), dtype=torch.float32, device=ref.device)
    _launch("spynet_level_input_forward", ref.contiguous(), supp.contiguous(), fp, out, n, h, w,
            fp.shape[2] if fp is not None else 0, fp.shape[3] if fp is not None else 0)
    return out


# ------------------------------------------------------------------------------------------
# backwarp (train-time PWC-Net path)
# ------------------------------------------------------------------------------------------
class _BackwarpFn(Function):
    @staticmethod
    def forward(ctx, x, flow):
        xd = _dense(x)
        flow32 = _param(flow, torch.float32)
        n, c, h, w = xd.shape
        out = _empty_like_layout(xd)
        mask = torch.empty((n, 1, h, w), dtype=xd.dtype, device=xd.device)
        _launch("backwarp_forward", xd, _strides(xd), flow32, out, _strides(out), mask, n, c, h, w,
                _dtype_code("backwarp", xd))
        ctx.save_for_backward(xd, flow32)
        ctx.flow_dtype = flow.dtype
        ctx.mark_non_differentiable(mask)
        return out, mask

    @staticmethod
    @once_differentiable
    def backward(ctx, gout, _gmask):
        xd, flow32 = ctx.saved_tensors
        g = _dense(gout.to(xd.dtype))
        gx32 = _empty_like_layout(xd, dtype=torch.float32) if ctx.needs_input_grad[0] else None
        gflow = torch.empty_like(flow32) if ctx.needs_input_grad[1] else None
        n, c, h, w = xd.shape
        _launch("backwarp_backward", g, _strides(g), xd, _strides(xd), flow32, gx32, _strides(gx32), gflow, n, c, h, w,
                _dtype_code("backwarp", xd))
        return _grad(gx32, xd.dtype), _grad(gflow, ctx.flow_dtype)


def _backwarp(name, tenInput, tenFlow):
    _require_cuda(name, tenInput, tenFlow)
    if tenInput.dim() != 4 or tenFlow.dim() != 4 or tenFlow.shape[1] != 2 or tenFlow.shape[0] != tenInput.shape[0] \
            or tenFlow.shape[2:] != tenInput.shape[2:]:
        raise ValueError(f"eavsr_b200.{name}: expected input (n,c,h,w) and flow (n,2,h,w), got "
                         f"{tuple(tenInput.shape)} / {tuple(tenFlow.shape)}")
    return _BackwarpFn.apply(tenInput, tenFlow)


def backwarp(tenInput, tenFlow):
    """Drop-in for ``PWCNET.Decoder.backwarp`` (models/pwc_net.py:184-207): bilinear warp with
    ``align_corners=False`` semantics, multiplied by the validity mask (warped ones > 0.999)."""
    return _backwarp("backwarp", tenInput, tenFlow)[0]


def get_backwarp(tenSecond, flow):
    """The ``flow is not None`` branch of ``BaseModel.get_backwarp`` (models/base_model.py:344-354):
    returns ``(backwarp(tenSecond, flow) * mask, mask)`` with ``mask`` (n,1,h,w) in {0,1}."""
    return _backwarp("get_backwarp", tenSecond, flow)


# ------------------------------------------------------------------------------------------
# DCNv2
# ------------------------------------------------------------------------------------------
def _dcn_prepare_x(x: torch.Tensor, weight: torch.Tensor, groups: int) -> torch.Tensor:
    """64->64 3x3 features go to the tensor-core kernel, which wants NHWC."""
    if x.shape[1] == 64 and weight.shape[0] == 64 and groups == 1 and tuple(weight.shape[2:]) == (3, 3):
        return x.contiguous(memory_format=torch.channels_last)
    return _dense(x)


def dcn_uses_tensor_cores(x, weight, stride=1, padding=0, dilation=1, groups=1, deform_groups=1) -> bool:
    """True when this call would run the tcgen05 implicit-GEMM kernel (tests/bench assert it)."""
    lib = L.load()
    sh, sw = _pair(stride)
    ph, pw = _pair(padding)
    dh, dw = _pair(dilation)
    xd = _dcn_prepare_x(x, weight, groups)
    cout, _, kh, kw = weight.shape
    out = _empty_like_layout(xd, channels=cout)
    return bool(lib.eavsr_dcn_forward_uses_tensor_cores(_strides(xd), _strides(out), xd.shape[1], cout, kh, kw,
                                                        sh, sw, ph, pw, dh, dw, groups, deform_groups, 0))


DCN_WS_PACKED = L.DCN_WS_PACKED
_DCN_STATIC_WEIGHT = 1 << 20  # Python-side only: the caller promises `weight` is constant (see _dcn_workspace)
_DCN_WS_CACHE = {}          # (id(weight), stream) -> (weakref(weight), version, dtype, workspace)
_DCN_WS_LOCK = threading.Lock()   # nn.DataParallel calls the ops from one thread per GPU


def _dcn_workspace(weight, dtype, ws_bytes, static):
    """Workspace for eavsr_dcn_forward.  Weights the caller declares constant (``static_weight=True``,
    inference only) keep their packed image: an entry is valid only while it is the same tensor object at the
    same version counter on the same stream (the pack kernel is ordered against later launches by stream
    order only), so an optimizer step / load_state_dict / in-place edit re-packs; writes through ``.data``
    do not bump the version counter -- call `invalidate_caches` after those.
    Returns (workspace, already_packed, commit); ``commit()`` records the entry and must be called only
    after the launch that packed the workspace succeeded."""
    nothing = lambda: None      # noqa: E731
    if not static or (torch.is_grad_enabled() and weight.requires_grad):
        return torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=weight.device), False, nothing
    key = (id(weight), torch.cuda.current_stream(weight.device))
    with _DCN_WS_LOCK:
        hit = _DCN_WS_CACHE.get(key)
    if hit is not None:
        ref, version, dt, ws = hit
        if ref() is weight and version == weight._version and dt == dtype and ws.numel() >= ws_bytes \
                and ws.device == weight.device:
            return ws, True, nothing
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=weight.device)

    def commit():
        with _DCN_WS_LOCK:
            if len(_DCN_WS_CACHE) > 256:
                for k in [k for k, v in _DCN_WS_CACHE.items() if v[0]() is None]:
                    del _DCN_WS_CACHE[k]
                if len(_DCN_WS_CACHE) > 256:
                    _DCN_WS_CACHE.clear()
            _DCN_WS_CACHE[key] = (weakref.ref(weight), weight._version, dtype, ws)
    return ws, False, commit


def invalidate_caches(module: Optional[nn.Module] = None) -> None:
    """Drop every cached packed-weight image (DCN workspaces, tcgen05 conv3x3 tiles, merged offset-conv
    weights).  The caches are keyed on the parameters' version counters, which writes through ``param.data``
    (EMA swaps, ``init_weights``) do not bump: call this after such a write.  ``module``: also clear the
    per-module entries below it."""
    with _DCN_WS_LOCK:
        _DCN_WS_CACHE.clear()
    if module is not None:
        for m in module.modules():
            for attr in ("_eavsr_packed", "_merged", "_merged_bias"):
                if attr in m.__dict__:
                    del m.__dict__[attr]


class _ModulatedDeformConv2dFn(Function):
    @staticmethod
    def forward(ctx, input, offset, mask, weight, bias, stride, padding, dilation, groups, deform_groups,
                flags=0):
        if input is not None and input.dim() != 4:
            raise ValueError(f'Expected 4D tensor as input, got {input.dim()}D tensor instead.')
        _require_cuda("modulated_deform_conv2d", input, offset, mask, weight, bias)
        lib = L.load()
        sh, sw = _pair(stride)
        ph, pw = _pair(padding)
        dh, dw = _pair(dilation)
        cout, cin_g, kh, kw = weight.shape
        n, cin, h, w = input.shape
        ho = (h + 2 * ph - (dh * (kh - 1) + 1)) // sh + 1
        wo = (w + 2 * pw - (dw * (kw - 1) + 1)) // sw + 1
        K = kh * kw
        if cin_g * groups != cin:
            raise ValueError(f"modulated_deform_conv2d: weight {tuple(weight.shape)} does not match "
                             f"{cin} input channels with groups={groups}")
        if tuple(offset.shape) != (n, deform_groups * 2 * K, ho, wo):
            raise ValueError(f"modulated_deform_conv2d: offset shape {tuple(offset.shape)}, expected "
                             f"{(n, deform_groups * 2 * K, ho, wo)}")
        if tuple(mask.shape) != (n, deform_groups * K, ho, wo):
            raise ValueError(f"modulated_deform_conv2d: mask shape {tuple(mask.shape)}, expected "
                             f"{(n, deform_groups * K, ho, wo)}")
        code = _dtype_code("modulated_deform_conv2d", input)
        xd = _dcn_prepare_x(input, weight, groups)
        off32 = _param(offset, torch.float32)
        msk32 = _param(mask, torch.float32)
        wd = _param(weight, input.dtype)
        out = _empty_like_layout(xd, channels=cout, hw=(ho, wo))
        ws_bytes = lib.eavsr_dcn_forward_workspace(cin, cout, kh, kw, groups, deform_groups, code)
        ws, packed, commit = _dcn_workspace(weight, input.dtype, ws_bytes, bool(flags & _DCN_STATIC_WEIGHT))
        flags &= ~_DCN_STATIC_WEIGHT
        if packed:
            flags |= DCN_WS_PACKED
        _launch("dcn_forward", xd, _strides(xd), off32, msk32, wd, _param(bias, input.dtype), out, _strides(out),
                n, cin, h, w, cout, kh, kw, sh, sw, ph, pw, dh, dw, groups, deform_groups, code, ws, ws.numel(), flags)
        if ws_bytes and lib.eavsr_dcn_forward_uses_tensor_cores(
                _strides(xd), _strides(out), cin, cout, kh, kw, sh, sw, ph, pw, dh, dw, groups, deform_groups, flags):
            commit()        # only a tensor-core launch has packed the workspace
        ctx.save_for_backward(xd, off32, msk32, wd)
        ctx.geom = (sh, sw, ph, pw, dh, dw, groups, deform_groups)
        ctx.bwd_flags = flags & (L.DCN_FORCE_GENERIC | L.DCN_BWD_GENERIC_DATA | L.DCN_BWD_GENERIC_WEIGHT)
        ctx.has_bias = bias is not None
        ctx.in_dtypes = (offset.dtype, mask.dtype, weight.dtype, bias.dtype if bias is not None else None)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        xd, off32, msk32, wd = ctx.saved_tensors
        sh, sw, ph, pw, dh, dw, groups, dg = ctx.geom
        need = ctx.needs_input_grad
        n, cin, h, w = xd.shape
        cout, _, kh, kw = wd.shape
        fmt = torch.channels_last if _is_channels_last(xd) else torch.contiguous_format
        g = gout.to(xd.dtype).contiguous(memory_format=fmt)
        gx32 = _empty_like_layout(xd, dtype=torch.float32) if need[0] else None
        goff = torch.empty_like(off32) if need[1] else None
        gmsk = torch.empty_like(msk32) if need[2] else None
        gw32 = torch.empty(wd.shape, dtype=torch.float32, device=xd.device) if need[3] else None
        gb32 = torch.empty(cout, dtype=torch.float32, device=xd.device) if (need[4] and ctx.has_bias) else None
        code = _dtype_code("modulated_deform_conv2d", xd)
        ws_bytes = L.load().eavsr_dcn_backward_workspace(cin, cout, kh, kw, groups, dg, code)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=xd.device) if ws_bytes else None
        _launch("dcn_backward", g, _strides(g), xd, _strides(xd), off32, msk32, wd, gx32, _strides(gx32), goff, gmsk,
                gw32, gb32, n, cin, h, w, cout, kh, kw, sh, sw, ph, pw, dh, dw, groups, dg, code, ws, ws_bytes,
                ctx.bwd_flags)
        od, md, wdt, bdt = ctx.in_dtypes
        return (_grad(gx32, xd.dtype), _grad(goff, od), _grad(gmsk, md), _grad(gw32, wdt), _grad(gb32, bdt),
                None, None, None, None, None, None)


def modulated_deform_conv2d(input, offset, mask, weight, bias=None, stride=1, padding=0, dilation=1,
                            groups=1, deform_groups=1, *, static_weight=False):
    """Drop-in for ``mmcv.ops.modulated_deform_conv2d`` with the positional order the reference
    uses at models/networks.py:627-630.  ``static_weight=True`` (extension, inference only) lets the
    packed tensor-core image of ``weight`` be kept between calls while the tensor is unchanged."""
    return _ModulatedDeformConv2dFn.apply(input, offset, mask, weight, bias, stride, padding, dilation,
                                          groups, deform_groups, _DCN_STATIC_WEIGHT if static_weight else 0)


class ModulatedDeformConv2d(nn.Module):
    """Drop-in for ``mmcv.ops.ModulatedDeformConv2d`` (parameter container + forward), subclassable
    exactly as ``MultiAdSTN`` does (models/networks.py:575-583).  Parameter names, shapes and
    initialisation follow mmcv-full 1.x: weight ~ U(+-1/sqrt(in*kh*kw)), bias = 0."""

    _version = 2

    def __init__(self, in_channels: int, out_channels: int, kernel_size: Union[int, Tuple[int, int]],
                 stride: int = 1, padding: int = 0, dilation: int = 1, groups: int = 1,
                 deform_groups: int = 1, bias: Union[bool, str] = True):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _pair(kernel_size)
        self.stride = _pair(stride)
        self.padding = _pair(padding)
        self.dilation = _pair(dilation)
        self.groups = groups
        self.deform_groups = deform_groups
        self.transposed = False
        self.output_padding = _pair(0)
        self.weight = nn.Parameter(torch.Tensor(out_channels, in_channels // groups, *self.kernel_size))
        if bias:
            self.bias = nn.Parameter(torch.Tensor(out_channels))
        else:
            self.register_parameter('bias', None)
        self.init_weights()

    def init_weights(self):
        n = self.in_channels
        for k in self.kernel_size:
            n *= k
        stdv = 1. / math.sqrt(n)
        self.weight.data.uniform_(-stdv, stdv)
        if self.bias is not None:
            self.bias.data.zero_()

    def forward(self, x, offset, mask):
        return modulated_deform_conv2d(x, offset, mask, self.weight, self.bias, self.stride, self.padding,
                                       self.dilation, self.groups, self.deform_groups)


# ------------------------------------------------------------------------------------------
# correlation
# ------------------------------------------------------------------------------------------
# Opt-in: fp32 cost volumes larger than 16x16 (w % 4 == 0) as a banded GEMM on tcgen05 in tf32.  tf32 truncates the
# inputs to 10 mantissa bits (max-abs error 0.8e-3 .. 2.5e-3 on unit-variance features, the fp32 bound is 1e-3) and
# the kernel is no faster than the exact fp32 path yet (csrc/correlation.cu), so the default stays exact.
CORRELATION_TF32 = False


class _FunctionCorrelation(Function):
    @staticmethod
    def forward(ctx, first, second):
        assert first.is_contiguous() is True    # pwc/correlation/correlation.py:286-287
        assert second.is_contiguous() is True
        if not first.is_cuda:
            raise NotImplementedError()          # pwc/correlation/correlation.py:324-325
        if first.shape != second.shape or first.dim() != 4:
            raise ValueError(f"correlation: shapes {tuple(first.shape)} / {tuple(second.shape)}")
        n, c, h, w = first.shape
        code = _dtype_code("FunctionCorrelation", first)
        second = second.to(first.dtype)
        out = first.new_empty((n, 81, h, w))
        _launch("correlation_forward_ex", first, second, out, n, c, h, w, code, L.CORR_TF32 if CORRELATION_TF32 else 0)
        ctx.save_for_backward(first, second)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        first, second = ctx.saved_tensors
        n, c, h, w = first.shape
        g1 = torch.empty_like(first) if ctx.needs_input_grad[0] else None
        g2 = torch.empty_like(second) if ctx.needs_input_grad[1] else None
        if g1 is not None or g2 is not None:
            _launch("correlation_backward", first, second, gout.to(first.dtype).contiguous(), g1, g2, n, c, h, w,
                    _dtype_code("FunctionCorrelation", first))
        return g1, g2


def FunctionCorrelation(tenFirst, tenSecond):
    """Drop-in for ``pwc.correlation.correlation.FunctionCorrelation`` (keyword names as used at
    models/pwc_net.py:157-158,165-167)."""
    return _FunctionCorrelation.apply(tenFirst, tenSecond)


class ModuleCorrelation(nn.Module):
    def forward(self, tenFirst, tenSecond):
        return _FunctionCorrelation.apply(tenFirst, tenSecond)


# ------------------------------------------------------------------------------------------
# fused inference-only producers / consumers around the hot path (no autograd: the callers in
# eavsr_b200.model use the PyTorch modules whenever a gradient is required)
# ------------------------------------------------------------------------------------------
def fused_inference_ok(*tensors) -> bool:
    """True when the fused (non-differentiable) kernels may be used: autograd is off (``torch.no_grad()`` /
    ``inference_mode``) and every tensor is a CUDA fp32 / bf16 tensor."""
    if torch.is_grad_enabled():
        # the fused kernels have no backward; callers only see a subset of the parameters a fused op consumes,
        # so "none of these requires grad" would not be a safe test (frozen encoder, trainable alignment)
        return False
    ts = [t for t in tensors if t is not None]
    if not all(t.is_cuda for t in ts):
        return False
    return all(t.dtype in _DTYPES for t in ts)


def adapt_mix(a, b, w1, b1, w2, b2, negative_slope: float = 0.2):
    """``concat2(concat(cat[a, b]))`` of the reference's AdaptBlocks (models/networks.py:289-290,299):
    depthwise 3x3 + LeakyReLU + grouped (2->1) 3x3 + LeakyReLU in one pass.  a, b: (n,64,h,w)."""
    _require_cuda("adapt_mix", a, b, w1, b1, w2, b2)
    n, c, h, w = a.shape
    ad = a.contiguous(memory_format=torch.channels_last)
    out = torch.empty_like(ad)
    _launch("adapt_mix_forward", ad, b.to(a.dtype).contiguous(memory_format=torch.channels_last),
            *(_param(t, a.dtype) for t in (w1, b1, w2, b2)), out, n, c, h, w, float(negative_slope),
            _dtype_code("adapt_mix", ad))
    return out


def affine_offsets_mask(transform, translation, mask_logits, deform_groups: int, transform_bias=None,
                        translation_bias=None, mask_bias=None):
    """Per-group affine offset expansion ``T*R - R + t`` and ``sigmoid(mask_logits)``
    (models/networks.py:302-313) -> fp32 NCHW (offset (n,18D,h,w), mask (n,9D,h,w) or None).
    The optional biases are added to T / t / logits first (bias-free producing convolutions)."""
    _require_cuda("affine_offsets_mask", transform, translation, mask_logits)
    n, _, h, w = transform.shape
    D = deform_groups
    translation = translation.to(transform.dtype)
    offset = torch.empty((n, 18 * D, h, w), dtype=torch.float32, device=transform.device)
    mask = None
    if mask_logits is not None:
        mask_logits = mask_logits.to(transform.dtype)
        mask = torch.empty((n, 9 * D, h, w), dtype=torch.float32, device=transform.device)
    biases = [_param(t, transform.dtype) for t in (transform_bias, translation_bias, mask_bias)]
    _launch("affine_offsets_forward", transform, _strides(transform), translation, _strides(translation),
            mask_logits, _strides(mask_logits), *biases, offset, mask, n, D, h, w,
            _dtype_code("affine_offsets_mask", transform))
    return offset, mask


def dcn_affine_eligible(x, affine, weight, deform_groups: int) -> bool:
    """True when `dcn_affine` can run: inference, bf16 channels_last 64-channel features, a dense
    (n, 15*dg, h, w) channels_last bf16 affine block, 64->64 3x3 weights, deform_groups = 8."""
    return (deform_groups == 8 and x.dim() == 4 and x.shape[1] == 64 and x.dtype == torch.bfloat16
            and tuple(weight.shape) == (64, 64, 3, 3) and affine.dtype == torch.bfloat16
            and affine.shape[1] == 15 * deform_groups and affine.shape[0] == x.shape[0]
            and affine.shape[2:] == x.shape[2:] and x.shape[2] * x.shape[3] <= (1 << 24)
            and affine.is_contiguous(memory_format=torch.channels_last) and affine.data_ptr() % 16 == 0
            and fused_inference_ok(x, affine, weight))


def dcn_affine(x, affine, affine_bias, weight, bias, deform_groups: int = 8, static_weight: bool = False,
               flags: int = 0, out=None):
    """DCNv2 with the offset generation fused in (SURVEY.md section 8 row f1): equals
    ``modulated_deform_conv2d(x, *affine_offsets_mask(T, t, m, dg, bT, bt, bm), weight, bias, 1, 1, 1, 1, dg)``
    with ``T, t, m = affine[:, :4dg], affine[:, 4dg:6dg], affine[:, 6dg:]`` (the raw outputs of
    AdaptBlockOffset's three convolutions, models/networks.py:302-315) and ``affine_bias`` their
    concatenated biases -- without the (n, 27*dg, h, w) fp32 offset / mask tensors in HBM.
    Inference only; check `dcn_affine_eligible` first.  ``out`` may be a 64-channel slice (dim 1) of a wider
    channels_last bf16 buffer: the result is written in place there (no torch.cat copy afterwards)."""
    _require_cuda("dcn_affine", x, affine, weight)
    n, c, h, w = x.shape
    xd = x.contiguous(memory_format=torch.channels_last)
    if out is None:
        out = torch.empty_like(xd)
    else:
        assert out.shape == xd.shape and out.dtype == xd.dtype and out.stride(1) == 1, "dcn_affine: bad out view"
    code = _dtype_code("dcn_affine", xd)
    ws_bytes = L.load().eavsr_dcn_forward_workspace(64, 64, 3, 3, 1, deform_groups, code)
    ws, packed, commit = _dcn_workspace(weight, x.dtype, ws_bytes, static_weight)
    if packed:
        flags |= DCN_WS_PACKED
    _launch("dcn_affine_forward", xd, _strides(xd), affine, _param(affine_bias, x.dtype), _param(weight, x.dtype),
            _param(bias, x.dtype), out, _strides(out), n, h, w, deform_groups, code, ws, ws.numel(), flags)
    commit()
    return out


def ca_residual(res, skip, w1, b1, w2, b2, reduction: int = 16, res_bias=None):
    """``r * CALayer(r) + skip`` with ``r = res + res_bias`` -- the tail of the reference's RCABlock
    (models/networks.py:449-465) with two kernels (channel sums; MLP + scale + residual).
    ``res_bias`` lets the producing convolution run bias-free.  res, skip: (n,64,h,w)."""
    _require_cuda("ca_residual", res, skip, w1, b1, w2, b2)
    n, c, h, w = res.shape
    rd = res.contiguous(memory_format=torch.channels_last)
    out = torch.empty_like(rd)
    sums = torch.empty((n, c), dtype=torch.float32, device=res.device)
    _launch("ca_residual_forward", rd, skip.to(res.dtype).contiguous(memory_format=torch.channels_last),
            *(_param(t, res.dtype) for t in (w1, b1, w2, b2, res_bias)), out, sums, n, c, h, w, reduction,
            _dtype_code("ca_residual", rd))
    return out


def bias_act_(x, bias, negative_slope: float = 1.0):
    """In place ``x = LeakyReLU_slope(x + bias[c])`` on a channels_last tensor (slope 1: bias only,
    0: ReLU).  Returns x."""
    _require_cuda("bias_act_", x, bias)
    n, c, h, w = x.shape
    if not x.is_contiguous(memory_format=torch.channels_last):
        raise ValueError("bias_act_: x must be dense channels_last")
    _launch("bias_act_forward", x, _param(bias, x.dtype), c, n * h * w, float(negative_slope),
            _dtype_code("bias_act_", x))
    return x


class _GroupedConv3x3Fn(Function):
    """Grouped 3x3 convolution (groups = out channels, 1 or 2 inputs per group) with its backward on the library's
    kernels (csrc/grouped_conv.cu).  NHWC, fp32 / bf16; gradients of weight and bias are accumulated in fp32."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        n, cin, h, w = x.shape
        cout = weight.shape[0]
        xd = x.contiguous(memory_format=torch.channels_last)
        wd = _param(weight, xd.dtype)
        out = torch.empty((n, cout, h, w), dtype=xd.dtype, device=xd.device, memory_format=torch.channels_last)
        _launch("grouped_conv3x3_forward", xd, wd, _param(bias, xd.dtype), out, n, cin, cout, h, w,
                _dtype_code("grouped_conv3x3", xd))
        ctx.save_for_backward(xd, wd)
        ctx.has_bias, ctx.wdtype, ctx.bdtype = bias is not None, weight.dtype, None if bias is None else bias.dtype
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        xd, wd = ctx.saved_tensors
        n, cin, h, w = xd.shape
        cout = wd.shape[0]
        need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2])
        g = gout.to(xd.dtype).contiguous(memory_format=torch.channels_last)
        gx = torch.empty_like(xd) if need_x else None
        gw = torch.zeros(wd.shape, dtype=torch.float32, device=xd.device) if need_w else None
        gb = torch.zeros(cout, dtype=torch.float32, device=xd.device) if need_w else None
        _launch("grouped_conv3x3_backward", g, xd, wd, gx, gw, gb, n, cin, cout, h, w, _dtype_code("grouped_conv3x3", xd))
        return gx, _grad(gw, ctx.wdtype), (_grad(gb, ctx.bdtype) if ctx.has_bias else None)


def grouped_conv3x3_eligible(conv: nn.Conv2d, x) -> bool:
    """True for the grouped 3x3 convolutions of the AdaptBlocks (groups = out channels, 1 or 2 inputs per group,
    stride 1, padding 1) on CUDA fp32 / bf16 tensors with channel counts that are multiples of 8."""
    return (isinstance(conv, nn.Conv2d) and x.is_cuda and x.dim() == 4 and conv.kernel_size == (3, 3)
            and conv.stride == (1, 1) and conv.padding == (1, 1) and conv.dilation == (1, 1) and conv.padding_mode == "zeros"
            and conv.groups == conv.out_channels and conv.in_channels // conv.out_channels in (1, 2)
            and conv.in_channels % conv.out_channels == 0 and conv.out_channels % 8 == 0 and conv.in_channels % 8 == 0
            and 256 % (conv.in_channels // 8) == 0 and x.shape[1] == conv.in_channels)


def grouped_conv3x3(conv: nn.Conv2d, x):
    """``conv(x)`` for an eligible grouped 3x3 convolution, differentiable, on the library's kernels; follows
    torch.autocast like nn.Conv2d does (inputs and parameters are cast to the autocast dtype)."""
    w, b = conv.weight, conv.bias
    if torch.is_autocast_enabled():
        dt = torch.get_autocast_dtype("cuda") if hasattr(torch, "get_autocast_dtype") else torch.get_autocast_gpu_dtype()
        x, w, b = x.to(dt), w.to(dt), None if b is None else b.to(dt)
        with torch.autocast("cuda", enabled=False):
            return _GroupedConv3x3Fn.apply(x, w, b)
    if x.dtype not in _DTYPES:
        raise TypeError(f"eavsr_b200.grouped_conv3x3: dtype {x.dtype} not supported (float32 / bfloat16)")
    return _GroupedConv3x3Fn.apply(x, w.to(x.dtype), None if b is None else b.to(x.dtype))


def _channel_sums(x):
    """(n, 64) fp32 sums over (h, w) of a CUDA channels_last 64-channel fp32 / bf16 tensor."""
    n, c, h, w = x.shape
    sums = torch.empty((n, c), dtype=torch.float32, device=x.device)
    _launch("channel_sum_forward", x, sums, n, c, h * w, _dtype_code("channel_sum", x))
    return sums


def _channel_sum_ok(x) -> bool:
    return (x.is_cuda and x.dim() == 4 and x.shape[1] == 64 and x.dtype in _DTYPES and x.shape[0] <= 65535
            and x.is_contiguous(memory_format=torch.channels_last) and x.data_ptr() % 16 == 0)


class _AddBiasFn(Function):
    """y + bias[c] whose bias gradient is the library's channel sum (fp32) instead of ATen's reduction."""

    @staticmethod
    def forward(ctx, y, bias):
        ctx.bdtype = bias.dtype
        return y + bias.to(y.dtype).view(1, -1, 1, 1)

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        gb = None
        if ctx.needs_input_grad[1]:
            g = gout if gout.is_contiguous(memory_format=torch.channels_last) else gout.contiguous(memory_format=torch.channels_last)
            gb = (_channel_sums(g).sum(0) if _channel_sum_ok(g) else g.float().sum((0, 2, 3))).to(ctx.bdtype)
        return gout, gb


def conv2d_native_bias_grad(conv: nn.Conv2d, x):
    """``conv(x)`` (differentiable) with the bias gradient computed by the library's channel-sum kernel: for the
    64-output convolutions of the residual backbone ATen's `grad.sum((0, 2, 3))` on channels_last tensors was 12 %
    of the training step.  Any other convolution runs unchanged."""
    if conv.bias is None or conv.out_channels != 64 or not x.is_cuda or not torch.is_grad_enabled():
        return conv(x)
    y = F.conv2d(x, conv.weight, None, conv.stride, conv.padding, conv.dilation, conv.groups)
    return _AddBiasFn.apply(y, conv.bias)


class _ChannelMeanFn(Function):
    """adaptive_avg_pool2d(x, 1) for channels_last 64-channel maps on the library's channel-sum kernel."""

    @staticmethod
    def forward(ctx, x):
        ctx.shape = x.shape
        n, c, h, w = x.shape
        return (_channel_sums(x) * (1.0 / (h * w))).to(x.dtype).view(n, c, 1, 1)

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        n, c, h, w = ctx.shape
        g = (gout * (1.0 / (h * w))).expand(n, c, h, w)
        return g.contiguous(memory_format=torch.channels_last)


class _ScaleResidualFn(Function):
    """res * scale + skip (scale broadcast over h, w) whose scale gradient sum_hw(grad * res) is one pass of the
    library's channel-dot kernel instead of a multiply + ATen reduction."""

    @staticmethod
    def forward(ctx, res, scale, skip):
        ctx.save_for_backward(res, scale)
        return torch.addcmul(skip, res, scale)

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        res, scale = ctx.saved_tensors
        g = gout if gout.is_contiguous(memory_format=torch.channels_last) else gout.contiguous(memory_format=torch.channels_last)
        gres = g * scale if ctx.needs_input_grad[0] else None
        gscale = None
        if ctx.needs_input_grad[1]:
            n, c, h, w = res.shape
            sums = torch.empty((n, c), dtype=torch.float32, device=res.device)
            _launch("channel_dot_forward", g, res, sums, n, c, h * w, _dtype_code("scale_residual", res))
            gscale = sums.to(scale.dtype).view(n, c, 1, 1)
        return gres, gscale, gout if ctx.needs_input_grad[2] else None


def scale_residual(res, scale, skip):
    """``res * scale + skip`` (differentiable) for RCABlock's channel attention; native scale gradient for CUDA
    channels_last 64-channel maps."""
    if (_channel_sum_ok(res) and scale.shape == (res.shape[0], 64, 1, 1) and skip.shape == res.shape
            and res.dtype == scale.dtype == skip.dtype and skip.is_contiguous(memory_format=torch.channels_last)):
        return _ScaleResidualFn.apply(res, scale, skip)
    return res * scale + skip


def channel_mean(x):
    """``F.adaptive_avg_pool2d(x, 1)`` (differentiable); native reduction for CUDA channels_last 64-channel maps."""
    if _channel_sum_ok(x):
        return _ChannelMeanFn.apply(x)
    return F.adaptive_avg_pool2d(x, 1)


def cat_channels(tensors, out=None, channel_offset: int = 0):
    """``torch.cat(tensors, 1)`` for channels_last tensors in one coalesced pass (inference: no autograd), optionally
    straight into the channel slice ``[channel_offset, +sum C_i)`` of an existing channels_last buffer ``out``
    (returned).  Falls back to ``torch.cat`` / ``copy_`` whenever the layout, dtype or a needed gradient rules the
    kernel out (models/eavsrp_model.py:271-324, 350-364)."""
    ts = list(tensors)
    x0 = ts[0]
    vec = 16 // x0.element_size() if x0.dtype in (torch.float32, torch.bfloat16) else 0
    ok = (vec > 0 and 1 <= len(ts) <= 8 and x0.is_cuda and fused_inference_ok(*ts)
          and all(t.dim() == 4 and t.dtype == x0.dtype and t.device == x0.device and t.shape[0] == x0.shape[0]
                  and t.shape[2:] == x0.shape[2:] and t.shape[1] % vec == 0
                  and t.is_contiguous(memory_format=torch.channels_last) and t.data_ptr() % 16 == 0 for t in ts))
    ctot = sum(t.shape[1] for t in ts)
    if out is not None:
        ok = ok and (out.dtype == x0.dtype and out.device == x0.device and out.dim() == 4 and out.shape[0] == x0.shape[0]
                     and out.shape[2:] == x0.shape[2:] and out.is_contiguous(memory_format=torch.channels_last)
                     and out.shape[1] % vec == 0 and channel_offset % vec == 0 and channel_offset + ctot <= out.shape[1])
    if not ok:
        if out is None:
            return torch.cat(ts, 1)
        out[:, channel_offset:channel_offset + ctot].copy_(torch.cat(ts, 1) if len(ts) > 1 else x0)
        return out
    n, _, h, w = x0.shape
    if out is None:
        out = torch.empty((n, ctot, h, w), dtype=x0.dtype, device=x0.device, memory_format=torch.channels_last)
    ptrs = (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    chans = (ctypes.c_int * len(ts))(*[t.shape[1] for t in ts])
    _launch("nhwc_cat_forward", ptrs, chans, len(ts), out, out.shape[1], channel_offset, n * h * w,
            _dtype_code("cat_channels", x0))
    return out


def conv2d_bias_act(conv: nn.Conv2d, x, negative_slope: float = 1.0):
    """cuDNN convolution with its bias add and (Leaky)ReLU folded into one vectorised epilogue pass
    (inference).  Falls back to ``act(conv(x))`` whenever a gradient is needed or the layout does
    not allow the fused epilogue."""
    vec = 16 // x.element_size()
    if (conv.bias is None or conv.out_channels % vec != 0 or not fused_inference_ok(x, conv.weight)
            or not x.is_contiguous(memory_format=torch.channels_last)):
        y = conv2d_native_bias_grad(conv, x)      # (== conv(x); training: bias gradient on the channel-sum kernel)
        if negative_slope == 1.0:
            return y
        return torch.relu_(y) if negative_slope == 0.0 else torch.nn.functional.leaky_relu_(y, negative_slope)
    y = torch.nn.functional.conv2d(x, conv.weight, None, conv.stride, conv.padding, conv.dilation, conv.groups)
    if not y.is_contiguous(memory_format=torch.channels_last):
        y = y.contiguous(memory_format=torch.channels_last)
    return bias_act_(y, conv.bias, negative_slope)


# ------------------------------------------------------------------------------------------
# tcgen05 3x3 convolution 64 -> 64 (bf16 NHWC) with fused bias / activation / channel sums
# ------------------------------------------------------------------------------------------
def conv3x3_64_eligible(conv: nn.Conv2d, x) -> bool:
    return (isinstance(conv, nn.Conv2d) and conv.in_channels == 64 and conv.out_channels == 64
            and conv.kernel_size == (3, 3) and conv.stride == (1, 1) and conv.padding == (1, 1)
            and conv.dilation == (1, 1) and conv.groups == 1 and conv.padding_mode == "zeros"
            and x.dtype == torch.bfloat16 and x.dim() == 4 and x.shape[1] == 64
            and fused_inference_ok(x, conv.weight))


def _packed_conv_weight(conv: nn.Conv2d, device, kind: str = "conv3x3") -> torch.Tensor:
    """Weights re-packed once into the swizzled bf16 tiles the MMA of ``eavsr_<kind>_*`` reads: 9 64x64 tiles for
    ``conv3x3``, 9 16x64 tiles for ``sr_tail`` (cached on the module, invalidated by the parameter's version
    counter / storage)."""
    w = conv.weight
    key = (kind, w.data_ptr(), w._version, str(device))
    hit = getattr(conv, "_eavsr_packed", None)
    if hit is not None and hit[0] == key:
        return hit[1]
    packed = torch.empty(getattr(L.load(), f"eavsr_{kind}_packed_weight_bytes")(), dtype=torch.uint8, device=device)
    _launch(f"{kind}_pack_weight", _param(w.to(device), torch.bfloat16), packed, conv.in_channels, conv.out_channels,
            L.BF16)
    conv._eavsr_packed = (key, packed)
    return packed


def conv3x3_64(conv: nn.Conv2d, x, negative_slope: float = 1.0, want_sums: bool = False, sums_out=None):
    """``LeakyReLU_slope(conv(x))`` for a 64->64 3x3 stride-1 pad-1 convolution on tcgen05 (bf16
    channels_last, inference).  With ``want_sums`` also returns the per-(n, channel) sums of the
    output over (h, w) in fp32, computed in the epilogue; ``sums_out`` is an already ZEROED (n, 64)
    fp32 buffer to accumulate them into (one memset for a whole residual group instead of one per
    convolution).  Check `conv3x3_64_eligible` first."""
    n, c, h, w = x.shape
    xd = x.contiguous(memory_format=torch.channels_last)
    out = torch.empty_like(xd)
    sums = None
    if want_sums:
        if sums_out is not None:
            assert sums_out.shape == (n, 64) and sums_out.dtype == torch.float32 and sums_out.is_contiguous()
            sums = sums_out
        else:
            sums = torch.empty((n, 64), dtype=torch.float32, device=x.device)
    _launch("conv3x3_forward", xd, _packed_conv_weight(conv, x.device), _param(conv.bias, torch.bfloat16), out, sums,
            n, 64, 64, h, w, float(negative_slope), L.BF16,
            L.CONV_SUMS_PREZEROED if (want_sums and sums_out is not None) else 0)
    return (out, sums) if want_sums else out


def conv3x3_64_ca(conv: nn.Conv2d, skip, res, res_sums, w1, b1, w2, b2, negative_slope: float = 1.0,
                  want_sums: bool = False, sums_out=None):
    """``y = res * sigmoid(MLP(mean(res))) + skip`` (the tail of the previous RCABlock) folded into
    ``LeakyReLU_slope(conv(y))``: returns ``(out, y)`` or ``(out, y, sums)``.  ``res_sums`` are the channel
    sums of ``res`` from the `conv3x3_64(..., want_sums=True)` call that produced it.  Same eligibility as
    `conv3x3_64`, batch <= 8."""
    n, c, h, w = skip.shape
    sd = skip.contiguous(memory_format=torch.channels_last)
    out = torch.empty_like(sd)
    y = torch.empty_like(sd)
    sums = None
    if want_sums:
        sums = sums_out if sums_out is not None else torch.empty((n, 64), dtype=torch.float32, device=skip.device)
    _launch("conv3x3_ca_forward", sd, res.contiguous(memory_format=torch.channels_last), res_sums,
            *(_param(t, skip.dtype) for t in (w1, b1, w2, b2)), y, _packed_conv_weight(conv, skip.device),
            _param(conv.bias, torch.bfloat16), out, sums, n, h, w, float(negative_slope), L.BF16,
            L.CONV_SUMS_PREZEROED if (want_sums and sums_out is not None) else 0)
    return (out, y, sums) if want_sums else (out, y)


def conv3x3_chain_eligible(convs, x) -> bool:
    """True when `rca_group_chain` can run the whole residual group in one launch."""
    return (len(convs) >= 2 and len(convs) <= 64 and x.dim() == 4 and x.shape[0] <= 8
            and all(conv3x3_64_eligible(c, x) for c in convs))


def rca_group_chain(blocks, tail_conv, x):
    """``tail_conv(RCAB_k(...RCAB_1(x)))`` of an RCAGroup (models/networks.py:449-482; the caller adds the group's
    skip) as ONE cooperative launch of the tcgen05 convolution (eavsr_conv3x3_chain_forward): 2 layers per block --
    conv + ReLU with the previous block's channel attention folded into its input, conv + channel sums -- and the
    closing convolution.  ``blocks``: modules with ``res[0]``, ``res[2]`` (3x3 convs) and ``ca.conv_du`` (the
    squeeze-excite 1x1 convs); inference only (check `conv3x3_chain_eligible`)."""
    n, c, h, w = x.shape
    dev = x.device
    xd = x.contiguous(memory_format=torch.channels_last)
    # activations: h (conv1 output), res (conv2 output), y ping-pong (block outputs); sums one row per block
    hbuf, rbuf, out = torch.empty_like(xd), torch.empty_like(xd), torch.empty_like(xd)
    ybuf = [torch.empty_like(xd), torch.empty_like(xd)]
    pool = torch.zeros((len(blocks), n, 64), dtype=torch.float32, device=dev)
    sync = torch.empty(1, dtype=torch.int32, device=dev)
    keep = []                      # `arr` holds raw addresses: converted parameters must outlive the launch

    def par(t):
        t = _param(t, torch.bfloat16)
        keep.append(t)
        return t.data_ptr()

    layers = []
    y = xd
    for i, blk in enumerate(blocks):
        c1, c2 = blk.res[0], blk.res[2]
        if i == 0:
            layers.append(dict(x=y, conv=c1, out=hbuf, slope=0.0))
        else:
            du = blocks[i - 1].ca.conv_du
            ynew = ybuf[i & 1]
            layers.append(dict(x=y, conv=c1, out=hbuf, slope=0.0, res=rbuf, res_sums=pool[i - 1], du=du, y_out=ynew))
            y = ynew
        layers.append(dict(x=hbuf, conv=c2, out=rbuf, slope=1.0, sums=pool[i]))
    du = blocks[-1].ca.conv_du
    layers.append(dict(x=y, conv=tail_conv, out=out, slope=1.0, res=rbuf, res_sums=pool[len(blocks) - 1], du=du,
                       y_out=ybuf[len(blocks) & 1]))
    arr = (L.ConvLayer * len(layers))()
    for a, d in zip(arr, layers):
        conv = d["conv"]
        a.x, a.out = d["x"].data_ptr(), d["out"].data_ptr()
        a.packed_weight = _packed_conv_weight(conv, dev).data_ptr()
        a.bias = par(conv.bias) if conv.bias is not None else None
        a.channel_sums = d["sums"].data_ptr() if "sums" in d else None
        a.negative_slope = d["slope"]
        if "res" in d:
            du = d["du"]
            a.res, a.res_sums, a.y_out = d["res"].data_ptr(), d["res_sums"].data_ptr(), d["y_out"].data_ptr()
            a.w1, a.b1, a.w2, a.b2 = par(du[0].weight), par(du[0].bias), par(du[2].weight), par(du[2].bias)
    _launch("conv3x3_chain_forward", arr, len(layers), n, h, w, L.BF16, sync)
    return out


def ca_scale(res, skip, sums, w1, b1, w2, b2, reduction: int = 16, res_bias=None):
    """``(res + res_bias) * sigmoid(MLP(sums / HW + res_bias)) + skip`` with channel sums that were
    produced by the convolution's epilogue (see `conv3x3_64`)."""
    n, c, h, w = res.shape
    rd = res.contiguous(memory_format=torch.channels_last)
    out = torch.empty_like(rd)
    _launch("ca_scale_forward", rd, skip.to(res.dtype).contiguous(memory_format=torch.channels_last), sums,
            *(_param(t, res.dtype) for t in (w1, b1, w2, b2, res_bias)), out, n, c, h, w, reduction,
            _dtype_code("ca_scale", rd))
    return out


def conv2d_bias_act_shuffle(conv: nn.Conv2d, x, negative_slope: float = 1.0):
    """``PixelShuffle(2)(LeakyReLU_slope(conv(x)))`` (LeakyReLU commutes with the shuffle): bias-free cuDNN
    convolution, then bias + activation + shuffle in one NHWC pass.  Falls back to the PyTorch ops whenever
    a gradient is needed or the layout does not allow it."""
    cout = conv.out_channels
    vec = 16 // x.element_size()
    if (cout % (4 * vec) != 0 or not fused_inference_ok(x, conv.weight)
            or not x.is_contiguous(memory_format=torch.channels_last)):
        y = torch.nn.functional.pixel_shuffle(conv(x), 2)
        return y if negative_slope == 1.0 else torch.nn.functional.leaky_relu(y, negative_slope)
    y = torch.nn.functional.conv2d(x, conv.weight, None, conv.stride, conv.padding, conv.dilation, conv.groups)
    if not y.is_contiguous(memory_format=torch.channels_last):
        y = y.contiguous(memory_format=torch.channels_last)
    n, _, h, w = y.shape
    out = torch.empty((n, cout // 4, 2 * h, 2 * w), dtype=y.dtype, device=y.device, memory_format=torch.channels_last)
    _launch("bias_act_shuffle_forward", y, _param(conv.bias, y.dtype), out, n, cout // 4, h, w, float(negative_slope),
            _dtype_code("bias_act_shuffle", y))
    return out


# ------------------------------------------------------------------------------------------
# reconstruction tail -> uint8 frames on tcgen05 (conv_last + bilinear base + visuals)
# ------------------------------------------------------------------------------------------
def sr_tail_u8_eligible(conv_last: nn.Conv2d, x) -> bool:
    """True when `sr_tail_u8` can run: ``conv_last`` is a 64 -> 3 3x3 stride-1 pad-1 convolution, ``x`` a dense
    channels_last bf16 CUDA map of 64 channels, and no gradient is needed."""
    return (isinstance(conv_last, nn.Conv2d) and conv_last.in_channels == 64 and conv_last.out_channels == 3
            and conv_last.kernel_size == (3, 3) and conv_last.stride == (1, 1) and conv_last.padding == (1, 1)
            and conv_last.dilation == (1, 1) and conv_last.groups == 1 and conv_last.padding_mode == "zeros"
            and x.dtype == torch.bfloat16 and x.dim() == 4 and x.shape[1] == 64
            and x.is_contiguous(memory_format=torch.channels_last) and fused_inference_ok(x, conv_last.weight))


def _check_tail_lr(name: str, x, lr, scale: int) -> None:
    n, c, h, w = x.shape
    if lr.dtype != torch.float32 or tuple(lr.shape) != (n, 3, h // scale, w // scale):
        raise ValueError(f"eavsr_b200.{name}: lr must be fp32 (n, 3, H/s, W/s), got {lr.dtype} {tuple(lr.shape)}")


def sr_tail_u8(conv_last: nn.Conv2d, x, lr, scale: int, out, out_h: int, out_w: int):
    """``out[n, y, x, :] = round(clamp(255 * (conv_last(x) + interpolate(lr, scale, bilinear)), 0, 255))`` for
    ``y < out_h``, ``x < out_w`` in one kernel (models/eavsrp_model.py:350-364 and the visuals of
    models/base_model.py:146-150).  ``x``: (n, 64, H, W) bf16 channels_last; ``lr``: (n, 3, H/scale, W/scale) fp32,
    any strides; ``out``: (n, out_h, out_w, 3) uint8, any strides (e.g. ``clip[:, i]`` of an (n, t, Ho, Wo, 3)
    tensor).  The residual is accumulated and added in fp32, never rounded to bf16.  Check `sr_tail_u8_eligible`
    first.  Returns ``out``."""
    _require_cuda("sr_tail_u8", x, lr, out)
    n, c, h, w = x.shape
    _check_tail_lr("sr_tail_u8", x, lr, scale)
    if out.dtype != torch.uint8 or tuple(out.shape) != (n, out_h, out_w, 3):
        raise ValueError(f"eavsr_b200.sr_tail_u8: out must be uint8 (n, out_h, out_w, 3), got {out.dtype} "
                         f"{tuple(out.shape)}")
    _launch("sr_tail_u8_forward", x, _strides(x), _packed_conv_weight(conv_last, x.device, "sr_tail"),
            _param(conv_last.bias, torch.bfloat16), lr, L.Strides(*lr.stride()), out, L.Strides(*out.stride()),
            n, c, h, w, int(scale), int(out_h), int(out_w), L.BF16)
    return out


def sr_tail_yuv420(conv_last: nn.Conv2d, x, lr, scale: int, y_out, u_out, v_out, out_h: int, out_w: int, kr: float,
                   kb: float):
    """The tail of `sr_tail_u8` written as 8-bit limited-range Y'CbCr 4:2:0 planes: ``rgb_to_yuv420(conv_last(x) +
    interpolate(lr, scale, bilinear), kr, kb)`` (`eavsr_b200.yuv`) cropped to ``out_h`` x ``out_w``, in one kernel.
    ``y_out``: (n, out_h, out_w) uint8; ``u_out``, ``v_out``: (n, out_h/2, out_w/2) uint8; any strides, so I420
    planes or the interleaved chroma of NV12 (``uv[..., 0::2]``, ``uv[..., 1::2]``) are written in place.  ``x`` and
    ``lr`` as for `sr_tail_u8`, with the same eligibility (`sr_tail_u8_eligible`).  Returns ``(y_out, u_out, v_out)``."""
    if out_h % 2 or out_w % 2:
        raise ValueError(f"eavsr_b200.sr_tail_yuv420: 4:2:0 needs an even crop, got {out_h}x{out_w}")
    n = x.shape[0]
    _check_tail_lr("sr_tail_yuv420", x, lr, scale)
    for name, p, shape in (("y_out", y_out, (n, out_h, out_w)), ("u_out", u_out, (n, out_h // 2, out_w // 2)),
                           ("v_out", v_out, (n, out_h // 2, out_w // 2))):
        if p.dtype != torch.uint8 or tuple(p.shape) != shape:
            raise ValueError(f"eavsr_b200.sr_tail_yuv420: {name} must be uint8 {shape}, got {p.dtype} {tuple(p.shape)}")
    _require_cuda("sr_tail_yuv420", x, lr, y_out, u_out, v_out)
    planes = [a for p in (y_out, u_out, v_out) for a in (p, L.Strides(*p.unsqueeze(1).stride()))]
    _launch("sr_tail_yuv420_forward", x, _strides(x), _packed_conv_weight(conv_last, x.device, "sr_tail"),
            _param(conv_last.bias, torch.bfloat16), lr, L.Strides(*lr.stride()), *planes,
            n, x.shape[1], x.shape[2], x.shape[3], int(scale), int(out_h), int(out_w), float(kr), float(kb), L.BF16)
    return y_out, u_out, v_out


def sr_tail_u16(conv_last: nn.Conv2d, x, lr, scale: int, out, out_h: int, out_w: int, bits: int):
    """`sr_tail_u8` at 10, 12 or 16 bits: ``out[n, y, x, :] = round(clamp(M * (conv_last(x) + interpolate(lr, scale,
    bilinear)), 0, M))`` with ``M = 2**bits - 1``, the code in the low bits.  ``out``: (n, out_h, out_w, 3) uint16,
    any strides.  ``x`` and ``lr`` as for `sr_tail_u8`, with the same eligibility (`sr_tail_u8_eligible`).
    Returns ``out``."""
    check_bits("eavsr_b200.sr_tail_u16", bits, 0, allowed=(10, 12, 16))
    n, c, h, w = x.shape
    _check_tail_lr("sr_tail_u16", x, lr, scale)
    if out.dtype != torch.uint16 or tuple(out.shape) != (n, out_h, out_w, 3):
        raise ValueError(f"eavsr_b200.sr_tail_u16: out must be uint16 (n, out_h, out_w, 3), got {out.dtype} "
                         f"{tuple(out.shape)}")
    _require_cuda("sr_tail_u16", x, lr, out)
    _launch("sr_tail_u16_forward", x, _strides(x), _packed_conv_weight(conv_last, x.device, "sr_tail"),
            _param(conv_last.bias, torch.bfloat16), lr, L.Strides(*lr.stride()), out, L.Strides(*out.stride()),
            n, c, h, w, int(scale), int(out_h), int(out_w), int(bits), L.BF16)
    return out


def sr_tail_yuv420_u16(conv_last: nn.Conv2d, x, lr, scale: int, y_out, u_out, v_out, out_h: int, out_w: int,
                       kr: float, kb: float, bits: int, shift: int):
    """`sr_tail_yuv420` at 10, 12 or 16 bits: ``rgb_to_yuv420(conv_last(x) + interpolate(lr, scale, bilinear), kr, kb,
    bits, shift)`` (`eavsr_b200.yuv`) cropped to ``out_h`` x ``out_w``, in one kernel.  ``y_out``: (n, out_h, out_w)
    uint16; ``u_out``, ``v_out``: (n, out_h/2, out_w/2) uint16; any strides, so planar ``yuv420p10le`` (``shift=0``)
    or the interleaved chroma of P010 (``shift=6``, ``uv[..., 0::2]``, ``uv[..., 1::2]``) are written in place.
    ``x`` and ``lr`` as for `sr_tail_u8`, with the same eligibility.  Returns ``(y_out, u_out, v_out)``."""
    check_bits("eavsr_b200.sr_tail_yuv420_u16", bits, shift, allowed=(10, 12, 16))
    if out_h % 2 or out_w % 2:
        raise ValueError(f"eavsr_b200.sr_tail_yuv420_u16: 4:2:0 needs an even crop, got {out_h}x{out_w}")
    n = x.shape[0]
    _check_tail_lr("sr_tail_yuv420_u16", x, lr, scale)
    for name, p, shape in (("y_out", y_out, (n, out_h, out_w)), ("u_out", u_out, (n, out_h // 2, out_w // 2)),
                           ("v_out", v_out, (n, out_h // 2, out_w // 2))):
        if p.dtype != torch.uint16 or tuple(p.shape) != shape:
            raise ValueError(f"eavsr_b200.sr_tail_yuv420_u16: {name} must be uint16 {shape}, got {p.dtype} "
                             f"{tuple(p.shape)}")
    _require_cuda("sr_tail_yuv420_u16", x, lr, y_out, u_out, v_out)
    planes = [a for p in (y_out, u_out, v_out) for a in (p, L.Strides(*p.unsqueeze(1).stride()))]
    _launch("sr_tail_yuv420_u16_forward", x, _strides(x), _packed_conv_weight(conv_last, x.device, "sr_tail"),
            _param(conv_last.bias, torch.bfloat16), lr, L.Strides(*lr.stride()), *planes,
            n, x.shape[1], x.shape[2], x.shape[3], int(scale), int(out_h), int(out_w), float(kr), float(kb),
            int(bits), int(shift), L.BF16)
    return y_out, u_out, v_out


def sr_tail_u8_sse(conv_last: nn.Conv2d, x, lr, scale: int, hr, sse, out_h: int, out_w: int, out=None):
    """The squared error of `sr_tail_u8`'s frame against a ground-truth frame, in one kernel: ``sse[n] += sum over
    y < out_h, x < out_w, c of (q[n, y, x, c] - hr[n, y, x, c])**2``, exact in int64, where ``q`` is the frame
    `sr_tail_u8` writes; with ``out`` given, ``q`` is also written there, bit for bit as `sr_tail_u8` writes it.
    ``hr``: (n, out_h, out_w, 3) uint8, any strides; ``sse``: (n,) int64, any stride (e.g. ``sums[:, i]`` of an
    (n, t) tensor), added to and not overwritten; ``out``: as for `sr_tail_u8`, or None.  ``x`` and ``lr`` as for
    `sr_tail_u8`, with the same eligibility (`sr_tail_u8_eligible`).  Returns ``sse``."""
    n, c, h, w = x.shape
    _check_tail_lr("sr_tail_u8_sse", x, lr, scale)
    if hr.dtype != torch.uint8 or tuple(hr.shape) != (n, out_h, out_w, 3):
        raise ValueError(f"eavsr_b200.sr_tail_u8_sse: hr must be uint8 (n, out_h, out_w, 3), got {hr.dtype} "
                         f"{tuple(hr.shape)}")
    if sse.dtype != torch.int64 or tuple(sse.shape) != (n,):
        raise ValueError(f"eavsr_b200.sr_tail_u8_sse: sse must be int64 (n,), got {sse.dtype} {tuple(sse.shape)}")
    if out is not None and (out.dtype != torch.uint8 or tuple(out.shape) != (n, out_h, out_w, 3)):
        raise ValueError(f"eavsr_b200.sr_tail_u8_sse: out must be uint8 (n, out_h, out_w, 3), got {out.dtype} "
                         f"{tuple(out.shape)}")
    _require_cuda("sr_tail_u8_sse", x, lr, hr, sse, out)
    _launch("sr_tail_u8_sse_forward", x, _strides(x), _packed_conv_weight(conv_last, x.device, "sr_tail"),
            _param(conv_last.bias, torch.bfloat16), lr, L.Strides(*lr.stride()), hr, L.Strides(*hr.stride()),
            out, None if out is None else L.Strides(*out.stride()), sse, sse.stride(0),
            n, c, h, w, int(scale), int(out_h), int(out_w), L.BF16)
    return sse
