"""CPU tests of the PSNR evaluation: the ctypes prototype of eavsr_sr_tail_u8_sse_forward derived from the header, the
PSNR formula, and the input checks of EAVSRP.psnr_uint8 and ops.sr_tail_u8_sse, which must fail before anything is
launched."""
import math
from ctypes import POINTER, c_int, c_int64, c_longlong, c_void_p

import pytest
import torch
import torch.nn as nn

from eavsr_b200 import _lib as L
from eavsr_b200 import ops
from eavsr_b200.model import EAVSRP, psnr_from_sse


def test_prototype_comes_from_the_header():
    assert "eavsr_sr_tail_u8_sse_forward" in L.EXPORTED_SYMBOLS
    res, args = L._signatures()["eavsr_sr_tail_u8_sse_forward"]
    strides = POINTER(c_int64)
    assert res is c_int and len(args) == 21
    # x, x_strides, packed_weight, bias, lr, lr_strides, gt, gt_strides, out, out_strides, sse, sse_stride,
    # n, c, h, w, scale, out_h, out_w, dtype, stream
    assert args == ([c_void_p, strides, c_void_p, c_void_p, c_void_p, strides, c_void_p, strides, c_void_p, strides,
                     c_void_p, c_longlong] + [c_int] * 8 + [c_void_p])


def test_psnr_formula():
    samples = 3 * 64 * 96
    sse = torch.tensor([[0, 1, samples], [samples * 255 ** 2, 12345, 2 ** 40]], dtype=torch.int64)
    got = psnr_from_sse(sse, samples)
    assert got.dtype == torch.float64 and got.shape == sse.shape
    assert got[0, 0].item() == math.inf
    assert got[0, 2].item() == pytest.approx(20 * math.log10(255), abs=1e-12)          # an MSE of one level
    assert got[1, 0].item() == pytest.approx(0, abs=1e-12)
    for v, s in zip(got.flatten().tolist()[1:], sse.flatten().tolist()[1:]):
        assert v == pytest.approx(-10 * math.log10(s / samples / 255 ** 2), abs=1e-12)


# ------------------------------------------------------------------------------------------------
# input checks: nothing is launched
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def net():
    return EAVSRP(4, n_resblock=1).eval()


@pytest.fixture
def no_trunk(net, monkeypatch):
    def trunk(lrs):
        raise AssertionError("the trunk ran on rejected input")
    monkeypatch.setattr(net, "_trunk", trunk)
    return net


def u8(*shape, dtype=torch.uint8):
    return torch.zeros(shape, dtype=dtype)


FRAMES, HR = u8(1, 2, 64, 96, 3), u8(1, 2, 256, 384, 3)


@pytest.mark.parametrize("args, kwargs, err", [
    ((u8(1, 2, 64, 96, 3, dtype=torch.float32), HR), {}, TypeError),                  # float frames
    ((u8(1, 2, 64, 96, 3, dtype=torch.uint16), HR), {}, TypeError),
    ((FRAMES, u8(1, 2, 256, 384, 3, dtype=torch.float32)), {}, TypeError),             # float ground truth
    ((FRAMES, u8(1, 2, 256, 384, 3, dtype=torch.int16)), {}, TypeError),
    ((FRAMES, HR.numpy()), {}, TypeError),
    ((FRAMES, HR), {"out": u8(1, 2, 256, 384, 3, dtype=torch.int32)}, TypeError),
    ((u8(2, 64, 96, 3), HR), {}, ValueError),                                         # no batch dimension
    ((u8(1, 2, 64, 96, 4), HR), {}, ValueError),                                      # RGBA
    ((u8(1, 2, 3, 64, 96), HR), {}, ValueError),                                      # channels first
    ((u8(1, 2, 62, 96, 3), u8(1, 2, 248, 384, 3)), {}, ValueError),                   # under 64
    ((FRAMES, u8(1, 2, 128, 192, 3)), {}, ValueError),                                # ground truth at x2 for a x4 net
    ((FRAMES, u8(1, 3, 256, 384, 3)), {}, ValueError),                                # another clip length
    ((FRAMES, u8(2, 2, 256, 384, 3)), {}, ValueError),                                # another batch
    ((FRAMES, u8(1, 2, 256, 384, 4)), {}, ValueError),
    ((FRAMES, u8(1, 2, 3, 256, 384)), {}, ValueError),                                # planar ground truth
    ((FRAMES, HR), {"out": u8(1, 2, 256, 380, 3)}, ValueError),                       # out of the wrong size
    ((FRAMES, HR), {"out": u8(1, 2, 256, 384)}, ValueError),
    ((FRAMES, HR), {}, NotImplementedError),                                          # CPU tensors
    ((FRAMES, HR), {"out": u8(1, 2, 256, 384, 3)}, NotImplementedError),
    ((u8(1, 2, 65, 97, 3), u8(1, 2, 260, 388, 3)), {}, NotImplementedError),          # odd sizes are padded
])
def test_psnr_uint8_rejects_bad_input_before_any_launch(no_trunk, args, kwargs, err):
    before = L.launch_count()
    with pytest.raises(err):
        no_trunk.psnr_uint8(*args, **kwargs)
    assert L.launch_count() == before


def _op_args(**over):
    a = dict(conv_last=nn.Conv2d(64, 3, 3, 1, 1), x=torch.zeros(2, 64, 40, 48), lr=torch.zeros(2, 3, 10, 12), scale=4,
             hr=u8(2, 40, 48, 3), sse=torch.zeros(2, dtype=torch.int64), out_h=40, out_w=48)
    a.update(over)
    return a


@pytest.mark.parametrize("over, err", [
    ({"hr": u8(2, 40, 48, 3, dtype=torch.int16)}, ValueError),
    ({"hr": u8(2, 40, 47, 3)}, ValueError),
    ({"sse": torch.zeros(2, dtype=torch.int32)}, ValueError),                          # 32 bits overflow
    ({"sse": torch.zeros(2, 1, dtype=torch.int64)}, ValueError),
    ({"sse": torch.zeros(3, dtype=torch.int64)}, ValueError),
    ({"out": u8(2, 40, 48, 3, dtype=torch.uint16)}, ValueError),
    ({"out": u8(2, 40, 48, 4)}, ValueError),
    ({"lr": torch.zeros(2, 3, 20, 24)}, ValueError),                                 # LR of a x2 map
    ({}, NotImplementedError),                                                        # CPU tensors
    ({"out": u8(2, 40, 48, 3)}, NotImplementedError),
])
def test_sr_tail_u8_sse_rejects_bad_input_before_any_launch(over, err):
    before = L.launch_count()
    with pytest.raises(err):
        ops.sr_tail_u8_sse(**_op_args(**over))
    assert L.launch_count() == before
