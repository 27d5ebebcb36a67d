"""CPU tests of Y'CbCr 4:2:0 inference: the conversions of eavsr_b200/yuv.py, the ctypes prototype of
eavsr_sr_tail_yuv420_forward derived from the header, and the input checks of EAVSRP.forward_yuv420 and
ops.sr_tail_yuv420, which must fail before anything is launched."""
from ctypes import POINTER, c_float, c_int, c_int64, c_void_p

import numpy as np
import pytest
import torch
import torch.nn as nn

from eavsr_b200 import _lib as L
from eavsr_b200 import ops
from eavsr_b200.model import EAVSRP
from eavsr_b200.yuv import MATRICES, coefficients, rgb_to_yuv420, yuv420_to_rgb

# textbook 8-bit limited-range codes (Y', Cb, Cr) of white, black and the primaries
CODES = {
    "bt709": {(1, 1, 1): (235, 128, 128), (0, 0, 0): (16, 128, 128), (1, 0, 0): (63, 102, 240),
              (0, 1, 0): (173, 42, 26), (0, 0, 1): (32, 240, 118)},
    "bt601": {(1, 1, 1): (235, 128, 128), (0, 0, 0): (16, 128, 128), (1, 0, 0): (81, 90, 240),
              (0, 1, 0): (145, 54, 34), (0, 0, 1): (41, 240, 110)},
}


def flat(colours, size=2):
    """(k, 3) colours -> (k, 3, size, size) flat images."""
    return torch.as_tensor(colours, dtype=torch.float32)[:, :, None, None].expand(-1, -1, size, size).contiguous()


@pytest.mark.parametrize("matrix", sorted(MATRICES))
def test_known_codes(matrix):
    kr, kb = MATRICES[matrix]
    rgb, codes = zip(*CODES[matrix].items())
    y, u, v = rgb_to_yuv420(flat(rgb, 4), kr, kb)
    assert y.dtype == u.dtype == v.dtype == torch.uint8
    assert y.shape == (5, 4, 4) and u.shape == v.shape == (5, 2, 2)
    got = torch.stack([y[:, 0, 0], u[:, 0, 0], v[:, 0, 0]], 1)
    assert got.tolist() == [list(c) for c in codes]
    assert (y == y[:, :1, :1]).all() and (u == u[:, :1, :1]).all() and (v == v[:, :1, :1]).all()
    # and back: (n, t) = (1, 5)
    planes = [p.view(1, 5, *p.shape[1:]).expand(1, 5, *p.shape[1:]) for p in (y, u, v)]
    back = yuv420_to_rgb(*planes, kr, kb)
    assert back.shape == (1, 5, 3, 4, 4) and back.dtype == torch.float32
    assert (back[0] - flat(rgb, 4)).abs().max().item() < 0.01


@pytest.mark.parametrize("matrix", sorted(MATRICES))
def test_round_trip_of_flat_blocks_stays_within_quantisation(matrix):
    kr, kb = MATRICES[matrix]
    kg = 1 - kr - kb
    g = torch.Generator().manual_seed(3)
    rgb = flat(torch.rand(4096, 3, generator=g))                    # one flat 2x2 image per colour
    y, u, v = rgb_to_yuv420(rgb, kr, kb)
    back = yuv420_to_rgb(y[None], u[None], v[None], kr, kb)[0]
    dy, dc = 0.5 / 219, 0.5 / 224                                   # half a level of Y' and of Cb / Cr
    bound = torch.tensor([dy + 2 * (1 - kr) * dc, dy + (2 * kr * (1 - kr) + 2 * kb * (1 - kb)) / kg * dc,
                          dy + 2 * (1 - kb) * dc]).view(1, 3, 1, 1)
    err = (back - rgb).abs()
    assert (err <= bound + 1e-5).all(), (err / bound).max()


def _rgb_to_yuv420_np32(rgb, kr, kb):
    """rgb_to_yuv420 restated in numpy float32, one rounded operation at a time."""
    f = np.float32
    kr, kg, kb, cu, cv = (f(c) for c in coefficients(kr, kb))
    p = np.clip(rgb.astype(f), f(0), f(1))
    luma = lambda a: (kr * a[0] + kg * a[1]) + kb * a[2]           # noqa: E731
    y = np.rint(f(16) + f(219) * luma(p))
    m = ((p[:, 0::2, 0::2] + p[:, 0::2, 1::2]) + (p[:, 1::2, 0::2] + p[:, 1::2, 1::2])) * f(0.25)
    ym = luma(m)
    return y, np.rint(f(128) + (m[2] - ym) * cu), np.rint(f(128) + (m[0] - ym) * cv)


def _rgb_to_yuv420_f64(rgb, kr, kb):
    """the same conversion in float64 without rounding; returns the unrounded codes."""
    kg = 1 - kr - kb
    p = np.clip(rgb.astype(np.float64), 0, 1)
    luma = lambda a: kr * a[0] + kg * a[1] + kb * a[2]              # noqa: E731
    m = (p[:, 0::2, 0::2] + p[:, 0::2, 1::2] + p[:, 1::2, 0::2] + p[:, 1::2, 1::2]) / 4
    return 16 + 219 * luma(p), 128 + 224 * (m[2] - luma(m)) / (2 * (1 - kb)), 128 + 224 * (m[0] - luma(m)) / (2 * (1 - kr))


@pytest.mark.parametrize("matrix", sorted(MATRICES))
def test_fp32_order_of_operations(matrix):
    kr, kb = MATRICES[matrix]
    g = torch.Generator().manual_seed(11)
    rgb = torch.rand(3, 96, 128, generator=g) * 1.2 - 0.1           # both clamps are hit
    got = [p.numpy().astype(np.float64) for p in rgb_to_yuv420(rgb, kr, kb)]
    for a, b in zip(got, _rgb_to_yuv420_np32(rgb.numpy(), kr, kb)):
        assert np.array_equal(a, b)                                  # the stated fp32 order, bit for bit
    for a, exact in zip(got, _rgb_to_yuv420_f64(rgb.numpy(), kr, kb)):
        d = np.abs(a - np.rint(exact))
        clear = np.abs(exact - np.floor(exact) - 0.5) > 1e-3        # away from rounding ties
        assert d.max() <= 1 and (d[clear] == 0).all()


def test_coefficients_are_fp32():
    kr, kg, kb, cu, cv = coefficients(*MATRICES["bt709"])
    f = np.float32
    assert kg == float((f(1) - f(0.2126)) - f(0.0722))
    assert cu == float(f(112) / (f(1) - f(0.0722))) and cv == float(f(112) / (f(1) - f(0.2126)))


def test_rgb_to_yuv420_rejects_odd_sizes():
    with pytest.raises(ValueError):
        rgb_to_yuv420(torch.zeros(3, 4, 5), *MATRICES["bt709"])
    with pytest.raises(ValueError):
        rgb_to_yuv420(torch.zeros(4, 4, 4), *MATRICES["bt709"])


def test_prototype_comes_from_the_header():
    assert "eavsr_sr_tail_yuv420_forward" in L.EXPORTED_SYMBOLS
    res, args = L._signatures()["eavsr_sr_tail_yuv420_forward"]
    strides = POINTER(c_int64)
    # x, x_strides, packed_weight, bias, lr, lr_strides, (plane, strides) x 3, n, c, h, w, scale, out_h, out_w, kr, kb,
    # dtype, stream
    assert res is c_int
    assert args == ([c_void_p, strides, c_void_p, c_void_p, c_void_p, strides] + [c_void_p, strides] * 3
                    + [c_int] * 7 + [c_float, c_float, c_int, c_void_p])


# ------------------------------------------------------------------------------------------------
# input checks: nothing is launched
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def net():
    return EAVSRP(4, n_resblock=1).eval()


def u8(*shape, dtype=torch.uint8):
    return torch.zeros(shape, dtype=dtype)


GOOD = (u8(1, 2, 64, 96), u8(1, 2, 32, 48), u8(1, 2, 32, 48))
OUT = (u8(1, 2, 256, 384), u8(1, 2, 128, 192), u8(1, 2, 128, 192))


@pytest.mark.parametrize("args, kwargs, err", [
    ((u8(1, 2, 64, 96, dtype=torch.float32),) + GOOD[1:], {}, TypeError),          # float Y
    (GOOD[:1] + (u8(1, 2, 32, 48, dtype=torch.int16), GOOD[2]), {}, TypeError),     # int16 U
    (GOOD, {"out": OUT[:2] + (u8(1, 2, 128, 192, dtype=torch.float32),)}, TypeError),
    (GOOD, {"matrix": "bt2020"}, ValueError),
    ((u8(2, 64, 96), u8(2, 32, 48), u8(2, 32, 48)), {}, ValueError),                 # no batch dimension
    ((u8(1, 2, 65, 96), u8(1, 2, 32, 48), u8(1, 2, 32, 48)), {}, ValueError),        # odd height
    ((u8(1, 2, 64, 97), u8(1, 2, 32, 48), u8(1, 2, 32, 48)), {}, ValueError),        # odd width
    ((u8(1, 2, 62, 96), u8(1, 2, 31, 48), u8(1, 2, 31, 48)), {}, ValueError),        # under 64
    (GOOD[:2] + (u8(1, 2, 32, 96),), {}, ValueError),                                # V at full width
    ((u8(1, 2, 64, 96), u8(1, 2, 64, 96), u8(1, 2, 64, 96)), {}, ValueError),        # 4:4:4
    (GOOD, {"out": OUT[:2]}, ValueError),
    (GOOD, {"out": (u8(1, 2, 128, 192),) + OUT[1:]}, ValueError),                    # output at x2 for a x4 net
    (GOOD, {"out": OUT[:1] + (u8(1, 2, 256, 384),) + OUT[2:]}, ValueError),
    (GOOD, {}, NotImplementedError),                                                  # CPU planes
    (GOOD, {"out": OUT, "matrix": "bt601"}, NotImplementedError),
])
def test_forward_yuv420_rejects_bad_input_before_any_launch(net, monkeypatch, args, kwargs, err):
    def no_trunk(lrs):
        raise AssertionError("the trunk ran on rejected input")
    monkeypatch.setattr(net, "_trunk", no_trunk)
    before = L.launch_count()
    with pytest.raises(err):
        net.forward_yuv420(*args, **kwargs)
    assert L.launch_count() == before


def _op_args(**over):
    a = dict(conv_last=nn.Conv2d(64, 3, 3, 1, 1), x=torch.zeros(2, 64, 40, 48), lr=torch.zeros(2, 3, 10, 12), scale=4,
             y_out=u8(2, 40, 48), u_out=u8(2, 20, 24), v_out=u8(2, 20, 24), out_h=40, out_w=48, kr=0.2126, kb=0.0722)
    a.update(over)
    return a


@pytest.mark.parametrize("over, err", [
    ({"out_h": 39, "y_out": u8(2, 39, 48)}, ValueError),                             # odd crop
    ({"out_w": 47, "y_out": u8(2, 40, 47)}, ValueError),
    ({"lr": torch.zeros(2, 3, 10, 12, dtype=torch.float64)}, ValueError),
    ({"lr": torch.zeros(2, 3, 20, 24)}, ValueError),                                 # LR of a x2 map
    ({"y_out": u8(2, 40, 48, dtype=torch.int16)}, ValueError),
    ({"y_out": u8(2, 40, 48, 1)}, ValueError),
    ({"u_out": u8(2, 40, 48)}, ValueError),                                          # full-size chroma
    ({"v_out": u8(1, 20, 24)}, ValueError),
    ({}, NotImplementedError),                                                        # CPU tensors
])
def test_sr_tail_yuv420_rejects_bad_input_before_any_launch(over, err):
    before = L.launch_count()
    with pytest.raises(err):
        ops.sr_tail_yuv420(**_op_args(**over))
    assert L.launch_count() == before
