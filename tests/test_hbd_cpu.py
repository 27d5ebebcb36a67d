"""CPU tests of 10-, 12- and 16-bit inference: the generalised conversions of eavsr_b200/yuv.py, the ctypes prototypes
of eavsr_sr_tail_u16_forward and eavsr_sr_tail_yuv420_u16_forward derived from the header, and the input checks of
EAVSRP.forward_uint16, EAVSRP.forward_yuv420_u16, ops.sr_tail_u16 and ops.sr_tail_yuv420_u16, which must fail before
anything is launched."""
from ctypes import POINTER, c_float, c_int, c_int64, c_void_p

import numpy as np
import pytest
import torch
import torch.nn as nn

from eavsr_b200 import _lib as L
from eavsr_b200 import ops
from eavsr_b200.model import EAVSRP
from eavsr_b200.yuv import HBD_MATRICES, MATRICES, coefficients, rgb_to_yuv420, yuv420_to_rgb

COLOURS = [(1, 1, 1), (0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1)]
# textbook limited-range codes (Y', Cb, Cr) of white, black and the primaries
CODES = {
    10: {"bt709": [(940, 512, 512), (64, 512, 512), (250, 409, 960), (691, 167, 105), (127, 960, 471)],
         "bt601": [(940, 512, 512), (64, 512, 512), (326, 361, 960), (578, 215, 137), (164, 960, 439)],
         "bt2020": [(940, 512, 512), (64, 512, 512), (294, 387, 960), (658, 189, 100), (116, 960, 476)]},
    12: {"bt709": [(3760, 2048, 2048), (256, 2048, 2048), (1001, 1637, 3840), (2762, 667, 420), (509, 3840, 1884)],
         "bt601": [(3760, 2048, 2048), (256, 2048, 2048), (1304, 1443, 3840), (2313, 861, 547), (655, 3840, 1757)],
         "bt2020": [(3760, 2048, 2048), (256, 2048, 2048), (1177, 1548, 3840), (2632, 756, 400), (464, 3840, 1904)]},
}


def flat(colours, size=2):
    """(k, 3) colours -> (k, 3, size, size) flat images."""
    return torch.as_tensor(colours, dtype=torch.float32)[:, :, None, None].expand(-1, -1, size, size).contiguous()


@pytest.mark.parametrize("bits", sorted(CODES))
@pytest.mark.parametrize("matrix", sorted(HBD_MATRICES))
def test_textbook_codes_match_the_definitions(bits, matrix):
    """The table above against Y' = 16k + 219k Yc, Cb = 128k + 112k (B - Yc) / (1 - Kb), Cr likewise, in float64."""
    kr, kb = HBD_MATRICES[matrix]
    k = 2 ** (bits - 8)
    for (r, g, b), codes in zip(COLOURS, CODES[bits][matrix]):
        yc = kr * r + (1 - kr - kb) * g + kb * b
        assert codes == (round(16 * k + 219 * k * yc), round(128 * k + 112 * k * (b - yc) / (1 - kb)),
                         round(128 * k + 112 * k * (r - yc) / (1 - kr)))


@pytest.mark.parametrize("bits", sorted(CODES))
@pytest.mark.parametrize("matrix", sorted(HBD_MATRICES))
@pytest.mark.parametrize("high", [False, True])
def test_known_codes(bits, matrix, high):
    shift = 16 - bits if high else 0
    kr, kb = HBD_MATRICES[matrix]
    y, u, v = rgb_to_yuv420(flat(COLOURS, 4), kr, kb, bits=bits, shift=shift)
    assert y.dtype == u.dtype == v.dtype == torch.uint16
    assert y.shape == (5, 4, 4) and u.shape == v.shape == (5, 2, 2)
    got = torch.stack([y[:, 0, 0], u[:, 0, 0], v[:, 0, 0]], 1).int()
    assert got.tolist() == [[c << shift for c in codes] for codes in CODES[bits][matrix]]
    for p in (y, u, v):
        assert (p.int() == p[:, :1, :1].int()).all()
    planes = [p.view(1, 5, *p.shape[1:]) for p in (y, u, v)]
    back = yuv420_to_rgb(*planes, kr, kb, bits=bits, shift=shift)
    assert back.shape == (1, 5, 3, 4, 4) and back.dtype == torch.float32
    assert (back[0] - flat(COLOURS, 4)).abs().max().item() < 2e-3


def test_input_codes_are_the_high_bits():
    """P010 input keeps floor(sample / 64): the low 6 bits are ignored."""
    kr, kb = HBD_MATRICES["bt2020"]
    y, u, v = rgb_to_yuv420(flat(torch.rand(6, 3, generator=torch.Generator().manual_seed(1))), kr, kb, bits=10)
    planes = [p.view(1, 6, *p.shape[1:]) for p in (y, u, v)]
    want = yuv420_to_rgb(*planes, kr, kb, bits=10)
    junk = [((p.int() << 6) + torch.randint(0, 64, p.shape)).to(torch.uint16) for p in planes]
    assert torch.equal(yuv420_to_rgb(*junk, kr, kb, bits=10, shift=6), want)


@pytest.mark.parametrize("bits", [10, 12, 16])
@pytest.mark.parametrize("matrix", sorted(HBD_MATRICES))
def test_round_trip_of_flat_blocks_stays_within_quantisation(bits, matrix):
    kr, kb = HBD_MATRICES[matrix]
    kg = 1 - kr - kb
    k = 2 ** (bits - 8)
    rgb = flat(torch.rand(4096, 3, generator=torch.Generator().manual_seed(3)))
    y, u, v = rgb_to_yuv420(rgb, kr, kb, bits=bits, shift=16 - bits)
    back = yuv420_to_rgb(y[None], u[None], v[None], kr, kb, bits=bits, shift=16 - bits)[0]
    dy, dc = 0.5 / (219 * k), 0.5 / (224 * k)                       # half a level of Y' and of Cb / Cr
    bound = torch.tensor([dy + 2 * (1 - kr) * dc, dy + (2 * kr * (1 - kr) + 2 * kb * (1 - kb)) / kg * dc,
                          dy + 2 * (1 - kb) * dc]).view(1, 3, 1, 1)
    err = (back - rgb).abs()
    assert (err <= bound + 1e-6).all(), (err / bound).max()


def _rgb_to_yuv420_np32(rgb, kr, kb, bits):
    """rgb_to_yuv420 at `bits` restated in numpy float32, one rounded operation at a time."""
    f = np.float32
    k = f(2 ** (bits - 8))
    kr, kg, kb, cu, cv = (f(c) for c in coefficients(kr, kb))
    p = np.clip(rgb.astype(f), f(0), f(1))
    luma = lambda a: (kr * a[0] + kg * a[1]) + kb * a[2]           # noqa: E731
    y = np.rint(f(16) * k + (f(219) * k) * luma(p))
    m = ((p[:, 0::2, 0::2] + p[:, 0::2, 1::2]) + (p[:, 1::2, 0::2] + p[:, 1::2, 1::2])) * f(0.25)
    ym = luma(m)
    return y, np.rint(f(128) * k + (m[2] - ym) * (cu * k)), np.rint(f(128) * k + (m[0] - ym) * (cv * k))


@pytest.mark.parametrize("bits", [10, 12, 16])
@pytest.mark.parametrize("matrix", sorted(HBD_MATRICES))
def test_fp32_order_of_operations(bits, matrix):
    kr, kb = HBD_MATRICES[matrix]
    rgb = torch.rand(3, 96, 128, generator=torch.Generator().manual_seed(11)) * 1.2 - 0.1
    for shift in sorted({0, 16 - bits}):
        got = [p.int().numpy() for p in rgb_to_yuv420(rgb, kr, kb, bits=bits, shift=shift)]
        for a, b in zip(got, _rgb_to_yuv420_np32(rgb.numpy(), kr, kb, bits)):
            assert np.array_equal(a, b.astype(np.int64) << shift)


def test_scaled_coefficients_are_exact():
    """cu_b = 112k / (1 - kb) rounded to fp32 is k times the 8-bit cu: the kernel computes k * cu."""
    for kr, kb in HBD_MATRICES.values():
        _, _, _, cu, cv = coefficients(kr, kb)
        f = np.float32
        for k in (4, 16, 256):
            assert f(f(112 * k) / (f(1) - f(kb))) == f(cu) * f(k)
            assert f(f(112 * k) / (f(1) - f(kr))) == f(cv) * f(k)


def _rgb_to_yuv420_8bit(rgb, kr, kb):
    """The 8-bit rgb_to_yuv420 before it took bits and shift, verbatim."""
    kr, kg, kb, cu, cv = coefficients(kr, kb)
    p = rgb.float().clamp(0, 1)
    r, g, b = p.unbind(-3)
    luma = lambda r, g, b: (kr * r + kg * g) + kb * b                 # noqa: E731
    y = torch.round(16 + 219 * luma(r, g, b))
    m = ((p[..., 0::2, 0::2] + p[..., 0::2, 1::2]) + (p[..., 1::2, 0::2] + p[..., 1::2, 1::2])) * 0.25
    mr, mg, mb = m.unbind(-3)
    ym = luma(mr, mg, mb)
    return y.to(torch.uint8), torch.round(128 + (mb - ym) * cu).to(torch.uint8), \
        torch.round(128 + (mr - ym) * cv).to(torch.uint8)


def _yuv420_to_rgb_8bit(y, u, v, kr, kb):
    """The 8-bit yuv420_to_rgb before it took bits and shift, verbatim."""
    n, t, h, w = y.shape
    kg = 1 - kr - kb
    yn = (y.float() - 16) / 219
    pbr = (torch.stack([u, v], 2).float() - 128) / 224
    pbr = torch.nn.functional.interpolate(pbr.reshape(n * t, 2, h // 2, w // 2), scale_factor=2, mode="bilinear",
                                          align_corners=False)
    pb, pr = pbr.view(n, t, 2, h, w).unbind(2)
    r = yn + 2 * (1 - kr) * pr
    b = yn + 2 * (1 - kb) * pb
    g = (yn - kr * r - kb * b) / kg
    return torch.stack([r, g, b], 2).clamp_(0, 1)


@pytest.mark.parametrize("matrix", sorted(MATRICES))
def test_8bit_results_are_unchanged(matrix):
    kr, kb = MATRICES[matrix]
    g = torch.Generator().manual_seed(5)
    rgb = torch.rand(2, 3, 3, 64, 96, generator=g) * 1.2 - 0.1
    want = _rgb_to_yuv420_8bit(rgb, kr, kb)
    for got in (rgb_to_yuv420(rgb, kr, kb), rgb_to_yuv420(rgb, kr, kb, bits=8, shift=0)):
        assert all(a.dtype == torch.uint8 and torch.equal(a, b) for a, b in zip(got, want))
    back = _yuv420_to_rgb_8bit(*want, kr, kb)
    assert torch.equal(yuv420_to_rgb(*want, kr, kb), back)
    assert torch.equal(yuv420_to_rgb(*want, kr, kb, bits=8, shift=0), back)


@pytest.mark.parametrize("bits, shift", [(8, 8), (9, 0), (14, 0), (10, 4), (12, 6), (16, 1)])
def test_conversions_reject_bad_bits(bits, shift):
    with pytest.raises(ValueError):
        rgb_to_yuv420(torch.zeros(3, 4, 4), *MATRICES["bt709"], bits=bits, shift=shift)
    z = torch.zeros(1, 1, 4, 4, dtype=torch.uint16)
    with pytest.raises(ValueError):
        yuv420_to_rgb(z, z[..., :2, :2], z[..., :2, :2], *MATRICES["bt709"], bits=bits, shift=shift)


def test_prototypes_come_from_the_header():
    strides = POINTER(c_int64)
    head = [c_void_p, strides, c_void_p, c_void_p, c_void_p, strides]
    assert "eavsr_sr_tail_u16_forward" in L.EXPORTED_SYMBOLS
    assert L._signatures()["eavsr_sr_tail_u16_forward"] == (
        c_int, head + [c_void_p, strides] + [c_int] * 7 + [c_int, c_int, c_void_p])
    assert "eavsr_sr_tail_yuv420_u16_forward" in L.EXPORTED_SYMBOLS
    # ..., (plane, strides) x 3, n, c, h, w, scale, out_h, out_w, kr, kb, bits, shift, dtype, stream
    assert L._signatures()["eavsr_sr_tail_yuv420_u16_forward"] == (
        c_int, head + [c_void_p, strides] * 3 + [c_int] * 7 + [c_float, c_float, c_int, c_int, c_int, c_void_p])


# ------------------------------------------------------------------------------------------------
# input checks: nothing is launched
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def net():
    return EAVSRP(4, n_resblock=1).eval()


def u16(*shape, dtype=torch.uint16):
    return torch.zeros(shape, dtype=dtype)


@pytest.fixture
def no_trunk(net, monkeypatch):
    def trunk(lrs):
        raise AssertionError("the trunk ran on rejected input")
    monkeypatch.setattr(net, "_trunk", trunk)
    return net


@pytest.mark.parametrize("args, kwargs, err", [
    ((u16(1, 2, 64, 96, 3, dtype=torch.uint8),), {}, TypeError),
    ((u16(1, 2, 64, 96, 3, dtype=torch.float32),), {}, TypeError),
    ((u16(1, 2, 64, 96, 3),), {"bits": 8}, ValueError),
    ((u16(1, 2, 64, 96, 3),), {"bits": 9}, ValueError),
    ((u16(1, 2, 64, 96, 3),), {"bits": 14}, ValueError),
    ((u16(2, 64, 96, 3),), {}, ValueError),                                          # no batch dimension
    ((u16(1, 2, 3, 64, 96),), {}, ValueError),                                       # planar RGB
    ((u16(1, 2, 62, 96, 3),), {}, ValueError),                                       # under 64
    ((u16(1, 2, 64, 96, 3),), {}, NotImplementedError),                               # CPU frames
    ((u16(1, 2, 65, 97, 3),), {"bits": 10}, NotImplementedError),                     # odd sizes are padded
])
def test_forward_uint16_rejects_bad_input_before_any_launch(no_trunk, args, kwargs, err):
    before = L.launch_count()
    with pytest.raises(err):
        no_trunk.forward_uint16(*args, **kwargs)
    assert L.launch_count() == before


GOOD = (u16(1, 2, 64, 96), u16(1, 2, 32, 48), u16(1, 2, 32, 48))
OUT = (u16(1, 2, 256, 384), u16(1, 2, 128, 192), u16(1, 2, 128, 192))


@pytest.mark.parametrize("args, kwargs, err", [
    ((u16(1, 2, 64, 96, dtype=torch.uint8),) + GOOD[1:], {}, TypeError),             # 8-bit planes
    (GOOD[:1] + (u16(1, 2, 32, 48, dtype=torch.uint8), GOOD[2]), {}, TypeError),
    (GOOD[:2] + (u16(1, 2, 32, 48, dtype=torch.int16),), {}, TypeError),
    (GOOD, {"out": OUT[:2] + (u16(1, 2, 128, 192, dtype=torch.uint8),)}, TypeError),
    (GOOD, {"bits": 8}, ValueError),
    (GOOD, {"bits": 9}, ValueError),
    (GOOD, {"bits": 14, "shift": 2}, ValueError),
    (GOOD, {"bits": 10, "shift": 4}, ValueError),                                      # shift of 12-bit codes
    (GOOD, {"bits": 12, "shift": 6}, ValueError),
    (GOOD, {"bits": 16, "shift": 6}, ValueError),
    (GOOD, {"matrix": "smpte240m"}, ValueError),
    ((u16(2, 64, 96), u16(2, 32, 48), u16(2, 32, 48)), {}, ValueError),              # no batch dimension
    ((u16(1, 2, 65, 96), u16(1, 2, 32, 48), u16(1, 2, 32, 48)), {}, ValueError),     # odd height
    ((u16(1, 2, 64, 97), u16(1, 2, 32, 48), u16(1, 2, 32, 48)), {}, ValueError),     # odd width
    ((u16(1, 2, 62, 96), u16(1, 2, 31, 48), u16(1, 2, 31, 48)), {}, ValueError),     # under 64
    (GOOD[:2] + (u16(1, 2, 32, 96),), {}, ValueError),                                # V at full width
    (GOOD, {"out": OUT[:2]}, ValueError),
    (GOOD, {"out": (u16(1, 2, 128, 192),) + OUT[1:]}, ValueError),                    # output at x2 for a x4 net
    (GOOD, {}, NotImplementedError),                                                   # CPU planes
    (GOOD, {"matrix": "bt2020", "bits": 10, "shift": 6}, NotImplementedError),        # BT.2020 P010 is accepted
    (GOOD, {"matrix": "bt2020", "bits": 12, "shift": 4, "out": OUT}, NotImplementedError),
    (GOOD, {"bits": 16}, NotImplementedError),
])
def test_forward_yuv420_u16_rejects_bad_input_before_any_launch(no_trunk, args, kwargs, err):
    before = L.launch_count()
    with pytest.raises(err):
        no_trunk.forward_yuv420_u16(*args, **kwargs)
    assert L.launch_count() == before


def _op_args(**over):
    a = dict(conv_last=nn.Conv2d(64, 3, 3, 1, 1), x=torch.zeros(2, 64, 40, 48), lr=torch.zeros(2, 3, 10, 12), scale=4,
             out=u16(2, 40, 48, 3), out_h=40, out_w=48, bits=16)
    a.update(over)
    return a


@pytest.mark.parametrize("over, err", [
    ({"bits": 8}, ValueError),
    ({"bits": 9}, ValueError),
    ({"bits": 14}, ValueError),
    ({"out": u16(2, 40, 48, 3, dtype=torch.uint8)}, ValueError),
    ({"out": u16(2, 40, 48, 4)}, ValueError),
    ({"lr": torch.zeros(2, 3, 20, 24)}, ValueError),                                 # LR of a x2 map
    ({}, NotImplementedError),                                                        # CPU tensors
])
def test_sr_tail_u16_rejects_bad_input_before_any_launch(over, err):
    before = L.launch_count()
    with pytest.raises(err):
        ops.sr_tail_u16(**_op_args(**over))
    assert L.launch_count() == before


def _yuv_op_args(**over):
    a = dict(conv_last=nn.Conv2d(64, 3, 3, 1, 1), x=torch.zeros(2, 64, 40, 48), lr=torch.zeros(2, 3, 10, 12), scale=4,
             y_out=u16(2, 40, 48), u_out=u16(2, 20, 24), v_out=u16(2, 20, 24), out_h=40, out_w=48,
             kr=0.2627, kb=0.0593, bits=10, shift=6)
    a.update(over)
    return a


@pytest.mark.parametrize("over, err", [
    ({"bits": 8, "shift": 0}, ValueError),
    ({"bits": 9, "shift": 0}, ValueError),
    ({"bits": 14, "shift": 2}, ValueError),
    ({"bits": 12, "shift": 6}, ValueError),                                          # shift of 10-bit codes
    ({"out_h": 39, "y_out": u16(2, 39, 48)}, ValueError),                            # odd crop
    ({"lr": torch.zeros(2, 3, 10, 12, dtype=torch.float64)}, ValueError),
    ({"y_out": u16(2, 40, 48, dtype=torch.uint8)}, ValueError),                      # 8-bit plane
    ({"u_out": u16(2, 40, 48)}, ValueError),                                          # full-size chroma
    ({"v_out": u16(1, 20, 24)}, ValueError),
    ({}, NotImplementedError),                                                        # CPU tensors
    ({"bits": 12, "shift": 0}, NotImplementedError),
])
def test_sr_tail_yuv420_u16_rejects_bad_input_before_any_launch(over, err):
    before = L.launch_count()
    with pytest.raises(err):
        ops.sr_tail_yuv420_u16(**_yuv_op_args(**over))
    assert L.launch_count() == before
