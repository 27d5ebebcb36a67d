"""The 16-bit reconstruction tails (eavsr_sr_tail_u16_forward, eavsr_sr_tail_yuv420_u16_forward) and
EAVSRP.forward_uint16 / EAVSRP.forward_yuv420_u16 against float64.

At 16 bits a level is 1.5e-5, so "exact away from 1 % of a level around a tie" is no longer obviously wider than the
fp32 error of the kernel.  The tie window is derived per element from an error bound instead (`tail64`)."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from eavsr_b200 import ops
from eavsr_b200.model import EAVSRP, pad_clip
from eavsr_b200.synthetic import clip_inputs, gen, seeded_parameters
from eavsr_b200.yuv import HBD_MATRICES, rgb_to_yuv420, yuv420_to_rgb

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
# Error of the kernel's fp32 value v = (t + bias) + up, in units of U * (sum |w x| + |bias| + |up|).  The products of
# bf16 operands are exact in fp32; t is 12 tensor-core steps of 16 products added to an fp32 accumulator, each step
# taken within 2 ulp (truncating alignment, 4 U) of the sum of the magnitudes so far (48 U), then two shuffled sums,
# the bias and the base are added (4 U) and the base carries ~4 roundings of its own (4 U); the multiplication by M
# adds one more (1 U).  64 bounds the 57 with room.
C_ERR = 64


def tail64(conv, x, lr, s, out_h, out_w):
    """float64 ``sr = conv(x) + up_s(lr)`` cropped, and the bound ``E`` of the kernel's error on it (same shape)."""
    w = conv.weight.to(torch.bfloat16).double()
    b = conv.bias.to(torch.bfloat16).double()
    xd = x.double().contiguous()
    base = F.interpolate(lr.double(), scale_factor=s, mode="bilinear", align_corners=False)
    sr = F.conv2d(xd, w, b, 1, 1) + base
    mag = F.conv2d(xd.abs(), w.abs(), None, 1, 1) + b.abs().view(1, 3, 1, 1) + base.abs()
    return sr[..., :out_h, :out_w], (C_ERR * U) * mag[..., :out_h, :out_w]


def check_codes(got, exact, window, what=""):
    """Integer codes against unrounded float64 ones: within one level everywhere, exact where ``exact`` is farther than
    ``window`` from a rounding tie, and exact for more than 99 % of the values."""
    want = torch.round(exact)
    diff = (got.double() - want).abs()
    clear = ((exact - exact.floor()) - 0.5).abs() > window
    frac = (diff > 0).double().mean().item()
    print(f"{what}: {frac:.5f} off by one, window {window.max().item():.4f} levels, "
          f"{clear.double().mean().item():.3f} of the values outside it")
    assert diff.max().item() <= 1
    assert (diff[clear] == 0).all(), f"{int((diff[clear] != 0).sum())} values off outside the window"
    assert frac < 0.01


def check_rgb(got, sr, err, bits):
    m = 2 ** bits - 1
    check_codes(got.int().permute(0, 3, 1, 2), m * sr.clamp(0, 1), m * err, f"rgb {bits} bits")


def check_yuv(planes, sr, err, kr, kb, bits, shift):
    """``planes`` (Y, U, V) of `rgb_to_yuv420(sr, kr, kb, bits, shift)` against float64.  The conversion's own fp32
    roundings (a few per code, relative to the code's scale) are covered by 8 U each side."""
    k = 2 ** (bits - 8)
    p = sr.clamp(0, 1)
    luma = lambda a: kr * a[:, 0] + (1 - kr - kb) * a[:, 1] + kb * a[:, 2]          # noqa: E731
    m = F.avg_pool2d(p, 2)
    e = err.amax(1)
    e2 = F.max_pool2d(e[:, None], 2)[:, 0]
    cu, cv = 112 * k / (1 - kb), 112 * k / (1 - kr)
    for q in planes:
        assert (q.int() % 2 ** shift == 0).all()
    y, u, v = (q.int() >> shift for q in planes)
    check_codes(y, 16 * k + 219 * k * luma(p), 219 * k * e + 235 * k * 8 * U, f"Y {bits}/{shift}")
    check_codes(u, 128 * k + cu * (m[:, 2] - luma(m)), 2 * cu * e2 + 240 * k * 16 * U, f"U {bits}/{shift}")
    check_codes(v, 128 * k + cv * (m[:, 0] - luma(m)), 2 * cv * e2 + 240 * k * 16 * U, f"V {bits}/{shift}")


def full16(shape, value, dev):
    return torch.full(shape, value, dtype=torch.uint16).to(dev)


def _operands(cuda, n, h, w, s, seed):
    """Residuals of a few 1e-2 (the model's are ~8e-3 RMS) around a base in [-0.1, 1.1]: both clamps are hit, most
    values are not clamped."""
    g = gen(seed)
    conv = nn.Conv2d(64, 3, 3, 1, 1)
    with torch.no_grad():
        conv.weight.copy_((torch.rand(conv.weight.shape, generator=g) * 2 - 1) * 0.004)
        conv.bias.copy_((torch.rand(3, generator=g) * 2 - 1) * 0.01)
    conv = conv.to(cuda, torch.bfloat16).eval()
    x = torch.randn(n, 64, h, w, generator=g).to(cuda, torch.bfloat16).contiguous(memory_format=torch.channels_last)
    lr = (torch.rand(n, 2, 3, h // s, w // s, generator=g) * 1.2 - 0.1).to(cuda)[:, 1]      # a strided LR frame
    return conv, x, lr


SHAPES = [
    (3, 72, 100, 4, 72, 100),        # W not a multiple of the 30-pixel tile or the 32-pixel halo
    (3, 70, 94, 2, 70, 94),          # H not a multiple of the 4-row tile
    (3, 40, 24, 4, 40, 24),          # W < 32: the halo box is wider than the map
    (3, 66, 130, 2, 64, 126),        # crop in both directions
    (2, 1088, 1920, 4, 1080, 1920),  # one frame of the benchmark batch: 272x480 -> 1088x1920, cropped to 1080
]


# ------------------------------------------------------------------------------------------------
# the operators against float64
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bits", [10, 16])
@pytest.mark.parametrize("n, h, w, s, out_h, out_w", SHAPES)
def test_rgb_op_matches_float64(cuda, bits, n, h, w, s, out_h, out_w):
    conv, x, lr = _operands(cuda, n, h, w, s, 3000 + h + w + bits)
    clip = full16((n, 2, out_h, out_w + 5, 3), 77, cuda)              # frame 1 of 2, rows padded by 5 pixels
    out = clip[:, 1, :, :out_w]
    with torch.no_grad():
        ops.sr_tail_u16(conv, x, lr, s, out, out_h, out_w, bits)
        sr, err = tail64(conv, x, lr, s, out_h, out_w)
    torch.cuda.synchronize()
    assert (sr < 0).any() and (sr > 1).any() and ((sr > 0) & (sr < 1)).double().mean() > 0.5
    check_rgb(out, sr, err, bits)
    assert (clip[:, 0].int() == 77).all() and (clip[:, 1, :, out_w:].int() == 77).all()


@pytest.mark.parametrize("bits, shift, matrix", [(10, 0, "bt709"), (10, 6, "bt2020"), (16, 0, "bt601"),
                                                 (12, 4, "bt2020")])
@pytest.mark.parametrize("n, h, w, s, out_h, out_w", SHAPES)
def test_yuv_op_matches_float64(cuda, bits, shift, matrix, n, h, w, s, out_h, out_w):
    kr, kb = HBD_MATRICES[matrix]
    conv, x, lr = _operands(cuda, n, h, w, s, 4000 + h + w + bits)
    # frame 1 of a 2-frame Y clip, and the chroma interleaved as P010 with 8 padding samples per row
    y_clip = full16((n, 2, out_h, out_w + 8), 77, cuda)
    uv_clip = full16((n, 2, out_h // 2, out_w + 8), 77, cuda)
    planes = y_clip[:, 1, :, :out_w], uv_clip[:, 1, :, 0:out_w:2], uv_clip[:, 1, :, 1:out_w:2]
    with torch.no_grad():
        ops.sr_tail_yuv420_u16(conv, x, lr, s, *planes, out_h, out_w, kr, kb, bits, shift)
        sr, err = tail64(conv, x, lr, s, out_h, out_w)
    torch.cuda.synchronize()
    check_yuv(planes, sr, err, kr, kb, bits, shift)
    assert (y_clip[:, 0].int() == 77).all() and (uv_clip[:, 0].int() == 77).all()      # the other frame
    assert (y_clip[:, 1, :, out_w:].int() == 77).all() and (uv_clip[:, 1, :, out_w:].int() == 77).all()  # padding


# ------------------------------------------------------------------------------------------------
# the model
# ------------------------------------------------------------------------------------------------
def _net(cuda, scale, dtype):
    net = EAVSRP(scale).eval()
    seeded_parameters(net)
    return net.to(cuda).prepare(dtype)


def _memoised_hr_features(net):
    """Every run sees the same HR features: the channel-attention sums of the propagation and reconstruction groups
    use float atomics, so two runs agree to rounding only (DESIGN.md section 4), and these tests are about the tail."""
    hr_features, memo = net._hr_features, {}

    def hr_once(feats, i):
        if i not in memo:
            memo[i] = hr_features(feats, i)
        return memo[i]
    net._hr_features = hr_once
    return memo


def _rgb16(cuda, t, h, w, seed, bits):
    m = 2 ** bits - 1
    return torch.round(clip_inputs(1, t, h, w, seed=seed) * m).permute(0, 1, 3, 4, 2).to(torch.uint16).to(cuda)


def _yuv16(cuda, t, h, w, seed, matrix, bits, shift):
    return [p.to(cuda) for p in rgb_to_yuv420(clip_inputs(1, t, h, w, seed=seed), *HBD_MATRICES[matrix], bits, shift)]


def _tails64(net, memo, lrs, h, w):
    """float64 tail of every frame from the memoised HR features: (sr, err) stacked over frames on dim 1."""
    s = net.scale
    with torch.no_grad():
        parts = [tail64(net.conv_last, memo[i], lrs[:, i], s, s * h, s * w) for i in range(lrs.shape[1])]
    return torch.stack([p[0] for p in parts], 1), torch.stack([p[1] for p in parts], 1)


@pytest.mark.parametrize("scale", [4, 2])
@pytest.mark.parametrize("t, h, w", [(4, 64, 64), (3, 70, 90)])       # 70x90: padded to 72x92, cropped back
def test_model_uint16_bf16_matches_float64_tail(cuda, scale, t, h, w):
    bits = 16
    net = _net(cuda, scale, torch.bfloat16)
    frames = _rgb16(cuda, t, h, w, 21, bits)
    memo = _memoised_hr_features(net)
    try:
        got = net.forward_uint16(frames, bits=bits)
    finally:
        del net._hr_features
    assert got.shape == (1, t, scale * h, scale * w, 3) and got.dtype == torch.uint16
    lrs = pad_clip(frames.permute(0, 1, 4, 2, 3).float().div(2 ** bits - 1))
    sr, err = _tails64(net, memo, lrs, h, w)
    check_rgb(got.flatten(0, 1), sr.flatten(0, 1), err.flatten(0, 1), bits)


@pytest.mark.parametrize("scale", [4, 2])
@pytest.mark.parametrize("t, h, w", [(4, 64, 64), (3, 70, 90)])
def test_model_yuv420_u16_bf16_matches_float64_tail(cuda, scale, t, h, w):
    bits, shift, matrix = 10, 6, "bt2020"
    kr, kb = HBD_MATRICES[matrix]
    net = _net(cuda, scale, torch.bfloat16)
    y, u, v = _yuv16(cuda, t, h, w, 22, matrix, bits, shift)
    memo = _memoised_hr_features(net)
    try:
        got = net.forward_yuv420_u16(y, u, v, bits=bits, shift=shift, matrix=matrix)
    finally:
        del net._hr_features
    assert [tuple(p.shape) for p in got] == [(1, t, scale * h, scale * w)] + [(1, t, scale * h // 2, scale * w // 2)] * 2
    assert all(p.dtype == torch.uint16 for p in got)
    sr, err = _tails64(net, memo, pad_clip(yuv420_to_rgb(y, u, v, kr, kb, bits, shift)), h, w)
    check_yuv([p.flatten(0, 1) for p in got], sr.flatten(0, 1), err.flatten(0, 1), kr, kb, bits, shift)


@pytest.mark.parametrize("scale", [4, 2])
def test_model_fp32_matches_the_composed_path_exactly(cuda, scale):
    net = _net(cuda, scale, torch.float32)
    t, h, w = 3, 70, 90
    s = scale
    kr, kb = HBD_MATRICES["bt2020"]
    frames = _rgb16(cuda, t, h, w, 5, 12)
    y, u, v = _yuv16(cuda, t, h, w, 6, "bt2020", 10, 6)
    memo = _memoised_hr_features(net)
    try:
        got = net.forward_uint16(frames, bits=12)
        with torch.no_grad():
            sr = net(pad_clip(frames.permute(0, 1, 4, 2, 3).float().div(4095)))[..., :s * h, :s * w]
        assert len(memo) == t
        assert torch.equal(got.int(), torch.clamp(sr * 4095, 0, 4095).round().permute(0, 1, 3, 4, 2).int())

        memo.clear()                                                    # the 4:2:0 clip has HR features of its own
        got = net.forward_yuv420_u16(y, u, v, bits=10, shift=6, matrix="bt2020")
        with torch.no_grad():
            sr = net(pad_clip(yuv420_to_rgb(y, u, v, kr, kb, 10, 6)))[..., :s * h, :s * w]
        assert len(memo) == t
        for a, b in zip(got, rgb_to_yuv420(sr, kr, kb, 10, 6)):
            assert torch.equal(a.int(), b.int())
    finally:
        del net._hr_features


def test_p010_views_match_planar_10bit(cuda):
    """P010 in (codes << 6, chroma interleaved) and out (row pitch > width) gives the planar shift=0 codes times 64."""
    net = _net(cuda, 4, torch.bfloat16)
    t, h, w, s = 3, 64, 96, 4
    y, u, v = _yuv16(cuda, t, h, w, 9, "bt709", 10, 0)
    y10 = (y.int() << 6).to(torch.uint16)
    uv = (torch.stack([u.int(), v.int()], -1) << 6).to(torch.uint16).view(1, t, h // 2, w)
    y_p010 = full16((1, t, s * h, s * w + 16), 77, cuda)
    uv_p010 = full16((1, t, s * h // 2, s * w + 16), 77, cuda)
    out = (y_p010[..., :s * w], uv_p010[..., 0:s * w:2], uv_p010[..., 1:s * w:2])
    _memoised_hr_features(net)
    try:
        planar = net.forward_yuv420_u16(y, u, v, bits=10, shift=0)
        ret = net.forward_yuv420_u16(y10, uv[..., 0::2], uv[..., 1::2], bits=10, shift=6, out=out)
    finally:
        del net._hr_features
    assert all(a is b for a, b in zip(ret, out))
    assert max(p.int().max().item() for p in planar) < 1024
    for a, b in zip(planar, out):
        assert torch.equal(a.int() * 64, b.int())
    assert (y_p010[..., s * w:].int() == 77).all() and (uv_p010[..., s * w:].int() == 77).all()


def test_graph_capture(cuda):
    net = _net(cuda, 4, torch.bfloat16)
    a = _yuv16(cuda, 4, 64, 64, 7, "bt2020", 10, 6)
    b = _yuv16(cuda, 4, 64, 64, 8, "bt2020", 10, 6)
    fa, fb = _rgb16(cuda, 4, 64, 64, 7, 16), _rgb16(cuda, 4, 64, 64, 8, 16)
    static = [p.clone() for p in a] + [fa.clone()]

    def run():
        return net.forward_yuv420_u16(*static[:3], bits=10, shift=6, matrix="bt2020") + (net.forward_uint16(static[3]),)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        run()                                              # warm-up outside capture (packed weights, cuDNN)
    torch.cuda.current_stream().wait_stream(st)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run()
    for p, q in zip(static, b + [fb]):
        p.copy_(q)
    graph.replay()
    torch.cuda.synchronize()
    eager = net.forward_yuv420_u16(*b, bits=10, shift=6, matrix="bt2020") + (net.forward_uint16(fb),)
    # two runs of the trunk agree to rounding only (float atomics), and an 8-bit output moves by at most one level
    # between them (test_gpu_yuv.py): allow one 8-bit level plus one level of the codes
    for o, e in zip(out[:3], eager[:3]):
        assert ((o.int() >> 6) - (e.int() >> 6)).abs().max().item() <= 4 + 1
    assert (out[3].int() - eager[3].int()).abs().max().item() <= 257 + 1
    first = net.forward_yuv420_u16(*a, bits=10, shift=6, matrix="bt2020")[0]
    assert not torch.equal(out[0].int(), first.int())       # the replay computed clip b, not the captured a
