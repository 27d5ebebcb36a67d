"""The 4:2:0 reconstruction tail (eavsr_sr_tail_yuv420_forward) against a float64 reference, and
EAVSRP.forward_yuv420 against rgb_to_yuv420 of EAVSRP.forward (eavsr_b200/yuv.py)."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from eavsr_b200 import ops
from eavsr_b200.model import EAVSRP, pad_clip
from eavsr_b200.synthetic import clip_inputs, gen, seeded_parameters
from eavsr_b200.yuv import MATRICES, rgb_to_yuv420, yuv420_to_rgb

pytestmark = pytest.mark.gpu


def check_codes(got, exact):
    """uint8 codes against unrounded float64 ones: within one level, exact away from rounding ties."""
    want = torch.round(exact)
    diff = (got.double() - want).abs()
    clear = ((exact - exact.floor()) - 0.5).abs() > 1e-2             # not within 1 % of a level of a tie
    assert diff.max().item() <= 1
    assert (diff[clear] == 0).all(), f"{int((diff[clear] != 0).sum())} values off away from ties"


# ------------------------------------------------------------------------------------------------
# the operator against float64
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("matrix", sorted(MATRICES))
@pytest.mark.parametrize("n, h, w, s, out_h, out_w", [
    (3, 72, 100, 4, 72, 100),        # W not a multiple of the 30-pixel tile or the 32-pixel halo
    (3, 70, 94, 2, 70, 94),          # H not a multiple of the 4-row tile
    (3, 40, 24, 4, 40, 24),          # W < 32: the halo box is wider than the map
    (3, 66, 130, 2, 64, 126),        # crop in both directions
    (2, 1088, 1920, 4, 1080, 1920),  # one frame of the benchmark batch: 272x480 -> 1088x1920, cropped to 1080
])
def test_op_matches_float64(cuda, matrix, n, h, w, s, out_h, out_w):
    kr, kb = MATRICES[matrix]
    g = gen(2000 + h + w)
    conv = nn.Conv2d(64, 3, 3, 1, 1)
    with torch.no_grad():
        # residuals of O(1) around a [0, 1] base: both clamps are hit, most pixels are not clamped
        conv.weight.copy_((torch.rand(conv.weight.shape, generator=g) * 2 - 1) * 0.05)
        conv.bias.copy_((torch.rand(3, generator=g) * 2 - 1) * 0.2)
    conv = conv.to(cuda, torch.bfloat16).eval()
    x = torch.randn(n, 64, h, w, generator=g).to(cuda, torch.bfloat16).contiguous(memory_format=torch.channels_last)
    lr = torch.rand(n, 2, 3, h // s, w // s, generator=g).to(cuda)[:, 1]          # a strided LR frame
    # frame 1 of a 2-frame Y clip, and the chroma as NV12 of frame 1 with 8 padding bytes per row
    y_clip = torch.full((n, 2, out_h, out_w), 77, dtype=torch.uint8, device=cuda)
    uv_clip = torch.full((n, 2, out_h // 2, out_w + 8), 77, dtype=torch.uint8, device=cuda)
    y, u, v = y_clip[:, 1], uv_clip[:, 1, :, 0:out_w:2], uv_clip[:, 1, :, 1:out_w:2]
    with torch.no_grad():
        ops.sr_tail_yuv420(conv, x, lr, s, y, u, v, out_h, out_w, kr, kb)
        sr = (F.conv2d(x.double().contiguous(), conv.weight.double(), conv.bias.double(), 1, 1)
              + F.interpolate(lr.double(), scale_factor=s, mode="bilinear", align_corners=False))[..., :out_h, :out_w]
    torch.cuda.synchronize()
    assert (sr < 0).any() and (sr > 1).any() and ((sr > 0) & (sr < 1)).double().mean() > 0.3
    p = sr.clamp(0, 1)
    luma = lambda a: kr * a[:, 0] + (1 - kr - kb) * a[:, 1] + kb * a[:, 2]       # noqa: E731
    m = F.avg_pool2d(p, 2)
    check_codes(y, 16 + 219 * luma(p))
    check_codes(u, 128 + 112 * (m[:, 2] - luma(m)) / (1 - kb))
    check_codes(v, 128 + 112 * (m[:, 0] - luma(m)) / (1 - kr))
    assert (y_clip[:, 0] == 77).all() and (uv_clip[:, 0] == 77).all()            # the other frame is untouched
    assert (uv_clip[:, 1, :, out_w:] == 77).all()                                 # and so is the NV12 row padding


# ------------------------------------------------------------------------------------------------
# the model
# ------------------------------------------------------------------------------------------------
def _net(cuda, scale, dtype):
    net = EAVSRP(scale).eval()
    seeded_parameters(net)
    return net.to(cuda).prepare(dtype)


def _planes(cuda, t, h, w, seed, matrix="bt709"):
    y, u, v = rgb_to_yuv420(clip_inputs(1, t, h, w, seed=seed), *MATRICES[matrix])
    return y.to(cuda), u.to(cuda), v.to(cuda)


def _yuv_of_forward(net, y, u, v, matrix):
    kr, kb = MATRICES[matrix]
    h, w = y.shape[-2:]
    s = net.scale
    with torch.no_grad():
        sr = net(pad_clip(yuv420_to_rgb(y, u, v, kr, kb)))[..., :s * h, :s * w]
    return rgb_to_yuv420(sr, kr, kb)


def _memoised_hr_features(net):
    """Both forwards see the same HR features: the channel-attention sums of the propagation and reconstruction
    groups use float atomics, so two runs agree to rounding only (DESIGN.md section 4), and these tests are about
    the tail."""
    hr_features, memo = net._hr_features, {}

    def hr_once(feats, i):
        if i not in memo:
            memo[i] = hr_features(feats, i)
        return memo[i]
    net._hr_features = hr_once
    return memo


@pytest.mark.parametrize("matrix", sorted(MATRICES))
@pytest.mark.parametrize("scale", [4, 2])
@pytest.mark.parametrize("t, h, w", [(4, 64, 64), (3, 70, 90)])       # 70x90: padded to 72x92, cropped back
def test_model_bf16_matches_yuv_of_forward(cuda, matrix, scale, t, h, w):
    net = _net(cuda, scale, torch.bfloat16)
    y, u, v = _planes(cuda, t, h, w, 21, matrix)
    got = net.forward_yuv420(y, u, v, matrix=matrix)
    assert [tuple(p.shape) for p in got] == [(1, t, scale * h, scale * w)] + [(1, t, scale * h // 2, scale * w // 2)] * 2
    assert all(p.dtype == torch.uint8 for p in got)
    want = _yuv_of_forward(net, y, u, v, matrix)
    for name, a, b in zip("YUV", got, want):
        diff = (a.float() - b.float()).abs()
        frac = (diff > 0).double().mean().item()
        # forward rounds conv_last's output to bf16 before adding the base; the fused tail keeps it in fp32
        print(f"{matrix} x{scale} {t}x{h}x{w} {name}: {frac:.5f} of the values differ by one level")
        assert diff.max().item() <= 1
        assert frac <= 0.01


@pytest.mark.parametrize("scale", [4, 2])
def test_model_fp32_matches_yuv_of_forward_exactly(cuda, scale):
    net = _net(cuda, scale, torch.float32)
    y, u, v = _planes(cuda, 3, 70, 90, 5)
    memo = _memoised_hr_features(net)
    try:
        got = net.forward_yuv420(y, u, v)
        want = _yuv_of_forward(net, y, u, v, "bt709")
    finally:
        del net._hr_features
    assert len(memo) == 3
    for a, b in zip(got, want):
        assert torch.equal(a, b)


def test_nv12_views_match_i420_planes(cuda):
    net = _net(cuda, 4, torch.bfloat16)
    t, h, w, s = 3, 64, 96, 4
    y, u, v = _planes(cuda, t, h, w, 9, "bt601")
    uv = torch.stack([u, v], -1).view(1, t, h // 2, w)                   # NV12 input: interleaved chroma
    y_nv = torch.full((1, t, s * h, s * w + 16), 77, dtype=torch.uint8, device=cuda)    # row pitch > width
    uv_nv = torch.full((1, t, s * h // 2, s * w + 16), 77, dtype=torch.uint8, device=cuda)
    out = (y_nv[..., :s * w], uv_nv[..., 0:s * w:2], uv_nv[..., 1:s * w:2])
    _memoised_hr_features(net)
    try:
        i420 = net.forward_yuv420(y, u, v, matrix="bt601")
        ret = net.forward_yuv420(y, uv[..., 0::2], uv[..., 1::2], matrix="bt601", out=out)
    finally:
        del net._hr_features
    assert all(a is b for a, b in zip(ret, out))
    for a, b in zip(i420, out):
        assert torch.equal(a, b)
    assert (y_nv[..., s * w:] == 77).all() and (uv_nv[..., s * w:] == 77).all()


def test_forward_yuv420_graph_capture(cuda):
    net = _net(cuda, 4, torch.bfloat16)
    a = _planes(cuda, 4, 64, 64, 7)
    b = _planes(cuda, 4, 64, 64, 8)
    static = [p.clone() for p in a]
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        net.forward_yuv420(*static)                         # warm-up outside capture (packed weights, cuDNN)
    torch.cuda.current_stream().wait_stream(st)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = net.forward_yuv420(*static)
    for p, q in zip(static, b):
        p.copy_(q)
    graph.replay()
    torch.cuda.synchronize()
    eager = net.forward_yuv420(*b)
    for o, e in zip(out, eager):
        assert (o.int() - e.int()).abs().max().item() <= 1
    assert not torch.equal(out[0], net.forward_yuv420(*a)[0])   # the replay computed clip b, not the captured a
