"""The squared-error tail (eavsr_sr_tail_u8_sse_forward) against sr_tail_u8 and an int64 sum in PyTorch, and
EAVSRP.psnr_uint8 against forward_uint8 (bf16) and the visuals of forward (fp32)."""
import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from eavsr_b200 import ops
from eavsr_b200.model import EAVSRP, pad_clip, psnr_from_sse
from eavsr_b200.synthetic import clip_inputs, gen, seeded_parameters

pytestmark = pytest.mark.gpu

SENTINEL = 7_000_000_000_123                      # more than 32 bits, in every sum slot the kernel must not touch


def sse64(frames, hr):
    """Exact int64 sum of (frames - hr)**2 over the last three dimensions (y, x, c)."""
    d = frames.int() - hr.int()
    return (d * d).flatten(frames.dim() - 3).sum(-1, dtype=torch.int64)


def _operands(cuda, n, h, w, s, seed):
    """As tests/test_gpu_sr_tail.py: residuals of O(1) around a [0, 1] base, so both clamps are hit."""
    g = gen(seed)
    conv = nn.Conv2d(64, 3, 3, 1, 1)
    with torch.no_grad():
        conv.weight.copy_((torch.rand(conv.weight.shape, generator=g) * 2 - 1) * 0.05)
        conv.bias.copy_((torch.rand(3, generator=g) * 2 - 1) * 0.2)
    conv = conv.to(cuda, torch.bfloat16).eval()
    # drawn on the device, (n, h, w, 64) viewed as channels_last (n, 64, h, w): the largest maps are 0.8 GB
    gd = torch.Generator(device=cuda).manual_seed(seed)
    x = torch.randn(n, h, w, 64, generator=gd, device=cuda, dtype=torch.bfloat16).permute(0, 3, 1, 2)
    lr = torch.rand(n, 2, 3, h // s, w // s, generator=g).to(cuda)[:, 1]                   # a strided LR frame
    return conv, x, lr, g


# ------------------------------------------------------------------------------------------------
# the operator
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n, h, w, s, out_h, out_w", [
    (3, 72, 100, 4, 72, 100),        # W not a multiple of the 30-pixel tile or the 32-pixel halo
    (3, 70, 94, 2, 70, 94),          # H not a multiple of the 4-row tile
    (3, 40, 24, 4, 40, 24),          # W < 32: the halo box is wider than the map
    (3, 66, 130, 2, 63, 125),        # crop in both directions
    (2, 1088, 1920, 4, 1080, 1920),  # one frame of the benchmark batch: 272x480 -> 1088x1920, cropped to 1080
])
def test_op_matches_sr_tail_u8_and_int64_sum(cuda, n, h, w, s, out_h, out_w):
    conv, x, lr, g = _operands(cuda, n, h, w, s, 5000 + h + w)
    # ground truth: frame 1 of 2, rows padded by 3 pixels
    hr = torch.randint(0, 256, (n, 2, out_h, out_w + 3, 3), generator=g, dtype=torch.uint8).to(cuda)[:, 1, :, :out_w]
    ref = torch.empty((n, out_h, out_w, 3), dtype=torch.uint8, device=cuda)
    clip = torch.full((n, 2, out_h, out_w + 5, 3), 77, dtype=torch.uint8, device=cuda)
    out = clip[:, 1, :, :out_w]                             # frame 1 of 2, rows padded by 5 pixels
    sums = torch.full((n, 4), SENTINEL, dtype=torch.int64, device=cuda)
    sums[:, 1] = 5                                          # added to, not overwritten
    sums[:, 2] = 0
    with torch.no_grad():
        ops.sr_tail_u8(conv, x, lr, s, ref, out_h, out_w)
        ops.sr_tail_u8_sse(conv, x, lr, s, hr, sums[:, 1], out_h, out_w, out=out)
        ops.sr_tail_u8_sse(conv, x, lr, s, hr, sums[:, 2], out_h, out_w)
    torch.cuda.synchronize()
    assert torch.equal(out, ref)
    want = sse64(ref, hr)
    assert torch.equal(sums[:, 1], want + 5)
    assert torch.equal(sums[:, 2], want)
    assert (sums[:, 0] == SENTINEL).all() and (sums[:, 3] == SENTINEL).all()
    assert (clip[:, 0] == 77).all() and (clip[:, 1, :, out_w:] == 77).all()
    assert (ref == 0).any() and (ref == 255).any()


@pytest.mark.parametrize("n", [2, 3])
def test_op_sums_beyond_32_bits_are_exact(cuda, n):
    """hr = 255 - frame: every sample adds (2q - 255)^2, and each image's sum passes 2^32.  With more tiles than fit
    in whole images per CTA, many CTAs have tiles of two images in their sequence."""
    h, w, s = 1088, 1920, 4
    conv, x, lr, _ = _operands(cuda, n, h, w, s, 6000 + n)
    frame = torch.empty((n, h, w, 3), dtype=torch.uint8, device=cuda)
    sums = torch.zeros((n, 3), dtype=torch.int64, device=cuda)
    with torch.no_grad():
        ops.sr_tail_u8(conv, x, lr, s, frame, h, w)
        hr = 255 - frame
        ops.sr_tail_u8_sse(conv, x, lr, s, hr, sums[:, 1], h, w)
    torch.cuda.synchronize()
    want = sse64(frame, hr)
    assert (want > 2 ** 32).all(), want
    assert torch.equal(sums[:, 1], want)
    assert (sums[:, 0] == 0).all() and (sums[:, 2] == 0).all()


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


def _clip(cuda, n, t, h, w, s, seed):
    """uint8 LR frames (n, t, h, w, 3) and their ground truth (n, t, s*h, s*w, 3), a strided view of planar frames:
    the LR frames are the ground truth's s x s means."""
    hr = clip_inputs(n, t, s * h, s * w, seed=seed)
    lr = F.avg_pool2d(hr.flatten(0, 1), s).view(n, t, 3, h, w)
    to_u8 = lambda a: (a * 255).round().to(torch.uint8).to(cuda)          # noqa: E731
    return to_u8(lr).permute(0, 1, 3, 4, 2).contiguous(), to_u8(hr).permute(0, 1, 3, 4, 2)


def _psnr64(sse, samples):
    return 10 * np.log10(255.0 ** 2 * samples / sse.cpu().numpy().astype(np.float64))


@pytest.mark.parametrize("scale", [4, 2])
@pytest.mark.parametrize("t, h, w", [(4, 64, 64), (3, 70, 90)])       # 70x90: padded to 72x92, cropped back
def test_model_bf16_matches_forward_uint8(cuda, scale, t, h, w):
    n, s = 2, scale
    net = _net(cuda, scale, torch.bfloat16)
    frames, hr = _clip(cuda, n, t, h, w, s, 31)
    clip = torch.full((n, t, s * h, s * w + 4, 3), 77, dtype=torch.uint8, device=cuda)
    out = clip[..., :s * w, :]
    memo = _memoised_hr_features(net)
    try:
        want = net.forward_uint8(frames)
        psnr, sse = net.psnr_uint8(frames, hr, out=out)
        psnr2, sse2 = net.psnr_uint8(frames, hr)
    finally:
        del net._hr_features
    assert len(memo) == t
    assert sse.shape == (n, t) and sse.dtype == torch.int64 and psnr.shape == (n, t) and psnr.dtype == torch.float64
    assert torch.equal(out, want)
    assert (clip[..., s * w:, :] == 77).all()
    assert torch.equal(sse, sse64(want, hr))
    assert torch.equal(sse2, sse) and torch.equal(psnr2, psnr)
    np.testing.assert_allclose(psnr.cpu().numpy(), _psnr64(sse, 3 * s * h * s * w), rtol=1e-12)
    print(f"x{scale} {t}x{h}x{w}: PSNR {psnr.mean().item():.2f} dB")
    assert (psnr > 15).all() and (psnr < 60).all()


@pytest.mark.parametrize("scale", [4, 2])
def test_model_fp32_matches_visuals_of_forward_exactly(cuda, scale):
    n, t, h, w, s = 1, 3, 70, 90, scale
    net = _net(cuda, scale, torch.float32)
    frames, hr = _clip(cuda, n, t, h, w, s, 32)
    out = torch.empty((n, t, s * h, s * w, 3), dtype=torch.uint8, device=cuda)
    memo = _memoised_hr_features(net)
    try:
        psnr, sse = net.psnr_uint8(frames, hr, out=out)
        with torch.no_grad():
            sr = net(pad_clip(frames.permute(0, 1, 4, 2, 3).float() / 255))[..., :s * h, :s * w]
    finally:
        del net._hr_features
    assert len(memo) == t
    visuals = torch.clamp(sr.float() * 255, 0, 255).round().permute(0, 1, 3, 4, 2).to(torch.uint8)
    assert torch.equal(out, visuals)
    assert torch.equal(sse, sse64(visuals, hr))
    assert torch.equal(psnr, psnr_from_sse(sse, 3 * s * h * s * w))


def test_graph_capture(cuda):
    n, t, h, w, s = 1, 4, 64, 64, 4
    net = _net(cuda, s, torch.bfloat16)
    fa, ha = _clip(cuda, n, t, h, w, s, 7)
    fb, hb = _clip(cuda, n, t, h, w, s, 8)
    static_f, static_h = fa.clone(), ha.clone()
    out = torch.empty((n, t, s * h, s * w, 3), dtype=torch.uint8, device=cuda)

    def run():
        return net.psnr_uint8(static_f, static_h, out=out)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        run()                                              # warm-up outside capture (packed weights, cuDNN)
    torch.cuda.current_stream().wait_stream(st)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        psnr, sse = run()
    static_f.copy_(fb)
    static_h.copy_(hb)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(sse, sse64(out, hb))                 # the replay measured the frames it wrote against hb
    assert torch.equal(psnr, psnr_from_sse(sse, 3 * s * h * s * w))
    eager_out = torch.empty_like(out)
    eager_psnr, eager_sse = net.psnr_uint8(fb, hb, out=eager_out)
    # two runs of the trunk agree to rounding only (float atomics): the frames by one level at most
    assert (out.int() - eager_out.int()).abs().max().item() <= 1
    assert (psnr - eager_psnr).abs().max().item() <= 0.01
    first_psnr, _ = net.psnr_uint8(fa, ha)
    assert not torch.equal(psnr, first_psnr)                # the replay computed clip b, not the captured a
