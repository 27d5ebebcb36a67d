"""`ops.adapt_mix` against a reference that rounds the intermediate the way the kernel does: stage 1 in fp64, y
rounded to the dtype, stage 2 in fp64.  The kernel sums each accumulator in fp32, so fp32 results agree to a few
ulps and bf16 results are nearly all the exactly rounded value; a wrong tap or channel moves far more elements."""
import pytest
import torch
import torch.nn.functional as F

from eavsr_b200 import ops

pytestmark = pytest.mark.gpu


def _cl(t):
    return t.contiguous(memory_format=torch.channels_last)


def _operands(n, h, w, dtype, dev, seed=5):
    g = torch.Generator(device=dev).manual_seed(seed)
    mk = lambda *s: torch.randn(*s, generator=g, device=dev)      # noqa: E731
    a, b = _cl(mk(n, 64, h, w).to(dtype)), _cl(mk(n, 64, h, w).to(dtype))
    params = [(mk(128, 1, 3, 3) * 0.3).to(dtype), (mk(128) * 0.1).to(dtype),
              (mk(64, 2, 3, 3) * 0.3).to(dtype), (mk(64) * 0.1).to(dtype)]
    return a, b, params


def _reference(a, b, w1, b1, w2, b2, dtype):
    """(reference, magnitude): the magnitude sums |term| over both stages and bounds what rounding can move."""
    d = lambda t: t.double()                                       # noqa: E731
    x = torch.cat([d(a), d(b)], 1)
    y = F.leaky_relu(F.conv2d(x, d(w1), d(b1), padding=1, groups=128), 0.2)
    y = y.to(dtype).double()                                       # the kernel keeps y in the dtype
    ref = F.leaky_relu(F.conv2d(y, d(w2), d(b2), padding=1, groups=64), 0.2)
    mag1 = F.conv2d(x.abs(), d(w1).abs(), d(b1).abs(), padding=1, groups=128)
    mag = F.conv2d(mag1, d(w2).abs(), d(b2).abs(), padding=1, groups=64)
    return ref, mag


def _check(out, ref, mag, dtype):
    assert out.shape == ref.shape and out.dtype == dtype
    err = (out.double() - ref).abs()
    if dtype == torch.float32:
        # fp32 sums of 10 (stage 1) and 19 (stage 2) terms
        assert (err <= 32 * torch.finfo(dtype).eps * mag).all(), err.max().item()
        return
    # bf16: the fp32 sums round to the bf16 of the exact value except near a rounding boundary, where y or the
    # output may land one bf16 step away
    assert (out == ref.to(dtype)).double().mean().item() > 0.99
    assert (err <= torch.finfo(dtype).eps * (ref.abs() + mag)).all(), err.max().item()


SHAPES = [(1, 17, 23), (2, 8, 16), (1, 67, 120), (1, 5, 3), (3, 1, 1), (2, 9, 33), (1, 16, 2),
          # more work items than one wave of persistent CTAs, with partial tiles on both edges
          (5, 41, 77)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_adapt_mix_rounded_reference(cuda, shape, dtype):
    a, b, p = _operands(*shape, dtype, cuda)
    with torch.no_grad():
        out = ops.adapt_mix(a, b, *p, 0.2)
    _check(out, *_reference(a, b, *p, dtype), dtype)


@pytest.mark.parametrize("shape", [(8, 272, 480), (8, 136, 240), (8, 68, 120)])
def test_adapt_mix_operating_shapes(cuda, shape):
    """The three resolutions MultiAdSTN runs at in the benchmark, 8 images each (bf16)."""
    dtype = torch.bfloat16
    a, b, p = _operands(*shape, dtype, cuda)
    with torch.no_grad():
        out = ops.adapt_mix(a, b, *p, 0.2)
        for i in range(shape[0]):                                  # fp64 reference one image at a time
            _check(out[i:i + 1], *_reference(a[i:i + 1], b[i:i + 1], *p, dtype), dtype)


def test_adapt_mix_graph_capture(cuda):
    a, b, p = _operands(2, 37, 45, torch.bfloat16, cuda)
    with torch.no_grad():
        eager = ops.adapt_mix(a, b, *p, 0.2)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            ops.adapt_mix(a, b, *p, 0.2)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = ops.adapt_mix(a, b, *p, 0.2)
        a.copy_(a.flip(3))                                         # replays read the buffers' current contents
        g.replay()
        torch.cuda.synchronize()
    assert torch.equal(out, ops.adapt_mix(a, b, *p, 0.2))
    assert not torch.equal(out, eager)
