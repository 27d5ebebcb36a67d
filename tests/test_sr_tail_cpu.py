"""CPU tests of the uint8 reconstruction tail: the ctypes prototypes derived from the header, and the input
checks of EAVSRP.forward_uint8, which must fail before anything is launched."""
from ctypes import POINTER, c_int, c_int64, c_size_t, c_void_p

import pytest
import torch

from eavsr_b200 import _lib as L
from eavsr_b200.model import EAVSRP

NAMES = ("eavsr_sr_tail_packed_weight_bytes", "eavsr_sr_tail_pack_weight", "eavsr_sr_tail_u8_forward")


def test_prototypes_come_from_the_header():
    assert set(NAMES) <= set(L.EXPORTED_SYMBOLS)
    sigs = L._signatures()
    assert sigs["eavsr_sr_tail_packed_weight_bytes"] == (c_size_t, [])
    assert sigs["eavsr_sr_tail_pack_weight"] == (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p])
    res, args = sigs["eavsr_sr_tail_u8_forward"]
    assert res is c_int and len(args) == 17
    strides = POINTER(c_int64)
    # x, x_strides, packed_weight, bias, lr, lr_strides, out, out_strides, n, c, h, w, scale, out_h, out_w, dtype, stream
    assert args == [c_void_p, strides, c_void_p, c_void_p, c_void_p, strides, c_void_p, strides] + [c_int] * 8 + [c_void_p]


@pytest.fixture(scope="module")
def net():
    return EAVSRP(4, n_resblock=1).eval()


@pytest.mark.parametrize("frames, err", [
    (torch.zeros(1, 2, 64, 64, 3), TypeError),                          # float frames
    (torch.zeros(1, 2, 64, 64, 3, dtype=torch.int16), TypeError),
    (torch.zeros(2, 64, 64, 3, dtype=torch.uint8), ValueError),         # no batch dimension
    (torch.zeros(1, 2, 64, 64, 4, dtype=torch.uint8), ValueError),      # RGBA
    (torch.zeros(1, 2, 3, 64, 64, dtype=torch.uint8), ValueError),      # channels first
    (torch.zeros(1, 2, 64, 64, 3, dtype=torch.uint8), NotImplementedError),   # CPU tensor
])
def test_forward_uint8_rejects_bad_input_before_any_launch(net, monkeypatch, frames, err):
    def no_trunk(lrs):
        raise AssertionError("the trunk ran on rejected input")
    monkeypatch.setattr(net, "_trunk", no_trunk)
    before = L.launch_count()
    with pytest.raises(err):
        net.forward_uint8(frames)
    assert L.launch_count() == before
