"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol declared in
include/eavsr_b200.h, and the Python mirror keeps the reference's error behaviour.  No compute."""
import ctypes
import os
import re

import pytest
import torch

import eavsr_b200 as E
from eavsr_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_text():
    text = open(os.path.join(ROOT, "include", "eavsr_b200.h")).read()
    return re.sub(r"/\*.*?\*/", "", text, flags=re.S)


def declared_symbols():
    return sorted(set(re.findall(r"\b(eavsr_[a-z0-9_]+)\s*\(", header_text())))


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(str(L.lib_path()))
    names = declared_symbols()
    assert len(names) >= 11
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(L.EXPORTED_SYMBOLS) == names      # the ctypes binding covers the whole header


def test_constants_match_the_header_defines():
    defines = {k: int(v) for k, v in re.findall(r"#define EAVSR_(\w+) (\d+)u?\b", header_text())}
    consts = {k: v for k, v in vars(L).items() if k.isupper() and type(v) is int}
    assert len(consts) >= 15
    for name, value in consts.items():
        assert defines.get(name) == value, name


@pytest.mark.parametrize("cls, c_name", [(L.FlowTerm, "EavsrFlowTerm"), (L.ConvLayer, "EavsrConvLayer")])
def test_structures_match_the_header_typedefs(cls, c_name):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (c_name, c_name), header_text(), flags=re.S).group(1)
    fields = []
    for decl in body.split(";")[:-1]:
        first, *more = decl.split(",")            # "int h, w" declares two fields
        fields += [first.split()[-1].lstrip("*")] + [m.strip() for m in more]
    assert [f for f, _ in cls._fields_] == fields


def test_unreadable_header_fails_loudly(monkeypatch, tmp_path):
    header = tmp_path / "eavsr_b200.h"
    monkeypatch.setattr(L, "_HEADER", header)
    L._signatures.cache_clear()
    try:
        with pytest.raises(L.EavsrError, match="not found"):
            L._signatures()
        header.write_text("int eavsr_f(const double x[4],\n            void* stream);\n")
        with pytest.raises(L.EavsrError, match=r"eavsr_f uses `const double\[4\]`"):
            L._signatures()
    finally:
        L._signatures.cache_clear()


def test_library_loads_and_reports_version():
    lib = L.load()
    assert lib.eavsr_version() >= 100
    assert isinstance(L.launch_count(), int)


def test_invalid_arguments_are_rejected_without_a_gpu():
    lib = L.load()
    s = L.Strides(1, 1, 1, 1)
    rc = lib.eavsr_flow_warp_forward(None, s, None, 0, None, s, 1, 1, 1, 1, 0, 0, None)
    assert rc == 1 and b"null pointer" in lib.eavsr_last_error()
    rc = lib.eavsr_correlation_forward(1, 1, 1, 0, 4, 4, 4, 0, None)
    assert rc == 1 and b"empty" in lib.eavsr_last_error()
    with pytest.raises(L.EavsrError):
        L.check(rc, "x")
    assert lib.eavsr_dcn_forward_workspace(64, 64, 3, 3, 1, 8, L.BF16) == 9 * 8192
    assert lib.eavsr_dcn_forward_workspace(64, 64, 3, 3, 1, 8, L.F32) == 2 * 9 * 8192
    assert lib.eavsr_dcn_forward_workspace(32, 64, 3, 3, 1, 8, L.F32) == 0
    nhwc = L.Strides(64 * 80, 1, 64 * 10, 64)
    nchw = L.Strides(64 * 80, 80, 10, 1)
    geo = (64, 64, 3, 3, 1, 1, 1, 1, 1, 1, 1, 8)
    assert lib.eavsr_dcn_forward_uses_tensor_cores(nhwc, nhwc, *geo, 0) == 1
    assert lib.eavsr_dcn_forward_uses_tensor_cores(nchw, nhwc, *geo, 0) == 0
    assert lib.eavsr_dcn_forward_uses_tensor_cores(nhwc, nhwc, *geo, L.DCN_FORCE_GENERIC) == 0
    assert lib.eavsr_dcn_forward_uses_tensor_cores(nhwc, nhwc, 64, 64, 3, 3, 2, 2, 1, 1, 1, 1, 1, 8, 0) == 0


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setenv("EAVSR_B200_LIB", str(tmp_path / "nope.so"))
    monkeypatch.setattr(L, "_lib", None)
    with pytest.raises(L.EavsrError, match="no CPU or PyTorch fallback"):
        L.load()


def test_cpu_tensors_raise_like_the_reference():
    x = torch.zeros(1, 4, 8, 8)
    with pytest.raises(NotImplementedError):
        E.flow_warp(x, torch.zeros(1, 2, 8, 8))
    with pytest.raises(NotImplementedError):                 # pwc/correlation/correlation.py:324-325
        E.FunctionCorrelation(tenFirst=x, tenSecond=x)
    with pytest.raises(NotImplementedError):
        E.modulated_deform_conv2d(torch.zeros(1, 64, 8, 8), torch.zeros(1, 144, 8, 8), torch.zeros(1, 72, 8, 8),
                                  torch.zeros(64, 64, 3, 3), None, 1, 1, 1, 1, 8)


def test_flow_warp_error_conventions():
    x = torch.zeros(1, 4, 8, 8)
    with pytest.raises(ValueError, match="spatial sizes"):   # models/networks.py:719-721
        E.flow_warp(x, torch.zeros(1, 2, 8, 9))
    with pytest.raises(ValueError, match="spatial sizes"):   # models/eavsrp_model.py:606-608
        E.flow_warp_nhw2(x, torch.zeros(1, 9, 8, 2))


def test_dcn_module_mirrors_mmcv_interface():
    class Sub(E.ModulatedDeformConv2d):                       # as MultiAdSTN does, models/networks.py:575-583
        def __init__(self):
            super().__init__(64, 64, kernel_size=3, padding=1, stride=1, dilation=1, deform_groups=8)

    m = Sub()
    assert m.weight.shape == (64, 64, 3, 3) and m.bias.shape == (64,)
    assert (m.stride, m.padding, m.dilation, m.groups, m.deform_groups) == ((1, 1), (1, 1), (1, 1), 1, 8)
    assert m.weight.abs().max() <= 1 / 24 and m.bias.abs().sum() == 0
    assert sorted(m.state_dict()) == ["bias", "weight"]
    with pytest.raises(ValueError, match="Expected 4D tensor"):
        E.modulated_deform_conv2d(torch.zeros(64, 8, 8), None, None, m.weight, m.bias, 1, 1, 1, 1, 8)
