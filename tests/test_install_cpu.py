"""The drop-in route: with eavsr_b200.install the UNMODIFIED reference imports and builds its
EAVSRP with our ModulatedDeformConv2d / flow_warp / correlation.  Needs a checkout of the reference
(HITRainer/EAVSR), named by EAVSR_REFERENCE; the forward itself needs a GPU (there is no CPU fallback),
which is asserted."""
import os
import subprocess
import sys
import textwrap

import pytest

REF = os.environ.get("EAVSR_REFERENCE", "")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "models")),
                                reason="EAVSR_REFERENCE does not name a checkout of the reference")


def test_reference_builds_on_our_ops():
    code = textwrap.dedent(f"""
        import sys, types
        sys.path[:0] = [{ROOT!r}, {REF!r}]
        import torch, torchvision.models.vgg as vgg
        _o = vgg.vgg16
        vgg.vgg16 = lambda pretrained=False, **kw: _o(weights=None, **kw)
        import eavsr_b200.install as I
        import eavsr_b200 as E
        I.install()
        import models.networks as N
        import models.eavsrp_model as M
        from pwc.correlation import correlation
        assert N.ModulatedDeformConv2d is E.ModulatedDeformConv2d
        assert N.modulated_deform_conv2d is E.modulated_deform_conv2d
        assert correlation.FunctionCorrelation is E.FunctionCorrelation
        assert sorted(I.rebind_flow_warp()) == ["models.eavsrp_model", "models.networks"]
        assert N.flow_warp is E.flow_warp and M.flow_warp is E.flow_warp_nhw2
        net = M.EAVSRP(types.SimpleNamespace(scale=4, predict=False, n_frame=3, n_flow=5), None)
        assert isinstance(net.deform_align["backward_1"], E.ModulatedDeformConv2d)
        from eavsr_b200.model import EAVSRP
        ours = EAVSRP(4)
        assert sorted(ours.state_dict()) == sorted(net.state_dict())
        ours.load_state_dict(net.state_dict(), strict=True)
        try:
            net(torch.rand(1, 3, 3, 64, 64))
        except NotImplementedError as e:
            assert "no CPU fallback" in str(e)
        else:
            raise SystemExit("expected NotImplementedError on CPU tensors")
        print("OK")
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
