"""EAVSR+ (x4 / x2) forward on the B200 alignment kernels -- the callers of the hot path.

This is the host-side orchestration that sits directly above the hot path in the reference
(SURVEY.md section 8 row a8): ``EAVSRP.forward / compute_flow / propagate / upsample``
(models/eavsrp_model.py:179-364, x2 twin models/eavsrpx2_model.py), ``MultiAdSTN.forward``
(models/networks.py:597-631), ``AdaptBlockOffset`` / ``AdaptBlock2_3x3`` (:280-348) and the live
``SPyNet`` (models/eavsrp_model.py:402-585).  The module tree reproduces the reference's parameter
names and shapes, so a reference ``EAVSRP_model_*.pth`` state dict loads with ``strict=True``.

What is B200-specific here:
  * every bilinear warp and the DCNv2 run in libeavsr_b200.so (no grid tensors, no im2col buffer);
  * activations are channels_last and (by default) bf16, flows / offsets / masks stay fp32;
  * SPyNet runs once on both directions stacked in one batch;
  * the per-group affine offset expansion is a broadcast expression, not a (n*P*D) x 2x2 bmm with
    four permute copies.
Dense 3x3/5x5/7x7 convolutions stay on cuDNN (out of scope, SURVEY.md section 2).
"""
from __future__ import annotations

from collections import OrderedDict

import torch
import torch.nn as nn
import torch.nn.functional as F

from .ops import (ModulatedDeformConv2d, adapt_mix, grouped_conv3x3, grouped_conv3x3_eligible, channel_mean, scale_residual,
                  conv2d_native_bias_grad, affine_offsets_mask, ca_residual, ca_scale, cat_channels, conv2d_bias_act,
                  conv2d_bias_act_shuffle,
                  dcn_affine, dcn_affine_eligible,
                  conv3x3_64, conv3x3_64_ca, conv3x3_64_eligible, conv3x3_chain_eligible, rca_group_chain,
                  flow_warp, flow_warp2, flow_warp_nhw2, flow_warp_pyramid, flow_warp_pyramid_eligible, fused_inference_ok,
                  spynet_level_input, sr_tail_u8, sr_tail_u8_eligible, sr_tail_yuv420,
                  sr_tail_u16, sr_tail_yuv420_u16, sr_tail_u8_sse,
                  modulated_deform_conv2d)
from .yuv import HBD_MATRICES, MATRICES, check_bits, rgb_to_yuv420, yuv420_to_rgb

__all__ = ["EAVSRP", "MultiAdSTN", "SPyNet"]


# --------------------------------------------------------------------------------------------
# small blocks (names chosen so that state-dict keys equal the reference's)
# --------------------------------------------------------------------------------------------
class _CALayer(nn.Module):
    def __init__(self, ch=64, reduction=16):
        super().__init__()
        self.conv_du = nn.Sequential(nn.Conv2d(ch, ch // reduction, 1), nn.ReLU(inplace=True),
                                     nn.Conv2d(ch // reduction, ch, 1), nn.Sigmoid())

    def forward(self, x):
        return x * self.conv_du(channel_mean(x))      # (native channel sums for CUDA channels_last maps)


class _RCABlock(nn.Module):
    def __init__(self, ch=64):
        super().__init__()
        self.res = nn.Sequential(nn.Conv2d(ch, ch, 3, 1, 1), nn.ReLU(inplace=True), nn.Conv2d(ch, ch, 3, 1, 1))
        self.ca = _CALayer(ch)

    def forward(self, x, sums_buf=None):
        du = self.ca.conv_du
        if conv3x3_64_eligible(self.res[0], x):
            # both convolutions on tcgen05: bias+ReLU in the first epilogue, bias + the channel sums of
            # the attention layer in the second; then one scale+residual pass.  3 kernels per block.
            h = conv3x3_64(self.res[0], x, 0.0)
            res, sums = conv3x3_64(self.res[2], h, 1.0, want_sums=True, sums_out=sums_buf)
            return ca_scale(res, x, sums, du[0].weight, du[0].bias, du[2].weight, du[2].bias, 16)
        if x.shape[1] == 64 and fused_inference_ok(x, self.res[0].weight):
            # conv+bias+ReLU epilogue in one pass, second conv bias-free (its bias is folded into the
            # channel-attention kernels), then reduce + MLP + scale + residual add in 2 kernels
            h = conv2d_bias_act(self.res[0], x, 0.0)
            c2 = self.res[2]
            res = F.conv2d(h, c2.weight, None, c2.stride, c2.padding)
            return ca_residual(res, x, du[0].weight, du[0].bias, du[2].weight, du[2].bias, 16, res_bias=c2.bias)
        # differentiable path (training): cuDNN convolutions, bias gradients and the attention's pooling on the
        # library's channel-sum kernel
        h = F.relu(conv2d_native_bias_grad(self.res[0], x), inplace=True)
        r = conv2d_native_bias_grad(self.res[2], h)
        return scale_residual(r, self.ca.conv_du(channel_mean(r)), x)      # == self.ca(r) + x


class _RCAGroup(nn.Module):
    def __init__(self, ch=64, nb=30):
        super().__init__()
        self.rg = nn.Sequential(*[_RCABlock(ch) for _ in range(nb)], nn.Conv2d(ch, ch, 3, 1, 1))
        self.chain = True          # inference: run the group as one chained launch when eligible

    def forward(self, x):
        blocks = self.rg[:-1]
        if self.chain and len(blocks) > 0 and conv3x3_chain_eligible(
                [c for b in blocks for c in (b.res[0], b.res[2])] + [self.rg[-1]], x):
            # the whole group -- 2 convolutions per block + the closing one -- as ONE cooperative tcgen05 launch
            return rca_group_chain(list(blocks), self.rg[-1], x) + x
        if conv3x3_64_eligible(self.rg[-1], x) and x.shape[0] <= 8 and len(blocks) > 0:
            # tcgen05 chain with the channel attention of block i folded into the first convolution of block
            # i+1 (and of the last block into the group's closing convolution): 2 launches per block,
            # y_i = y_{i-1} + res_i * scale_i is produced by the consumer's loader warps.
            pool = torch.zeros((len(blocks), x.shape[0], 64), dtype=torch.float32, device=x.device)
            y, res, sums, prev = x, None, None, None
            for i, blk in enumerate(blocks):
                if prev is None:
                    h = conv3x3_64(blk.res[0], y, 0.0)
                else:
                    du = prev.ca.conv_du
                    h, y = conv3x3_64_ca(blk.res[0], y, res, sums, du[0].weight, du[0].bias, du[2].weight, du[2].bias, 0.0)
                res, sums = conv3x3_64(blk.res[2], h, 1.0, want_sums=True, sums_out=pool[i])
                prev = blk
            du = prev.ca.conv_du
            out, _ = conv3x3_64_ca(self.rg[-1], y, res, sums, du[0].weight, du[0].bias, du[2].weight, du[2].bias, 1.0)
            return out + x
        y = x
        for blk in blocks:
            y = blk(y)
        if conv3x3_64_eligible(self.rg[-1], y):
            return conv3x3_64(self.rg[-1], y, 1.0) + x
        if torch.is_grad_enabled():
            return conv2d_native_bias_grad(self.rg[-1], y) + x
        return conv2d_bias_act(self.rg[-1], y, 1.0) + x


class _ResidualStack(nn.Module):
    """conv3x3 + LeakyReLU(0.1) + RCAGroup (reference: ResidualBlocksWithInputConv)."""

    def __init__(self, cin, ch=64, nb=30):
        super().__init__()
        self.main = nn.Sequential(nn.Conv2d(cin, ch, 3, 1, 1), nn.LeakyReLU(0.1, inplace=True), _RCAGroup(ch, nb))

    def forward(self, x):
        return self.main[2](conv2d_bias_act(self.main[0], x, 0.1))


class _Encoder(nn.Module):
    """VGG16 conv1_1..conv3_1 with the pools removed + 3x3 tail (reference: ContrasExtractorLayer)."""

    def __init__(self, ch=64):
        super().__init__()
        spec = (("conv1_1", 3, 64), ("conv1_2", 64, 64), ("conv2_1", 64, 128), ("conv2_2", 128, 128),
                ("conv3_1", 128, 256))
        layers = OrderedDict()
        for i, (name, ci, co) in enumerate(spec):
            layers[name] = nn.Conv2d(ci, co, 3, 1, 1)
            if i + 1 < len(spec):
                layers[name.replace("conv", "relu")] = nn.ReLU(inplace=True)
        self.model = nn.Sequential(layers)
        self.tail = nn.Conv2d(256, ch, 3, 1, 1)
        self.register_buffer("mean", torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1))
        self.register_buffer("std", torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1))

    def forward(self, x):
        x = (x - self.mean) / self.std
        convs = [m for m in self.model if isinstance(m, nn.Conv2d)]
        for i, conv in enumerate(convs):
            x = conv2d_bias_act(conv, x, 0.0 if i + 1 < len(convs) else 1.0)   # no ReLU after conv3_1
        return conv2d_bias_act(self.tail, x, 1.0)


_R = ((-1., -1., -1., 0., 0., 0., 1., 1., 1.), (-1., 0., 1., -1., 0., 1., -1., 0., 1.))


def _affine_offsets(T, t, D, R=None):
    """offset[n, (g*9+k)*2+i] = sum_j T[n,g,i,j] * R[j,k] - R[i,k] + t[n,g,i]
    (reference: matmul + 4 permute/reshape copies at models/networks.py:302-310).
    R is the module's `regular_matrix` buffer (already on the device: no H2D copy, graph-safe)."""
    n, _, h, w = T.shape
    R = T.new_tensor(_R) if R is None else R.to(T.dtype)   # (2, 9)
    T = T.reshape(n, D, 1, 2, 2, h, w)                     # g, -, i, j
    Rk = R.t().reshape(1, 1, 9, 1, 2, 1, 1)                # -, -, k, -, j
    off = (T * Rk).sum(4) - R.t().reshape(1, 1, 9, 2, 1, 1) + t.reshape(n, D, 1, 2, h, w)
    return off.reshape(n, D * 18, h, w)


class _AdaptBase(nn.Module):
    native_grouped = True      # differentiable grouped 3x3 convolutions on the library's kernels (False: nn.Conv2d)

    def __init__(self, ch, n_mat, n_trans, k):
        super().__init__()
        self.register_buffer("regular_matrix", torch.tensor(_R))
        self.concat = nn.Sequential(nn.Conv2d(2 * ch, 2 * ch, 3, 1, 1, groups=2 * ch), nn.LeakyReLU(0.2, inplace=True))
        self.concat2 = nn.Sequential(nn.Conv2d(2 * ch, ch, 3, 1, 1, groups=ch), nn.LeakyReLU(0.2, inplace=True))
        self.transform_matrix_conv = nn.Conv2d(ch, n_mat, k, 1, k // 2)
        self.translation_conv = nn.Conv2d(ch, n_trans, k, 1, k // 2)

    def _merged_weight(self):
        ws = [self.transform_matrix_conv.weight, self.translation_conv.weight]
        if hasattr(self, "mask_conv"):
            ws.append(self.mask_conv.weight)
        key = tuple((w.data_ptr(), w._version, w.dtype) for w in ws)
        hit = getattr(self, "_merged", None)
        if hit is None or hit[0] != key:
            hit = (key, torch.cat([w.detach() for w in ws], 0).contiguous(memory_format=torch.channels_last))
            self._merged = hit
        return hit[1]

    def _mix(self, x, ref):
        if x.shape[1] == 64 and fused_inference_ok(x, ref):      # both grouped convs in one pass
            return adapt_mix(x, ref, self.concat[0].weight, self.concat[0].bias, self.concat2[0].weight,
                             self.concat2[0].bias, 0.2)
        xr = torch.cat([x, ref], 1)
        c1, c2 = self.concat[0], self.concat2[0]
        if self.native_grouped and grouped_conv3x3_eligible(c1, xr) and xr.dtype in (torch.float32, torch.bfloat16):
            # training path: cuDNN's grouped kernels (forward, and above all backward: 647 us per call on 8 MB
            # tensors + layout transforms) were ~30 % of the training step
            y = F.leaky_relu(grouped_conv3x3(c1, xr), 0.2)
            if grouped_conv3x3_eligible(c2, y):
                return F.leaky_relu(grouped_conv3x3(c2, y), 0.2)
            return self.concat2(y)
        return self.concat2(self.concat(xr))


class _AdaptBlock2_3x3(_AdaptBase):
    """One affine matrix + translation -> 18-channel offset (models/networks.py:318-348)."""

    def __init__(self, ch=64):
        super().__init__(ch, 4, 2, 3)

    def forward(self, x, ref):
        f = self._mix(x, ref)
        if fused_inference_ok(f, self.transform_matrix_conv.weight):
            ct, cr = self.transform_matrix_conv, self.translation_conv      # bias-free; biases added in-kernel
            y = F.conv2d(f, self._merged_weight(), None, 1, ct.padding)     # one 64 -> 6 convolution
            return affine_offsets_mask(y[:, :4], y[:, 4:6], None, 1, ct.bias, cr.bias)[0]
        T, t = self.transform_matrix_conv(f), self.translation_conv(f)
        return _affine_offsets(T.float(), t.float(), 1, self.regular_matrix)


class _AdaptBlockOffset(_AdaptBase):
    """Per-deformable-group affine offsets + sigmoid mask (models/networks.py:280-315)."""

    def __init__(self, ch=64, D=8):
        super().__init__(ch, 4 * D, 2 * D, 5)
        self.D = D
        self.mask_conv = nn.Conv2d(ch, 9 * D, 5, 1, 2)

    def raw(self, x, ref):
        """(n, 15*D, h, w) output of the merged bias-free convolution and the concatenated biases: the
        operands of `dcn_affine` (row f1), which expands offsets and masks inside the DCN kernel."""
        f = self._mix(x, ref)
        ct, cr, cm = self.transform_matrix_conv, self.translation_conv, self.mask_conv
        y = F.conv2d(f, self._merged_weight(), None, 1, ct.padding)
        key = tuple((b.data_ptr(), b._version) for b in (ct.bias, cr.bias, cm.bias))
        hit = getattr(self, "_merged_bias", None)
        if hit is None or hit[0] != key:
            hit = (key, torch.cat([ct.bias.detach(), cr.bias.detach(), cm.bias.detach()]).contiguous())
            self._merged_bias = hit
        return y, hit[1]

    def forward(self, x, ref):
        f = self._mix(x, ref)
        if fused_inference_ok(f, self.mask_conv.weight):
            # the three 5x5 convolutions read the same input: ONE bias-free 64 -> 15*D convolution, whose
            # channel slices (strided views, no copies) feed the expansion kernel; biases are added there
            ct, cr, cm = self.transform_matrix_conv, self.translation_conv, self.mask_conv
            y = F.conv2d(f, self._merged_weight(), None, 1, ct.padding)
            D = self.D
            return affine_offsets_mask(y[:, :4 * D], y[:, 4 * D:6 * D], y[:, 6 * D:], D, ct.bias, cr.bias, cm.bias)
        T, t, m = self.transform_matrix_conv(f), self.translation_conv(f), self.mask_conv(f)
        off = _affine_offsets(T.float(), t.float(), self.D, self.regular_matrix)
        return off, torch.sigmoid(m.float())


class _TransOffset(nn.Module):
    def __init__(self):
        super().__init__()
        self.conv_first = nn.Conv2d(18, 2, 3, 1, 1)

    def forward(self, off):
        return self.conv_first(off)


def _resize_flow(flow, scale):
    """bilinear, align_corners=True resize of a flow field, magnitudes scaled with it."""
    return F.interpolate(flow, scale_factor=scale, mode="bilinear", align_corners=True) * scale


class MultiAdSTN(ModulatedDeformConv2d):
    """Coarse-to-fine flow refinement on a 3-level pyramid, then DCNv2 with per-group affine
    offsets (reference: models/networks.py:575-631)."""

    def __init__(self, ch=64, deformable_groups=8):
        super().__init__(ch, ch, kernel_size=3, padding=1, stride=1, dilation=1, deform_groups=deformable_groups)
        for i in (1, 2, 3):
            setattr(self, f"flow_l{i}", _AdaptBlock2_3x3(ch))
        self.adastn = _AdaptBlockOffset(ch, deformable_groups)
        self.fuse_offsets = True     # inference: expand offsets / masks inside the DCN kernel (dcn_affine)
        self.fold_pyramid = True     # inference: evaluate the pyramid flows inside the warp kernels (row f2)
        for i in (3, 2, 1):
            setattr(self, f"trans_l{i}", _TransOffset())

    def _residual(self, lvl, warped, ref):
        off18 = getattr(self, f"flow_l{lvl}")(warped, ref)
        return getattr(self, f"trans_l{lvl}")(off18.to(warped.dtype)).float()

    def forward(self, nbr, ref, feat_prop, flow, out=None):
        """`out`: optional 64-channel slice of a wider channels_last buffer that receives the result when the
        fused-offset DCN runs (saves the torch.cat copy of the caller); the returned tensor is what to use."""
        flow = flow.float()
        if self.fold_pyramid and flow_warp_pyramid_eligible(nbr[0], feat_prop) and flow_warp_pyramid_eligible(nbr[1]) \
                and flow_warp_pyramid_eligible(nbr[2]) and nbr[0].dtype == torch.bfloat16:
            # row f2: the resized / rescaled / summed flows of the three pyramid levels are evaluated inside the warps
            w3 = flow_warp_pyramid(nbr[2], [(flow, 0.25)])
            p1 = self._residual(3, w3, ref[2])
            w2, p1_up = flow_warp_pyramid(nbr[1], [(flow, 0.5), (p1, 2.0)], keep=(1,))
            p2 = self._residual(2, w2, ref[1])
            w1, flow_p2 = flow_warp_pyramid(nbr[0], [(flow, 1.0), (p2, 2.0), (p1_up, 2.0)], want_flow=True)
            p3 = self._residual(1, w1, ref[0])
            nbr_w, feat = flow_warp_pyramid(nbr[0], [(flow_p2, 1.0), (p3, 1.0)], x2=feat_prop)
            return self._deform(nbr_w, feat, ref, out)
        f4 = _resize_flow(flow, 0.25)
        f2 = _resize_flow(flow, 0.5)
        p1 = self._residual(3, flow_warp(nbr[2], f4), ref[2])
        p1_up = _resize_flow(p1, 2)
        p2 = self._residual(2, flow_warp(nbr[1], f2 + p1_up), ref[1])
        p2_up = _resize_flow(p2 + p1_up, 2)
        p3 = self._residual(1, flow_warp(nbr[0], flow + p2_up), ref[0])
        flow = p3 + p2_up + flow
        if fused_inference_ok(nbr[0], feat_prop, flow):
            nbr_w, feat = flow_warp2(nbr[0], feat_prop, flow)     # one launch when eligible (row f2)
        else:
            nbr_w = flow_warp(nbr[0], flow)
            feat = flow_warp(feat_prop, flow)
        return self._deform(nbr_w, feat, ref, out)

    def _deform(self, nbr_w, feat, ref, out=None):
        """offsets / masks from the warped neighbour and the reference, then DCNv2 (models/networks.py:625-630)."""
        if (self.fuse_offsets and fused_inference_ok(nbr_w, self.adastn.mask_conv.weight)
                and nbr_w.dtype == torch.bfloat16 and tuple(self.weight.shape) == (64, 64, 3, 3)):
            y, yb = self.adastn.raw(nbr_w, ref[0])
            if dcn_affine_eligible(feat, y, self.weight, self.deform_groups):
                return dcn_affine(feat, y, yb, self.weight, self.bias, self.deform_groups, static_weight=True,
                                  out=out)
            D = self.deform_groups
            offset, mask = affine_offsets_mask(y[:, :4 * D], y[:, 4 * D:6 * D], y[:, 6 * D:], D, yb[:4 * D],
                                               yb[4 * D:6 * D], yb[6 * D:])
        else:
            offset, mask = self.adastn(nbr_w, ref[0])
        return modulated_deform_conv2d(feat, offset, mask, self.weight, self.bias, self.stride, self.padding,
                                       self.dilation, self.groups, self.deform_groups,
                                       static_weight=not torch.is_grad_enabled())


class _ConvModule(nn.Module):
    def __init__(self, cin, cout, act):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, 7, 1, 3)
        self.activate = nn.ReLU(inplace=True) if act else None

    def forward(self, x):
        return conv2d_bias_act(self.conv, x, 0.0 if self.activate is not None else 1.0)


class _SPyNetLevel(nn.Module):
    def __init__(self):
        super().__init__()
        chans = (8, 32, 64, 32, 16, 2)
        self.basic_module = nn.Sequential(*[_ConvModule(chans[i], chans[i + 1], i < 4) for i in range(5)])

    def forward(self, x):
        return self.basic_module(x)


class SPyNet(nn.Module):
    """6-level SPyNet (reference: models/eavsrp_model.py:402-585); always evaluated in fp32."""

    def __init__(self):
        super().__init__()
        self.basic_module = nn.ModuleList([_SPyNetLevel() for _ in range(6)])
        self.fuse_level_input = True    # inference: warp + upsampled flow + concat of a level in one launch (row f4)
        self.register_buffer("mean", torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1))
        self.register_buffer("std", torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1))

    def compute_flow(self, ref, supp):
        n, _, h, w = ref.shape
        ref = [(ref - self.mean) / self.std]
        supp = [(supp - self.mean) / self.std]
        for _ in range(5):
            ref.append(F.avg_pool2d(ref[-1], 2, 2, count_include_pad=False))
            supp.append(F.avg_pool2d(supp[-1], 2, 2, count_include_pad=False))
        ref, supp = ref[::-1], supp[::-1]
        if self.fuse_level_input and fused_inference_ok(ref[0], supp[0]) and ref[0].dtype == torch.float32:
            flow = None                                   # row f4: one launch builds each level's 8-channel input
            for lvl in range(6):
                x8 = spynet_level_input(ref[lvl], supp[lvl], flow)
                flow = x8[:, 6:] + self.basic_module[lvl](x8)
            return flow
        flow = ref[0].new_zeros(n, 2, h // 32, w // 32)
        for lvl in range(6):
            up = flow if lvl == 0 else _resize_flow(flow, 2)
            warped = flow_warp_nhw2(supp[lvl], up.permute(0, 2, 3, 1), padding_mode="border")
            flow = up + self.basic_module[lvl](torch.cat([ref[lvl], warped, up], 1))
        return flow

    def forward(self, ref, supp):
        h, w = ref.shape[2:]
        hu, wu = -(-h // 32) * 32, -(-w // 32) * 32
        ref = F.interpolate(ref, size=(hu, wu), mode="bilinear", align_corners=False)
        supp = F.interpolate(supp, size=(hu, wu), mode="bilinear", align_corners=False)
        flow = F.interpolate(self.compute_flow(ref, supp), size=(h, w), mode="bilinear", align_corners=False)
        return torch.cat([flow[:, :1] * (w / wu), flow[:, 1:] * (h / hu)], 1)


_BRANCHES = ("backward_1", "forward_1", "backward_2", "forward_2")


class EAVSRP(nn.Module):
    """EAVSR+ generator, scale 4 (models/eavsrp_model.py:121-364) or 2 (models/eavsrpx2_model.py)."""

    def __init__(self, scale=4, n_feats=64, n_resblock=30, deformable_groups=8):
        super().__init__()
        assert scale in (2, 4)
        self.scale, self.n_feats = scale, n_feats
        self.spynet = SPyNet()
        for p in self.spynet.parameters():
            p.requires_grad = False
        self.encoder = _Encoder(n_feats)
        self.deform_align, self.backbone, self.fusion = nn.ModuleDict(), nn.ModuleDict(), nn.ModuleDict()
        for i, b in enumerate(_BRANCHES):
            self.deform_align[b] = MultiAdSTN(n_feats, deformable_groups)
            self.backbone[b] = _ResidualStack((2 + i) * n_feats, n_feats, n_resblock)
            self.fusion[b] = nn.Conv2d(3 * n_feats, n_feats, 1)
        self.reconstruction = _ResidualStack(5 * n_feats, n_feats, 5)
        self.upsample1 = nn.Sequential(nn.Conv2d(n_feats, 4 * n_feats, 3, 1, 1), nn.PixelShuffle(2))
        if scale == 4:
            self.upsample2 = nn.Sequential(nn.Conv2d(n_feats, 4 * n_feats, 3, 1, 1), nn.PixelShuffle(2))
        self.conv_hr = nn.Conv2d(64, 64, 3, 1, 1)
        self.conv_last = nn.Conv2d(64, 3, 3, 1, 1)
        self.compute_dtype = torch.float32

    # -- precision / layout policy ---------------------------------------------------------
    def prepare(self, dtype=torch.bfloat16):
        """channels_last everywhere; features in `dtype`; SPyNet stays fp32 (flows are coordinates)."""
        self.to(memory_format=torch.channels_last)
        for name, child in self.named_children():
            if name != "spynet":
                child.to(dtype)
        self.compute_dtype = dtype
        return self

    # -- flows -------------------------------------------------------------------------------
    def compute_flow(self, lrs):
        n, t, c, h, w = lrs.shape
        # TIME-major batches (frame pairs of all clips are contiguous): the per-frame flow `flows[i]` below is then a
        # dense (n, 2, h, w) tensor for any batch size instead of a view strided over the clips
        lt = lrs.transpose(0, 1)
        a = lt[:-1].reshape(-1, c, h, w)
        b = lt[1:].reshape(-1, c, h, w)
        m = a.shape[0]
        # both directions in one batch: [backward (a<-b); forward (b<-a)].  Flows are coordinates: SPyNet stays
        # fp32 even when the caller trains under torch.autocast
        with torch.autocast(lrs.device.type, enabled=False):
            flows = self.spynet(torch.cat([a, b]).float(), torch.cat([b, a]).float())
        return flows[m:].view(t - 1, n, 2, h, w), flows[:m].view(t - 1, n, 2, h, w)   # forward, backward: (t-1, n, 2, h, w)

    # -- one propagation branch ----------------------------------------------------------------
    def _propagate(self, feats, flows, branch):
        tm1, n, _, h, w = flows.shape
        t = tm1 + 1
        backward = branch.startswith("backward")
        order = range(t - 1, -1, -1) if backward else range(t)
        step = 1 if backward else -1                     # index offset of the previously visited frame
        align, fuse, body = self.deform_align[branch], self.fusion[branch], self.backbone[branch]
        others = [k for k in feats if k not in ("spatial", "spatial_d2", "spatial_d4", branch)]
        pyr = lambda j: [feats["spatial"][j], feats["spatial_d2"][j], feats["spatial_d4"][j]]   # noqa: E731
        prop = feats["spatial"][0].new_zeros(n, self.n_feats, h, w).contiguous(memory_format=torch.channels_last)
        outs = []
        prev_flow = None
        for i, idx in enumerate(order):
            cur = feats["spatial"][idx]
            if i > 0:
                flow1 = flows[idx if backward else idx - 1]
                # [cond1 | cur | cond2]: the aligned features are written straight into their slices of the
                # fusion convolution's input when the fused-offset DCN runs (no torch.cat pass)
                cat3 = None
                if fused_inference_ok(cur, prop) and cur.dtype == torch.bfloat16:
                    cat3 = torch.empty((n, 3 * self.n_feats, h, w), dtype=cur.dtype, device=cur.device,
                                       memory_format=torch.channels_last)
                nf = self.n_feats
                cond1 = align(pyr(idx + step), pyr(idx), prop, flow1, out=None if cat3 is None else cat3[:, :nf])
                if i > 1:
                    flow2 = flow1 + flow_warp_nhw2(prev_flow, flow1.permute(0, 2, 3, 1))
                    cond2 = align(pyr(idx + 2 * step), pyr(idx), outs[-2], flow2,
                                  out=None if cat3 is None else cat3[:, 2 * nf:])
                else:
                    cond2 = torch.zeros_like(cond1)
                if cat3 is not None:
                    if cond1.data_ptr() != cat3.data_ptr():
                        cat_channels([cond1], out=cat3, channel_offset=0)
                    cat_channels([cur], out=cat3, channel_offset=nf)
                    if cond2.data_ptr() != cat3[:, 2 * nf:].data_ptr():
                        cat_channels([cond2], out=cat3, channel_offset=2 * nf)
                    prop = conv2d_bias_act(fuse, cat3, 1.0)
                else:
                    prop = conv2d_bias_act(fuse, torch.cat([cond1, cur, cond2], 1), 1.0)
                prev_flow = flow1
            x = cat_channels([cur] + [feats[k][idx] for k in others] + [prop])
            prop = prop + body(x)
            outs.append(prop)
        feats[branch] = outs[::-1] if backward else outs
        return feats

    def _hr_features(self, feats, i):
        """HR feature map of frame i: reconstruction, the pixel-shuffle stages and conv_hr + LeakyReLU -- everything
        of the reconstruction up to conv_last."""
        x = cat_channels([feats["spatial"][i]] + [feats[b][i] for b in _BRANCHES])
        x = self.reconstruction(x)
        # LeakyReLU commutes with PixelShuffle: fold it into the conv epilogue
        x = conv2d_bias_act_shuffle(self.upsample1[0], x, 0.1)
        if self.scale == 4:
            x = conv2d_bias_act_shuffle(self.upsample2[0], x, 0.1)
        return conv3x3_64(self.conv_hr, x, 0.1) if conv3x3_64_eligible(self.conv_hr, x) else \
            conv2d_bias_act(self.conv_hr, x, 0.1)

    def _sr_frame(self, lrs, x, i):
        # the image-domain tail is fp32: residual (small) + bilinear base (the [0,1] frame itself)
        base = F.interpolate(lrs[:, i].float(), scale_factor=self.scale, mode="bilinear", align_corners=False)
        return self.conv_last(x).float() + base

    def _upsample(self, lrs, feats):
        return torch.stack([self._sr_frame(lrs, self._hr_features(feats, i), i) for i in range(lrs.shape[1])], 1)

    def forward(self, lrs):
        return self._upsample(lrs, self._trunk(lrs))

    def forward_uint8(self, frames):
        """8-bit frames in, 8-bit SR frames out: ``frames`` (n, t, h, w, 3) uint8 RGB on the GPU -> (n, t, s*h, s*w, 3)
        uint8, the reference's visuals ``clamp(sr * 255, 0, 255).round()`` (models/base_model.py:146-150) of the
        forward on ``frames / 255``.  The clip is replicate-padded to multiples of 4 (`pad_clip`) and the output
        cropped back.  With bf16 features, conv_last, the bilinear base and the quantisation run as one kernel per
        frame that writes straight into the output (`ops.sr_tail_u8`); otherwise they are composed in PyTorch and the
        result equals the visuals of `forward` bit for bit.  Inference only (runs under ``no_grad``); no host
        synchronisation, so it can be captured in a CUDA graph like `forward`."""
        if not isinstance(frames, torch.Tensor) or frames.dtype != torch.uint8:
            raise TypeError(f"EAVSRP.forward_uint8 takes a uint8 tensor, got {getattr(frames, 'dtype', type(frames))}")
        if frames.dim() != 5 or frames.shape[-1] != 3:
            raise ValueError(f"EAVSRP.forward_uint8 takes (n, t, h, w, 3) RGB frames, got {tuple(frames.shape)}")
        if not frames.is_cuda:
            raise NotImplementedError("EAVSRP.forward_uint8: CUDA tensors only (the B200 library has no CPU fallback)")
        n, t, h, w, _ = frames.shape
        assert h >= 64 and w >= 64, f"The height and width of inputs should be at least 64, but got {h} and {w}."
        s = self.scale
        with torch.no_grad():
            lrs = frames.permute(0, 1, 4, 2, 3).float().div(255).contiguous()
            out = torch.empty((n, t, s * h, s * w, 3), dtype=torch.uint8, device=frames.device)

            def fused(i, x, lr):
                sr_tail_u8(self.conv_last, x, lr, s, out[:, i], s * h, s * w)

            def composed(i, sr):
                out[:, i] = torch.clamp(sr * 255, 0, 255).round().permute(0, 2, 3, 1)
            self._sr_frames(lrs, fused, composed)
        return out

    def forward_yuv420(self, y, u, v, matrix="bt709", out=None):
        """8-bit limited-range Y'CbCr 4:2:0 frames in and out, as video decoders and encoders exchange them.

        ``y`` (n, t, h, w) and ``u``, ``v`` (n, t, h/2, w/2) are uint8 planes on the GPU with any strides (I420
        planes, or the NV12 views ``uv[..., 0::2]``, ``uv[..., 1::2]``); h and w are even and at least 64.  Returns
        ``(Y, U, V)``: (n, t, s*h, s*w) and (n, t, s*h/2, s*w/2) uint8, or writes into ``out = (Y, U, V)``, caller
        planes of those shapes with any strides (NV12 output).  ``matrix`` is "bt709" or "bt601" (`yuv.MATRICES`).

        The result is ``rgb_to_yuv420(crop(forward(pad_clip(yuv420_to_rgb(y, u, v)))))`` (`eavsr_b200.yuv`,
        centre-sited chroma).  With bf16 features conv_last, the bilinear base and the conversion run as one kernel
        per frame that writes the three planes (`ops.sr_tail_yuv420`), keeping the residual in fp32; otherwise they
        are composed in PyTorch.  Inference only (``no_grad``); no host synchronisation, so it can be captured in a
        CUDA graph."""
        planes = (y, u, v) + (tuple(out) if out is not None else ())
        for p in planes:
            if not isinstance(p, torch.Tensor) or p.dtype != torch.uint8:
                raise TypeError(f"EAVSRP.forward_yuv420 takes uint8 planes, got {getattr(p, 'dtype', type(p))}")
        if matrix not in MATRICES:
            raise ValueError(f"EAVSRP.forward_yuv420: matrix must be one of {sorted(MATRICES)}, got {matrix!r}")
        if y.dim() != 4:
            raise ValueError(f"EAVSRP.forward_yuv420 takes an (n, t, h, w) Y plane, got {tuple(y.shape)}")
        n, t, h, w = y.shape
        if h % 2 or w % 2 or h < 64 or w < 64:
            raise ValueError(f"EAVSRP.forward_yuv420 needs an even height and width of at least 64, got {h}x{w}")
        s = self.scale
        shapes = [(n, t, h, w), (n, t, h // 2, w // 2), (n, t, h // 2, w // 2)]
        if out is not None:
            if len(out) != 3:
                raise ValueError(f"EAVSRP.forward_yuv420: out must be three planes (Y, U, V), got {len(out)}")
            shapes += [(n, t, s * h, s * w), (n, t, s * h // 2, s * w // 2), (n, t, s * h // 2, s * w // 2)]
        for name, p, shape in zip(("y", "u", "v", "out Y", "out U", "out V"), planes, shapes):
            if tuple(p.shape) != shape:
                raise ValueError(f"EAVSRP.forward_yuv420: {name} must be {shape}, got {tuple(p.shape)}")
        if not all(p.is_cuda for p in planes):
            raise NotImplementedError("EAVSRP.forward_yuv420: CUDA tensors only (the B200 library has no CPU fallback)")
        kr, kb = MATRICES[matrix]
        with torch.no_grad():
            if out is None:
                out = (torch.empty((n, t, s * h, s * w), dtype=torch.uint8, device=y.device),) + tuple(
                    torch.empty((n, t, s * h // 2, s * w // 2), dtype=torch.uint8, device=y.device) for _ in range(2))
            Y, U, V = out

            def fused(i, x, lr):
                sr_tail_yuv420(self.conv_last, x, lr, s, Y[:, i], U[:, i], V[:, i], s * h, s * w, kr, kb)

            def composed(i, sr):
                Y[:, i], U[:, i], V[:, i] = rgb_to_yuv420(sr, kr, kb)
            self._sr_frames(yuv420_to_rgb(y, u, v, kr, kb), fused, composed)
        return tuple(out)

    def forward_uint16(self, frames, bits=16):
        """16-bit RGB frames in and out, for 10-, 12- or 16-bit codes: ``frames`` (n, t, h, w, 3) uint16 on the GPU,
        codes 0 .. M = 2**bits - 1 in the low bits -> (n, t, s*h, s*w, 3) uint16, ``round(clamp(sr * M, 0, M))`` of
        the forward on ``frames / M``.  As `forward_uint8` otherwise: padded to multiples of 4 and cropped back; with
        bf16 features one kernel per frame (`ops.sr_tail_u16`) keeps the residual in fp32 and writes the codes,
        otherwise PyTorch composes the tail.  Inference only (``no_grad``); no host synchronisation, so codes above M
        are not rejected (they scale past 1 as they are) and it can be captured in a CUDA graph."""
        if not isinstance(frames, torch.Tensor) or frames.dtype != torch.uint16:
            raise TypeError(f"EAVSRP.forward_uint16 takes a uint16 tensor, got {getattr(frames, 'dtype', type(frames))}")
        check_bits("EAVSRP.forward_uint16", bits, 0, allowed=(10, 12, 16))
        if frames.dim() != 5 or frames.shape[-1] != 3:
            raise ValueError(f"EAVSRP.forward_uint16 takes (n, t, h, w, 3) RGB frames, got {tuple(frames.shape)}")
        n, t, h, w, _ = frames.shape
        if h < 64 or w < 64:
            raise ValueError(f"EAVSRP.forward_uint16 needs a height and width of at least 64, got {h}x{w}")
        if not frames.is_cuda:
            raise NotImplementedError("EAVSRP.forward_uint16: CUDA tensors only (the B200 library has no CPU fallback)")
        s, m = self.scale, float(2 ** bits - 1)
        with torch.no_grad():
            lrs = frames.permute(0, 1, 4, 2, 3).float().div(m).contiguous()
            out = torch.empty((n, t, s * h, s * w, 3), dtype=torch.uint16, device=frames.device)

            def fused(i, x, lr):
                sr_tail_u16(self.conv_last, x, lr, s, out[:, i], s * h, s * w, bits)

            def composed(i, sr):
                out[:, i] = torch.clamp(sr * m, 0, m).round().permute(0, 2, 3, 1).to(torch.uint16)
            self._sr_frames(lrs, fused, composed)
        return out

    def forward_yuv420_u16(self, y, u, v, bits=10, shift=0, matrix="bt709", out=None):
        """Limited-range Y'CbCr 4:2:0 frames of 10, 12 or 16 bits in and out, as HEVC Main10 / AV1 decoders and
        encoders exchange them.

        ``y`` (n, t, h, w) and ``u``, ``v`` (n, t, h/2, w/2) are uint16 planes on the GPU with any strides; h and w
        are even and at least 64.  Each sample holds a ``bits``-bit code times ``2**shift``: ``shift=0`` is planar
        ``yuv420p10le`` (codes in the low bits), ``shift = 16 - bits`` is P010 / P012 (codes in the high bits, chroma
        interleaved: pass the views ``uv[..., 0::2]``, ``uv[..., 1::2]``).  Returns ``(Y, U, V)``: (n, t, s*h, s*w) and
        (n, t, s*h/2, s*w/2) uint16 in the same packing, or writes into ``out = (Y, U, V)``, caller planes of those
        shapes with any strides.  ``matrix`` is a key of `yuv.HBD_MATRICES` ("bt709", "bt601", "bt2020").

        The result is ``rgb_to_yuv420(crop(forward(pad_clip(yuv420_to_rgb(y, u, v, bits=bits, shift=shift)))),
        bits=bits, shift=shift)`` (`eavsr_b200.yuv`).  With bf16 features conv_last, the bilinear base and the
        conversion run as one kernel per frame (`ops.sr_tail_yuv420_u16`), keeping the residual in fp32; otherwise
        they are composed in PyTorch.  Inference only (``no_grad``); no host synchronisation, so the code range is not
        checked (out-of-range codes are converted as they are) and it can be captured in a CUDA graph."""
        planes = (y, u, v) + (tuple(out) if out is not None else ())
        for p in planes:
            if not isinstance(p, torch.Tensor) or p.dtype != torch.uint16:
                raise TypeError(f"EAVSRP.forward_yuv420_u16 takes uint16 planes, got {getattr(p, 'dtype', type(p))}")
        check_bits("EAVSRP.forward_yuv420_u16", bits, shift, allowed=(10, 12, 16))
        if matrix not in HBD_MATRICES:
            raise ValueError(f"EAVSRP.forward_yuv420_u16: matrix must be one of {sorted(HBD_MATRICES)}, got {matrix!r}")
        if y.dim() != 4:
            raise ValueError(f"EAVSRP.forward_yuv420_u16 takes an (n, t, h, w) Y plane, got {tuple(y.shape)}")
        n, t, h, w = y.shape
        if h % 2 or w % 2 or h < 64 or w < 64:
            raise ValueError(f"EAVSRP.forward_yuv420_u16 needs an even height and width of at least 64, got {h}x{w}")
        s = self.scale
        shapes = [(n, t, h, w), (n, t, h // 2, w // 2), (n, t, h // 2, w // 2)]
        if out is not None:
            if len(out) != 3:
                raise ValueError(f"EAVSRP.forward_yuv420_u16: out must be three planes (Y, U, V), got {len(out)}")
            shapes += [(n, t, s * h, s * w), (n, t, s * h // 2, s * w // 2), (n, t, s * h // 2, s * w // 2)]
        for name, p, shape in zip(("y", "u", "v", "out Y", "out U", "out V"), planes, shapes):
            if tuple(p.shape) != shape:
                raise ValueError(f"EAVSRP.forward_yuv420_u16: {name} must be {shape}, got {tuple(p.shape)}")
        if not all(p.is_cuda for p in planes):
            raise NotImplementedError("EAVSRP.forward_yuv420_u16: CUDA tensors only (the B200 library has no CPU "
                                      "fallback)")
        kr, kb = HBD_MATRICES[matrix]
        with torch.no_grad():
            if out is None:
                out = (torch.empty((n, t, s * h, s * w), dtype=torch.uint16, device=y.device),) + tuple(
                    torch.empty((n, t, s * h // 2, s * w // 2), dtype=torch.uint16, device=y.device) for _ in range(2))
            Y, U, V = out

            def fused(i, x, lr):
                sr_tail_yuv420_u16(self.conv_last, x, lr, s, Y[:, i], U[:, i], V[:, i], s * h, s * w, kr, kb, bits,
                                   shift)

            def composed(i, sr):
                Y[:, i], U[:, i], V[:, i] = rgb_to_yuv420(sr, kr, kb, bits, shift)
            self._sr_frames(yuv420_to_rgb(y, u, v, kr, kb, bits, shift), fused, composed)
        return tuple(out)

    def psnr_uint8(self, frames, hr, out=None):
        """Per-frame PSNR of the 8-bit SR frames against ground-truth frames, the evaluation of the reference's
        test_basic.py (``calc_psnr`` of util/util.py on the visuals), without materialising the SR clip.

        ``frames`` (n, t, h, w, 3) and ``hr`` (n, t, s*h, s*w, 3) are uint8 RGB on the GPU, ``hr`` with any strides.
        Returns ``(psnr, sse)``, both (n, t) on the device: ``sse`` (int64) is the sum over pixels and channels of
        ``(q - hr)**2``, exact, where ``q`` is the frame `forward_uint8` returns, and ``psnr`` (float64) is
        ``10 * log10(255**2 * 3 * s*h * s*w / sse)`` (`psnr_from_sse`), ``+inf`` where ``sse == 0``.  A per-clip PSNR
        is then either the mean of ``psnr`` or `psnr_from_sse` of ``sse.sum(1)``, as the evaluation protocol asks.
        With ``out``, a caller clip of `forward_uint8`'s shape with any strides, the frames are written there too.

        With bf16 features, conv_last, the bilinear base, the quantisation and the squared-error sum run as one kernel
        per frame (`ops.sr_tail_u8_sse`), which reads each ground-truth byte once and writes nothing else unless
        ``out`` is given; otherwise the tail is composed in PyTorch as in `forward_uint8`, and ``sse`` equals the int64
        error of the visuals of `forward` exactly.  Inference only (``no_grad``); no host synchronisation, so it can be
        captured in a CUDA graph."""
        named = (("frames", frames), ("hr", hr)) + ((("out", out),) if out is not None else ())
        for name, p in named:
            if not isinstance(p, torch.Tensor) or p.dtype != torch.uint8:
                raise TypeError(f"EAVSRP.psnr_uint8: {name} must be a uint8 tensor, got "
                                f"{getattr(p, 'dtype', type(p))}")
        if frames.dim() != 5 or frames.shape[-1] != 3:
            raise ValueError(f"EAVSRP.psnr_uint8 takes (n, t, h, w, 3) RGB frames, got {tuple(frames.shape)}")
        n, t, h, w, _ = frames.shape
        if h < 64 or w < 64:
            raise ValueError(f"EAVSRP.psnr_uint8 needs a height and width of at least 64, got {h}x{w}")
        s = self.scale
        for name, p in named[1:]:
            if tuple(p.shape) != (n, t, s * h, s * w, 3):
                raise ValueError(f"EAVSRP.psnr_uint8: {name} must be {(n, t, s * h, s * w, 3)}, got {tuple(p.shape)}")
        if not all(p.is_cuda for _, p in named):
            raise NotImplementedError("EAVSRP.psnr_uint8: CUDA tensors only (the B200 library has no CPU fallback)")
        with torch.no_grad():
            lrs = frames.permute(0, 1, 4, 2, 3).float().div(255).contiguous()
            sse = torch.zeros((n, t), dtype=torch.int64, device=frames.device)

            def fused(i, x, lr):
                sr_tail_u8_sse(self.conv_last, x, lr, s, hr[:, i], sse[:, i], s * h, s * w,
                               None if out is None else out[:, i])

            def composed(i, sr):
                q = torch.clamp(sr * 255, 0, 255).round().permute(0, 2, 3, 1).to(torch.uint8)
                if out is not None:
                    out[:, i] = q
                d = q.int() - hr[:, i].int()
                sse[:, i] = (d * d).sum((1, 2, 3), dtype=torch.int64)
            self._sr_frames(lrs, fused, composed)
            return psnr_from_sse(sse, 3 * s * h * s * w), sse

    def _sr_frames(self, lrs, fused, composed):
        """The frame-in, frame-out forwards' common part, under ``no_grad``: pad the (n, t, 3, h, w) clip `lrs` (`pad_clip`), run
        `_trunk`, then per frame i `_hr_features` and the tail -- ``fused(i, x, lr_i)`` when the fused tail kernel can
        run on the HR features ``x`` (`ops.sr_tail_u8_eligible`), else ``composed(i, sr_i)`` with the SR frame of
        `_sr_frame` cropped to (s*h, s*w)."""
        h, w = lrs.shape[-2:]
        s = self.scale
        lrs = pad_clip(lrs)
        feats = self._trunk(lrs)
        for i in range(lrs.shape[1]):
            x = self._hr_features(feats, i)
            if sr_tail_u8_eligible(self.conv_last, x):
                fused(i, x, lrs[:, i])
            else:
                composed(i, self._sr_frame(lrs, x, i)[..., :s * h, :s * w])

    def _trunk(self, lrs):
        """Flows, encoder and the four propagation branches of a padded clip: the features `_hr_features` reads."""
        n, t, c, h, w = lrs.shape
        assert h >= 64 and w >= 64, f"The height and width of inputs should be at least 64, but got {h} and {w}."
        if h % 4 or w % 4:
            raise ValueError(f"EAVSRP needs H and W divisible by 4 (3-level pyramid), got {h}x{w}; "
                             "replicate-pad the clip (see eavsr_b200.model.pad_clip)")
        with torch.no_grad():
            flows_fwd, flows_bwd = self.compute_flow(lrs)
        # the encoder runs on a TIME-major batch, so that frame i of all n clips is one dense channels_last tensor:
        # with the clip-major order of the reference (`lrs.view(-1, c, h, w)`, models/eavsrp_model.py:213-215) the
        # per-frame features of a batch of clips are views strided over the clips, which every native operator
        # (and cuDNN) first copies into a dense buffer -- 6 % of the device time at 8 clips per batch
        x = lrs.transpose(0, 1).reshape(-1, c, h, w).to(self.compute_dtype).contiguous(memory_format=torch.channels_last)
        f1 = self.encoder(x)
        f2 = F.interpolate(f1, scale_factor=0.5, mode="bilinear", align_corners=False)
        f4 = F.interpolate(f1, scale_factor=0.25, mode="bilinear", align_corners=False)
        split = lambda f: list(f.view(t, n, *f.shape[1:]).unbind(0))      # noqa: E731
        feats = {"spatial": split(f1), "spatial_d2": split(f2), "spatial_d4": split(f4)}
        for b in _BRANCHES:
            feats = self._propagate(feats, flows_bwd if b.startswith("backward") else flows_fwd, b)
        return feats


def pad_clip(lrs, multiple=4):
    """Replicate-pad (n,t,c,h,w) so that h, w are multiples of `multiple` (270 -> 272; SURVEY.md F4)."""
    h, w = lrs.shape[-2:]
    ph, pw = (-h) % multiple, (-w) % multiple
    if ph == 0 and pw == 0:
        return lrs
    n, t, c = lrs.shape[:3]
    out = F.pad(lrs.reshape(n * t, c, h, w), (0, pw, 0, ph), mode="replicate")
    return out.view(n, t, c, h + ph, w + pw)


def psnr_from_sse(sse, samples):
    """PSNR of 8-bit frames from their integer squared-error sums over ``samples`` values each (pixels times
    channels): ``10 * log10(255**2 * samples / sse)`` in float64, as ``calc_psnr`` of the reference's util/util.py on
    the visuals; ``+inf`` where ``sse == 0``."""
    return 10 * torch.log10((255.0 ** 2 * samples) / sse.double())
