"""Host-side mirror of the reference's module surface (pytorch/bts.py) over the B200 kernels.

Same class names, constructor arguments, forward signatures, 5-tuple output and -- the checkpoint wire
format -- the same state_dict keys and shapes (SURVEY.md Appendix C), so the reference's bts_main.py /
bts_test.py import this as `bts` unchanged.  The arithmetic underneath is ours:
  * plane heads + LPG + /max_depth + nearest down-sample: one fused sm_100a kernel each way (ops.plane_head_lpg)
  * silog loss: two streaming kernels (ops.silog)
  * convolutions: the tcgen05 implicit-GEMM engine (bts_b200.conv) where enabled, cuDNN otherwise (scaffold)
Reference lines are cited per class.
"""
import math
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops


def bn_init_as_tf(m):
    """reference pytorch/bts.py:26-31 -- BN layers behave like TF {'is_training': False, 'scale': True}."""
    if isinstance(m, nn.BatchNorm2d):
        m.track_running_stats = True
        m.eval()
        m.affine = True
        m.requires_grad = True


def weights_init_xavier(m):
    """reference pytorch/bts.py:34-38 -- called as model.decoder.apply(weights_init_xavier) by bts_main.py:338."""
    if isinstance(m, nn.Conv2d):
        nn.init.xavier_uniform_(m.weight)
        if m.bias is not None:
            nn.init.zeros_(m.bias)


class silog_loss(nn.Module):
    """reference pytorch/bts.py:41-48."""

    def __init__(self, variance_focus):
        super().__init__()
        self.variance_focus = variance_focus

    def forward(self, depth_est, depth_gt, mask):
        return ops.silog(depth_est, depth_gt, mask, self.variance_focus)


def _require_cuda_fp32(x, what):
    """the product path has no CPU / eager / library fallback (north_star): fail loudly instead of silently diverging"""
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 4):
        raise RuntimeError("bts_b200.%s runs on CUDA fp32 NCHW/NHWC tensors only (got device=%s dtype=%s dim=%d); there is "
                           "no CPU or library fallback" % (what, x.device, x.dtype, x.dim()))


class Conv2dTC(nn.Conv2d):
    """nn.Conv2d whose forward/dgrad run on the tcgen05 engine.  It stays an nn.Conv2d subclass so that
    weights_init_xavier (bts_main.py:338), state_dict keys and optimizer groups behave exactly as in the reference."""

    def forward(self, x):
        if (x.is_cuda and x.dtype == torch.float32
                and self.bias is None and self.stride[0] == self.stride[1] and self.padding[0] == self.padding[1]
                and self.dilation[0] == self.dilation[1] and self.kernel_size[0] == self.kernel_size[1]
                and isinstance(self.padding, tuple) and self.padding_mode == "zeros" and self.stride[0] in (1, 2)):
            from . import conv
            if self.groups == 1:
                if conv.c1_eligible(self.weight, self.stride[0], self.padding[0], self.dilation[0]):
                    return conv.conv_c1(x, self.weight, sigmoid=False)
                return conv.conv2d(x, self.weight, self.stride[0], self.padding[0], self.dilation[0])
            cpg = self.in_channels // self.groups
            from . import glue
            if glue.dw_eligible(self):
                # depthwise 3x3 (MobileNetV2): CUDA-core streaming kernels, fwd / dgrad / wgrad
                return glue.dwconv(x, self.weight, self.stride[0])
            if (self.in_channels == self.out_channels and cpg >= 4 and conv.group_window(self.out_channels, cpg) == 128):
                # ResNeXt grouped 3x3 (32 groups): block-diagonal operator on the engine, fwd / dgrad / wgrad
                return conv.conv2d(x, self.weight, self.stride[0], self.padding[0], self.dilation[0], groups=self.groups)
        # shapes the engine does not cover (bias / asymmetric geometry): the library conv, pinned to true fp32 for parity
        with torch.backends.cudnn.flags(enabled=True, benchmark=torch.backends.cudnn.benchmark, allow_tf32=False):
            return super().forward(x)

    def forward_sigmoid(self, x):
        """conv + Sigmoid in one kernel when this is a single-output-channel head (get_depth, reduc1x1.final)."""
        if x.is_cuda and x.dtype == torch.float32:
            from . import conv
            if conv.c1_eligible(self.weight, self.stride[0], self.padding[0], self.dilation[0]):
                return conv.conv_c1(x, self.weight, sigmoid=True)
        return torch.sigmoid(self.forward(x))


def fuse_enabled(x):
    """the fused glue path (bts_b200/glue.py) is taken for fp32 CUDA tensors when the tensor-core backend is active"""
    from . import glue
    return glue.eligible(x)


class BatchNormTC(nn.BatchNorm2d):
    """nn.BatchNorm2d (same parameters / buffers / state_dict) whose forward + backward run on our streaming kernels;
    `_fuse_relu` folds the ReLU module that follows it in torchvision's `features` (norm0 -> relu0)."""
    _fuse_relu = False

    def forward(self, x):
        if fuse_enabled(x) and self.affine:
            from . import glue
            return glue.bn_act(x, self, relu=self._fuse_relu)
        y = super().forward(x)                     # non-affine / non-fp32 BatchNorm: not on the BTS path
        return F.relu(y) if self._fuse_relu else y


class ReluFolded(nn.Identity):
    """stands where torchvision's `relu0` was: the ReLU already ran inside the preceding BatchNormTC"""


class MaxPoolTC(nn.MaxPool2d):
    """the encoder stems' 3x3 / stride 2 / pad 1 max-pool (densenet `pool0`, resnet `maxpool`) on our NHWC kernels"""

    def forward(self, x):
        k = self.kernel_size if isinstance(self.kernel_size, int) else self.kernel_size[0]
        st = self.stride if isinstance(self.stride, int) else self.stride[0]
        pd = self.padding if isinstance(self.padding, int) else self.padding[0]
        if fuse_enabled(x) and (k, st, pd) == (3, 2, 1) and self.dilation in (1, (1, 1)) and not self.ceil_mode \
                and not self.return_indices:
            from . import glue
            return glue.maxpool3s2(x)
        return super().forward(x)


def _bottleneck_class():
    from torchvision.models.resnet import Bottleneck

    class BottleneckTC(Bottleneck):
        """torchvision ResNet / ResNeXt bottleneck [1x1 -> BN -> ReLU -> (grouped) 3x3 -> BN -> ReLU -> 1x1 -> BN -> +id ->
        ReLU]: every conv on the tcgen05 engine (the grouped 3x3 as a block-diagonal operator), BN(+ReLU) and the
        BN + residual + ReLU tail on our streaming kernels; parameters / buffers / state_dict untouched."""

        def forward(self, x):
            if not fuse_enabled(x):
                return super().forward(x)
            from . import glue
            out = glue.bn_act(self.conv1(x), self.bn1, relu=True)
            out = glue.bn_act(self.conv2(out), self.bn2, relu=True)
            out = self.conv3(out)
            identity = x if self.downsample is None else self.downsample(x)
            return glue.bn_add_relu(out, identity, self.bn3)

    return Bottleneck, BottleneckTC


def _transition_class():
    from torchvision.models.densenet import _Transition

    class TransitionTC(_Transition):
        """torchvision DenseNet transition [BN -> ReLU -> 1x1 conv -> 2x2 avg-pool]: BN + ReLU folded into the conv's
        A-operand prologue, pooling on our streaming kernel"""

        def forward(self, x):
            if fuse_enabled(x) and self.norm.affine and self.conv.bias is None:
                from . import glue
                return glue.avgpool2(glue.bn_relu_conv(x, self.norm, self.conv.weight))
            return super().forward(x)

    return _Transition, TransitionTC


def _dense_block_class():
    from torchvision.models.densenet import _DenseBlock

    class DenseBlockTC(_DenseBlock):
        """torchvision dense block whose forward/backward run as ONE fused, concat-free autograd Function
        (bts_b200/fused.py) when the tensor-core backend is active; identical parameters / buffers / state_dict."""

        def forward(self, init_features):
            from . import fused
            if fused.dense_block_eligible(self, init_features):
                return fused.dense_block_forward(self, init_features)
            return super().forward(init_features)

    return _DenseBlock, DenseBlockTC


def _mobilenet_classes():
    from torchvision.models.mobilenetv2 import InvertedResidual
    from torchvision.ops.misc import Conv2dNormActivation

    def conv_bn_relu6(seq):
        """(conv, bn) of a Conv2dNormActivation [Conv2d(no bias), affine BatchNorm2d, ReLU6], else None"""
        if len(seq) == 3 and isinstance(seq[0], nn.Conv2d) and seq[0].bias is None and type(seq[1]) is nn.BatchNorm2d \
                and seq[1].affine and isinstance(seq[2], nn.ReLU6):
            return seq[0], seq[1]
        return None

    class ConvBnReLU6TC(Conv2dNormActivation):
        """torchvision Conv2dNormActivation [conv -> BN -> ReLU6] (the MobileNetV2 stem and last 1x1 layer): the conv on the
        engine (or the depthwise kernels), BN + ReLU6 on our streaming kernels; parameters / buffers / state_dict untouched"""

        def forward(self, x):
            parts = conv_bn_relu6(self)
            if not (fuse_enabled(x) and parts):
                return super().forward(x)
            from . import glue
            return glue.bn_act(parts[0](x), parts[1], act="relu6")

    class InvertedResidualTC(InvertedResidual):
        """torchvision MobileNetV2 block [(1x1 -> BN -> ReLU6) -> dw 3x3 -> BN -> ReLU6 -> 1x1 -> BN (+ x)] as one fused
        autograd unit (glue.inverted_residual); parameters / buffers / state_dict untouched"""

        def _parts(self):
            layers = list(self.conv)
            if len(layers) not in (3, 4):
                return None
            expand = conv_bn_relu6(layers[0]) if len(layers) == 4 else (None, None)
            dw = conv_bn_relu6(layers[-3])
            project, bn3 = layers[-2], layers[-1]
            if expand is None or dw is None or not (isinstance(project, nn.Conv2d) and project.bias is None
                                                   and tuple(project.kernel_size) == (1, 1) and project.stride == (1, 1)
                                                   and type(bn3) is nn.BatchNorm2d and bn3.affine):
                return None
            if expand[0] is not None and (tuple(expand[0].kernel_size) != (1, 1) or expand[0].stride != (1, 1)
                                          or expand[0].groups != 1):
                return None
            return expand[0], expand[1], dw[0], dw[1], project, bn3

        def forward(self, x):
            from . import glue
            parts = self._parts()
            if not (fuse_enabled(x) and parts and glue.dw_eligible(parts[2])):
                return super().forward(x)
            return glue.inverted_residual(x, *parts, residual=self.use_res_connect)

    return InvertedResidual, InvertedResidualTC, Conv2dNormActivation, ConvBnReLU6TC


def adopt_convs(module):
    """Re-class every eligible nn.Conv2d (-> Conv2dTC), DenseNet block (-> fused DenseBlockTC), ResNet bottleneck and
    MobileNetV2 block / conv-BN-ReLU6 layer of a torchvision module tree in place -- parameter names, shapes and init are
    untouched."""
    base, fusedcls = _dense_block_class()
    tbase, tcls = _transition_class()
    bbase, bcls = _bottleneck_class()
    ibase, icls, cbase, ccls = _mobilenet_classes()
    resnet = any(type(m) is bbase for m in module.modules())
    for m in module.modules():
        if type(m) is nn.Conv2d:
            m.__class__ = Conv2dTC
        elif type(m) is ibase:
            m.__class__ = icls
        elif type(m) is cbase:
            m.__class__ = ccls
        elif type(m) is base:
            m.__class__ = fusedcls
        elif type(m) is tbase:
            m.__class__ = tcls
        elif type(m) is bbase:
            m.__class__ = bcls
        elif type(m) is nn.MaxPool2d:
            m.__class__ = MaxPoolTC
        elif resnet and type(m) is nn.BatchNorm2d:
            m.__class__ = BatchNormTC          # stem bn1, bottleneck BNs (when not fused), downsample BNs
    # ResNet stem: bn1 (+ relu folded: the module named `relu` -- the H/2 skip tap -- then passes the activated tensor on)
    if resnet and hasattr(module, "bn1") and isinstance(getattr(module, "relu", None), nn.ReLU):
        module.bn1._fuse_relu = True
        module.relu = ReluFolded()
    # DenseNet `features`: norm0 (+ relu0 folded) and norm5 on the streaming BatchNorm kernels
    if isinstance(module, nn.Sequential) and hasattr(module, "norm0") and type(module.norm0) is nn.BatchNorm2d:
        module.norm0.__class__ = BatchNormTC
        if isinstance(getattr(module, "relu0", None), nn.ReLU):
            module.norm0._fuse_relu = True
            module.relu0 = ReluFolded()
    if isinstance(module, nn.Sequential) and hasattr(module, "norm5") and type(module.norm5) is nn.BatchNorm2d:
        module.norm5.__class__ = BatchNormTC
    return module


def _conv(cin, cout, k, dilation=1):
    pad = dilation * (k // 2)
    return Conv2dTC(cin, cout, k, 1, pad, dilation=dilation, bias=False)


class atrous_conv(nn.Sequential):
    """reference pytorch/bts.py:51-66: [BN(eps 1.1e-5)] ReLU 1x1(C->2*out) BN ReLU 3x3 dilated (2*out->out)."""

    def __init__(self, in_channels, out_channels, dilation, apply_bn_first=True):
        super().__init__()
        body = nn.Sequential()
        if apply_bn_first:
            body.add_module("first_bn", nn.BatchNorm2d(in_channels, momentum=0.01, affine=True,
                                                       track_running_stats=True, eps=1.1e-5))
        body.add_module("aconv_sequence", nn.Sequential(
            nn.ReLU(),
            _conv(in_channels, out_channels * 2, 1),
            nn.BatchNorm2d(out_channels * 2, momentum=0.01, affine=True, track_running_stats=True),
            nn.ReLU(),
            _conv(out_channels * 2, out_channels, 3, dilation)))
        self.atrous_conv = body

    def forward(self, x):
        _require_cuda_fp32(x, "atrous_conv")
        from . import glue
        seq = self.atrous_conv.aconv_sequence
        if hasattr(self.atrous_conv, "first_bn"):
            b = glue.bn_relu_conv(x, self.atrous_conv.first_bn, seq[1].weight)
        else:
            b = glue.conv_act(x, seq[1].weight, pre_relu=True)
        return glue.bn_relu_conv(b, seq[2], seq[4].weight, seq[4].padding[0], seq[4].dilation[0])


class upconv(nn.Module):
    """reference pytorch/bts.py:69-80: nearest x ratio -> 3x3 conv -> ELU."""

    def __init__(self, in_channels, out_channels, ratio=2):
        super().__init__()
        self.elu = nn.ELU()
        self.conv = _conv(in_channels, out_channels, 3)
        self.ratio = ratio

    def forward(self, x, pre_relu=False):
        _require_cuda_fp32(x, "upconv")
        from . import glue
        if self.ratio == 2:                      # up-sample folded into the im2col map, ELU in the epilogue
            return glue.conv_act(x, self.conv.weight, 1, 1, pre_relu=pre_relu, up=True, act="elu")
        # other ratios never occur in BTS (bts.py:153-189 always uses 2): materialise the up-sample, conv + ELU on the engine
        if pre_relu:
            x = F.relu(x)
        x = F.interpolate(x, scale_factor=self.ratio, mode="nearest").contiguous(memory_format=torch.channels_last)
        return glue.conv_act(x, self.conv.weight, 1, 1, act="elu")


class reduction_1x1(nn.Sequential):
    """reference pytorch/bts.py:83-122.  `trunk()` runs the 1x1+ELU chain and the last 1x1 conv; the decoder
    feeds its 3-channel result to the fused head+LPG kernel.  `forward()` keeps the reference's public
    behaviour (4-vector (n1,n2,n3,n4) for plane heads, sigmoid map for the final head)."""

    def __init__(self, num_in_filters, num_out_filters, max_depth, is_final=False):
        super().__init__()
        self.max_depth = max_depth
        self.is_final = is_final
        self.sigmoid = nn.Sigmoid()
        self.reduc = nn.Sequential()
        cin, cout = num_in_filters, num_out_filters
        while cout >= 4:
            if cout < 8:
                if is_final:
                    self.reduc.add_module("final", nn.Sequential(_conv(cin, 1, 1), nn.Sigmoid()))
                else:
                    self.reduc.add_module("plane_params", _conv(cin, 3, 1))
                break
            self.reduc.add_module("inter_{}_{}".format(cin, cout), nn.Sequential(_conv(cin, cout, 1), nn.ELU()))
            cin, cout = cout, cout // 2

    def trunk(self, net):
        _require_cuda_fp32(net, "reduction_1x1")
        from . import glue
        for name, m in self.reduc.named_children():
            if name == "final":                 # Sequential(1x1 conv 8->1, Sigmoid): fused single-channel head kernel
                net = m[0].forward_sigmoid(net)
            elif name == "plane_params":
                net = m(net)
            else:                               # Sequential(1x1 conv, ELU): ELU in the conv epilogue
                net = glue.conv_act(net, m[0].weight, 0, 1, act="elu")
        return net

    def forward(self, net):
        net = self.trunk(net)
        if self.is_final:
            return net
        theta = torch.sigmoid(net[:, 0]) * math.pi / 3
        phi = torch.sigmoid(net[:, 1]) * math.pi * 2
        dist = torch.sigmoid(net[:, 2]) * self.max_depth
        st = torch.sin(theta)
        return torch.stack([st * torch.cos(phi), st * torch.sin(phi), torch.cos(theta), dist], dim=1)


class local_planar_guidance(nn.Module):
    """reference pytorch/bts.py:124-146.  `focal` is accepted and ignored, as in the reference (Q1)."""

    def __init__(self, upratio):
        super().__init__()
        self.upratio = float(upratio)
        k = torch.arange(int(upratio)).float()
        self.u = k.reshape(1, 1, -1)
        self.v = k.reshape(1, -1, 1)

    def forward(self, plane_eq, focal=None):
        return ops.lpg(plane_eq, int(self.upratio))


class bts(nn.Module):
    """The decoder, reference pytorch/bts.py:148-266."""

    def __init__(self, params, feat_out_channels, num_features=512):
        super().__init__()
        self.params = params
        f, nf = feat_out_channels, num_features
        self.upconv5 = upconv(f[4], nf)
        self.bn5 = nn.BatchNorm2d(nf, momentum=0.01, affine=True, eps=1.1e-5)
        self.conv5 = nn.Sequential(_conv(nf + f[3], nf, 3), nn.ELU())
        self.upconv4 = upconv(nf, nf // 2)
        self.bn4 = nn.BatchNorm2d(nf // 2, momentum=0.01, affine=True, eps=1.1e-5)
        self.conv4 = nn.Sequential(_conv(nf // 2 + f[2], nf // 2, 3), nn.ELU())
        self.bn4_2 = nn.BatchNorm2d(nf // 2, momentum=0.01, affine=True, eps=1.1e-5)
        self.daspp_3 = atrous_conv(nf // 2, nf // 4, 3, apply_bn_first=False)
        self.daspp_6 = atrous_conv(nf // 2 + nf // 4 + f[2], nf // 4, 6)
        self.daspp_12 = atrous_conv(nf + f[2], nf // 4, 12)
        self.daspp_18 = atrous_conv(nf + nf // 4 + f[2], nf // 4, 18)
        self.daspp_24 = atrous_conv(nf + nf // 2 + f[2], nf // 4, 24)
        self.daspp_conv = nn.Sequential(_conv(nf + nf // 2 + nf // 4, nf // 4, 3), nn.ELU())
        self.reduc8x8 = reduction_1x1(nf // 4, nf // 4, params.max_depth)
        self.lpg8x8 = local_planar_guidance(8)
        self.upconv3 = upconv(nf // 4, nf // 4)
        self.bn3 = nn.BatchNorm2d(nf // 4, momentum=0.01, affine=True, eps=1.1e-5)
        self.conv3 = nn.Sequential(_conv(nf // 4 + f[1] + 1, nf // 4, 3), nn.ELU())
        self.reduc4x4 = reduction_1x1(nf // 4, nf // 8, params.max_depth)
        self.lpg4x4 = local_planar_guidance(4)
        self.upconv2 = upconv(nf // 4, nf // 8)
        self.bn2 = nn.BatchNorm2d(nf // 8, momentum=0.01, affine=True, eps=1.1e-5)
        self.conv2 = nn.Sequential(_conv(nf // 8 + f[0] + 1, nf // 8, 3), nn.ELU())
        self.reduc2x2 = reduction_1x1(nf // 8, nf // 16, params.max_depth)
        self.lpg2x2 = local_planar_guidance(2)
        self.upconv1 = upconv(nf // 8, nf // 16)
        self.reduc1x1 = reduction_1x1(nf // 16, nf // 32, params.max_depth, is_final=True)
        self.conv1 = nn.Sequential(_conv(nf // 16 + 4, nf // 16, 3), nn.ELU())
        self.get_depth = nn.Sequential(_conv(nf // 16, 1, 3), nn.Sigmoid())

    def forward(self, features, focal):
        _require_cuda_fp32(features[4], "bts.forward")
        return self._forward_fused(features, focal)

    def _forward_fused(self, features, focal):
        """bts.forward (reference pytorch/bts.py:196-266) over the fused units of bts_b200/glue.py: no ATen BatchNorm /
        ReLU / ELU / interpolate / cat kernels; every conv (fwd, dgrad, wgrad) on the tcgen05 engine."""
        from . import glue as G
        skip0, skip1, skip2, skip3 = features[0], features[1], features[2], features[3]
        md = self.params.max_depth
        c3 = lambda seq: seq[0].weight          # Sequential(3x3 conv, ELU)
        x = G.bn_act(self.upconv5(features[4], pre_relu=True), self.bn5)                  # H/16
        x = G.conv_act(G.cat_nhwc([x, skip3]), c3(self.conv5), 1, 1, act="elu")
        cat4 = G.cat_nhwc([G.bn_act(self.upconv4(x), self.bn4), skip2])                   # H/8
        iconv4 = G.bn_act(G.conv_act(cat4, c3(self.conv4), 1, 1, act="elu"), self.bn4_2)
        d3 = self.daspp_3(iconv4)
        d6 = self.daspp_6(G.cat_nhwc([cat4, d3]))
        d12 = self.daspp_12(G.cat_nhwc([cat4, d3, d6]))
        d18 = self.daspp_18(G.cat_nhwc([cat4, d3, d6, d12]))
        d24 = self.daspp_24(G.cat_nhwc([cat4, d3, d6, d12, d18]))
        feat8 = G.conv_act(G.cat_nhwc([iconv4, d3, d6, d12, d18, d24]), c3(self.daspp_conv), 1, 1, act="elu")

        depth_8x8_scaled, d8_ds = ops.plane_head_lpg(self.reduc8x8.trunk(feat8), 8, md, ds_stride=4)
        x = G.bn_act(self.upconv3(feat8), self.bn3)                                       # H/4
        iconv3 = G.conv_act(G.cat_nhwc([x, skip1, d8_ds]), c3(self.conv3), 1, 1, act="elu")
        depth_4x4_scaled, d4_ds = ops.plane_head_lpg(self.reduc4x4.trunk(iconv3), 4, md, ds_stride=2)
        x = G.bn_act(self.upconv2(iconv3), self.bn2)                                      # H/2
        iconv2 = G.conv_act(G.cat_nhwc([x, skip0, d4_ds]), c3(self.conv2), 1, 1, act="elu")
        depth_2x2_scaled = ops.plane_head_lpg(self.reduc2x2.trunk(iconv2), 2, md)
        up1 = self.upconv1(iconv2)                                                        # H
        reduc1x1 = self.reduc1x1(up1)
        iconv1 = G.conv_act(G.cat_nhwc([up1, reduc1x1, depth_2x2_scaled, depth_4x4_scaled, depth_8x8_scaled]),
                            c3(self.conv1), 1, 1, act="elu")
        final_depth = md * self.get_depth[0].forward_sigmoid(iconv1)      # Sequential(3x3 conv 32->1, Sigmoid), fused
        if self.params.dataset == "kitti":
            final_depth = final_depth * focal.view(-1, 1, 1, 1).float() / 715.0873
        return depth_8x8_scaled, depth_4x4_scaled, depth_2x2_scaled, reduc1x1, final_depth


_ENCODERS = {
    # params.encoder: (torchvision ctor, use .features, skip tap names, skip channels)   reference bts.py:273-300
    "densenet121_bts": ("densenet121", True, ["relu0", "pool0", "transition1", "transition2", "norm5"], [64, 64, 128, 256, 1024]),
    "densenet161_bts": ("densenet161", True, ["relu0", "pool0", "transition1", "transition2", "norm5"], [96, 96, 192, 384, 2208]),
    "resnet50_bts": ("resnet50", False, ["relu", "layer1", "layer2", "layer3", "layer4"], [64, 256, 512, 1024, 2048]),
    "resnet101_bts": ("resnet101", False, ["relu", "layer1", "layer2", "layer3", "layer4"], [64, 256, 512, 1024, 2048]),
    "resnext50_bts": ("resnext50_32x4d", False, ["relu", "layer1", "layer2", "layer3", "layer4"], [64, 256, 512, 1024, 2048]),
    "resnext101_bts": ("resnext101_32x8d", False, ["relu", "layer1", "layer2", "layer3", "layer4"], [64, 256, 512, 1024, 2048]),
    "mobilenetv2_bts": ("mobilenet_v2", True, [], [16, 24, 32, 64, 1280]),
}


def _load_backbone(ctor, pretrained):
    """The reference builds the backbone with `pretrained=True` (bts.py:274-298), which torchvision maps to the
    IMAGENET1K_V1 weights and downloads into the torch-hub cache when they are not there yet.  Same here by default
    (params.pretrained absent / None / True).  Random init is OPT-IN: params.pretrained=False (bench.py, the tests) or
    BTS_B200_PRETRAINED=0.  If the weights can be neither found nor downloaded (offline box) the encoder falls back to
    random init with a loud warning -- or raises when params.pretrained is True."""
    import warnings
    import torchvision.models as tvm
    fn = getattr(tvm, ctor)
    if pretrained is False or (pretrained is None and os.environ.get("BTS_B200_PRETRAINED", "1") == "0"):
        return fn(weights=None)
    try:
        return fn(weights=tvm.get_model_weights(ctor).IMAGENET1K_V1)
    except Exception as e:
        if pretrained is True:
            raise
        msg = ("bts_b200: ImageNet (IMAGENET1K_V1) weights for %s could not be loaded or downloaded (%s: %s) -- the "
               "encoder is RANDOMLY INITIALISED, unlike the reference (pytorch/bts.py:274-298). Put the checkpoint into "
               "%s or pass params.pretrained=False to silence this." %
               (ctor, type(e).__name__, e, os.path.join(torch.hub.get_dir(), "checkpoints")))
        warnings.warn(msg, RuntimeWarning, stacklevel=2)
        print("WARNING: " + msg)
        return fn(weights=None)


class encoder(nn.Module):
    """reference pytorch/bts.py:268-320.  The backbone modules (and therefore parameter names, which
    bts_main.set_misc freezes by substring, bts_main.py:222-247) are torchvision's, as in the reference.
    params.pretrained: None (default, as the reference: ImageNet V1 weights, downloaded if needed; loud warning + random
    init when offline), True = must load, False = random init."""

    def __init__(self, params):
        super().__init__()
        self.params = params
        if params.encoder not in _ENCODERS:
            print("Not supported encoder: {}".format(params.encoder))
            return
        ctor, feats, names, ch = _ENCODERS[params.encoder]
        m = _load_backbone(ctor, getattr(params, "pretrained", None))
        self.base_model = adopt_convs(m.features if feats else m)
        self.feat_names = names
        self.feat_out_channels = ch
        if params.encoder == "mobilenetv2_bts":
            self.feat_inds = [2, 4, 7, 11, 19]

    def forward(self, x):
        skips = []
        mobile = self.params.encoder == "mobilenetv2_bts"
        for i, (k, v) in enumerate(self.base_model._modules.items(), start=1):
            if "fc" in k or "avgpool" in k:
                continue
            x = v(x)
            if mobile:
                if i in (2, 4, 7, 11, 19):
                    skips.append(x)
            elif any(n in k for n in self.feat_names):
                skips.append(x)
        return skips


class BtsModel(nn.Module):
    """reference pytorch/bts.py:323-331."""

    def __init__(self, params):
        super().__init__()
        self.encoder = encoder(params)
        self.decoder = bts(params, self.encoder.feat_out_channels, params.bts_size)

    def forward(self, x, focal):
        if x.is_cuda and x.dim() == 4:
            x = x.contiguous(memory_format=torch.channels_last)      # NHWC in memory for the whole path
        return self.decoder(self.encoder(x), focal)
