"""Composable fused autograd units for the BTS decoder and the encoder's non-dense-block stages (SURVEY 8a rows a5-a10,
a11 transitions/stem).  The reference (torch-eager, pytorch/bts.py:196-266) runs every BatchNorm, ReLU, ELU, nearest
up-sample and torch.cat as its own ATen/cuDNN kernel, forward and backward; here they are either folded into the tcgen05
conv engine (ELU in the epilogue, ReLU / BN-apply + ReLU in the A-operand prologue, the x2 up-sample in the im2col map) or
run as one of the streaming NHWC kernels of csrc/elem.cu / csrc/bn.cu:

  conv_act       y = act(conv(pre_relu?(up2?(x))))        upconv (bts.py:69-80), iconvs (:156-192), reduction chains (:83-108)
  bn_act         y = BN(x) [ReLU]                          decoder BNs (:154-182), torchvision norm0(+relu0) / norm5
  bn_relu_conv   y = conv(ReLU(BN(x)))                     atrous_conv halves (:51-66), DenseNet transitions
  cat_nhwc       channel concat into a 16-byte-aligned slab (the nine torch.cat of bts.forward); backward = views
  avgpool2       2x2 average pool of the transitions
  dwconv         depthwise 3x3 conv (padding 1, stride 1 / 2) on csrc/dwconv.cu, forward / dgrad / wgrad
  bn_add         y = BN(x) + res                           MobileNetV2 inverted-residual tail
  inverted_residual  torchvision InvertedResidual as ONE unit: expand 1x1 -> BN+ReLU6 folded into the depthwise conv's
                 prologue -> depthwise 3x3 (BN statistics in its epilogue) -> BN+ReLU6 -> project 1x1 -> BN [+ x]

Each unit is a torch.autograd.Function whose backward launches our kernels too (ELU', BN reductions, wgrad / dgrad on
the engine, 2x2 gradient fold of the up-sample).  Parameters stay the nn.Modules' own, BatchNorm running statistics are
updated with nn.BatchNorm2d semantics (momentum, unbiased variance, num_batches_tracked).
"""
import torch

from . import _lib, conv
from .ops import _ptr, _stream


def eligible(x):
    return x.is_cuda and x.dtype == torch.float32 and x.dim() == 4


def _nhwc(t):
    """(tensor, pixel stride) with NHWC memory; converts (one copy) when the layout is something else"""
    return conv._nhwc_view(t)


def _new(B, C, H, W, dev):
    return torch.empty((B, C, H, W), device=dev, dtype=torch.float32, memory_format=torch.channels_last)


# ------------------------------------------------------------------------------------------------ raw kernel wrappers
def bn_stats(x):
    x, xs = _nhwc(x)
    B, C, H, W = x.shape
    out = torch.empty((2, C), device=x.device, dtype=torch.float64)
    _lib.check(_lib.lib().bts_bn_stats(_ptr(x), xs, B * H * W, C, _ptr(out[0]), _ptr(out[1]), _stream()), "bts_bn_stats")
    _lib.count()
    return out


def bn_finalize(sums, n, bn, gamma, beta, training):
    """(scale, shift, mean, invstd) as a [4,C] tensor; in training also the module's running-stat update"""
    C = bn.num_features
    out = torch.empty((4, C), device=bn.running_mean.device if bn.running_mean is not None else gamma.device,
                      dtype=torch.float32)
    L = _lib.lib()
    g = gamma.detach() if gamma is not None else None
    b = beta.detach() if beta is not None else None
    if training:
        track = bn.track_running_stats and bn.running_mean is not None
        mom = bn.momentum if bn.momentum is not None else 0.1
        nbt = bn.num_batches_tracked if (track and bn.num_batches_tracked is not None) else None
        _lib.check(L.bts_bn_finalize_track(_ptr(sums[0]), _ptr(sums[1]), n, C, _ptr(g), _ptr(b), float(bn.eps), float(mom),
                                           _ptr(bn.running_mean) if track else None, _ptr(bn.running_var) if track else None,
                                           _ptr(nbt), _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]), _stream()),
                   "bts_bn_finalize_track")
    else:
        _lib.check(L.bts_bn_fold(C, _ptr(g), _ptr(b), float(bn.eps), _ptr(bn.running_mean), _ptr(bn.running_var),
                                 _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]), _stream()), "bts_bn_fold")
    _lib.count()
    return out


def bn_uses_batch_stats(bn):
    """nn.BatchNorm2d: batch statistics in train mode, or whenever no running statistics are tracked"""
    return bn.training or bn.running_mean is None


def bn_backward(x, g, st, use_stats, relu, out=None, accumulate=False):
    """d/dx of [relu](bn(x)) given g = d/d(output); returns (dx, S) with S = (dbeta, dgamma) as fp64 [2,C]"""
    x, xs = _nhwc(x)
    g, gs = _nhwc(g)
    B, C, H, W = x.shape
    if out is None:
        out = _new(B, C, H, W, x.device)
    o2, os_ = _nhwc(out)
    if o2 is not out:
        raise ValueError("bn_backward: out must be NHWC in memory")
    M = B * H * W
    L = _lib.lib()
    S = torch.empty((2, C), device=x.device, dtype=torch.float64)
    coef = torch.empty((2, C), device=x.device, dtype=torch.float32)
    _lib.check(L.bts_bn_bwd_reduce(_ptr(x), xs, _ptr(g), gs, M, C, _ptr(st[0]), _ptr(st[1]), _ptr(st[2]), _ptr(st[3]),
                                   int(relu), _ptr(S[0]), _ptr(S[1]), _ptr(coef), _stream()), "bts_bn_bwd_reduce")
    _lib.check(L.bts_bn_bwd_apply(_ptr(x), xs, _ptr(g), gs, M, C, _ptr(st[0]), _ptr(st[1]),
                                  _ptr(coef) if use_stats else None, int(relu), _ptr(out), os_, int(accumulate), _stream()),
               "bts_bn_bwd_apply")
    _lib.count(3)
    return out, S


def copy_channels(src, dst, accumulate=False):
    s, ss = _nhwc(src)
    d, ds = _nhwc(dst)
    if d is not dst:
        raise ValueError("copy_channels: dst must be NHWC in memory")
    B, C, H, W = s.shape
    _lib.check(_lib.lib().bts_copy_channels(_ptr(s), ss, B * H * W, C, _ptr(d), ds, int(accumulate), _stream()),
               "bts_copy_channels")
    _lib.count()


# ------------------------------------------------------------------------------------------------ conv (+ pre / act)
class _ConvAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, padding, dilation, pre_relu, up, act):
        y = conv.conv2d_tc(x, weight, 1, padding, dilation, pre_relu=pre_relu, upsample2=up, act=act)
        ctx.cfg = (padding, dilation, pre_relu, up, act)
        ctx.save_for_backward(x, weight, y if act == "elu" else None)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight, y = ctx.saved_tensors
        padding, dilation, pre_relu, up, act = ctx.cfg
        L = _lib.lib()
        g, gs = _nhwc(gy)
        B, Co, Ho, Wo = g.shape
        if act == "elu":
            ge = _new(B, Co, Ho, Wo, g.device)
            y2, ys = _nhwc(y)
            _lib.check(L.bts_elu_bwd(_ptr(g), gs, _ptr(y2), ys, B * Ho * Wo, Co, _ptr(ge), Co, _stream()), "bts_elu_bwd")
            _lib.count()
            g = ge
        elif act is not None:
            raise RuntimeError("conv_act backward supports act in (None, 'elu')")
        gx = gw = None
        KH = weight.shape[2]
        if ctx.needs_input_grad[1]:
            gw = conv.wgrad_tc(x, g, weight.shape, weight.stride(), 1, padding, dilation, pre_relu=pre_relu, upsample2=up)
        if ctx.needs_input_grad[0]:
            Ci = weight.shape[1]
            out = None
            if Ci % 4:        # keep the gradient's pixel rows 16-byte aligned (concat3 = 225, concat2 = 161 channels)
                Hf, Wf = (2 * x.shape[2], 2 * x.shape[3]) if up else (x.shape[2], x.shape[3])
                out = _new(x.shape[0], (Ci + 3) // 4 * 4, Hf, Wf, g.device)[:, :Ci]
            full = conv.conv2d_tc(g, weight, 1, dilation * (KH - 1) - padding, dilation, transpose_flip=True, out=out)
            if up:
                x2, xs = _nhwc(x)
                Bx, Ci, Hs, Ws = x2.shape
                gx = _new(Bx, Ci, Hs, Ws, g.device)
                full, fs = _nhwc(full)
                _lib.check(L.bts_upsample2_sum(_ptr(full), fs, Bx, Hs, Ws, Ci, _ptr(x2) if pre_relu else None, xs,
                                               _ptr(gx), Ci, _stream()), "bts_upsample2_sum")
                _lib.count()
            elif pre_relu:
                gx = torch.where(x > 0, full, torch.zeros((), device=full.device))
            else:
                gx = full
        return gx, gw, None, None, None, None, None


def conv_act(x, weight, padding=0, dilation=1, pre_relu=False, up=False, act=None):
    """act(conv2d(pre_relu ? relu(x) : x, nearest-x2 up-sampled when `up`)), stride 1, all three GEMMs on the engine"""
    return _ConvAct.apply(x, weight, int(padding), int(dilation), bool(pre_relu), bool(up), act)


# ------------------------------------------------------------------------------------------------ BatchNorm (+ ReLU)
_ACT_CODE = {None: 0, "relu": 1, "relu6": 2}      # the `relu` flag of bts_bn_apply / bts_bn_bwd_reduce / bts_bn_bwd_apply


def bn_apply(x, st, relu):
    """x*scale + shift [ReLU | ReLU6] with (scale, shift) = st[0], st[1]"""
    x, xs = _nhwc(x)
    B, C, H, W = x.shape
    y = _new(B, C, H, W, x.device)
    _lib.check(_lib.lib().bts_bn_apply(_ptr(x), xs, B * H * W, C, _ptr(st[0]), _ptr(st[1]), int(relu), _ptr(y), C, _stream()),
               "bts_bn_apply")
    _lib.count()
    return y


class _BnAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, bn, relu):
        x, xs = _nhwc(x)
        B, C, H, W = x.shape
        n = B * H * W
        batch = bn_uses_batch_stats(bn)
        st = bn_finalize(bn_stats(x) if batch else None, n, bn, gamma, beta, batch)
        y = _new(B, C, H, W, x.device)
        _lib.check(_lib.lib().bts_bn_apply(_ptr(x), xs, n, C, _ptr(st[0]), _ptr(st[1]), int(relu), _ptr(y), C, _stream()),
                   "bts_bn_apply")
        _lib.count()
        ctx.cfg = (batch, relu)
        ctx.save_for_backward(x, st)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, st = ctx.saved_tensors
        batch, relu = ctx.cfg
        gx, S = bn_backward(x, gy, st, batch, relu)
        return (gx if ctx.needs_input_grad[0] else None, S[1].float() if ctx.needs_input_grad[1] else None,
                S[0].float() if ctx.needs_input_grad[2] else None, None, None)


def bn_act(x, bn, relu=False, act=None):
    """nn.BatchNorm2d `bn` applied to x (batch statistics + running-stat update in train mode, folded running
    statistics in eval mode), optionally followed by ReLU (relu=True or act="relu") or ReLU6 (act="relu6") -- 3 streaming
    kernels forward, 3 backward"""
    if act not in _ACT_CODE:
        raise ValueError("bn_act: act must be one of %s" % sorted(k for k in _ACT_CODE if k))
    return _BnAct.apply(x, bn.weight, bn.bias, bn, _ACT_CODE[act] or int(bool(relu)))


# ------------------------------------------------------------------------------------------------ BN -> ReLU -> conv
class _BnReluConv(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, weight, bn, padding, dilation):
        x, _ = _nhwc(x)
        B, C, H, W = x.shape
        n = B * H * W
        batch = bn_uses_batch_stats(bn)
        st = bn_finalize(bn_stats(x) if batch else None, n, bn, gamma, beta, batch)
        y = conv.conv2d_tc(x, weight, 1, padding, dilation, pre_scale=st[0], pre_shift=st[1], pre_relu=True)
        ctx.cfg = (padding, dilation, batch)
        ctx.save_for_backward(x, weight, st)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight, st = ctx.saved_tensors
        padding, dilation, batch = ctx.cfg
        KH = weight.shape[2]
        gw = None
        if ctx.needs_input_grad[3]:
            gw = conv.wgrad_tc(x, gy, weight.shape, weight.stride(), 1, padding, dilation, pre_scale=st[0], pre_shift=st[1],
                               pre_relu=True)
        from . import fused
        if fused.EPI_BNBWD:
            gx, S = fused.dgrad_bn_relu_backward(gy, weight, padding, dilation, x, st, batch)   # sums in the dgrad epilogue
        else:
            g_a = conv.conv2d_tc(gy, weight, 1, dilation * (KH - 1) - padding, dilation, transpose_flip=True)
            gx, S = bn_backward(x, g_a, st, batch, True, out=g_a)          # in place on the dgrad result
        return (gx if ctx.needs_input_grad[0] else None, S[1].float() if ctx.needs_input_grad[1] else None,
                S[0].float() if ctx.needs_input_grad[2] else None, gw, None, None, None)


def bn_relu_conv(x, bn, weight, padding=0, dilation=1):
    """conv2d(relu(bn(x))): the normalisation + ReLU run inside the conv's A-operand prologue (never materialised)"""
    return _BnReluConv.apply(x, bn.weight, bn.bias, weight, bn, int(padding), int(dilation))


# ------------------------------------------------------------------------------------------------ concat
class _CatNHWC(torch.autograd.Function):
    @staticmethod
    def forward(ctx, *ts):
        B, _, H, W = ts[0].shape
        cs = [int(t.shape[1]) for t in ts]
        C = sum(cs)
        Cp = (C + 3) // 4 * 4
        slab = _new(B, Cp, H, W, ts[0].device)
        off = 0
        for t, c in zip(ts, cs):
            copy_channels(t, slab[:, off:off + c])
            off += c
        if Cp != C:
            _lib.check(_lib.lib().bts_zero_channels(_ptr(slab), Cp, B * H * W, C, Cp, _stream()), "bts_zero_channels")
            _lib.count()
        ctx.cs = cs
        return slab[:, :C] if Cp != C else slab

    @staticmethod
    def backward(ctx, g):
        out, off = [], 0
        for i, c in enumerate(ctx.cs):
            out.append(g[:, off:off + c] if ctx.needs_input_grad[i] else None)
            off += c
        return tuple(out)


def cat_nhwc(tensors):
    """torch.cat(tensors, 1) into a fresh NHWC slab whose pixel rows are 16-byte aligned (zero channels appended when the
    channel sum is not a multiple of 4: concat3 = 225, concat2 = 161); backward hands out channel-slice views"""
    return _CatNHWC.apply(*tensors)


# ------------------------------------------------------------------------------------------------ 2x2 average pool
class _AvgPool2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x, xs = _nhwc(x)
        B, C, H, W = x.shape
        if H % 2 or W % 2:
            raise ValueError("avgpool2 needs even spatial dims")
        y = _new(B, C, H // 2, W // 2, x.device)
        _lib.check(_lib.lib().bts_avgpool2_fwd(_ptr(x), xs, B, H // 2, W // 2, C, _ptr(y), C, _stream()), "bts_avgpool2_fwd")
        _lib.count()
        return y

    @staticmethod
    def backward(ctx, g):
        g, gs = _nhwc(g)
        B, C, Ho, Wo = g.shape
        gx = _new(B, C, 2 * Ho, 2 * Wo, g.device)
        _lib.check(_lib.lib().bts_avgpool2_bwd(_ptr(g), gs, B, Ho, Wo, C, _ptr(gx), C, _stream()), "bts_avgpool2_bwd")
        _lib.count()
        return gx


def avgpool2(x):
    return _AvgPool2.apply(x)


# ------------------------------------------------------------------------------------------------ ResNet / ResNeXt glue
class _MaxPool3s2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x, xs = _nhwc(x)
        B, C, H, W = x.shape
        Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        y = _new(B, C, Ho, Wo, x.device)
        arg = torch.empty(B * Ho * Wo * C, device=x.device, dtype=torch.uint8)
        _lib.check(_lib.lib().bts_maxpool3s2_fwd(_ptr(x), xs, B, H, W, C, _ptr(y), C, _ptr(arg), _stream()), "bts_maxpool3s2_fwd")
        _lib.count()
        ctx.shape = (B, C, H, W)
        ctx.save_for_backward(arg)
        return y

    @staticmethod
    def backward(ctx, g):
        (arg,) = ctx.saved_tensors
        B, C, H, W = ctx.shape
        g, gs = _nhwc(g)
        gx = _new(B, C, H, W, g.device)
        _lib.check(_lib.lib().bts_maxpool3s2_bwd(_ptr(g), gs, _ptr(arg), B, H, W, C, _ptr(gx), C, _stream()), "bts_maxpool3s2_bwd")
        _lib.count()
        return gx


def maxpool3s2(x):
    """3x3 / stride 2 / pad 1 max-pool (torchvision densenet `pool0`, resnet `maxpool`) on our NHWC kernels"""
    return _MaxPool3s2.apply(x)


class _BnAddRelu(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, res, gamma, beta, bn):
        x, xs = _nhwc(x)
        res, rs = _nhwc(res)
        B, C, H, W = x.shape
        n = B * H * W
        batch = bn_uses_batch_stats(bn)
        st = bn_finalize(bn_stats(x) if batch else None, n, bn, gamma, beta, batch)
        y = _new(B, C, H, W, x.device)
        _lib.check(_lib.lib().bts_bn_add_relu(_ptr(x), xs, n, C, _ptr(st[0]), _ptr(st[1]), _ptr(res), rs, _ptr(y), C, _stream()),
                   "bts_bn_add_relu")
        _lib.count()
        ctx.batch = batch
        ctx.save_for_backward(x, st, y)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, st, y = ctx.saved_tensors
        g, gs = _nhwc(gy)
        B, C, H, W = y.shape
        gm = _new(B, C, H, W, y.device)
        _lib.check(_lib.lib().bts_relu_bwd(_ptr(g), gs, _ptr(y), C, B * H * W, C, _ptr(gm), C, _stream()), "bts_relu_bwd")
        _lib.count()
        gx, S = bn_backward(x, gm, st, ctx.batch, False)
        return (gx if ctx.needs_input_grad[0] else None, gm if ctx.needs_input_grad[1] else None,
                S[1].float() if ctx.needs_input_grad[2] else None, S[0].float() if ctx.needs_input_grad[3] else None, None)


def bn_add_relu(x, res, bn):
    """relu(bn(x) + res): the tail of a torchvision Bottleneck, one streaming kernel after the statistics"""
    return _BnAddRelu.apply(x, res, bn.weight, bn.bias, bn)


class _BnAdd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, res, gamma, beta, bn):
        x, xs = _nhwc(x)
        res, rs = _nhwc(res)
        B, C, H, W = x.shape
        n = B * H * W
        batch = bn_uses_batch_stats(bn)
        st = bn_finalize(bn_stats(x) if batch else None, n, bn, gamma, beta, batch)
        y = _new(B, C, H, W, x.device)
        _lib.check(_lib.lib().bts_bn_add(_ptr(x), xs, n, C, _ptr(st[0]), _ptr(st[1]), _ptr(res), rs, _ptr(y), C, _stream()),
                   "bts_bn_add")
        _lib.count()
        ctx.batch = batch
        ctx.save_for_backward(x, st)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, st = ctx.saved_tensors
        gx, S = bn_backward(x, gy, st, ctx.batch, 0)
        return (gx if ctx.needs_input_grad[0] else None, gy if ctx.needs_input_grad[1] else None,
                S[1].float() if ctx.needs_input_grad[2] else None, S[0].float() if ctx.needs_input_grad[3] else None, None)


def bn_add(x, res, bn):
    """bn(x) + res: the tail of a MobileNetV2 inverted residual with its identity connection"""
    return _BnAdd.apply(x, res, bn.weight, bn.bias, bn)


# ------------------------------------------------------------------------------------------------ depthwise 3x3
def dw_eligible(conv_module):
    """a depthwise 3x3 / padding 1 / stride 1 or 2 nn.Conv2d without bias that csrc/dwconv.cu computes"""
    m = conv_module
    C = m.in_channels
    return (m.groups == C and m.out_channels == C and C % 4 == 0 and tuple(m.kernel_size) == (3, 3)
            and tuple(m.padding) == (1, 1) and tuple(m.dilation) == (1, 1) and m.stride[0] == m.stride[1]
            and m.stride[0] in (1, 2) and m.bias is None and m.padding_mode == "zeros")


def _dw_out(H, W, stride):
    return (H - 1) // stride + 1, (W - 1) // stride + 1


def dw_fwd(x, weight, stride, pre=None, post=None, stats=False):
    """depthwise 3x3 forward: (y, sums).  pre = [4,C] BN state -> input prologue clamp(x*st[0] + st[1], 0, 6);
    post = [4,C] eval BN state -> epilogue clamp(y*st[0] + st[1], 0, 6); stats -> sums = fp64 [2,C] (sum y, sum y^2)"""
    x, xs = _nhwc(x)
    B, C, H, W = x.shape
    Ho, Wo = _dw_out(H, W, stride)
    L = _lib.lib()
    y = _new(B, C, Ho, Wo, x.device)
    part = sums = None
    if stats:
        part = torch.empty(L.bts_dw_partials(B, Ho, Wo, C, 0), device=x.device, dtype=torch.float64)
        sums = torch.empty((2, C), device=x.device, dtype=torch.float64)
    w = weight.detach().contiguous()
    _lib.check(L.bts_dw_fwd(_ptr(x), xs, B, H, W, C, int(stride), _ptr(w),
                            _ptr(pre[0]) if pre is not None else None, _ptr(pre[1]) if pre is not None else None,
                            _ptr(post[0]) if post is not None else None, _ptr(post[1]) if post is not None else None,
                            _ptr(y), C, _ptr(part), _ptr(sums), _stream()), "bts_dw_fwd")
    _lib.count(2 if stats else 1)
    return y, sums


def dw_dgrad(g, weight, stride, H, W):
    """d/dx of the depthwise 3x3 conv (input H x W) given g = d/dy"""
    g, gs = _nhwc(g)
    B, C = g.shape[0], g.shape[1]
    gx = _new(B, C, H, W, g.device)
    w = weight.detach().contiguous()
    _lib.check(_lib.lib().bts_dw_dgrad(_ptr(g), gs, B, H, W, C, int(stride), _ptr(w), _ptr(gx), C, _stream()),
               "bts_dw_dgrad")
    _lib.count()
    return gx


def dw_wgrad(x, g, weight, stride, pre=None):
    """dW (shaped / strided like the weight) of the depthwise 3x3 conv, the input prologue `pre` recomputed from x"""
    x, xs = _nhwc(x)
    g, gs = _nhwc(g)
    B, C, H, W = x.shape
    L = _lib.lib()
    part = torch.empty(L.bts_dw_partials(B, g.shape[2], g.shape[3], C, 1), device=x.device, dtype=torch.float64)
    gw = torch.empty_strided(tuple(weight.shape), tuple(weight.stride()), device=x.device, dtype=torch.float32)
    s = weight.stride()
    _lib.check(L.bts_dw_wgrad(_ptr(x), xs, B, H, W, C, int(stride), _ptr(pre[0]) if pre is not None else None,
                              _ptr(pre[1]) if pre is not None else None, _ptr(g), gs, _ptr(part), _ptr(gw), s[0], s[2], s[3],
                              _stream()), "bts_dw_wgrad")
    _lib.count(2)
    return gw


class _DwConv(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, stride):
        y, _ = dw_fwd(x, weight, stride)
        ctx.stride = stride
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gx = dw_dgrad(gy, weight, ctx.stride, x.shape[2], x.shape[3]) if ctx.needs_input_grad[0] else None
        gw = dw_wgrad(x, gy, weight, ctx.stride) if ctx.needs_input_grad[1] else None
        return gx, gw, None


def dwconv(x, weight, stride=1):
    """depthwise 3x3 conv, padding 1, weight (C,1,3,3): forward, dgrad and wgrad on csrc/dwconv.cu"""
    return _DwConv.apply(x, weight, int(stride))


# ------------------------------------------------------------------------------------------------ MobileNetV2 block
def _zeros2(C, dev):
    return torch.zeros((2, C), device=dev, dtype=torch.float64)


class _InvertedResidual(torch.autograd.Function):
    """torchvision InvertedResidual [(1x1 -> BN1 -> ReLU6) -> dw 3x3 -> BN2 -> ReLU6 -> 1x1 -> BN3 (+ x)].  BN1 + ReLU6 run
    inside the depthwise conv's prologue (the expanded activation is never written), the depthwise conv's epilogue reduces
    BN2's batch statistics (or, in eval mode without autograd, applies BN2 + ReLU6), the 1x1 convs run on the tcgen05
    engine.  Saved for backward: x, the raw expand output e, the raw dw output d, the project conv's input a and its
    output p -- BN1 / BN2 activations are recomputed from e / d."""

    @staticmethod
    def forward(ctx, x, w1, g1, b1, wdw, g2, b2, w3, g3, b3, bns, stride, residual):
        bn1, bn2, bn3 = bns
        x, xs = _nhwc(x)
        B, _, H, W = x.shape
        dev = x.device
        grad = any(ctx.needs_input_grad)
        t1 = t2 = None
        st1 = e = None
        if w1 is not None:
            t1 = bn_uses_batch_stats(bn1)
            s1 = _zeros2(w1.shape[0], dev) if t1 and w1.shape[0] <= 256 else None      # stats in the engine epilogue
            e = conv.conv2d_tc(x, w1, stats=s1)
            st1 = bn_finalize((s1 if s1 is not None else bn_stats(e)) if t1 else None, B * H * W, bn1, g1, b1, t1)
        src = e if e is not None else x
        Ho, Wo = _dw_out(H, W, stride)
        t2 = bn_uses_batch_stats(bn2)
        d = None
        if not t2 and not grad:          # eval without autograd: BN2 + ReLU6 in the depthwise epilogue
            st2 = bn_finalize(None, B * Ho * Wo, bn2, g2, b2, False)
            a, _ = dw_fwd(src, wdw, stride, pre=st1, post=st2)
        else:
            d, s2 = dw_fwd(src, wdw, stride, pre=st1, stats=t2)
            st2 = bn_finalize(s2, B * Ho * Wo, bn2, g2, b2, t2)
            a = bn_apply(d, st2, 2)
        t3 = bn_uses_batch_stats(bn3)
        Co = w3.shape[0]
        s3 = _zeros2(Co, dev) if t3 and Co <= 256 else None
        p = conv.conv2d_tc(a, w3, stats=s3)
        st3 = bn_finalize((s3 if s3 is not None else bn_stats(p)) if t3 else None, B * Ho * Wo, bn3, g3, b3, t3)
        y = _new(B, Co, Ho, Wo, dev)
        L = _lib.lib()
        if residual:
            _lib.check(L.bts_bn_add(_ptr(p), Co, B * Ho * Wo, Co, _ptr(st3[0]), _ptr(st3[1]), _ptr(x), xs, _ptr(y), Co,
                                    _stream()), "bts_bn_add")
        else:
            _lib.check(L.bts_bn_apply(_ptr(p), Co, B * Ho * Wo, Co, _ptr(st3[0]), _ptr(st3[1]), 0, _ptr(y), Co, _stream()),
                       "bts_bn_apply")
        _lib.count()
        if grad:
            ctx.cfg = (stride, residual, t1, t2, t3)
            ctx.save_for_backward(x, e, d, a, p, st1, st2, st3, w1, wdw, w3)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, e, d, a, p, st1, st2, st3, w1, wdw, w3 = ctx.saved_tensors
        stride, residual, t1, t2, t3 = ctx.cfg
        need = ctx.needs_input_grad
        gy, _ = _nhwc(gy)
        gp, S3 = bn_backward(p, gy, st3, t3, 0)
        gw3 = conv.wgrad_tc(a, gp, w3.shape, w3.stride()) if need[7] else None
        ga = conv.conv2d_tc(gp, w3, 1, 0, 1, transpose_flip=True)
        gd, S2 = bn_backward(d, ga, st2, t2, 2, out=ga)                    # in place on the dgrad result
        src = e if e is not None else x
        gwdw = dw_wgrad(src, gd, wdw, stride, pre=st1) if need[4] else None
        gx = gw1 = S1 = None
        if e is not None:
            ge, S1 = bn_backward(e, dw_dgrad(gd, wdw, stride, e.shape[2], e.shape[3]), st1, t1, 2)
            gw1 = conv.wgrad_tc(x, ge, w1.shape, w1.stride()) if need[1] else None
            if need[0]:
                gx = conv.conv2d_tc(ge, w1, 1, 0, 1, transpose_flip=True)
        elif need[0]:
            gx = dw_dgrad(gd, wdw, stride, x.shape[2], x.shape[3])
        if gx is not None and residual:
            copy_channels(gy, gx, accumulate=True)
        f = lambda S, i, k: S[k].float() if (S is not None and need[i]) else None
        return (gx, gw1, f(S1, 2, 1), f(S1, 3, 0), gwdw, f(S2, 5, 1), f(S2, 6, 0), gw3, f(S3, 8, 1), f(S3, 9, 0),
                None, None, None)


def inverted_residual(x, expand, bn1, dw, bn2, project, bn3, residual):
    """torchvision InvertedResidual forward on our kernels; `expand` / `bn1` are None for the t = 1 block"""
    return _InvertedResidual.apply(x, expand.weight if expand is not None else None,
                                   bn1.weight if bn1 is not None else None, bn1.bias if bn1 is not None else None,
                                   dw.weight, bn2.weight, bn2.bias, project.weight, bn3.weight, bn3.bias, (bn1, bn2, bn3),
                                   int(dw.stride[0]), bool(residual))
