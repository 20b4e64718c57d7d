"""GPU tests of the MobileNetV2 encoder on native kernels: the depthwise 3x3 kernels (csrc/dwconv.cu), BatchNorm + ReLU6 and
BatchNorm + residual add, the fused InvertedResidual unit, the whole model against the reference's golden outputs, the
absence of library convolution / BatchNorm / hardtanh ops on the encoder path, and run-to-run determinism."""
import copy
import types

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

WIDTHS = (32, 96, 144, 192, 384, 576, 960)


def _max_err(got, want):
    """max abs error over the output scale (the bar of test_resnet_gpu.py)"""
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).abs().max() / want.abs().max().clamp_min(1e-30))


def _rel_norm(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).norm() / want.norm().clamp_min(1e-30))


def _bn_state(C, gen, dev):
    """[4,C] BN state (scale, shift, mean, invstd) whose affine maps many values below 0 and above 6"""
    scale = torch.rand(C, generator=gen) * 2 + 0.5
    shift = torch.randn(C, generator=gen) * 2 + 2
    return torch.stack([scale, shift, torch.zeros(C), torch.ones(C)]).to(dev)


# ---------------------------------------------------------------------------------------------------- depthwise kernels
@pytest.mark.parametrize("pre", [False, True])
@pytest.mark.parametrize("B", [1, 2])
@pytest.mark.parametrize("stride", [1, 2])
@pytest.mark.parametrize("C", WIDTHS)
def test_depthwise_vs_fp64(C, stride, B, pre):
    from bts_b200 import glue
    gen = torch.Generator().manual_seed(C * 10 + stride * 3 + B + 7 * pre)
    H, W = 9, 13
    x = (torch.randn(B, C, H, W, generator=gen) * 4 + 1).cuda().contiguous(memory_format=torch.channels_last)
    w = torch.randn(C, 1, 3, 3, generator=gen).cuda()
    st = _bn_state(C, gen, "cuda") if pre else None

    x64 = x.detach().double().cpu().requires_grad_(True)
    a64 = (x64 * st[0].double().cpu().view(1, -1, 1, 1) + st[1].double().cpu().view(1, -1, 1, 1)).clamp(0, 6) if pre else x64
    w64 = w.double().cpu().requires_grad_(True)
    y64 = F.conv2d(a64, w64, stride=stride, padding=1, groups=C)

    y, sums = glue.dw_fwd(x, w, stride, pre=st, stats=True)
    assert y.shape == y64.shape
    assert _max_err(y, y64) <= 2e-5
    y_plain, none = glue.dw_fwd(x, w, stride, pre=st)
    assert none is None and torch.equal(y_plain, y)          # the statistics epilogue does not change y
    r = y64.detach()
    for k, ref in enumerate((r.sum((0, 2, 3)), (r * r).sum((0, 2, 3)))):
        den = (r.abs() if k == 0 else r * r).sum((0, 2, 3)).max()
        assert float((sums[k].cpu() - ref).abs().max() / den) <= 2e-5, "statistics %d" % k

    # eval-mode epilogue: clamp(y*s + t, 0, 6)
    post = _bn_state(C, gen, "cuda")
    yq, _ = glue.dw_fwd(x, w, stride, pre=st, post=post)
    ref_q = (y64.detach() * post[0].double().cpu().view(1, -1, 1, 1) + post[1].double().cpu().view(1, -1, 1, 1)).clamp(0, 6)
    assert float((yq.double().cpu() - ref_q).abs().max()) <= 2e-5 * 3 * float(y64.abs().max())

    g = torch.randn(y64.shape, generator=gen)
    y64.backward(g.double())
    gc = g.cuda().contiguous(memory_format=torch.channels_last)
    gw = glue.dw_wgrad(x, gc, w, stride, pre=st)
    assert _max_err(gw, w64.grad) <= 2e-5
    if not pre:
        gx = glue.dw_dgrad(gc, w, stride, H, W)
        assert _max_err(gx, x64.grad) <= 2e-5
    assert torch.equal(glue.dw_wgrad(x, gc, w, stride, pre=st), gw)      # deterministic reduction


@pytest.mark.parametrize("stride", [1, 2])
def test_depthwise_conv2dtc_autograd(stride):
    """a depthwise nn.Conv2d re-classed to Conv2dTC runs on the native kernels with autograd (odd sizes)"""
    from bts_b200 import model
    gen = torch.Generator().manual_seed(stride)
    C = 96
    conv = nn.Conv2d(C, C, 3, stride, 1, groups=C, bias=False)
    ref = copy.deepcopy(conv).double()
    conv.__class__ = model.Conv2dTC
    conv.cuda()
    x = torch.randn(2, C, 11, 15, generator=gen)
    xc = x.cuda().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    x64 = x.double().requires_grad_(True)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        y = conv(xc)
        g = torch.randn(y.shape, generator=gen)
        y.backward(g.cuda())
    assert not [e.name for e in prof.events() if "convolution" in e.name]
    y64 = ref(x64)
    y64.backward(g.double())
    assert _max_err(y, y64) <= 2e-5
    assert _max_err(xc.grad, x64.grad) <= 2e-5
    assert _max_err(conv.weight.grad, ref.weight.grad) <= 2e-5


# ---------------------------------------------------------------------------------------------------- BN + ReLU6, bn_add
@pytest.mark.parametrize("mode", ["train", "eval"])
@pytest.mark.parametrize("kind", ["relu6", "add"])
def test_bn_relu6_and_bn_add_vs_fp64(kind, mode):
    from bts_b200 import glue
    gen = torch.Generator().manual_seed(3)
    B, C, H, W = 2, 96, 9, 13
    bn = nn.BatchNorm2d(C)
    with torch.no_grad():
        bn.weight.copy_(torch.rand(C, generator=gen) * 2 + 0.5)
        bn.bias.copy_(torch.randn(C, generator=gen) + 2)
        bn.running_mean.copy_(torch.randn(C, generator=gen))
        bn.running_var.copy_(torch.rand(C, generator=gen) + 0.5)
    ref = copy.deepcopy(bn).double()
    bn.cuda()
    getattr(bn, mode)()
    getattr(ref, mode)()
    x = torch.randn(B, C, H, W, generator=gen) * 3 + 1
    res = torch.randn(B, C, H, W, generator=gen)
    xc = x.cuda().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    rc = res.cuda().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    x64, r64 = x.double().requires_grad_(True), res.double().requires_grad_(True)
    if kind == "relu6":
        y = glue.bn_act(xc, bn, act="relu6")
        y64 = F.relu6(ref(x64))
        assert 0.05 < float((y64 == 0).double().mean()) and 0.01 < float((y64 == 6).double().mean())
    else:
        y = glue.bn_add(xc, rc, bn)
        y64 = ref(x64) + r64
    g = torch.randn(y64.shape, generator=gen)
    y.backward(g.cuda())
    y64.backward(g.double())
    assert _max_err(y, y64) <= 2e-5
    assert _rel_norm(xc.grad, x64.grad) <= 1e-4
    assert _rel_norm(bn.weight.grad, ref.weight.grad) <= 1e-4
    assert _rel_norm(bn.bias.grad, ref.bias.grad) <= 1e-4
    if kind == "add":
        assert torch.equal(rc.grad.cpu(), g)
    for k in ("running_mean", "running_var", "num_batches_tracked"):
        np.testing.assert_allclose(getattr(bn, k).cpu().double().numpy(), getattr(ref, k).numpy(), rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------------- InvertedResidualTC
@pytest.mark.parametrize("mode", ["train", "eval"])
@pytest.mark.parametrize("inp,oup,stride,t", [(32, 16, 1, 1), (24, 32, 2, 6), (24, 24, 1, 6)],
                         ids=["t1", "stride2", "residual"])
def test_inverted_residual_vs_torchvision_fp64(inp, oup, stride, t, mode):
    from torchvision.models.mobilenetv2 import InvertedResidual

    from bts_b200 import model
    torch.manual_seed(inp + oup + stride + t)
    blk = InvertedResidual(inp, oup, stride, t)
    with torch.no_grad():
        for m in blk.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.weight.uniform_(0.5, 2.5)
                m.bias.normal_(1.0, 1.0)
                m.running_mean.normal_(0, 0.5)
                m.running_var.uniform_(0.5, 1.5)
    ref = copy.deepcopy(blk).double()
    model.adopt_convs(nn.Sequential(blk))
    assert type(blk).__name__ == "InvertedResidualTC" and blk._parts() is not None
    assert blk.use_res_connect == (t == 6 and stride == 1)
    blk.cuda()
    getattr(blk, mode)()
    getattr(ref, mode)()
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(2, inp, 9, 13, generator=gen) * 2
    xc = x.cuda().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    x64 = x.double().requires_grad_(True)
    y = blk(xc)
    y64 = ref(x64)
    assert y.shape == y64.shape
    g = torch.randn(y64.shape, generator=gen)
    y.backward(g.cuda())
    y64.backward(g.double())
    assert _max_err(y, y64) <= 1e-4
    assert _rel_norm(xc.grad, x64.grad) <= 1e-3
    pr = dict(ref.named_parameters())
    for k, p in blk.named_parameters():
        assert _rel_norm(p.grad, pr[k].grad) <= 1e-3, k
    br = dict(ref.named_buffers())
    for k, b in blk.named_buffers():
        np.testing.assert_allclose(b.cpu().double().numpy(), br[k].numpy(), rtol=1e-4, atol=1e-6, err_msg=k)
    with torch.no_grad():                    # eval forward without autograd: BN2 + ReLU6 in the depthwise epilogue
        y_ng = blk(xc.detach())
        y64_ng = ref(x64.detach())
    assert _max_err(y_ng, y64_ng) <= 1e-4


# ---------------------------------------------------------------------------------------------------- whole model
def _mobilenet_model():
    import bts
    p = types.SimpleNamespace(encoder="mobilenetv2_bts", max_depth=10.0, dataset="nyu", bts_size=512, pretrained=False)
    torch.manual_seed(0)
    return bts.BtsModel(p)


def test_whole_model_vs_reference_golden(golden):
    from make_golden import model_inputs, seeded_state_dict
    g = golden("model_mobilenetv2_bts")
    m = _mobilenet_model()
    m.load_state_dict(seeded_state_dict(m), strict=True)
    m.cuda()
    for mode, x, focal in model_inputs():
        getattr(m, mode)()
        with torch.no_grad():
            outs = m(x.cuda(), focal.cuda())
        idx = g[mode + "_idx"]
        for i, o in enumerate(outs):
            v = o.reshape(-1).double().cpu().numpy()
            key = "%s_out%d" % (mode, i)
            np.testing.assert_allclose(v[idx], g[key], rtol=1e-3, atol=1e-3 * float(np.median(np.abs(g[key]))), err_msg=key)
            assert abs(v.sum() - float(g[key + "_sum"])) <= 1e-3 * float(g[key + "_abssum"]), key
            assert abs(np.abs(v).sum() - float(g[key + "_abssum"])) <= 1e-3 * float(g[key + "_abssum"]), key


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_encoder_path_has_no_library_ops(mode):
    m = _mobilenet_model().cuda()
    getattr(m, mode)()
    x = torch.randn(2, 3, 96, 128, generator=torch.Generator().manual_seed(0)).cuda()
    x = x.contiguous(memory_format=torch.channels_last)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        skips = m.encoder(x)
        sum(s.sum() for s in skips).backward()
        torch.cuda.synchronize()
    assert len(skips) == 5 and [s.shape[1] for s in skips] == [16, 24, 32, 64, 1280]
    names = {e.name for e in prof.events()}
    bad = sorted(n for n in names if any(k in n for k in ("convolution", "batch_norm", "hardtanh")))
    assert not bad, bad
    assert all(p.grad is not None for p in m.encoder.parameters())


def test_train_step_is_deterministic_and_graph_capturable():
    import bts
    from bts_b200.graph import GraphedTrainStep
    m = _mobilenet_model().cuda().train()
    state = copy.deepcopy(m.state_dict())
    gen = torch.Generator().manual_seed(4)
    x = torch.randn(2, 3, 96, 128, generator=gen).cuda()
    focal = torch.full((2,), 518.8579, device="cuda")
    gt = (torch.rand(2, 1, 96, 128, generator=gen) * 10).cuda()
    crit = bts.silog_loss(0.85)
    loss_fn = lambda out, gt: crit(out[4], gt, gt > 0.1)

    def eager():
        m.load_state_dict(state)
        for p in m.parameters():
            p.grad = None
        out = m(x, focal)
        loss = loss_fn(out, gt)
        loss.backward()
        torch.cuda.synchronize()
        return ([o.detach().clone() for o in out], loss.detach().clone(), [p.grad.clone() for p in m.parameters()],
                [b.clone() for b in m.buffers()])

    a, b = eager(), eager()
    for u, v in zip(a[0] + [a[1]] + a[2] + a[3], b[0] + [b[1]] + b[2] + b[3]):
        assert torch.equal(u, v)

    step = GraphedTrainStep(m, loss_fn, ((x, focal), (gt,)))
    m.load_state_dict(state)
    loss = step((x, focal), (gt,))
    torch.cuda.synchronize()
    assert torch.equal(loss, a[1])
    for p, want in zip(m.parameters(), a[2]):
        assert torch.equal(p.grad, want)
