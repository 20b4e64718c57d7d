"""CPU tests of the MobileNetV2 encoder's module surface: every InvertedResidual / Conv2dNormActivation is re-classed onto
the native units, every depthwise conv is a Conv2dTC, and the state_dict keys and shapes are the reference's."""
import types

import torch.nn as nn

import bts
from bts_b200 import glue, model


def _model():
    p = types.SimpleNamespace(encoder="mobilenetv2_bts", max_depth=10.0, dataset="nyu", bts_size=512, pretrained=False)
    return bts.BtsModel(p)


def test_mobilenet_blocks_are_reclassed():
    from torchvision.models.mobilenetv2 import InvertedResidual
    from torchvision.ops.misc import Conv2dNormActivation
    m = _model()
    blocks = [x for x in m.encoder.modules() if isinstance(x, InvertedResidual)]
    cnas = [x for x in m.encoder.modules() if isinstance(x, Conv2dNormActivation)]
    assert len(blocks) == 17 and len(cnas) == 2 + 17 + 16          # stem + last, one dw per block, 16 expand layers
    assert all(type(x).__name__ == "InvertedResidualTC" and x._parts() is not None for x in blocks)
    assert all(type(x).__name__ == "ConvBnReLU6TC" for x in cnas)
    ir, ir_tc, cna, cna_tc = model._mobilenet_classes()
    assert not any(type(x) in (ir, cna, nn.Conv2d) for x in m.encoder.modules())


def test_mobilenet_depthwise_convs_are_native():
    m = _model()
    dws = [x for x in m.encoder.modules() if isinstance(x, nn.Conv2d) and x.groups > 1]
    assert len(dws) == 17
    assert all(type(x) is model.Conv2dTC and glue.dw_eligible(x) for x in dws)
    assert sorted({(x.in_channels, x.stride[0]) for x in dws}) == [
        (32, 1), (96, 2), (144, 1), (144, 2), (192, 1), (192, 2), (384, 1), (576, 1), (576, 2), (960, 1)]


def test_mobilenet_state_dict_matches_reference_keys(golden):
    g = golden("model_mobilenetv2_bts")
    got = sorted("%s:%s" % (k, "x".join(map(str, v.shape))) for k, v in _model().state_dict().items())
    assert got == g["keys"].tolist()
