"""The ResNet-50 body is upstream maskrcnn_benchmark code the reference does not vendor: it is restated twice (nn.Module form
in oracle/shim for the golden generator, functional form in oracle/siammot_oracle.py).  This pins both restatements to an
independent implementation -- torchvision's ResNet-50 with the stage strides moved from the 3x3 to the first 1x1 (the Detectron
STRIDE_IN_1X1 convention) and BatchNorm in eval mode with a vanishing eps (FrozenBatchNorm2d has none) -- on the same weights."""
import os
import sys

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torchvision_twin(sd):
    tv = pytest.importorskip("torchvision")
    net = tv.models.resnet50(weights=None).eval()
    for li in (2, 3, 4):
        blk = getattr(net, "layer%d" % li)[0]
        blk.conv1.stride, blk.conv2.stride = (2, 2), (1, 1)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eps = 1e-12   # torch refuses 0; against running_var >= 1 this is below fp32 resolution
    mapped = {}
    for k, v in sd.items():
        if not k.startswith("backbone.body."):
            continue
        k = k[len("backbone.body."):]
        if k.startswith("stem."):
            k = k[len("stem."):]
        mapped[k] = v
    missing, unexpected = net.load_state_dict(mapped, strict=False)
    assert not unexpected, unexpected
    assert all(m.startswith("fc.") or m.endswith("num_batches_tracked") for m in missing), missing

    def body(x):
        x = net.maxpool(net.relu(net.bn1(net.conv1(x))))
        outs = []
        for li in (1, 2, 3, 4):
            x = getattr(net, "layer%d" % li)(x)
            outs.append(x)
        return outs
    return body


def _cfg_and_weights():
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from helpers import scenario_inputs
    cfg, sd, clip = scenario_inputs("emm_r50_192x320")
    return cfg, sd, clip


def test_oracle_resnet50_matches_torchvision_with_strides_on_the_1x1():
    from oracle import siammot_oracle as orc
    cfg, sd, clip = _cfg_and_weights()
    x = clip[0][None]
    with torch.no_grad():
        ref = _torchvision_twin(sd)(x)
        got = orc.resnet50_forward({k: v.float() for k, v in sd.items()}, x)
    assert [tuple(t.shape) for t in got] == [(1, 256, 48, 80), (1, 512, 24, 40), (1, 1024, 12, 20), (1, 2048, 6, 10)]
    for a, b in zip(got, ref):
        assert float((a - b).abs().max()) <= 1e-4 * float(b.abs().max())


def test_shim_resnet50_matches_oracle():
    """The nn.Module restatement the golden generator runs the reference on == the functional restatement that travels."""
    from oracle import reference_loader
    from oracle import siammot_oracle as orc
    cfg, sd, clip = _cfg_and_weights()
    reference_loader.use_shim()
    from maskrcnn_benchmark.config import cfg as ucfg
    from maskrcnn_benchmark.modeling.backbone import resnet
    c = ucfg.clone()
    c.MODEL.BACKBONE.CONV_BODY = "R-50-FPN"
    net = resnet.ResNet(c).eval()
    body = {k[len("backbone.body."):]: v for k, v in sd.items() if k.startswith("backbone.body.")}
    net.load_state_dict(body, strict=True)
    x = clip[1][None]
    with torch.no_grad():
        ref = net(x)
        got = orc.resnet50_forward({k: v.float() for k, v in sd.items()}, x)
    for a, b in zip(got, ref):
        assert torch.equal(a, b)
