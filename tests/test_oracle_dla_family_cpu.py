"""The DLA family beyond DLA-34 (dla.py:316-372: DLA-46-C / 60 / 102 / 169 -- bottleneck blocks, trees up to five levels deep,
residual roots): the oracle's functional restatement against the reference's own ``dla.py`` modules, and the synthetic weight
layout against the reference's state-dict keys.  The reference's keys and a fixed sample of its outputs on seeded weights are
stored in tests/golden/reference_modules.pt.gz (tests/golden/make_reference_golden.py)."""
import pytest
import torch

from helpers import load_golden

ARCHS = ["DLA-34-FPN", "DLA-46-C-FPN", "DLA-60-FPN", "DLA-102-FPN", "DLA-169-FPN"]


NO_DCN = (False,) * 6
DCN_345 = (False, False, False, True, True, True)      # the reference's "-DCN" models deform levels 3..5 (readme/model_zoo.md:54-55)
CASES = [(a, NO_DCN) for a in ARCHS] + [("DLA-60-FPN", DCN_345), ("DLA-102-FPN", DCN_345), ("DLA-34-FPN", DCN_345)]


def seeded_weights(keys):
    """Non-trivial FrozenBN buffers and weights for the (name, shape) list, in its order, and the 1x3x64x96 input."""
    g = torch.Generator().manual_seed(1)
    sd = {}
    for k, shape in keys:
        if k.endswith("running_var"):
            v = 1.0 + 0.1 * torch.rand(shape, generator=g)
        elif len(shape) == 1:
            v = torch.randn(shape, generator=g) * 0.1 + (1.0 if k.endswith("weight") else 0.0)
        else:
            v = torch.randn(shape, generator=g) * (2.0 / (shape[1] * shape[2] * shape[3])) ** 0.5
        sd[k] = v
    return sd, torch.randn(1, 3, 64, 96, generator=g)


def test_deform_conv_restatement_matches_torchvision():
    """oracle.deform_conv3x3 (written out from the published DCN v1 operator) against torchvision.ops.deform_conv2d."""
    from torchvision.ops import deform_conv2d
    from oracle import siammot_oracle as orc
    g = torch.Generator().manual_seed(0)
    for stride, (H, W), C in ((1, (19, 23), 24), (2, (20, 26), 16), (1, (5, 4), 8)):
        x = torch.randn(1, C, H, W, generator=g)
        w = torch.randn(C + 3, C, 3, 3, generator=g)
        OH, OW = (H - 1) // stride + 1, (W - 1) // stride + 1
        off = torch.randn(1, 18, OH, OW, generator=g) * 2.5      # many samples land outside the map
        ref = deform_conv2d(x, off, w, None, stride=stride, padding=1)
        got = orc.deform_conv3x3(x, off, w, stride)
        assert got.shape == ref.shape and float((got - ref).abs().max()) <= 1e-4 * float(ref.abs().max())


@pytest.mark.parametrize("arch,dcn", CASES)
def test_oracle_dla_family_matches_the_reference_modules(arch, dcn):
    from oracle import siammot_oracle as orc
    from siammot_b200.synthetic import dla_layout
    gold = load_golden("reference_modules")["dla"][(arch, dcn)]
    # the synthetic layout lists exactly the reference's parameter groups, in its module order, with its shapes
    keys = []
    for kind, name, shape in dla_layout(arch, dcn):
        if kind == "conv":
            keys.append((name + ".weight", tuple(shape)))
        elif kind == "convb":
            keys += [(name + ".weight", tuple(shape)), (name + ".bias", (shape[0],))]
        else:
            keys += [(name + "." + f, (shape,)) for f in ("weight", "bias", "running_mean", "running_var")]
    assert keys == gold["keys"]
    sd, x = seeded_weights(gold["keys"])
    with torch.no_grad():
        got = orc.dla_forward({"backbone.body." + k: v for k, v in sd.items()}, x, arch)
    assert len(got) == len(gold["maps"]) == 4
    for a, b in zip(got, gold["maps"]):
        assert tuple(a.shape) == b["shape"]
        a = a.reshape(-1)[b["idx"].long()]
        if any(dcn) and arch != "DLA-34-FPN":          # the deformable conv is summed in another order than torchvision's
            assert float((a - b["val"]).abs().max()) <= 1e-4 * float(b["val"].abs().max())
        else:
            assert torch.equal(a, b["val"])
