"""CPU tests: oracle/model_ref.py (the torch-CPU restatement of the reference Model) against the
golden head outputs produced by the UNMODIFIED reference Model (tests/golden/model_*.npz), and the
state_dict layout of the product against the reference's."""
import os

import numpy as np
import pytest
import torch

from oracle import model_ref
from retinanet_examples_b200.model import conv_specs, make_state_dict


@pytest.mark.parametrize("backbone", ["ResNet18FPN", "ResNet50FPN", "ResNeXt50_32x4dFPN", "MobileNetV2FPN"])
def test_model_ref_matches_reference_golden(golden_dir, backbone):
    g = np.load(os.path.join(golden_dir, "model_%s.npz" % backbone))
    sd = make_state_dict(backbone, int(g["classes"]), 9, False, int(g["seed"]))
    cls, box = model_ref.forward_heads(sd, backbone, torch.from_numpy(g["x"]))
    for i in range(5):
        np.testing.assert_allclose(cls[i].numpy(), g["cls%d" % i], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(box[i].numpy(), g["box%d" % i], rtol=1e-4, atol=1e-5)


def test_state_dict_layout_and_flop_count():
    specs = conv_specs("ResNet50FPN", 80, 9, False)
    convs = [s for s in specs if s[1].startswith("conv")]
    # SURVEY.md App. A counts conv CALLS (111 / 162 / 78): the 10 head convs run on 5 levels
    assert len(convs) - 10 + 50 == 111
    assert len([s for s in conv_specs("ResNet101FPN") if s[1].startswith("conv")]) - 10 + 50 == 162
    assert len([s for s in conv_specs("ResNet18FPN") if s[1].startswith("conv")]) - 10 + 50 == 78
    sd = make_state_dict("ResNet18FPN", 3, 9, False, 0)
    assert sd["cls_head.8.weight"].shape == (27, 256, 3, 3) and sd["box_head.8.weight"].shape == (36, 256, 3, 3)
    assert abs(float(sd["cls_head.8.bias"][0]) + np.log(99)) < 1e-5   # prior of odtk/model.py:115-118
    sdr = make_state_dict("ResNet50FPN", 80, 27, True, 0)
    assert sdr["cls_head.8.weight"].shape[0] == 2160 and sdr["box_head.8.weight"].shape[0] == 162


def test_model_ref_against_live_reference(golden_dir):
    """A second ResNet18FPN case (4 classes, another seed and input size): the unmodified reference Model's head outputs,
    stored in tests/golden/model_ResNet18FPN_seed77.npz by oracle/gen_golden.py."""
    g = np.load(os.path.join(golden_dir, "model_ResNet18FPN_seed77.npz"))
    x = torch.from_numpy(g["x"])
    assert torch.equal(x, torch.randn((1, 3, 128, 128), generator=torch.Generator().manual_seed(5)))
    mc, mb = model_ref.forward_heads(make_state_dict("ResNet18FPN", int(g["classes"]), 9, False, int(g["seed"])), "ResNet18FPN", x)
    for i in range(5):
        np.testing.assert_allclose(mc[i].numpy(), g["cls%d" % i], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(mb[i].numpy(), g["box%d" % i], rtol=1e-4, atol=1e-5)
