"""Golden vectors for the convolution stack: the UNMODIFIED reference Model (imported from
/root/reference) loaded with the deterministic synthetic state_dict of
retinanet_examples_b200.model.make_state_dict, run on a small seeded input.  TEST INFRASTRUCTURE ONLY.
Called by oracle/gen_golden.py ("model")."""
import os

import numpy as np
import torch

from retinanet_examples_b200.model import make_state_dict

CASES = [("ResNet18FPN", 3, 11, (1, 3, 128, 256)), ("ResNet50FPN", 3, 12, (1, 3, 128, 128)),
         ("ResNeXt50_32x4dFPN", 3, 13, (1, 3, 128, 128)),      # grouped 3x3 bottlenecks (torchvision groups=32)
         ("MobileNetV2FPN", 3, 14, (1, 3, 128, 128))]          # inverted residuals: depthwise 3x3, ReLU6 (odtk/backbones/mobilenet.py)


def reference_heads(odtk, backbone, classes, seed, x):
    m = odtk.model.Model(backbone, classes=classes)
    sd = make_state_dict(backbone, classes, 9, False, seed)
    full = m.state_dict()
    # (.fc. / features.18 / classifier: the classification tails the reference keeps in its state_dict but never runs)
    missing = [k for k in full if k not in sd and "num_batches_tracked" not in k and ".fc." not in k and
               ".features.18." not in k and ".classifier." not in k]
    assert not missing, missing[:5]
    full.update(sd)
    m.load_state_dict(full)
    m.eval()
    m.exporting = True
    with torch.no_grad():
        cls, box = m(x)
    return cls, box, m


def save(odtk, path, backbone, classes, seed, x):
    cls, box, m = reference_heads(odtk, backbone, classes, seed, x)
    d = {"x": x.numpy(), "classes": np.int32(classes), "seed": np.int32(seed)}
    for i, (c, b) in enumerate(zip(cls, box)):
        d["cls%d" % i] = c.numpy()
        d["box%d" % i] = b.numpy()
    np.savez_compressed(path, **d)


def main(odtk, out_dir):
    for backbone, classes, seed, shape in CASES:
        g = torch.Generator().manual_seed(seed)
        save(odtk, os.path.join(out_dir, "model_%s.npz" % backbone), backbone, classes, seed, torch.randn(shape, generator=g))
