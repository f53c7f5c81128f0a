"""Generate tests/golden/*.npz by running the REFERENCE's own Python (imported unmodified from
/root/reference, see oracle/ref_import.py) on small seeded inputs.  TEST INFRASTRUCTURE ONLY.

Run in the build container (the reference cannot travel to the GPU box):
    python oracle/gen_golden.py
The committed fixtures pin oracle/odtk_oracle.c, oracle/model_ref.py and the product's host code.

What each fixture is (reference function -> file):
  anchors.npz      odtk.box.generate_anchors / generate_anchors_rotated for strides 8..128, plus
                   the hard-coded tables of extras/cppapi/export.cpp:69-85 parsed from the source
  nms.npz          odtk.box.nms CPU path (odtk/box.py:319-367), unmodified
  nms_uniform.npz  the same on boxes scattered uniformly over the image (3 trials, 300 boxes, 3 classes)
  decode.npz       odtk.box.decode CPU path (odtk/box.py:266-309) with '/' -> '//' on the three
                   index divisions that crash on torch >= 1.6 (ref_import.patched_cpu_decode)
  focal.npz        odtk.loss.FocalLoss forward + autograd backward (odtk/loss.py:13-18)
  snap.npz         odtk.box.snap_to_anchors (odtk/box.py:134-186), unmodified, CPU
  model_*.npz      odtk.model.Model forward (exporting=True head outputs, and the full inference
                   branch with the patched CPU decode + unmodified CPU nms)
  model_ResNet18FPN_seed77.npz   one more ResNet18FPN head case (4 classes, state_dict seed 77, 128 x 128)
"""
import math
import os
import re
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def gen_anchors(odtk):
    ratios, scales = [1.0, 2.0, 0.5], [4 * 2 ** (i / 3) for i in range(3)]
    d = {}
    for s in (8, 16, 32, 64, 128):
        d["axis_%d" % s] = odtk.box.generate_anchors(s, ratios, scales).numpy()
    # rotated config of extras/cppapi/generate_anchors.py
    rr, rs = [0.25, 0.5, 1.0, 2.0, 4.0], [2 * 2 ** (2 * i / 3) for i in range(3)]
    ra = [-math.pi / 6, 0, math.pi / 6]
    for s in (8, 16, 32, 64, 128):
        ax, rot = odtk.box.generate_anchors_rotated(s, rr, rs, ra)
        d["rot_axis_%d" % s] = ax.numpy()
        d["rot_corners_%d" % s] = rot.numpy()
    # default rotated model config (odtk/model.py:44-45)
    for s in (8, 16, 32, 64, 128):
        ax, rot = odtk.box.generate_anchors_rotated(s, ratios, scales, ra)
        d["rotdef_axis_%d" % s] = ax.numpy()
        d["rotdef_corners_%d" % s] = rot.numpy()
    # known-answer tables hard-coded in the reference's C++ sample
    src = open(os.path.join(ref_import.REF_ROOT, "extras/cppapi/export.cpp")).read()
    rows = re.findall(r"^\s*\{(-?[0-9][^{}]*)\},?\s*$", src, flags=re.M)
    tables = [np.array([float(v) for v in r.split(",")], dtype=np.float32) for r in rows]
    assert len(tables) == 10, len(tables)
    for i, s in enumerate((8, 16, 32, 64, 128)):
        d["cpp_axis_%d" % s] = tables[i]
        d["cpp_rot_%d" % s] = tables[5 + i]
    np.savez_compressed(os.path.join(OUT, "anchors.npz"), **d)


def synth_nms_case(rng, batch, n, ncls, zero_frac, cluster):
    """Boxes clustered around a few centres so that suppression really happens."""
    ctr = rng.uniform(50, 600, size=(batch, cluster, 2)).astype(np.float32)
    which = rng.integers(0, cluster, size=(batch, n))
    c = np.take_along_axis(ctr, which[..., None].repeat(2, -1), axis=1) + rng.normal(0, 12, (batch, n, 2))
    wh = rng.uniform(20, 120, size=(batch, n, 2))
    boxes = np.concatenate([c - wh / 2, c + wh / 2], -1).astype(np.float32)
    scores = rng.uniform(0.05, 1.0, size=(batch, n)).astype(np.float32)
    scores[rng.uniform(size=(batch, n)) < zero_frac] = 0.0
    classes = rng.integers(0, ncls, size=(batch, n)).astype(np.float32)
    return scores, boxes, classes


def gen_nms(odtk):
    rng = np.random.default_rng(1234)
    d = {}
    cases = [(2, 400, 3, 0.1, 6, 0.5, 100), (1, 1500, 5, 0.3, 12, 0.5, 100), (3, 64, 2, 0.0, 2, 0.3, 16),
             (1, 300, 1, 0.2, 3, 0.7, 300)]
    for k, (b, n, ncls, zf, cl, thr, det) in enumerate(cases):
        s, bx, c = synth_nms_case(rng, b, n, ncls, zf, cl)
        os_, ob, oc = odtk.box.nms(torch.from_numpy(s), torch.from_numpy(bx), torch.from_numpy(c), thr, det)
        d.update({"c%d_scores" % k: s, "c%d_boxes" % k: bx, "c%d_classes" % k: c,
                  "c%d_thr" % k: np.float32(thr), "c%d_det" % k: np.int32(det),
                  "c%d_out_scores" % k: os_.numpy(), "c%d_out_boxes" % k: ob.numpy(),
                  "c%d_out_classes" % k: oc.numpy()})
    d["ncases"] = np.int32(len(cases))
    np.savez_compressed(os.path.join(OUT, "nms.npz"), **d)


def gen_nms_uniform(odtk):
    rng = np.random.default_rng(7)
    d = {}
    for k in range(3):
        n = 300
        ctr = rng.uniform(0, 300, (1, n, 2))
        wh = rng.uniform(20, 100, (1, n, 2))
        b = np.concatenate([ctr - wh / 2, ctr + wh / 2], -1).astype(np.float32)
        s = rng.uniform(0.01, 1, (1, n)).astype(np.float32)
        c = rng.integers(0, 3, (1, n)).astype(np.float32)
        os_, ob, oc = odtk.box.nms(torch.from_numpy(s), torch.from_numpy(b), torch.from_numpy(c), 0.5, 100)
        d.update({"c%d_scores" % k: s, "c%d_boxes" % k: b, "c%d_classes" % k: c, "c%d_out_scores" % k: os_.numpy(),
                  "c%d_out_boxes" % k: ob.numpy(), "c%d_out_classes" % k: oc.numpy()})
    d["ncases"] = np.int32(3)
    np.savez_compressed(os.path.join(OUT, "nms_uniform.npz"), **d)


def gen_decode(odtk):
    dec = ref_import.patched_cpu_decode()
    rng = np.random.default_rng(4321)
    ratios, scales = [1.0, 2.0, 0.5], [4 * 2 ** (i / 3) for i in range(3)]
    d = {}
    # (B, C, H, W, stride, top_n, mean logit)  -> count > top_n and count < top_n cases
    cases = [(2, 4, 10, 16, 8, 50, -2.0), (1, 3, 7, 10, 128, 100, -4.0), (2, 5, 13, 20, 64, 1000, -1.0)]
    for k, (b, c, h, w, stride, top_n, mu) in enumerate(cases):
        anchors = odtk.box.generate_anchors(stride, ratios, scales)
        a = anchors.shape[0]
        cls = 1 / (1 + np.exp(-rng.normal(mu, 1.6, size=(b, a * c, h, w)))).astype(np.float32)
        box = rng.normal(0, 0.2, size=(b, a * 4, h, w)).astype(np.float32)
        os_, ob, oc = dec(torch.from_numpy(cls), torch.from_numpy(box), stride, 0.05, top_n, anchors)
        d.update({"c%d_cls" % k: cls, "c%d_box" % k: box, "c%d_anchors" % k: anchors.numpy(),
                  "c%d_stride" % k: np.int32(stride), "c%d_top_n" % k: np.int32(top_n),
                  "c%d_out_scores" % k: os_.numpy(), "c%d_out_boxes" % k: ob.numpy(),
                  "c%d_out_classes" % k: oc.numpy()})
    d["ncases"] = np.int32(len(cases))
    np.savez_compressed(os.path.join(OUT, "decode.npz"), **d)


def gen_focal(odtk):
    rng = np.random.default_rng(99)
    x = rng.normal(-2.0, 3.0, size=(2, 9, 5, 6, 7)).astype(np.float32)
    t = (rng.uniform(size=x.shape) < 0.05).astype(np.float32)
    xt = torch.from_numpy(x).requires_grad_(True)
    loss = odtk.loss.FocalLoss()(xt, torch.from_numpy(t))
    loss.sum().backward()
    np.savez_compressed(os.path.join(OUT, "focal.npz"), x=x, t=t, loss=loss.detach().numpy(),
                        grad=xt.grad.numpy())


def gen_snap(odtk):
    """odtk.box.snap_to_anchors (odtk/box.py:134-186), unmodified, on CPU: seeded ground-truth boxes over small
    grids, incl. an image without boxes and boxes that exactly tile anchors (IoU ties / thresholds)."""
    rng = np.random.default_rng(77)
    ratios, scales = [1.0, 2.0, 0.5], [4 * 2 ** (i / 3) for i in range(3)]
    d = {}
    cases = [(12, 9, 8, 7, 5), (10, 16, 16, 12, 3), (5, 4, 32, 0, 4), (7, 6, 64, 300, 6), (16, 10, 8, 20, 80)]   # W, H, stride, #gt, classes
    for k, (w, h, stride, g, ncls) in enumerate(cases):
        anchors = odtk.box.generate_anchors(stride, ratios, scales)
        size = [w * stride, h * stride]
        if g:
            wh = rng.uniform(0.5 * stride, 12.0 * stride, size=(g, 2))
            xy = rng.uniform(-stride, [size[0], size[1]], size=(g, 2)) - wh / 4
            cls = rng.integers(0, ncls, size=(g, 1))
            boxes = np.concatenate([np.round(xy), np.round(wh) + 1, cls], 1).astype(np.float32)
            if g >= 5:      # boxes coinciding with anchors of some cells -> IoU exactly 1 and exact ties
                a = anchors.numpy()
                for j in range(3):
                    cx, cy = int(rng.integers(0, w)) * stride, int(rng.integers(0, h)) * stride
                    an = a[int(rng.integers(0, a.shape[0]))]
                    boxes[j, :4] = [cx + an[0], cy + an[1], an[2] - an[0] + 1, an[3] - an[1] + 1]
                boxes[4] = boxes[3]          # duplicate row: first maximum must win
                boxes[4, 4] = (boxes[3, 4] + 1) % ncls
        else:
            boxes = np.zeros((0, 5), np.float32)
        ct, bt, dp = odtk.box.snap_to_anchors(torch.from_numpy(boxes), size, stride, anchors, ncls, "cpu", [0.4, 0.5])
        d.update({"c%d_boxes" % k: boxes, "c%d_size" % k: np.int32(size), "c%d_stride" % k: np.int32(stride),
                  "c%d_anchors" % k: anchors.numpy(), "c%d_classes" % k: np.int32(ncls),
                  "c%d_cls_target" % k: ct.numpy().astype(np.uint8), "c%d_box_target" % k: bt.numpy(),
                  "c%d_depth" % k: dp.numpy()})
    d["ncases"] = np.int32(len(cases))
    np.savez_compressed(os.path.join(OUT, "snap.npz"), **d)


def main():
    os.makedirs(OUT, exist_ok=True)
    odtk = ref_import.import_reference()
    which = sys.argv[1:] or ["anchors", "nms", "nms_uniform", "decode", "focal", "snap", "model", "model_seed77"]
    if "anchors" in which: gen_anchors(odtk)
    if "nms" in which: gen_nms(odtk)
    if "nms_uniform" in which: gen_nms_uniform(odtk)
    if "decode" in which: gen_decode(odtk)
    if "focal" in which: gen_focal(odtk)
    if "snap" in which: gen_snap(odtk)
    if "model" in which:
        from oracle import gen_golden_model
        gen_golden_model.main(odtk, OUT)
    if "model_seed77" in which:
        from oracle import gen_golden_model
        x = torch.randn((1, 3, 128, 128), generator=torch.Generator().manual_seed(5))
        gen_golden_model.save(odtk, os.path.join(OUT, "model_ResNet18FPN_seed77.npz"), "ResNet18FPN", 4, 77, x)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def gen_l1_preproc(odtk):
    """SmoothL1Loss + autograd (odtk/loss.py:27-31) and the tensor maths of CocoDataset.__getitem__
    (odtk/data.py:113-123: float().div(255), per-channel sub_(mean).div_(std), F.pad to the stride) run
    verbatim on seeded inputs (the dataset class itself needs pycocotools + image files)."""
    import torch.nn.functional as F
    rng = np.random.default_rng(5)
    p = rng.normal(0, 0.3, size=(2, 36, 5, 7)).astype(np.float32)
    t = rng.normal(0, 0.3, size=p.shape).astype(np.float32)
    pt = torch.from_numpy(p).requires_grad_(True)
    loss = odtk.loss.SmoothL1Loss(beta=0.11)(pt, torch.from_numpy(t))
    loss.sum().backward()
    img = rng.integers(0, 256, size=(37, 53, 3), dtype=np.uint8)
    data = torch.from_numpy(img.copy()).float().div(255).permute(2, 0, 1).contiguous()
    for tt, mean, std in zip(data, [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]):
        tt.sub_(mean).div_(std)
    pw, ph = ((128 - d % 128) % 128 for d in (53, 37))
    data = F.pad(data, (0, pw, 0, ph))
    np.savez_compressed(os.path.join(OUT, "l1_preproc.npz"), p=p, t=t, loss=loss.detach().numpy(),
                        grad=pt.grad.numpy(), img=img, pre=data.numpy())


if __name__ == "__main__":
    main()
    if len(sys.argv) == 1 or "l1" in sys.argv[1:]:
        gen_l1_preproc(ref_import.import_reference())
