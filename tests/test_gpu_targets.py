"""GPU parity tests of the anchor target assignment kernel (targets.cu, SURVEY.md section 8f row 2) through the C ABI:
against the fixtures produced by the reference's own odtk.box.snap_to_anchors on CPU (tests/golden/snap.npz) and
against the numpy oracle on larger seeded cases.  Bars: depth, one-hot classes and class indices bit-exact (IoU in fp32
with the reference's operation order, IEEE division, no FMA contraction); box deltas within 1e-5 (logf vs torch.log)."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from retinanet_examples_b200 import box, loss as loss_mod

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def test_snap_to_anchors_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "snap.npz"))
    for k in range(int(g["ncases"])):
        boxes, size, stride = g["c%d_boxes" % k], g["c%d_size" % k].tolist(), int(g["c%d_stride" % k])
        anchors, ncls = torch.from_numpy(g["c%d_anchors" % k]), int(g["c%d_classes" % k])
        ct, bt, dp = box.snap_to_anchors(torch.from_numpy(boxes), size, stride, anchors, ncls, DEV, [0.4, 0.5])
        np.testing.assert_array_equal(dp.cpu().numpy(), g["c%d_depth" % k])
        np.testing.assert_array_equal(ct.cpu().numpy().astype(np.uint8), g["c%d_cls_target" % k])
        np.testing.assert_allclose(bt.cpu().numpy(), g["c%d_box_target" % k], rtol=1e-5, atol=1e-5)


def _random_targets(rng, batch, g, w, h, stride, ncls, pad_frac):
    wh = rng.uniform(0.5 * stride, 14.0 * stride, size=(batch, g, 2))
    xy = rng.uniform(-stride, [w * stride, h * stride], size=(batch, g, 2)) - wh / 4
    cls = rng.integers(0, ncls, size=(batch, g, 1)).astype(np.float64)
    cls[rng.uniform(size=(batch, g, 1)) < pad_frac] = -1          # padding rows, interleaved
    return np.concatenate([np.round(xy), np.round(wh) + 1, cls], 2).astype(np.float32)


@pytest.mark.parametrize("batch,g,w,h,stride,ncls", [(3, 40, 40, 25, 32, 80), (2, 300, 20, 13, 64, 5), (4, 64, 160, 100, 8, 80),
                                                     (2, 1, 10, 7, 128, 3)])
def test_snap_to_anchors_batched_matches_oracle(batch, g, w, h, stride, ncls):
    """Whole batch in one launch, padding rows (class -1) skipped on the device, > 256 boxes (two staging passes)."""
    rng = np.random.default_rng(w * 1000 + g)
    t = _random_targets(rng, batch, g, w, h, stride, ncls, 0.3)
    t[-1, :, 4] = -1 if batch > 2 else t[-1, :, 4]                 # one image without any valid box
    anchors = box.generate_anchors(stride, [1.0, 2.0, 0.5], [4 * 2 ** (i / 3) for i in range(3)])
    ct, bt, dp, ci = box.snap_to_anchors_batch(torch.from_numpy(t).to(DEV), (h, w), stride, anchors, ncls, [0.4, 0.5])
    _, _, dp2, ci2 = box.snap_to_anchors_batch(torch.from_numpy(t).to(DEV), (h, w), stride, anchors, ncls, [0.4, 0.5], dense=False)
    assert torch.equal(dp, dp2) and torch.equal(ci, ci2)
    for b in range(batch):
        oct_, obt, odp, oci = oracle.snap_to_anchors(t[b], [w * stride, h * stride], stride, anchors.numpy(), ncls, [0.4, 0.5])
        np.testing.assert_array_equal(dp[b].cpu().numpy(), odp)
        np.testing.assert_array_equal(ci[b].cpu().numpy(), oci)
        np.testing.assert_array_equal(ct[b].cpu().numpy(), oct_)
        np.testing.assert_allclose(bt[b].cpu().numpy(), obt, rtol=1e-5, atol=1e-5)
    if g >= 40:
        assert int((dp > 0).sum()) > 0          # the case is not vacuous: some anchors are foreground


def test_class_index_targets_feed_the_focal_loss():
    """Model._compute_loss (odtk/model.py:192-199): focal loss of the class head against the dense one-hot with the
    (depth >= 0) mask == the same kernel fed with the class-index targets (no one-hot, no mask tensor)."""
    rng = np.random.default_rng(5)
    batch, g, w, h, stride, ncls = 2, 30, 40, 25, 32, 20
    t = torch.from_numpy(_random_targets(rng, batch, g, w, h, stride, ncls, 0.2)).to(DEV)
    anchors = box.generate_anchors(stride, [1.0, 2.0, 0.5], [4 * 2 ** (i / 3) for i in range(3)])
    ct, _, dp, ci = box.snap_to_anchors_batch(t, (h, w), stride, anchors, ncls, [0.4, 0.5])
    logits = torch.randn((batch, 9, ncls, h, w), generator=torch.Generator().manual_seed(1)).to(DEV) * 2 - 3
    mask = (dp >= 0).expand_as(ct).float().contiguous()
    dense = loss_mod.focal_loss_sum(logits, ct, mask)
    indexed = loss_mod.focal_loss_sum(logits.reshape(batch * 9, ncls, h * w), cls_index=ci.reshape(batch * 9, h * w))
    np.testing.assert_allclose(float(indexed), float(dense), rtol=1e-5)


# ---- rotated target assignment: odtk_iou / _C.iou / box.snap_to_anchors_rotated (SURVEY.md section 8f row 2) ----------
def test_iou_matches_oracle_and_golden(golden_dir):
    """_C.iou (odtk_iou) == oracle_iou bit for bit on the committed quads (IEEE, no FMA contraction on both sides)."""
    from retinanet_examples_b200 import _C
    g = np.load(os.path.join(golden_dir, "snap_rotated.npz"))
    b, a = torch.from_numpy(g["iou_boxes"]).to(DEV), torch.from_numpy(g["iou_anchors"]).to(DEV)
    out = _C.iou(b.view(-1), a.view(-1))[0]
    assert tuple(out.shape) == (a.shape[0], b.shape[0])
    np.testing.assert_array_equal(out.cpu().numpy(), g["iou"])
    # larger seeded case: rotated rectangles (convex), > 64 boxes (two staging passes), 20 000 anchors
    rng = np.random.default_rng(3)

    def rects(n):
        c, wh, th = rng.uniform(0, 300, (n, 1, 2)), rng.uniform(4, 120, (n, 2)), rng.uniform(-1.2, 1.2, n)
        base = np.stack([np.stack([-wh[:, 0], -wh[:, 1]], 1), np.stack([wh[:, 0], -wh[:, 1]], 1),
                         np.stack([wh[:, 0], wh[:, 1]], 1), np.stack([-wh[:, 0], wh[:, 1]], 1)], 1) / 2
        R = np.stack([np.stack([np.cos(th), -np.sin(th)], 1), np.stack([np.sin(th), np.cos(th)], 1)], 1)
        return (np.einsum("nij,nkj->nki", R, base) + c).reshape(n, 8).astype(np.float32)
    bq, aq = rects(70), rects(20000)
    aq[:70] = bq                                                   # identical quads: the 0.001 jitter path
    out = _C.iou(torch.from_numpy(bq).to(DEV), torch.from_numpy(aq).to(DEV))[0].cpu().numpy()
    ref = oracle.iou(bq, aq)
    np.testing.assert_array_equal(out, ref)
    assert 0.9 < out[np.arange(70), np.arange(70)].min() and out.max() <= 1.01


def test_iou_matches_reference_cuda_kernel(golden_dir):
    """The reference's own iou_cuda_kernel (nms_iou.cu:324-387, compiled unmodified, --use_fast_math; its output is stored in
    tests/golden/refcuda.npz by oracle/gen_golden_refcuda.py) on the same quads: same [num_anchors, num_boxes] orientation
    (the swapped-argument quirk) and values within fast-math slack."""
    from oracle import gen_golden_refcuda as refcuda
    from retinanet_examples_b200 import _C
    ref = np.load(os.path.join(golden_dir, "refcuda.npz"))["iou"]
    b, a = refcuda.iou_case()
    mine = _C.iou(torch.from_numpy(b).to(DEV), torch.from_numpy(a).to(DEV))[0]
    assert tuple(mine.shape) == ref.shape
    np.testing.assert_allclose(mine.cpu().numpy(), ref, rtol=2e-3, atol=2e-4)
    assert float(mine.max()) > 0.1


def test_snap_to_anchors_rotated_matches_reference_golden(golden_dir):
    """box.snap_to_anchors_rotated on the GPU against the fixtures the unmodified reference function produced."""
    g = np.load(os.path.join(golden_dir, "snap_rotated.npz"))
    for k in range(int(g["ncases"])):
        boxes, size, stride = g["c%d_boxes" % k], g["c%d_size" % k].tolist(), int(g["c%d_stride" % k])
        anchors = (torch.from_numpy(g["c%d_anchors_axis" % k]), torch.from_numpy(g["c%d_anchors_rot" % k]))
        ct, bt, dp = box.snap_to_anchors_rotated(torch.from_numpy(boxes), size, stride, anchors, int(g["c%d_classes" % k]), DEV,
                                                 [0.4, 0.5])
        gd = g["c%d_depth" % k]
        # rotate_boxes runs torch sin/cos on the device: corners may differ from the CPU fixture in the last ulp, which can
        # flip an assignment that sits exactly on a threshold -- allow a handful out of thousands, the rest identical
        same = (dp.cpu().numpy() == gd)
        assert same.mean() > 0.998, same.mean()
        m = same[:, 0]
        np.testing.assert_array_equal(ct.cpu().numpy().astype(np.uint8)[m[:, None].repeat(ct.shape[1], 1)],
                                      g["c%d_cls_target" % k][m[:, None].repeat(ct.shape[1], 1)])
        fg = (gd[:, 0] > 0) & m
        np.testing.assert_allclose(bt.cpu().numpy().transpose(0, 2, 3, 1)[fg], g["c%d_box_target" % k].transpose(0, 2, 3, 1)[fg],
                                   rtol=1e-4, atol=1e-4)
