"""CPU tests: the oracle (oracle/odtk_oracle.c + oracle/oracle.py) against the fixtures generated
from the reference's own Python (tests/golden/, oracle/gen_golden.py) and the known-answer anchor
tables of extras/cppapi/export.cpp:69-85."""
import os

import numpy as np

from oracle import oracle

RATIOS, SCALES = oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def test_anchors_oracle_matches_reference_and_cpp_tables(golden_dir):
    g = _load(golden_dir, "anchors.npz")
    for s in (8, 16, 32, 64, 128):
        a = oracle.generate_anchors(s, RATIOS, SCALES)
        np.testing.assert_array_equal(a, g["axis_%d" % s])                      # bit-exact vs odtk.box
        np.testing.assert_allclose(np.round(a.reshape(-1), 2), g["cpp_axis_%d" % s], atol=6e-3)
        ax = oracle.generate_anchors_rotated_axis(s, [0.25, 0.5, 1.0, 2.0, 4.0],
                                                  [2 * 2 ** (2 * i / 3) for i in range(3)], oracle.DEFAULT_ANGLES)
        np.testing.assert_array_equal(ax, g["rot_axis_%d" % s])
        np.testing.assert_allclose(np.round(ax.reshape(-1), 2), g["cpp_rot_%d" % s], atol=6e-3)
        axd = oracle.generate_anchors_rotated_axis(s, RATIOS, SCALES, oracle.DEFAULT_ANGLES)
        np.testing.assert_array_equal(axd, g["rotdef_axis_%d" % s])


def test_nms_oracle_matches_reference_cpu_path(golden_dir):
    g = _load(golden_dir, "nms.npz")
    for k in range(int(g["ncases"])):
        s, b, c = g["c%d_scores" % k], g["c%d_boxes" % k], g["c%d_classes" % k]
        os_, ob, oc, oi = oracle.nms(s, b, c, float(g["c%d_thr" % k]), int(g["c%d_det" % k]), return_index=True)
        rs, rb, rc = g["c%d_out_scores" % k], g["c%d_out_boxes" % k], g["c%d_out_classes" % k]
        for img in range(s.shape[0]):
            keep = rs[img] > 0
            nk = int(keep.sum())
            assert nk > 0
            # CUDA semantics emit suppressed (score 0) entries after the kept ones; the reference's
            # CPU path leaves zeros there (SURVEY.md App. B5): compare the kept prefix exactly.
            assert int((os_[img] > 0).sum()) == nk
            np.testing.assert_array_equal(os_[img][:nk], rs[img][:nk])
            np.testing.assert_array_equal(ob[img][:nk], rb[img][:nk])
            np.testing.assert_array_equal(oc[img][:nk], rc[img][:nk])
            np.testing.assert_array_equal(s[img][oi[img][:nk]], rs[img][:nk])   # kept indices are consistent


def test_nms_oracle_tail_semantics():
    # 3 boxes, the 2nd suppressed by the 1st: output = kept(0, 2) then suppressed(1) with score 0
    s = np.array([[0.9, 0.8, 0.7]], np.float32)
    b = np.array([[[0, 0, 10, 10], [1, 1, 11, 11], [50, 50, 60, 60]]], np.float32)
    c = np.zeros((1, 3), np.float32)
    os_, ob, oc, oi = oracle.nms(s, b, c, 0.5, 4, return_index=True)
    np.testing.assert_array_equal(oi[0], [0, 2, 1, -1])
    np.testing.assert_array_equal(os_[0], np.array([0.9, 0.7, 0.0, 0.0], np.float32))
    np.testing.assert_array_equal(ob[0][2], [1, 1, 11, 11])


def test_decode_oracle_matches_reference_cpu_path(golden_dir):
    g = _load(golden_dir, "decode.npz")
    for k in range(int(g["ncases"])):
        cls, box, anchors = g["c%d_cls" % k], g["c%d_box" % k], g["c%d_anchors" % k]
        top_n, stride = int(g["c%d_top_n" % k]), int(g["c%d_stride" % k])
        os_, ob, oc = oracle.decode(cls, box, anchors.reshape(-1), stride, 0.05, top_n)
        rs, rb, rc = g["c%d_out_scores" % k], g["c%d_out_boxes" % k], g["c%d_out_classes" % k]
        for img in range(cls.shape[0]):
            n = int((rs[img] > 0).sum())
            assert int((os_[img] > 0).sum()) == n
            # the reference's CPU path always top-k sorts; CUDA semantics keep index order when
            # count <= top_n (SURVEY.md App. B2): compare after a descending sort by score
            # (exact score ties are ordered by index in CUDA, arbitrarily by torch.topk: break them
            # by class and box so both sides agree when the SETS agree)
            o = np.lexsort((ob[img][:n, 1], ob[img][:n, 0], oc[img][:n], -os_[img][:n]))
            r = np.lexsort((rb[img][:n, 1], rb[img][:n, 0], rc[img][:n], -rs[img][:n]))
            np.testing.assert_array_equal(os_[img][:n][o], rs[img][:n][r])
            np.testing.assert_array_equal(oc[img][:n][o], rc[img][:n][r])
            # CUDA clamps only the low side of (x1,y1) and the high side of (x2,y2) (decode.cu:151-154);
            # the CPU path clamps all four both ways (box.py:105-111, App. B3): apply the CPU clamp
            H, W = cls.shape[2], cls.shape[3]
            hi = np.array([W * stride - 1, H * stride - 1] * 2, np.float32)
            mine = np.clip(ob[img][:n][o], 0, hi)
            np.testing.assert_allclose(mine, rb[img][:n][r], atol=1e-3, rtol=0)


def test_focal_oracle_matches_reference(golden_dir):
    g = _load(golden_dir, "focal.npz")
    tot, loss, grad = oracle.focal_loss(g["x"], g["t"])
    np.testing.assert_allclose(loss.reshape(g["loss"].shape), g["loss"], rtol=2e-5, atol=1e-7)
    np.testing.assert_allclose(grad.reshape(g["grad"].shape), g["grad"], rtol=2e-5, atol=1e-7)
    np.testing.assert_allclose(tot, g["loss"].astype(np.float64).sum(), rtol=1e-6)


def test_rotated_overlap_basic_properties():
    # identical boxes: union_area is area_i + area_m (nms_iou.cu:240), so I / (U - I) is the IoU;
    # the 0.001 jitter of nms_iou.cu:210-217 keeps it just below 1
    a = np.array([10, 10, 50, 40, 0.0, 1.0], np.float32)
    assert 0.999 < oracle.rotated_overlap(a, a) <= 1.0
    b = np.array([20, 15, 60, 45, 0.0, 1.0], np.float32)   # no +1 convention in the polygon IoU
    assert abs(oracle.rotated_overlap(a, b) - (30 * 25) / (2 * 40 * 30 - 30 * 25)) < 1e-4
    far = np.array([200, 200, 240, 230, 0.0, 1.0], np.float32)
    assert oracle.rotated_overlap(a, far) == 0.0
    # the quirk: the max box is rotated with the CANDIDATE's angle unless fixed_angle
    c = np.array([10, 10, 50, 40, np.sin(0.5), np.cos(0.5)], np.float32)
    m = np.array([12, 8, 48, 44, 0.0, 1.0], np.float32)
    assert oracle.rotated_overlap(c, m, False) != oracle.rotated_overlap(c, m, True)


def test_oracle_against_live_reference_nms(golden_dir):
    """The reference's CPU nms (odtk.box.nms, unmodified) on boxes scattered uniformly over the image, 3 seeded trials:
    tests/golden/nms_uniform.npz (oracle/gen_golden.py)."""
    g = np.load(os.path.join(golden_dir, "nms_uniform.npz"))
    for k in range(int(g["ncases"])):
        s, b, c = g["c%d_scores" % k], g["c%d_boxes" % k], g["c%d_classes" % k]
        rs, rb = g["c%d_out_scores" % k], g["c%d_out_boxes" % k]
        os_, ob, oc = oracle.nms(s, b, c, 0.5, 100)
        nk = int((rs[0] > 0).sum())
        np.testing.assert_array_equal(os_[0][:nk], rs[0][:nk])
        np.testing.assert_array_equal(ob[0][:nk], rb[0][:nk])


def test_l1_and_preprocess_oracle_match_reference(golden_dir):
    """Fixture: reference odtk.loss.SmoothL1Loss(beta=.11) + autograd on seeded inputs, and the tensor maths of
    odtk/data.py:113-123 (float().div(255), per-channel sub_(mean).div_(std), F.pad to stride 128) run verbatim on a
    seeded uint8 image (generated in the build container with the reference imported from /root/reference)."""
    g = _load(golden_dir, "l1_preproc.npz")
    tot, lo, gr = oracle.smooth_l1(g["p"], g["t"])
    np.testing.assert_allclose(lo.reshape(g["loss"].shape), g["loss"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(gr.reshape(g["grad"].shape), g["grad"], rtol=1e-5, atol=1e-6)
    pre = oracle.preprocess_u8(g["img"])
    np.testing.assert_allclose(pre, g["pre"], rtol=1e-6, atol=1e-6)


def test_snap_to_anchors_oracle_matches_reference(golden_dir):
    """oracle.snap_to_anchors vs odtk.box.snap_to_anchors run unmodified on CPU (tests/golden/snap.npz): depth and
    one-hot classes bit-exact (IoU thresholds, first-maximum ties, the empty image), box deltas to 1e-6 (log)."""
    g = np.load(os.path.join(golden_dir, "snap.npz"))
    for k in range(int(g["ncases"])):
        ct, bt, dp, ci = oracle.snap_to_anchors(g["c%d_boxes" % k], g["c%d_size" % k].tolist(), int(g["c%d_stride" % k]),
                                                g["c%d_anchors" % k], int(g["c%d_classes" % k]), [0.4, 0.5])
        np.testing.assert_array_equal(dp, g["c%d_depth" % k])
        np.testing.assert_array_equal(ct.astype(np.uint8), g["c%d_cls_target" % k])
        np.testing.assert_allclose(bt, g["c%d_box_target" % k], rtol=1e-6, atol=1e-6)
        # the class-index form is the same assignment: foreground <=> depth > 0, ignored <=> depth == -1
        d = dp[:, 0]
        np.testing.assert_array_equal(ci >= 0, d > 0)
        np.testing.assert_array_equal(ci == -2, d == -1)
        np.testing.assert_array_equal(ci[ci >= 0], d[d > 0].astype(np.int32) - 1)


def test_oracle_iou_matches_golden_and_reference_rotated_snap(golden_dir):
    """oracle_iou (restated nms_iou.cu:324-387) against the committed known answers, and the host-side mirrors of
    odtk.utils.rotate_boxes / odtk.box.box2delta_rotated against what the unmodified reference produced
    (tests/golden/snap_rotated.npz, oracle/gen_golden_rotated.py)."""
    import torch
    from oracle import oracle
    from retinanet_examples_b200 import box
    g = np.load(os.path.join(golden_dir, "snap_rotated.npz"))
    np.testing.assert_array_equal(oracle.iou(g["iou_boxes"], g["iou_anchors"]), g["iou"])
    for k in range(int(g["ncases"])):
        b = torch.from_numpy(g["c%d_boxes" % k])
        axis, rot = box.rotate_boxes(b[:, :5])
        np.testing.assert_allclose(axis.numpy(), g["c%d_boxes_axis" % k], rtol=1e-6, atol=1e-5)
        np.testing.assert_allclose(rot.numpy(), g["c%d_boxes_rot" % k], rtol=1e-6, atol=2e-4)
        aa = torch.from_numpy(g["c%d_anchors_axis" % k])
        d = box.box2delta_rotated(axis[:1].expand(aa.shape[0], 6), aa)
        assert d.shape == (aa.shape[0], 6) and torch.isfinite(d).all()
