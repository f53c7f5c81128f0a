"""Fixture from the reference's own CUDA kernels: csrc/cuda/{decode,decode_rotate,nms,nms_iou}.cu compiled unmodified
for sm_100a (--use_fast_math, as its setup.py ships them) into oracle/_ref/libodtk_ref.so by oracle/Makefile, behind the
extern "C" doors of oracle/ref_shim.cu.  Needs that library and a GPU; TEST INFRASTRUCTURE ONLY.
    python oracle/gen_golden_refcuda.py [out_dir]  ->  <out_dir, default tests/golden>/refcuda.npz

What it stores, for rotated = 0 / 1 (keys r0_* / r1_*) and the seeded inputs of decode_case / iou_case below:
  dec_*     the reference decode of one level (scores, boxes, classes; top_n 1000, threshold 0.05)
  nms_in_*  the product's own decode of the same level: the input both NMS implementations are compared on
  nms_*     the reference NMS of nms_in_* (IoU 0.5, 100 detections)
  iou       the reference iou kernel on iou_case: [num_anchors, num_boxes] (its swapped-argument orientation)"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle  # noqa: E402

REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libodtk_ref.so")
TOP_N, THRESH, NMS_THRESH, DETECTIONS = 1000, 0.05, 0.5, 100


def decode_case(rotated):
    """One 25 x 40 level at stride 16, 10 classes, batch 2, ~3 % of the scores above the threshold.
    Returns (anchors as a flat list, stride, cls [2, A*10, 25, 40], deltas [2, A*nbox, 25, 40])."""
    rng = np.random.default_rng(31)
    a, nbox, stride = (27, 6, 16) if rotated else (9, 4, 16)
    anchors = (oracle.generate_anchors_rotated_axis(stride, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES, oracle.DEFAULT_ANGLES)
               if rotated else oracle.generate_anchors(stride, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES)).reshape(-1).tolist()
    cls = (1 / (1 + np.exp(-rng.normal(-3.5, 1.6, size=(2, a * 10, 25, 40))))).astype(np.float32)
    deltas = rng.normal(0, 0.2, size=(2, a * nbox, 25, 40)).astype(np.float32)
    if rotated:
        th = rng.uniform(-np.pi / 4, np.pi / 4, size=(2, a, 25, 40))
        d = deltas.reshape(2, a, 6, 25, 40)
        d[:, :, 4] = np.sin(th)
        d[:, :, 5] = np.cos(th)
    return anchors, stride, cls, deltas


def iou_case():
    """300 rectangles as corner lists [300, 8]: the first 5 are the boxes, the other 295 the anchors."""
    rng = np.random.default_rng(8)
    c = rng.uniform(0, 200, (300, 1, 2))
    quads = (c + np.array([[-20, -10], [20, -10], [20, 10], [-20, 10]]) * rng.uniform(0.5, 2, (300, 1, 1))).reshape(300, 8)
    quads = quads.astype(np.float32)
    return quads[:5].copy(), quads[5:].copy()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _two_phase(fn, args, torch):
    """The reference's workspace protocol: a size query (no workspace), then the call itself."""
    size = fn(*args, None, ctypes.c_longlong(0), None)
    ws = torch.zeros(max(int(size), 1), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    assert fn(*args, _ptr(ws), ctypes.c_longlong(size), None) == 0
    torch.cuda.synchronize()


def main():
    import torch
    from retinanet_examples_b200 import _C
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    L = ctypes.CDLL(REF_LIB)
    L.ref_decode.restype = L.ref_nms.restype = L.ref_iou.restype = ctypes.c_longlong
    d = {}
    for rotated in (0, 1):
        anchors, stride, cls, deltas = decode_case(rotated)
        nbox = 6 if rotated else 4
        b, ac, h, w = cls.shape
        na = len(anchors) // 4
        tc, td = torch.from_numpy(cls).cuda(), torch.from_numpy(deltas).cuda()
        s, bx, c = torch.zeros(b, TOP_N, device="cuda"), torch.zeros(b, TOP_N, nbox, device="cuda"), torch.zeros(b, TOP_N, device="cuda")
        anc = (ctypes.c_float * len(anchors))(*anchors)
        _two_phase(L.ref_decode, [b, _ptr(tc), _ptr(td), _ptr(s), _ptr(bx), _ptr(c), h, w, stride, na, ac // na, anc,
                                  len(anchors), ctypes.c_float(THRESH), TOP_N, rotated], torch)
        mine = _C.decode(tc, td, anchors, stride, THRESH, TOP_N, bool(rotated))
        os_, ob, oc = torch.zeros(b, DETECTIONS, device="cuda"), torch.zeros(b, DETECTIONS, nbox, device="cuda"), \
            torch.zeros(b, DETECTIONS, device="cuda")
        _two_phase(L.ref_nms, [b, _ptr(mine[0]), _ptr(mine[1]), _ptr(mine[2]), _ptr(os_), _ptr(ob), _ptr(oc), TOP_N,
                               DETECTIONS, ctypes.c_float(NMS_THRESH), rotated], torch)
        k = "r%d_" % rotated
        for name, t in (("dec_scores", s), ("dec_boxes", bx), ("dec_classes", c), ("nms_in_scores", mine[0]),
                        ("nms_in_boxes", mine[1]), ("nms_in_classes", mine[2]), ("nms_scores", os_), ("nms_boxes", ob),
                        ("nms_classes", oc)):
            d[k + name] = t.cpu().numpy()
    boxes, anchors = iou_case()
    tb, ta = torch.from_numpy(boxes).cuda(), torch.from_numpy(anchors).cuda()
    ref = torch.zeros((anchors.shape[0], boxes.shape[0]), device="cuda")
    torch.cuda.synchronize()
    assert L.ref_iou(_ptr(tb), _ptr(ta), _ptr(ref), boxes.shape[0], anchors.shape[0], None) == 0
    torch.cuda.synchronize()
    d["iou"] = ref.cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, "refcuda.npz"), **d)
    print({k: v.shape for k, v in d.items()})


if __name__ == "__main__":
    main()
