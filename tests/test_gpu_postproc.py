"""GPU parity tests (run with -m gpu on the B200 box): the sm_100a decode / nms kernels, called
through the C ABI (ctypes), against the CPU oracle on the same seeded inputs, against the
committed golden fixtures, and against the outputs of the reference's own CUDA kernels
(tests/golden/refcuda.npz).

Bars: kept indices / classes / scores bit-exact; box coordinates within 1e-3 absolute (the only
non-IEEE-exact operation is expf: CUDA's and glibc's differ by <= 2 ulp)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from retinanet_examples_b200 import _C, box, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"


def _gpu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _check_decode(cls, deltas, anchors, stride, thresh, top_n, rotated=False):
    os_, ob, oc = oracle.decode(cls, deltas, anchors, stride, thresh, top_n, rotated)
    gs, gb, gc = [t.cpu().numpy() for t in _C.decode(_gpu(cls), _gpu(deltas), list(anchors), stride, thresh, top_n, rotated)]
    np.testing.assert_array_equal(gs, os_)
    np.testing.assert_array_equal(gc, oc)
    np.testing.assert_allclose(gb, ob, atol=1e-3, rtol=0)
    return os_, ob, oc, gs, gb, gc


def _level_case(rng, b, c, h, w, a, mu, nbox=4):
    cls = (1 / (1 + np.exp(-rng.normal(mu, 1.6, size=(b, a * c, h, w))))).astype(np.float32)
    deltas = rng.normal(0, 0.2, size=(b, a * nbox, h, w)).astype(np.float32)
    return cls, deltas


@pytest.mark.parametrize("stride,h,w,mu,top_n", [(8, 25, 40, -4.0, 1000), (16, 13, 20, -2.0, 1000),
                                                 (128, 7, 10, -6.0, 1000), (32, 9, 7, -1.0, 37)])
def test_decode_matches_oracle(stride, h, w, mu, top_n):
    rng = np.random.default_rng(stride * 1000 + h)
    anchors = oracle.generate_anchors(stride, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES).reshape(-1)
    cls, deltas = _level_case(rng, 3, 20, h, w, 9, mu)
    os_, *_ = _check_decode(cls, deltas, anchors, stride, 0.05, top_n)
    assert (os_ > 0).any()


def test_decode_full_size_level_p4_batch2():
    """One full-size pyramid level of the BASELINE shape (P4: 720 x 50 x 80) incl. the sort path."""
    cls, box_ = synth.head_outputs(2, seed=3)
    anchors = oracle.generate_anchors(16, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES).reshape(-1)
    os_, *_ = _check_decode(cls[1].numpy(), box_[1].numpy(), anchors, 16, 0.05, 1000)
    assert (os_[:, -1] > 0).all()          # more than top_n candidates: the sorted path ran


def test_decode_edge_cases():
    rng = np.random.default_rng(5)
    anchors = oracle.generate_anchors(8, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES).reshape(-1)
    cls, deltas = _level_case(rng, 2, 3, 6, 5, 9, -3.0)
    # nothing passes
    _check_decode(np.zeros_like(cls), deltas, anchors, 8, 0.05, 100)
    # everything passes, ragged size (n % 4 != 0 -> scalar load path): 9*3*5*7 = 945
    c2, d2 = _level_case(rng, 1, 3, 5, 7, 9, 3.0)
    _check_decode(c2, d2, anchors, 8, 0.05, 64)
    # massive exact ties: the tie bin exceeds the sort capacity -> radix-select fallback
    c3 = np.full((1, 9 * 4, 16, 16), 0.5, np.float32)
    d3 = rng.normal(0, 0.2, size=(1, 36, 16, 16)).astype(np.float32)
    os_, ob, oc, gs, gb, gc = _check_decode(c3, d3, anchors, 8, 0.05, 1000)
    assert (os_ == 0.5).all()
    # threshold is strict '>' (decode.cu:97): scores == thresh are dropped
    c4 = np.full((1, 9, 4, 4), 0.05, np.float32)
    c4[0, 0, 0, 0] = 0.06
    os_, *_ = _check_decode(c4, rng.normal(0, 0.2, size=(1, 36, 4, 4)).astype(np.float32), anchors, 8, 0.05, 10)
    assert (os_ > 0).sum() == 1
    # no anchors: raw deltas come back (decode.cu:118 has_anchors)
    _check_decode(cls, deltas, np.zeros(0, np.float32), 8, 0.05, 100)


def test_decode_candidate_overflow_slow_path():
    """More than 2^20 survivors in one image overflow the candidate list: exact fallback."""
    rng = np.random.default_rng(11)
    anchors = oracle.generate_anchors(8, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES).reshape(-1)
    cls = rng.uniform(0.06, 1.0, size=(1, 9 * 20, 80, 100)).astype(np.float32)   # 1.44 M, all pass
    deltas = rng.normal(0, 0.2, size=(1, 36, 80, 100)).astype(np.float32)
    _check_decode(cls, deltas, anchors, 8, 0.05, 1000)


def test_decode_rotated_matches_oracle():
    rng = np.random.default_rng(21)
    anchors = oracle.generate_anchors_rotated_axis(16, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES,
                                                   oracle.DEFAULT_ANGLES).reshape(-1)
    cls, deltas = _level_case(rng, 2, 8, 13, 20, 27, -3.0, nbox=6)
    os_, ob, *_ = _check_decode(cls, deltas, anchors, 16, 0.05, 1000, rotated=True)
    assert ob.shape[-1] == 6 and (os_ > 0).any()


def test_decode_golden_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "decode.npz"))
    for k in range(int(g["ncases"])):
        cls, deltas, anchors = g["c%d_cls" % k], g["c%d_box" % k], g["c%d_anchors" % k]
        top_n, stride = int(g["c%d_top_n" % k]), int(g["c%d_stride" % k])
        gs, gb, gc = [t.cpu().numpy() for t in _C.decode(_gpu(cls), _gpu(deltas), anchors.reshape(-1).tolist(), stride, 0.05, top_n)]
        rs, rb, rc = g["c%d_out_scores" % k], g["c%d_out_boxes" % k], g["c%d_out_classes" % k]
        H, W = cls.shape[2], cls.shape[3]
        hi = np.array([W * stride - 1, H * stride - 1] * 2, np.float32)
        for img in range(cls.shape[0]):
            n = int((rs[img] > 0).sum())
            assert int((gs[img] > 0).sum()) == n
            o = np.lexsort((gb[img][:n, 1], gb[img][:n, 0], gc[img][:n], -gs[img][:n]))
            r = np.lexsort((rb[img][:n, 1], rb[img][:n, 0], rc[img][:n], -rs[img][:n]))
            np.testing.assert_array_equal(gs[img][:n][o], rs[img][:n][r])
            np.testing.assert_array_equal(gc[img][:n][o], rc[img][:n][r])
            np.testing.assert_allclose(np.clip(gb[img][:n][o], 0, hi), rb[img][:n][r], atol=1e-3, rtol=0)


# ------------------------------------------------------------------------------------------------
def _nms_case(rng, b, n, ncls, zero_frac, clusters, rotated=False):
    ctr = rng.uniform(50, 900, size=(b, clusters, 2))
    which = rng.integers(0, clusters, size=(b, n))
    c = np.take_along_axis(ctr, which[..., None].repeat(2, -1), axis=1) + rng.normal(0, 10, (b, n, 2))
    wh = rng.uniform(20, 120, size=(b, n, 2))
    boxes = np.concatenate([c - wh / 2, c + wh / 2], -1)
    if rotated:
        th = rng.uniform(-np.pi / 4, np.pi / 4, size=(b, n, 1))
        boxes = np.concatenate([boxes, np.sin(th), np.cos(th)], -1)
    scores = rng.uniform(0.05, 1.0, size=(b, n)).astype(np.float32)
    scores[rng.uniform(size=(b, n)) < zero_frac] = 0.0
    classes = rng.integers(0, ncls, size=(b, n)).astype(np.float32)
    return scores, boxes.astype(np.float32), classes


def _check_nms(s, b, c, thr, det, rotated=False, fixed_angle=False):
    os_, ob, oc, oi = oracle.nms(s, b, c, thr, det, rotated=rotated, fixed_angle=fixed_angle, return_index=True)
    gs, gb, gc, gi = [t.cpu().numpy() for t in _C.nms(_gpu(s), _gpu(b), _gpu(c), thr, det, rotated,
                                                      return_index=True, fixed_angle=fixed_angle)]
    np.testing.assert_array_equal(gi, oi)      # kept indices: bit-exact
    np.testing.assert_array_equal(gs, os_)
    np.testing.assert_array_equal(gb, ob)
    np.testing.assert_array_equal(gc, oc)
    return os_, oi


@pytest.mark.parametrize("b,n,ncls,zf,cl,thr,det", [(2, 400, 3, 0.1, 6, 0.5, 100), (3, 5000, 80, 0.15, 40, 0.5, 100),
                                                    (1, 6144, 2, 0.0, 3, 0.5, 100), (2, 777, 1, 0.3, 2, 0.3, 1000),
                                                    (1, 50, 4, 0.0, 50, 0.5, 100), (4, 33, 2, 0.5, 4, 0.7, 7)])
def test_nms_matches_oracle(b, n, ncls, zf, cl, thr, det):
    rng = np.random.default_rng(n * 7 + det)
    s, bx, c = _nms_case(rng, b, n, ncls, zf, cl)
    os_, oi = _check_nms(s, bx, c, thr, det)
    assert (os_ > 0).any()


@pytest.mark.parametrize("rotated", [False, True])
def test_nms_prefix_exhausted_falls_back_to_the_full_sort(rotated):
    """The kernel first orders only the ~512-2048 top-scoring candidates; when the greedy walk exhausts them without
    reaching D keepers (here: thousands of near-identical same-class boxes, so almost everything is suppressed) it must
    run the full sort and still return exactly the oracle's result -- including the suppressed tail entries."""
    rng = np.random.default_rng(41)
    n = 5000
    s = rng.uniform(0.06, 1.0, size=(2, n)).astype(np.float32)
    ctr = rng.integers(0, 3, size=(2, n, 1)) * 400.0 + rng.normal(0, 1.0, size=(2, n, 2))
    b = np.concatenate([ctr, ctr + 100.0], 2)
    if rotated:
        th = rng.uniform(-0.05, 0.05, size=(2, n, 1))
        b = np.concatenate([b, np.sin(th), np.cos(th)], 2)
    c = np.zeros((2, n), np.float32)
    os_, oi = _check_nms(s, b.astype(np.float32), c, 0.5, 100, rotated=rotated)
    assert 0 < int((os_[0] > 0).sum()) < 20          # a handful of keepers, the other output slots are suppressed entries
    assert (oi[0] >= 0).sum() == 100


def test_nms_edge_cases():
    rng = np.random.default_rng(3)
    s, bx, c = _nms_case(rng, 2, 200, 3, 0.0, 5)
    _check_nms(np.zeros_like(s), bx, c, 0.5, 100)                 # nothing valid
    s2 = s.copy(); s2[:, 1:] = 0
    _check_nms(s2, bx, c, 0.5, 100)                               # a single candidate
    s3 = np.full_like(s, 0.5)                                     # all scores tie: positional order
    _check_nms(s3, bx, c, 0.5, 100)
    bx4 = np.repeat(bx[:, :1], 200, axis=1)                       # identical boxes: 1 keeper per class
    os_, oi = _check_nms(s, bx4, c, 0.5, 100)
    assert (os_ > 0).sum(axis=1).max() <= 3


def test_nms_golden_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "nms.npz"))
    for k in range(int(g["ncases"])):
        s, b, c = g["c%d_scores" % k], g["c%d_boxes" % k], g["c%d_classes" % k]
        gs, gb, gc = [t.cpu().numpy() for t in _C.nms(_gpu(s), _gpu(b), _gpu(c), float(g["c%d_thr" % k]), int(g["c%d_det" % k]))]
        rs, rb, rc = g["c%d_out_scores" % k], g["c%d_out_boxes" % k], g["c%d_out_classes" % k]
        for img in range(s.shape[0]):
            nk = int((rs[img] > 0).sum())
            assert int((gs[img] > 0).sum()) == nk
            np.testing.assert_array_equal(gs[img][:nk], rs[img][:nk])
            np.testing.assert_array_equal(gb[img][:nk], rb[img][:nk])
            np.testing.assert_array_equal(gc[img][:nk], rc[img][:nk])


@pytest.mark.parametrize("fixed", [False, True])
def test_nms_rotated_matches_oracle(fixed):
    rng = np.random.default_rng(17)
    s, bx, c = _nms_case(rng, 2, 1500, 4, 0.1, 12, rotated=True)
    os_, oi = _check_nms(s, bx, c, 0.5, 100, rotated=True, fixed_angle=fixed)
    assert (os_ > 0).any()


def test_decode_then_nms_full_pipeline_batch2():
    """Five full-size levels -> concat -> nms at the BASELINE shapes (config 2 with batch 2)."""
    cls, deltas = synth.head_outputs(2, seed=1)
    outs_g, outs_o = [], []
    for lvl, stride in enumerate(synth.LEVEL_STRIDES):
        anchors = oracle.generate_anchors(stride, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES).reshape(-1)
        outs_g.append(_C.decode(cls[lvl].to(DEV), deltas[lvl].to(DEV), anchors.tolist(), stride, 0.05, 1000))
        if True:          # all five levels incl. P3 (23 M scores: ~1 s in the C oracle)
            o = oracle.decode(cls[lvl].numpy(), deltas[lvl].numpy(), anchors, stride, 0.05, 1000)
            np.testing.assert_array_equal(outs_g[-1][0].cpu().numpy(), o[0])
            np.testing.assert_allclose(outs_g[-1][1].cpu().numpy(), o[1], atol=1e-3, rtol=0)
    cat = [torch.cat(t, 1) for t in zip(*outs_g)]
    assert cat[0].shape == (2, 5000)
    # the all-levels entry point (3 launches) must equal the torch.cat of the per-level calls
    all_anchors = [oracle.generate_anchors(s, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES).reshape(-1).tolist()
                   for s in synth.LEVEL_STRIDES]
    fused = _C.decode_levels([c.to(DEV) for c in cls], [d.to(DEV) for d in deltas], all_anchors,
                             synth.LEVEL_STRIDES, 0.05, 1000)
    for f, c in zip(fused, cat):
        np.testing.assert_array_equal(f.cpu().numpy(), c.cpu().numpy())
    gs, gb, gc, gi = [t.cpu().numpy() for t in _C.nms(*cat, 0.5, 100, False, return_index=True)]
    os_, ob, oc, oi = oracle.nms(cat[0].cpu().numpy(), cat[1].cpu().numpy(), cat[2].cpu().numpy(), 0.5, 100, return_index=True)
    np.testing.assert_array_equal(gi, oi)
    np.testing.assert_array_equal(gs, os_)
    np.testing.assert_array_equal(gb, ob)


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rotated", [False, True])
def test_against_reference_cuda_kernels(golden_dir, rotated):
    """The reference's own csrc/cuda kernels (compiled unmodified for sm_100a, --use_fast_math as
    shipped; their outputs are stored in tests/golden/refcuda.npz by oracle/gen_golden_refcuda.py)
    on the same inputs: same kept set; coordinates within 1e-3 + fast-math slack."""
    from oracle import gen_golden_refcuda as refcuda
    g = np.load(os.path.join(golden_dir, "refcuda.npz"))
    k = "r%d_" % rotated
    anchors, stride, cls, deltas = refcuda.decode_case(rotated)
    mine = _C.decode(_gpu(cls), _gpu(deltas), anchors, stride, refcuda.THRESH, refcuda.TOP_N, rotated)
    np.testing.assert_array_equal(mine[0].cpu().numpy(), g[k + "dec_scores"])
    np.testing.assert_array_equal(mine[2].cpu().numpy(), g[k + "dec_classes"])
    np.testing.assert_allclose(mine[1].cpu().numpy(), g[k + "dec_boxes"], atol=2e-2, rtol=0)   # __expf
    # nms through both implementations on the decoded boxes the reference's nms was given (the product's own decode)
    nms_in = [_gpu(g[k + "nms_in_" + n]) for n in ("scores", "boxes", "classes")]
    gs, gb, gc = [t.cpu().numpy() for t in _C.nms(*nms_in, refcuda.NMS_THRESH, refcuda.DETECTIONS, rotated)]
    rs, rb, rc = g[k + "nms_scores"], g[k + "nms_boxes"], g[k + "nms_classes"]
    for img in range(2):
        nk = int((rs[img] > 0).sum())
        # fast-math division can flip a decision that sits within 1 ulp of the threshold: allow
        # at most one differing keeper, everything else identical
        same = (gs[img][:nk] == rs[img][:nk])
        assert same.mean() > 0.97, (img, same.mean())
        if same.all():
            np.testing.assert_array_equal(gb[img][:nk], rb[img][:nk])
            np.testing.assert_array_equal(gc[img][:nk], rc[img][:nk])


@pytest.mark.parametrize("rotated", [False, True])
def test_literal_drop_in_symbols_with_data(rotated):
    """The four literally-named drop-in entry points -- odtk_decode / odtk_decode_rotate / odtk_nms / odtk_nms_rotate, the
    argument lists of odtk::cuda::decode(_rotate) / nms(_rotate) (csrc/cuda/*.h) -- called through raw ctypes with DATA (the
    Python mirror and the other tests go through the _ex / _levels extensions): two-phase workspace, outputs pre-zeroed
    by the caller as the reference's pybind layer does (extensions.cpp:83-85), results equal to the oracle."""
    from retinanet_examples_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(99 + rotated)
    A, nbox, stride, top_n, det = (27 if rotated else 9), (6 if rotated else 4), 32, 300, 100
    anchors = (oracle.generate_anchors_rotated_axis(stride, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES, oracle.DEFAULT_ANGLES)
               if rotated else oracle.generate_anchors(stride, oracle.DEFAULT_RATIOS, oracle.DEFAULT_SCALES)).reshape(-1)
    cls, deltas = _level_case(rng, 2, 6, 13, 20, A, -3.0, nbox)
    if rotated:
        th = rng.uniform(-0.7, 0.7, size=(2, A, 13, 20))
        d = deltas.reshape(2, A, 6, 13, 20); d[:, :, 4] = np.sin(th); d[:, :, 5] = np.cos(th)
    tc, td = _gpu(cls), _gpu(deltas)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    s = torch.zeros((2, top_n), device=DEV); b = torch.zeros((2, top_n, nbox), device=DEV); c = torch.zeros((2, top_n), device=DEV)
    anc = (ctypes.c_float * len(anchors))(*anchors.tolist())
    dec = L.odtk_decode_rotate if rotated else L.odtk_decode
    args = (2, _lib.ptr_array([tc.data_ptr(), td.data_ptr()]), _lib.ptr_array([s.data_ptr(), b.data_ptr(), c.data_ptr()]),
            13, 20, stride, A, 6, anc, len(anchors), 0.05, top_n)
    size = dec(*args, None, 0, None)
    assert size > 0
    ws = torch.empty(size, dtype=torch.uint8, device=DEV)
    assert dec(*args, ctypes.c_void_p(ws.data_ptr()), size, st) == 0
    os_, ob, oc = oracle.decode(cls, deltas, anchors, stride, 0.05, top_n, rotated)
    np.testing.assert_array_equal(s.cpu().numpy(), os_)
    np.testing.assert_array_equal(c.cpu().numpy(), oc)
    np.testing.assert_allclose(b.cpu().numpy(), ob, atol=1e-3, rtol=0)
    assert (os_ > 0).sum() > 50
    ns = torch.zeros((2, det), device=DEV); nb = torch.zeros((2, det, nbox), device=DEV); nc = torch.zeros((2, det), device=DEV)
    nms = L.odtk_nms_rotate if rotated else L.odtk_nms
    nargs = (2, _lib.ptr_array([s.data_ptr(), b.data_ptr(), c.data_ptr()]), _lib.ptr_array([ns.data_ptr(), nb.data_ptr(), nc.data_ptr()]),
             top_n, det, 0.5)
    nsize = nms(*nargs, None, 0, None)
    assert nsize > 0
    nws = torch.empty(nsize, dtype=torch.uint8, device=DEV)
    assert nms(*nargs, ctypes.c_void_p(nws.data_ptr()), nsize, st) == 0
    rs, rb, rc = oracle.nms(s.cpu().numpy(), b.cpu().numpy(), c.cpu().numpy(), 0.5, det, rotated=rotated)
    np.testing.assert_array_equal(ns.cpu().numpy(), rs)
    np.testing.assert_array_equal(nb.cpu().numpy(), rb)
    np.testing.assert_array_equal(nc.cpu().numpy(), rc)
