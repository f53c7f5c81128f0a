"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/odtk_b200.h
declares, the cub-style size queries work without a GPU, the anchor tables of the product match the
reference's, and inputs that are not CUDA tensors are rejected like odtk._C does."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from retinanet_examples_b200 import _C, _lib, box, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "odtk_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(odtk_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    names = _declared_symbols()
    assert len(names) >= 7
    for n in names:
        assert hasattr(L, n), n
        assert n in _lib.SIGNATURES, "ctypes signature missing for %s" % n
    assert b"sm_100a" in L.odtk_b200_version()


def test_workspace_size_queries_need_no_gpu():
    L = _lib.lib()
    # decode: P3 of RetinaNet at 800x1280, batch 8 (SURVEY.md section 8)
    sz = L.odtk_decode_ex(8, None, None, 100, 160, 8, 9, 80, None, 36, 0.05, 1000, 4, 1000, 0, None, 0, None)
    assert sz > 8 * (1 << 20) * 8          # candidate lists dominate
    assert sz % 256 == 0
    assert L.odtk_decode(8, None, None, 100, 160, 8, 9, 80, None, 36, 0.05, 1000, None, 0, None) == sz
    assert L.odtk_nms(8, None, None, 5000, 100, 0.5, None, 0, None) == 256
    # argument validation happens before any CUDA call
    assert L.odtk_decode(0, None, None, 100, 160, 8, 9, 80, None, 36, 0.05, 1000, None, 0, None) == -1
    assert L.odtk_decode(1, None, None, 100, 160, 8, 9, 80, None, 36, 0.05, 5000, None, 0, None) == -3
    assert L.odtk_nms(1, None, None, 7000, 100, 0.5, None, 0, None) == -3
    assert L.odtk_nms_ex(1, None, None, 100, 10, 0.5, 5, 0, None, None, 0, None) == -1


def test_product_anchors_match_reference_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "anchors.npz"))
    for s in (8, 16, 32, 64, 128):
        a = box.generate_anchors(s, box.DEFAULT_RATIOS, box.DEFAULT_SCALES)
        np.testing.assert_array_equal(a.numpy(), g["axis_%d" % s])
        np.testing.assert_allclose(np.round(a.numpy().reshape(-1), 2), g["cpp_axis_%d" % s], atol=6e-3)
        ax, rot = box.generate_anchors_rotated(s, box.DEFAULT_RATIOS, box.DEFAULT_SCALES, box.DEFAULT_ANGLES)
        np.testing.assert_allclose(ax.numpy(), g["rotdef_axis_%d" % s], atol=1e-5)
        np.testing.assert_allclose(rot.numpy(), g["rotdef_corners_%d" % s], atol=1e-4)
        ax, rot = box.generate_anchors_rotated(s, [0.25, 0.5, 1.0, 2.0, 4.0], [2 * 2 ** (2 * i / 3) for i in range(3)],
                                               box.DEFAULT_ANGLES)
        np.testing.assert_allclose(ax.numpy(), g["rot_axis_%d" % s], atol=1e-5)
        np.testing.assert_allclose(np.round(ax.numpy().reshape(-1), 2), g["cpp_rot_%d" % s], atol=6e-3)
        np.testing.assert_allclose(rot.numpy(), g["rot_corners_%d" % s], atol=1e-4)


def test_cpu_tensors_are_rejected_no_fallback():
    s = torch.zeros(1, 9 * 2, 4, 4)
    b = torch.zeros(1, 36, 4, 4)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        _C.decode(s, b, [0.0] * 36, 8, 0.05, 10)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        _C.nms(torch.zeros(1, 8), torch.zeros(1, 8, 4), torch.zeros(1, 8), 0.5, 4)


def test_level_sizes_match_survey():
    assert synth.level_sizes(800, 1280) == [(100, 160), (50, 80), (25, 40), (13, 20), (7, 10)]


def test_layer_table_tool_reproduces_committed_profile(tmp_path):
    """tools/layer_table.py joins the committed ncu launch list with the engine trace of the same step; the
    committed summary (which bench.py reads for roofline.traffic) must be what the tool computes from them
    with the peaks the summary records."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    prof = os.path.join(root, "profiles")
    out = str(tmp_path / "table")
    old = json.load(open(os.path.join(prof, "r01_layer_table.json")))["summary"]
    subprocess.run([sys.executable, os.path.join(root, "tools", "layer_table.py"), os.path.join(prof, "r01_step_launches.csv"),
                    os.path.join(prof, "r01_step_trace.json"), "--out", out, "--tensor-tflops", repr(old["tensor_peak_tflops"]),
                    "--hbm-gbs", repr(old["hbm_peak_gbs"])], check=True, capture_output=True)
    new = json.load(open(out + ".json"))["summary"]
    for k in ("launches", "sum_us", "sum_ideal_us", "conv_dram_bytes"):
        assert new[k] == old[k], k
    assert 0.5 < new["frac"] <= 1.0
    trace = json.load(open(os.path.join(prof, "r01_step_trace.json")))
    assert sum(l["flops"] for l in trace) == 15266307768320      # 477.07 GFLOP/image x 32 (DESIGN.md section 4)


def test_plugin_shaped_wrappers_compile_and_query_sizes(tmp_path):
    """plugins/odtk_b200_plugin.h (TensorRT-plugin-shaped enqueue / getWorkspaceSize / configurePlugin over the C ABI,
    mirroring csrc/plugins/DecodePlugin.h:141-161 and NMSPlugin.h:120-138) compiles with stub NvInfer types, links against
    libodtk_b200.so and answers the workspace queries without a GPU."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "retinanet-examples_b200")
    exe = str(tmp_path / "plugin_check")
    subprocess.run(["g++", "-std=c++17", "-Wall", "-Werror", "-I", os.path.join(root, "plugins"),
                    os.path.join(root, "plugins", "plugin_check.cpp"), "-o", exe, "-L", libdir, "-lodtk_b200",
                    "-Wl,-rpath," + libdir], check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    assert "decode_ws=" in out and "format_ok=1" in out


def test_header_is_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: include/odtk_b200.h must compile as C (no C++-isms, no torch / CUDA types)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "abi_check.c"
    src.write_text('#include "odtk_b200.h"\nint main(void) { odtk_conv_t c; odtk_bneck_t b; odtk_gather_t g; (void)c; (void)b; (void)g; return 0; }\n')
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(root, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_state_dict_layouts_match_torchvision():
    """make_state_dict / conv_specs follow the reference's key layout: `backbones.<Name>.features.` + the torchvision module's
    own keys (odtk/backbones/resnet.py:7-22, mobilenet.py:5-13), same shapes; only the classification tails the reference
    never runs (fc / features.18 / classifier) are absent."""
    import torchvision.models as tvm
    from retinanet_examples_b200.model import make_state_dict
    for name, ctor in (("ResNet50FPN", tvm.resnet50), ("ResNeXt50_32x4dFPN", tvm.resnext50_32x4d), ("MobileNetV2FPN", tvm.mobilenet_v2)):
        ref = ctor(weights=None).state_dict()
        sd = make_state_dict(name, 3, 9, False, seed=0)
        pre = "backbones.%s.features." % name
        ours = {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}
        skip = ("num_batches_tracked", "fc.", "features.18.", "classifier.")
        want = {k: v for k, v in ref.items() if not any(t in k for t in skip)}
        assert set(ours) == set(want), (name, sorted(set(want) ^ set(ours))[:5])
        for k, v in want.items():
            assert tuple(ours[k].shape) == tuple(v.shape), (name, k)


def test_bench_dump_outputs_writes_float_arrays_and_caps_their_size(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one DIR/<name>.npy per returned array; past the size cap, the rows of a fixed seeded
    sample of images and their positions in the batch (the same sample on every run)."""
    import bench
    rows = {"scores": np.arange(40, dtype=np.float32).reshape(10, 4), "boxes": np.ones((10, 4, 4), np.float32)}
    bench.dump_outputs(str(tmp_path / "all"), rows)
    assert sorted(os.listdir(tmp_path / "all")) == ["boxes.npy", "scores.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "scores.npy"), rows["scores"])
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 3 * (16 + 64))          # room for 3 of the 10 images
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), rows)
    idx = np.load(tmp_path / "a" / "image_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 3
    np.testing.assert_array_equal(idx, np.load(tmp_path / "b" / "image_index.npy"))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "scores.npy"), rows["scores"][idx.astype(int)])
    assert np.load(tmp_path / "a" / "boxes.npy").dtype == np.float32
