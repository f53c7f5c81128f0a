"""oracle/model_ref.py -- TEST INFRASTRUCTURE ONLY.

Pure-PyTorch fp32 CPU restatement of the reference's Model.forward for ResNet-FPN backbones, written
against the reference's state_dict key layout.  It is the CPU "port" used (a) to check the CUDA
convolution stack (the reference itself runs nn.Conv2d: torch is the arithmetic oracle here), and
(b) as bench.py's cpu_baseline / --impl reference leg on the GPU box, where /root/reference does
not exist.  Pinned against the unmodified reference Model by tests/golden/model_*.npz
(oracle/gen_golden_model.py).

Follows: odtk/model.py:125-165 (forward), odtk/backbones/fpn.py:45-61 (FPN),
odtk/backbones/resnet.py:24-39 (feature extractor), torchvision/models/resnet.py BasicBlock :59-105,
Bottleneck :108-163 (stride on the 3x3: "v1.5"), stem/maxpool :197-200, eps = 1e-5."""
import numpy as np
import torch
import torch.nn.functional as F

from . import oracle

LAYERS = {"ResNet18FPN": ("basic", [2, 2, 2, 2]), "ResNet34FPN": ("basic", [3, 4, 6, 3]),
          "ResNet50FPN": ("bottleneck", [3, 4, 6, 3]), "ResNet101FPN": ("bottleneck", [3, 4, 23, 3]),
          "ResNet152FPN": ("bottleneck", [3, 8, 36, 3]),
          "ResNeXt50_32x4dFPN": ("bottleneck", [3, 4, 6, 3]), "ResNeXt101_32x8dFPN": ("bottleneck", [3, 4, 23, 3])}
GROUPS = {"ResNeXt50_32x4dFPN": 32, "ResNeXt101_32x8dFPN": 32}     # odtk/backbones/fpn.py:85-91 (torchvision groups=32)


def _bn(sd, p, x):
    return F.batch_norm(x, sd[p + ".running_mean"], sd[p + ".running_var"], sd[p + ".weight"], sd[p + ".bias"],
                        training=False, eps=1e-5)


def _conv(sd, p, x, stride=1, padding=0, groups=1):
    return F.conv2d(x, sd[p + ".weight"], sd.get(p + ".bias"), stride=stride, padding=padding, groups=groups)


# ---- fp16-emulating mode ------------------------------------------------------------------------------------------
# The product path stores activations and weights in fp16 and accumulates in fp32 (what "fp16" means for the reference
# too: apex AMP O2 / a TensorRT FP16 engine, SURVEY.md App. B item 10).  With fp16=True this oracle performs the SAME
# roundings -- BatchNorm folded into the weights in fp32, weights rounded to fp16 once, every layer's output (after bias,
# residual / upsample add and ReLU, all in fp32) rounded to fp16, head outputs kept in fp32 -- and sums each convolution
# in the product's K order (_conv_fp32_steps), so that what remains between it and the CUDA path is the rounding inside
# one tensor-core step (plus the rare 1-ulp fp16 rounding flip it causes): the conv stack can then be held to
# 2e-3 * max|ref| and detections to 1e-3 instead of the 3e-2 an all-fp32 oracle allows.
def _q(x, fp16):
    return x.half().float() if fp16 else x


def _add_rz(acc, step):
    """fp32 accumulator + float64 step, rounded toward zero (the tensor cores truncate when they accumulate: Fasi, Higham,
    Mikaitis, Pranesh, "Numerical behavior of NVIDIA tensor cores", PeerJ CS 2021)."""
    s = acc.double() + step
    f = s.float()
    return torch.where(f.double().abs() > s.abs(), torch.nextafter(f, torch.zeros_like(f)), f)


def _conv_fp32_steps(x, w, b, stride, padding, groups):
    """fp16 mode: the convolution summed in the order of the product's tensor-core kernels (csrc/conv.cu) -- 64-channel
    chunks, then taps, then the 16-channel steps of one MMA -- each step's 16 products summed exactly (float64) and added
    to the fp32 accumulator with truncation (_add_rz), the bias added last.  torch's own CPU convolution splits its fp32
    sums by the host's thread count, which moves the fp16 roundings downstream by as much as the parity bars allow.
    Grouped and depthwise convolutions (at most a few hundred products per output) are summed exactly and rounded once."""
    xd, wd = x.double(), w.double()
    if groups > 1:
        acc = F.conv2d(xd, wd, None, stride=stride, padding=padding, groups=groups).float()
    else:
        n, c, h, wi = x.shape
        o, _, kh, kw = w.shape
        cols = F.unfold(xd, (kh, kw), padding=padding, stride=stride)
        cols = cols.view(n, c, kh * kw, cols.shape[-1])
        wd = wd.reshape(o, c, kh * kw)
        acc = torch.zeros((n, o, cols.shape[-1]), dtype=torch.float32)
        for c64 in range(0, c, 64):
            for tap in range(kh * kw):
                for c0 in range(c64, min(c64 + 64, c), 16):
                    step = torch.einsum("ncl,oc->nol", cols[:, c0:c0 + 16, tap], wd[:, c0:c0 + 16, tap])
                    acc = _add_rz(acc, step)
        acc = acc.view(n, o, (h + 2 * padding - kh) // stride + 1, (wi + 2 * padding - kw) // stride + 1)
    if b is not None:
        acc = (acc.double() + b.double().view(1, -1, 1, 1)).float()
    return acc


def _cb(sd, pconv, pbn, x, stride=1, padding=0, fp16=False, groups=1):
    """conv (+ eval BatchNorm).  fp16: folded weights rounded to fp16, fp32 accumulation in the product's order
    (_conv_fp32_steps), fp32 shift added after."""
    if not fp16:
        y = _conv(sd, pconv, x, stride, padding, groups)
        return _bn(sd, pbn, y) if pbn else y
    w, b = sd[pconv + ".weight"], sd.get(pconv + ".bias")
    if pbn:
        scale = sd[pbn + ".weight"] / torch.sqrt(sd[pbn + ".running_var"] + 1e-5)
        w = w * scale.view(-1, 1, 1, 1)
        b = sd[pbn + ".bias"] - sd[pbn + ".running_mean"] * scale
    return _conv_fp32_steps(x, w.half().float(), b, stride, padding, groups)


# MobileNetV2 (odtk/backbones/mobilenet.py:5-25 over torchvision mobilenetv2.py: features[0] 3x3 s2 conv + BN + ReLU6,
# features[1..17] InvertedResidual = [1x1 expand + BN + ReLU6 unless t == 1] + depthwise 3x3 + BN + ReLU6 + 1x1 project + BN,
# residual when stride 1 and cin == cout; FPN taps after features[6], [13], [17] (fpn.py:92-93))
MOBILENET = {"MobileNetV2FPN": [(1, 16, 1, 1), (6, 24, 2, 2), (6, 32, 3, 2), (6, 64, 4, 2), (6, 96, 3, 1), (6, 160, 3, 2), (6, 320, 1, 1)]}


def _features_mobilenet(sd, backbone, x, fp16):
    f = "backbones.%s.features.features." % backbone
    x = _q(x, fp16)
    x = _q(F.relu6(_cb(sd, f + "0.0", f + "0.1", x, 2, 1, fp16)), fp16)
    taps, cin, idx = {}, 32, 1
    for t, c, n, s in MOBILENET[backbone]:
        for i in range(n):
            stride, p, k = (s if i == 0 else 1), f + "%d.conv." % idx, 0
            h = x
            if t != 1:
                h = _q(F.relu6(_cb(sd, p + "0.0", p + "0.1", h, 1, 0, fp16)), fp16)
                k = 1
            h = _q(F.relu6(_cb(sd, p + "%d.0" % k, p + "%d.1" % k, h, stride, 1, fp16, groups=h.shape[1])), fp16)
            h = _cb(sd, p + "%d" % (k + 1), p + "%d" % (k + 2), h, 1, 0, fp16)
            x = _q(h + x if (stride == 1 and cin == c) else h, fp16)
            if idx in (6, 13, 17):
                taps[idx] = x
            cin, idx = c, idx + 1
    return taps[6], taps[13], taps[17]


def features(sd, backbone, x, fp16=False):
    if backbone in MOBILENET:
        c3, c4, c5 = _features_mobilenet(sd, backbone, x, fp16)
        return _fpn(sd, backbone, c3, c4, c5, fp16)
    block, layers = LAYERS[backbone]
    f = "backbones.%s.features." % backbone
    x = _q(x, fp16)
    x = _q(F.relu(_cb(sd, f + "conv1", f + "bn1", x, 2, 3, fp16)), fp16)
    x = F.max_pool2d(x, 3, 2, 1)
    outs = []
    for li, nblocks in enumerate(layers):
        for b in range(nblocks):
            stride = 2 if (b == 0 and li > 0) else 1
            p = f + "layer%d.%d." % (li + 1, b)
            identity = x
            if block == "bottleneck":
                out = _q(F.relu(_cb(sd, p + "conv1", p + "bn1", x, 1, 0, fp16)), fp16)
                out = _q(F.relu(_cb(sd, p + "conv2", p + "bn2", out, stride, 1, fp16, GROUPS.get(backbone, 1))), fp16)
                out = _cb(sd, p + "conv3", p + "bn3", out, 1, 0, fp16)
            else:
                out = _q(F.relu(_cb(sd, p + "conv1", p + "bn1", x, stride, 1, fp16)), fp16)
                out = _cb(sd, p + "conv2", p + "bn2", out, 1, 1, fp16)
            if (p + "downsample.0.weight") in sd:
                identity = _cb(sd, p + "downsample.0", p + "downsample.1", x, stride, 0, fp16)
                # the product path computes the stride-1 projection of layer1's first bottleneck block inside the fused
                # block kernel (bottleneck.cu) and adds it in fp32; every other projected identity is stored in fp16
                if not (block == "bottleneck" and stride == 1 and backbone not in GROUPS):
                    identity = _q(identity, fp16)
            x = _q(F.relu(out + identity), fp16)
        if li >= 1:
            outs.append(x)
    c3, c4, c5 = outs
    return _fpn(sd, backbone, c3, c4, c5, fp16)


def _fpn(sd, backbone, c3, c4, c5, fp16):
    n = "backbones.%s." % backbone
    p5 = _q(_cb(sd, n + "lateral5", None, c5, 1, 0, fp16), fp16)
    p4 = _q(F.interpolate(p5, scale_factor=2) + _cb(sd, n + "lateral4", None, c4, 1, 0, fp16), fp16)
    p3 = _q(F.interpolate(p4, scale_factor=2) + _cb(sd, n + "lateral3", None, c3, 1, 0, fp16), fp16)
    p6 = _q(_cb(sd, n + "pyramid6", None, c5, 2, 1, fp16), fp16)
    p7 = _q(_cb(sd, n + "pyramid7", None, F.relu(p6), 2, 1, fp16), fp16)
    return [_q(_cb(sd, n + "smooth3", None, p3, 1, 1, fp16), fp16), _q(_cb(sd, n + "smooth4", None, p4, 1, 1, fp16), fp16),
            _q(_cb(sd, n + "smooth5", None, p5, 1, 1, fp16), fp16), p6, p7]


def head(sd, name, t, fp16=False):
    for i in (0, 2, 4, 6):
        t = _q(F.relu(_cb(sd, "%s.%d" % (name, i), None, t, 1, 1, fp16)), fp16)
    return _cb(sd, "%s.8" % name, None, t, 1, 1, fp16)            # head outputs stay fp32


def forward_heads(sd, backbone, x, sigmoid=True, fp16=False):
    """== reference Model.forward with exporting=True (odtk/model.py:130-144); fp16=True: with the product path's
    roundings (see above)."""
    with torch.no_grad():
        sd = {k: v.float() for k, v in sd.items()}
        feats = features(sd, backbone, x.float(), fp16)
        cls = [head(sd, "cls_head", t, fp16) for t in feats]
        box = [head(sd, "box_head", t, fp16) for t in feats]
        if sigmoid:
            cls = [c.sigmoid() for c in cls]
    return cls, box


def postprocess(cls_heads, box_heads, width, ratios=None, scales=None, angles=None, rotated=False,
                threshold=0.05, top_n=1000, nms=0.5, detections=100, return_index=False):
    """odtk/model.py:146-165 with the CUDA semantics of decode / nms (oracle/odtk_oracle.c)."""
    ratios = ratios or oracle.DEFAULT_RATIOS
    scales = scales or oracle.DEFAULT_SCALES
    outs = []
    for c, b in zip(cls_heads, box_heads):
        c = c.numpy() if torch.is_tensor(c) else c
        b = b.numpy() if torch.is_tensor(b) else b
        stride = width // c.shape[-1]
        anchors = (oracle.generate_anchors_rotated_axis(stride, ratios, scales, angles or oracle.DEFAULT_ANGLES)
                   if rotated else oracle.generate_anchors(stride, ratios, scales))
        outs.append(oracle.decode(c, b, anchors.reshape(-1), stride, threshold, top_n, rotated))
    cat = [np.concatenate(t, 1) for t in zip(*outs)]
    return oracle.nms(cat[0], cat[1], cat[2], nms, detections, rotated=rotated, return_index=return_index), cat


def forward(sd, backbone, x, fp16=False, **kw):
    cls, box = forward_heads(sd, backbone, x, fp16=fp16)
    return postprocess(cls, box, x.shape[-1], **kw)[0]
