#!/usr/bin/env python
"""bench.py -- the driver-facing benchmark of the RetinaNet inference hot path (see DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload full|postproc] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One JSON line on rank 0.  A "step" is one pass of the hot path over one batch of synthetic input:
`full` (default, BASELINE.json configs[2]) = Model.forward: backbone + FPN + heads + decode + NMS
on [B, 3, 800, 1280] fp16; `postproc` (configs[1]) = decode + NMS on pre-computed head outputs.
`value` is device-timed whole-job throughput with inputs resident in HBM; `e2e` is the same metric
through the public API with HOST (pinned) buffers and the host<->device copies inside the timed
region; `roofline` describes the dominant kernel (live CUDA-event timing on the launching stream);
`cpu_baseline` is the CPU oracle timed on this box's host cores (rank 0, N=1).  With N > 1 every rank
runs the same per-GPU batch on its own images (weak scaling, image-wise sharding) and the detections
of all ranks are gathered with one NCCL all-gather per step inside the timed region.
Every timed loop runs exactly --steps steps.  --dump-outputs DIR writes what the last step of the measured pass
returned (scores, boxes, classes of every image; see dump_outputs) as DIR/<name>.npy; the inputs and weights are
seeded, so two builds of the project can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": d["hbm_gbs"], "tensor": d["bf16_tflops"], "tensor_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured"}
    return {"hbm": 6650.0, "tensor": 1590.0, "tensor_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], None, set(), []
        for (t, line) in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                mx = float(f[1])
                if t0 - 0.05 <= t <= t1 + 0.05:
                    sm.append(float(f[0]))
                    power.append(float(f[2]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                pass
        if not sm:   # region shorter than the sampling period: use every sample we have
            for (t, line) in self.rows:
                try:
                    sm.append(float(line.split(",")[0]))
                except ValueError:
                    pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


def _prof_get(lib, tag):
    ms, n = ctypes.c_double(0), ctypes.c_longlong(0)
    lib.odtk_prof_get(tag, ctypes.byref(ms), ctypes.byref(n))
    return ms.value, n.value


# =================================================================================================
# workload: full model (BASELINE.json configs[2]: ResNet50FPN fp16, batch 32 per GPU, 3x800x1280)
# =================================================================================================
class FullWorkload:
    metric = "images/sec (3x800x1280 fp16, backbone+FPN+heads+decode+NMS)"
    dtype = "f16"
    H, W = 800, 1280

    def __init__(self, backbone, batch, rank, device, rotated=False):
        import torch
        from retinanet_examples_b200 import engine, synth
        from retinanet_examples_b200.model import Model, make_state_dict
        self.torch, self.batch, self.device, self.engine = torch, batch, device, engine
        self.backbone = backbone
        self.rotated, self.nbox, na = rotated, (6 if rotated else 4), (27 if rotated else 9)
        self.name = "%s fp16%s, batch %d per GPU, full backbone+FPN+heads+decode+NMS, 3x800x1280 (BASELINE configs[%d])" % (
            backbone, " --rotated-bbox (27 anchors, 5-param boxes, rotated-IoU NMS)" if rotated else "", batch, 4 if rotated else 2)
        g = torch.Generator().manual_seed(1000 + rank)
        self.host_x = torch.randn((batch, 3, self.H, self.W), generator=g).to(torch.float16) \
            .contiguous(memory_format=torch.channels_last).pin_memory()
        self.dev_x = self.host_x.to(device)
        sd = make_state_dict(backbone, 80, na, rotated, seed=0)
        model = Model(backbone, classes=80, rotated_bbox=rotated)

        def gpu_logits(s):   # probe: 2 images through the CUDA engine
            model.load_state_dict(s).cuda(device.index)
            return model.forward_heads(self.dev_x[:2], sigmoid=False)[0]
        self.sd = synth.calibrate_cls_head(sd, gpu_logits)
        self.model = model.load_state_dict(self.sd).cuda(device.index)
        if os.environ.get("ODTK_BENCH_CUDA_GRAPH", "1") != "0":
            self.model.enable_cuda_graph()
        self.det = self.model.detections
        self.h2d_bytes = self.host_x.numel() * 2
        self.d2h_bytes = batch * self.det * (2 + self.nbox) * 4
        self.host_out = torch.empty((batch, self.det, 2 + self.nbox), dtype=torch.float32).pin_memory()
        self.out = None
        self.world_gather = None
        self.peer = None
        engine.STATS["launches"] = engine.STATS["conv_flops"] = 0
        engine.STATS["trace"] = []
        self.model.parallel_heads = False         # trace in the order step_profile() launches
        self.model.forward(self.dev_x)            # eager pass: counts launches / algorithmic FLOPs
        self.model.parallel_heads = True
        torch.cuda.synchronize()
        self.trace, engine.STATS["trace"] = engine.STATS["trace"], None
        if os.environ.get("ODTK_BENCH_TRACE"):
            json.dump(self.trace, open(os.environ["ODTK_BENCH_TRACE"], "w"))
        # + decode (filter, gather, select: the filter launch disappears when the class head's last
        #   convolution appends the candidates itself) + nms (1); memsets are not counted
        self.launches_per_step = engine.STATS["launches"] + (3 if self.model.fused_candidates else 4)
        self.flops_per_step = engine.STATS["conv_flops"]

    def enable_gather(self, world):
        """Image-wise sharding over `world` ranks.  Default: the NMS kernel itself pushes this rank's detections into every
        rank's gather buffer over NVLink peer memory (peer.PeerGather; inside the CUDA graph, no collective launch);
        ODTK_BENCH_GATHER=nccl keeps round 1's host-launched ncclAllGather per step."""
        self.world_gather = world
        if os.environ.get("ODTK_BENCH_GATHER", "peer") != "nccl":
            from retinanet_examples_b200 import peer
            self.peer = peer.PeerGather(self.batch, detections=self.det, nbox=self.nbox)
            self.model.attach_gather(self.peer)

    def _gather(self, out):
        if self.peer is not None:
            from retinanet_examples_b200 import infer
            return infer.split_packed(self.peer.gathered())      # views of the rows the kernels already delivered
        if self.world_gather:
            from retinanet_examples_b200 import infer
            return infer.gather_detections(*out, world=self.world_gather)
        return out

    def step(self):
        self.out = self._gather(self.model(self.dev_x, static_input=True))

    def step_profile(self):
        """Same step launched eagerly (a CUDA-graph replay runs no host code, so the per-kernel
        CUDA events of the roofline pass can only be recorded around eager launches)."""
        self.model.parallel_heads = False       # one stream: per-kernel event times must not overlap
        try:
            self.out = self._gather(self.model.forward(self.dev_x))
        finally:
            self.model.parallel_heads = True

    def step_e2e(self):
        """One end-to-end step through the public API: this step's images travel pinned host -> device,
        Model.forward runs, the packed detections travel device -> pinned host.  The upload of step k+1
        is issued on a copy stream while step k computes (double-buffered, like any input pipeline;
        the reference overlaps its loader the same way), every byte still moves inside the timed region."""
        torch = self.torch
        main = torch.cuda.current_stream()
        if not hasattr(self, "_e2e"):
            self._e2e = {"copy": torch.cuda.Stream(), "buf": [torch.empty_like(self.dev_x), torch.empty_like(self.dev_x)],
                         "ready": [torch.cuda.Event(), torch.cuda.Event()], "free": [torch.cuda.Event(), torch.cuda.Event()],
                         "k": 0, "primed": False}
        e = self._e2e

        def upload(i):
            with torch.cuda.stream(e["copy"]):
                e["copy"].wait_event(e["free"][i])          # the step that last read this buffer is done
                e["buf"][i].copy_(self.host_x, non_blocking=True)
                e["ready"][i].record(e["copy"])
        if not e["primed"]:
            e["free"][0].record(main); e["free"][1].record(main)
            upload(0)
            e["primed"] = True
        i = e["k"] & 1
        upload(i ^ 1)                                       # next step's input, overlapped with this step
        main.wait_event(e["ready"][i])
        s, b, c = self.model(e["buf"][i], static_input=True)      # graph reads the upload buffer in place
        e["free"][i].record(main)
        lag = os.environ.get("ODTK_BENCH_E2E_LAG", "0") == "1"   # experimental (off): read step k's result back while
        if lag and "hout" not in e:                               # step k+1 computes, instead of idling the GPU on it
            e["hout"] = [self.host_out, torch.empty_like(self.host_out).pin_memory()]
            e["done"] = [torch.cuda.Event(), torch.cuda.Event()]
        hout = e["hout"][e["k"] & 1] if lag else self.host_out
        hout.copy_(self.model.last_packed, non_blocking=True)      # the NMS kernel wrote the packed rows itself
        self._gather((s, b, c))
        if lag:
            e["done"][e["k"] & 1].record(main)
            if e["k"] > 0:
                e["done"][(e["k"] - 1) & 1].synchronize()         # the PREVIOUS step's result is on the host
            e["k"] += 1
            return
        e["k"] += 1
        main.synchronize()                                  # the step's result is on the host

    def latency(self, reps):
        """Single-request latency of one batch, input resident, host-blocking per call (what a caller at batch 1 sees):
        CUDA-graph replay and eager launches (the eager path re-uses cached tensor maps, csrc/conv.cu)."""
        torch = self.torch
        out = {}
        for name, fn in (("graph_ms", lambda: self.model(self.dev_x, static_input=True)), ("eager_ms", lambda: self.model.forward(self.dev_x))):
            if self.peer is not None and name == "eager_ms":
                continue                 # all ranks must run the same number of gathering steps
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) * 1e3)
            out[name] = round(sorted(ts)[len(ts) // 2], 3)
        return out

    def units_per_step(self):
        return self.batch

    def config(self):
        n_det = int((self.out[0] > 0).sum().item())
        return {"workload": self.name, "images_per_gpu": self.batch, "classes": 80, "anchors": 27 if self.rotated else 9,
                "conv_gflop_per_image": round(self.flops_per_step / self.batch / 1e9, 2),
                "weights": "random init (seed 0), BatchNorm folded, class head calibrated to ~0.56% scores > 0.05",
                "cuda_graph": getattr(self.model, "_graphs", None) is not None,
                "detections_in_last_step": n_det,
                "l2": "activations of a step (GBs) exceed the 126 MB L2; input batch %.0f MB" % (self.h2d_bytes / 1e6)}

    PROFILE = "r02_layer_table.json"

    def _profiled_traffic(self):
        if not (self.backbone == "ResNet50FPN" and self.batch == 32 and not self.rotated):
            return None
        try:
            return int(json.load(open(os.path.join(ROOT, "profiles", self.PROFILE)))["summary"]["conv_dram_bytes"])
        except (OSError, KeyError, ValueError):
            return None

    def roofline(self, lib, peaks, steps):
        ms, n = _prof_get(lib, 3)
        if n == 0:
            return None
        flops = float(self.flops_per_step) * steps
        achieved = flops / (ms * 1e-3) / 1e12
        peak = peaks["tensor_sustained"] or peaks["tensor"]
        # layer-by-layer speed of light: every launch at max(FLOPs / tensor peak, algorithmic bytes / HBM peak)
        t_tc = [l["flops"] / (peak * 1e12) for l in self.trace]
        t_hbm = [l["bytes"] / (peaks["hbm"] * 1e9) for l in self.trace]
        ideal = [max(a, b) for a, b in zip(t_tc, t_hbm)]
        self.layerwise = {"ideal_ms_per_step": round(sum(ideal) * 1e3, 3),
                          "tensor_bound_ms": round(sum(i for i, a, b in zip(ideal, t_tc, t_hbm) if a >= b) * 1e3, 3),
                          "hbm_bound_ms": round(sum(i for i, a, b in zip(ideal, t_tc, t_hbm) if a < b) * 1e3, 3),
                          "algorithmic_bytes_per_step": int(sum(l["bytes"] for l in self.trace)),
                          "note": "sum over the step's launches of max(FLOPs/tensor peak, operand+output bytes/HBM peak): "
                                  "the bound of layer-by-layer execution; frac_of_step = ideal / measured ms_per_step"}
        return {"kernel": "conv_gemm_kernel + bottleneck_tail_kernel + stem_pool_kernel (tcgen05, all %d conv launches of a step)" % (n // steps), "bound": "tensor",
                "achieved": round(achieved, 1), "peak": peak, "unit": "TFLOP/s", "frac": round(achieved / peak, 4),
                # dram__bytes_read.sum + dram__bytes_write.sum summed over the conv launches of ONE step, from the
                # committed ncu capture of this workload (tools/capture_step.py -> profiles/r02_layer_table.json)
                "traffic": self._profiled_traffic(),
                "traffic_note": "bytes per step (all conv launches), from profiles/%s (ncu, same workload)" % self.PROFILE,
                "peak_source": peaks["source"] + " (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)",
                "avg_launch_ms": round(ms / n, 5), "launches_timed": n,
                "algorithmic_flops_per_step": int(self.flops_per_step),
                "conv_share_of_step": None}

    # ---- CPU legs (oracle port of the reference's PyTorch-CPU path; rank 0 only) --------------------
    @staticmethod
    def cpu_threads():
        """A FIXED thread count for every CPU leg: the cores this process may run on, capped at 32 (one image's
        convolutions stop scaling there and the GPU boxes' hosts are shared)."""
        try:
            n = len(os.sched_getaffinity(0))
        except AttributeError:
            n = os.cpu_count() or 1
        return max(1, min(n, 32))

    @staticmethod
    def cpu_run(backbone, sd, nimg, reps, H=800, W=1280, rotated=False, warmup=1):
        """`reps` timed passes of the CPU oracle port over `nimg` images each (after `warmup` untimed ones).
        Returns (list of per-pass seconds, threads used)."""
        import torch
        from oracle import model_ref
        nt = FullWorkload.cpu_threads()
        torch.set_num_threads(nt)
        x = torch.randn((nimg, 3, H, W), generator=torch.Generator().manual_seed(7))
        for _ in range(max(1, warmup)):
            model_ref.forward(sd, backbone, x, rotated=rotated)
        times = []
        for _ in range(reps):
            t0 = time.perf_counter()
            model_ref.forward(sd, backbone, x, rotated=rotated)
            times.append(time.perf_counter() - t0)
        return times, torch.get_num_threads()

    def cpu_baseline(self):
        times, cores = self.cpu_run(self.backbone, self.sd, 1, 5, rotated=self.rotated, warmup=2)
        med = sorted(times)[len(times) // 2]
        return {"value": round(1.0 / med, 3), "unit": "images/sec", "cores": cores, "kind": "port",
                "sample": "median of 5 x 1 image 3x800x1280 fp32 (2 warm-up), oracle/model_ref.py (torch CPU convs, same "
                          "weights) + oracle decode/nms, %d threads; the reference's own PyTorch-CPU path restated" % cores}


# =================================================================================================
# workload: decode + NMS only (BASELINE.json configs[1]: RN50FPN head shapes, batch 8 per GPU)
# =================================================================================================
class PostprocWorkload:
    metric = "decode+NMS images/sec (3x800x1280 head outputs, fp32 NCHW entry point)"
    dtype = "f32"

    def __init__(self, batch, rank, device, rotated=False):
        import torch
        from retinanet_examples_b200 import box, synth
        self.torch, self.batch, self.device = torch, batch, device
        self.rotated, self.nbox = rotated, (6 if rotated else 4)
        self.name = "decode+nms only, ResNet50FPN head shapes 3x800x1280, 80 classes, %d anchors%s, batch %d (BASELINE configs[%d])" % (
            27 if rotated else 9, ", rotated 5-param boxes + rotated-IoU NMS" if rotated else "", batch, 4 if rotated else 1)
        cls, deltas = synth.head_outputs(batch, seed=rank, rotated=rotated, anchors=27 if rotated else 9)
        self.host = [(c.pin_memory(), d.pin_memory()) for c, d in zip(cls, deltas)]
        self.dev = [(c.to(device), d.to(device)) for c, d in self.host]
        if rotated:
            self.anchors = [box.generate_anchors_rotated(s, box.DEFAULT_RATIOS, box.DEFAULT_SCALES, box.DEFAULT_ANGLES)[0]
                            .reshape(-1).tolist() for s in synth.LEVEL_STRIDES]
        else:
            self.anchors = [box.generate_anchors(s, box.DEFAULT_RATIOS, box.DEFAULT_SCALES).reshape(-1).tolist()
                            for s in synth.LEVEL_STRIDES]
        self.strides = synth.LEVEL_STRIDES
        self.top_n, self.det = 1000, 100
        self.h2d_bytes = sum(c.numel() * 4 + d.numel() * 4 for c, d in self.host)
        self.d2h_bytes = batch * self.det * (2 + self.nbox) * 4
        self.out = None
        self.host_out = torch.empty((batch, self.det, 2 + self.nbox), dtype=torch.float32).pin_memory()
        self.launches_per_step = 3 + 1   # filter, gather, select+decode (all levels), nms
        self.level_score_bytes = [c.numel() * 4 for c, _ in self.host]
        self.world_gather = None
        # throughput mode: consecutive batches alternate between CUDA streams, so the HBM-bound score filter of batch k+1
        # runs next to the latency-bound select + NMS of batch k (a few CTAs); per-batch latency is unchanged
        self.nstreams = int(os.environ.get("ODTK_BENCH_POSTPROC_STREAMS", "3"))
        self.streams = [torch.cuda.Stream(device=device) for _ in range(self.nstreams)] if self.nstreams > 1 else []
        self.k = 0
        self.graphs = []

    def _capture(self):
        """One CUDA graph of the step per stream (its own output / workspace buffers): the five launches of a step take
        less GPU time than their host-side enqueue, so the pipelined mode replays graphs."""
        torch = self.torch
        for s in self.streams:
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self._run(self.dev)
            s.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                out = self._run(self.dev)
            self.graphs.append((g, out))

    def _run(self, tensors):
        from retinanet_examples_b200 import _C
        scores, boxes, classes = _C.decode_levels([c for c, _ in tensors], [d for _, d in tensors], self.anchors,
                                                  self.strides, 0.05, self.top_n, self.rotated)
        return _C.nms(scores, boxes, classes, 0.5, self.det, self.rotated)

    def step(self):
        if not self.streams:
            self.out = self._run(self.dev)
            return
        torch = self.torch
        if not self.graphs:
            self._capture()
        i = self.k % self.nstreams
        main, side = torch.cuda.current_stream(), self.streams[i]
        self.k += 1
        side.wait_stream(main)                    # ordered after whatever the caller enqueued (the timing start event)
        with torch.cuda.stream(side):
            self.graphs[i][0].replay()
        self.out = self.graphs[i][1]

    def step_profile(self):
        """Eager, one stream: the library's per-kernel event brackets see every launch (roofline pass, latency)."""
        self.out = self._run(self.dev)

    def drain(self):
        """The caller's stream waits for every batch still in flight (called before the timing end event)."""
        for s in self.streams:
            self.torch.cuda.current_stream().wait_stream(s)

    def step_e2e(self):
        torch = self.torch
        dev = [(c.to(self.device, non_blocking=True), d.to(self.device, non_blocking=True)) for c, d in self.host]
        s, b, c = self._run(dev)
        packed = torch.cat([s[..., None], b, c[..., None]], dim=2)
        self.host_out.copy_(packed, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def units_per_step(self):
        return self.batch

    def config(self):
        return {"workload": self.name, "images_per_gpu": self.batch, "top_n": 1000, "detections": 100,
                "threshold": 0.05, "nms": 0.5, "batches_in_flight": max(1, self.nstreams),
                "l2": "inputs (%.0f MB per step per GPU) exceed the 126 MB L2" % (self.h2d_bytes / 1e6)}

    def roofline(self, lib, peaks, steps):
        ms, n = _prof_get(lib, 0)
        if n == 0:
            return None
        bytes_per_launch = float(sum(self.level_score_bytes))
        avg_ms = ms / n
        achieved = bytes_per_launch / (avg_ms * 1e-3) / 1e9
        return {"kernel": "score_filter_kernel", "bound": "hbm", "achieved": round(achieved, 1),
                "peak": peaks["hbm"], "unit": "GB/s", "frac": round(achieved / peaks["hbm"], 4),
                # ncu --set full capture of this kernel at batch 8 (profiles/r01_score_filter_ncu_summary.json)
                "traffic": 497508352 if (self.batch == 8 and not self.rotated) else None, "peak_source": peaks["source"] + " (MEASURED_PEAKS.json hbm_gbs, burst copy)",
                "avg_launch_ms": round(avg_ms, 5), "launches_timed": n,
                "algorithmic_bytes_per_launch": int(bytes_per_launch),
                "note": "one launch per step streams the scores of all 5 levels of the batch"}

    def cpu_once(self, nimg):
        import numpy as np
        from oracle import oracle
        outs = []
        t0 = time.perf_counter()
        for lvl, (c, d) in enumerate(self.host):
            outs.append(oracle.decode(c[:nimg].numpy(), d[:nimg].numpy(), np.asarray(self.anchors[lvl], np.float32),
                                      self.strides[lvl], 0.05, self.top_n, getattr(self, "rotated", False)))
        cat = [np.concatenate(t, 1) for t in zip(*outs)]
        oracle.nms(cat[0], cat[1], cat[2], 0.5, self.det, rotated=getattr(self, "rotated", False))
        return time.perf_counter() - t0

    def cpu_baseline(self):
        nimg = min(self.batch, 4)
        self.cpu_once(1)
        dt = self.cpu_once(nimg)
        return {"value": round(nimg / dt, 3), "unit": "images/sec", "cores": 1, "kind": "port",
                "sample": "%d images of the same batch, all 5 levels, oracle/odtk_oracle.c decode+nms, 1 thread" % nimg}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """arrays: name -> float32 [B, ...] numpy array, one row per image, written as out_dir/<name>.npy.  Past DUMP_LIMIT_BYTES
    in all, the rows of a fixed seeded sample of images are written instead and their positions in the batch go to
    out_dir/image_index.npy (float64)."""
    import numpy as np
    n = next(iter(arrays.values())).shape[0]
    per_image = sum(v.nbytes for v in arrays.values()) // max(n, 1)
    keep = min(n, DUMP_LIMIT_BYTES // max(per_image, 1))
    if keep < n:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["image_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


# BASELINE.json `configs` (and north_star's batch 1 / 8 / 32) as presets of the flags below
CONFIGS = {
    "b1": {"workload": "full", "batch": 1}, "b8": {"workload": "full", "batch": 8}, "b32": {"workload": "full", "batch": 32},
    "rn101x8": {"workload": "full", "backbone": "ResNet101FPN", "batch": 8},      # configs[3]: launch with --gpus 8 (64 images / step)
    "rotated": {"workload": "full", "batch": 8, "rotated": True},                  # configs[4]
    "postproc": {"workload": "postproc", "batch": 8},                              # configs[1]
    "postproc_rotated": {"workload": "postproc", "batch": 8, "rotated": True},
}


def postproc_sub(device, peaks, lib, steps, rotated=False, batch=8):
    """decode + NMS alone (the second half of BASELINE.json's metric, configs[1]: head outputs of 8 images, fp32 NCHW entry
    points): microseconds per image, device-timed -- throughput with 3 batches in flight (CUDA graphs on 3 streams) and
    one batch at a time (eager, per-kernel event brackets) -- plus the streaming kernel's HBM roofline."""
    import torch
    wl = PostprocWorkload(batch, 0, device, rotated)
    for _ in range(3):
        wl.step()
    wl.drain()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        wl.step()
    wl.drain()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    # the same batches one after the other on one stream, eagerly, every kernel bracketed by events
    for _ in range(2):
        wl.step_profile()
    lib.odtk_prof_reset()
    lib.odtk_prof_enable(1)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        wl.step_profile()
    e1.record()
    torch.cuda.synchronize()
    lib.odtk_prof_enable(0)
    serial_ms = e0.elapsed_time(e1)
    roof = wl.roofline(lib, peaks, steps)
    nms_ms, nms_n = _prof_get(lib, 2)
    sel_ms, sel_n = _prof_get(lib, 1)
    return {"workload": wl.name, "us_per_image": round(ms * 1e3 / steps / batch, 2), "images_per_gpu": batch, "steps": steps,
            "batches_in_flight": max(1, wl.nstreams), "latency_us_per_batch": round(serial_ms * 1e3 / steps, 1),
            "us_per_image_one_batch_at_a_time": round(serial_ms * 1e3 / steps / batch, 2),
            "images_per_sec": round(batch * steps / (ms * 1e-3), 1),
            "hbm_floor_us_per_image": round(sum(wl.level_score_bytes) / batch / (peaks["hbm"] * 1e9) * 1e6, 2),
            "nms_us_per_launch": round(nms_ms * 1e3 / max(nms_n, 1), 2), "select_decode_us_per_step": round(sel_ms * 1e3 / steps, 2),
            "note": "per-kernel times come from event-bracketed launches of the one-batch-at-a-time loop", "roofline": roof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="full", choices=["full", "postproc"])
    ap.add_argument("--backbone", default="ResNet50FPN")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: 32 full, 8 postproc)")
    ap.add_argument("--rotated", action="store_true", help="BASELINE configs[4]: --rotated-bbox model / rotated decode+NMS")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-postproc", action="store_true", help="skip the decode+NMS sub-measurement of the default line")
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS),
                    help="BASELINE.json matrix presets: " + ", ".join("%s = %s" % kv for kv in sorted(CONFIGS.items())))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the scores / boxes / classes the last measured step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    if args.config:
        for k, v in CONFIGS[args.config].items():
            setattr(args, k, v)
    args.warmup = max(args.warmup, 3)
    if not args.batch:
        args.batch = 32 if args.workload == "full" else 8

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        return reference_arm(args, rank, world)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    from retinanet_examples_b200 import _lib
    lib = _lib.lib()
    peaks = _peaks()

    wl = FullWorkload(args.backbone, args.batch, rank, device, args.rotated) if args.workload == "full" else \
        PostprocWorkload(args.batch, rank, device, args.rotated)
    if world > 1:
        if hasattr(wl, "enable_gather"):
            wl.enable_gather(world)
        else:
            wl.world_gather = world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile):
        lib.odtk_prof_reset()
        lib.odtk_prof_enable(1 if profile else 0)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            fn()
        if getattr(wl, "drain", None):
            wl.drain()
        e1.record()
        barrier()
        t1 = time.time()
        lib.odtk_prof_enable(0)
        ms = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), t0, t1

    with torch.no_grad():
        for _ in range(args.warmup):
            wl.step()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
            time.sleep(0.3)
        # pass 1: the measured value (no per-kernel events in the stream)
        ms, t0, t1 = timed(wl.step, args.steps, profile=False)
        last = {k: t.float().cpu().numpy() for k, t in zip(("scores", "boxes", "classes"), wl.out)} \
            if args.dump_outputs and rank == 0 else None
        clocks = sampler.stop(t0, t1) if rank == 0 else None
        # pass 2: same steps with the dominant kernel bracketed by CUDA events (roofline numbers)
        ms_prof, _, _ = timed(getattr(wl, "step_profile", wl.step), args.steps, profile=True)
        roof = wl.roofline(lib, peaks, args.steps)
        if roof is not None and "conv_share_of_step" in roof:
            # share of the step's summed KERNEL time (every launch of the eager, single-stream step is bracketed by
            # events: decode 0-1, nms 2, conv 3, pad / max-pool / lowering 5) -- comparable with the ncu launch list
            cms, _ = _prof_get(lib, 3)
            kernel_ms = sum(_prof_get(lib, t)[0] for t in (0, 1, 2, 3, 5))
            roof["conv_share_of_step"] = round(cms / kernel_ms, 4)
            roof["kernel_ms_per_step"] = round(kernel_ms / args.steps, 4)
            roof["eager_ms_per_step"] = round(ms_prof / args.steps, 4)
        if roof is not None and os.environ.get("ODTK_BENCH_INSTEP") and hasattr(wl, "trace"):
            # in-step per-layer table: per-launch event times of the LAST eager step (tags: conv 3, small layers 5), joined
            # with the engine trace of one step in launch order
            per = {}
            for tag, kinds in ((3, ("conv1x1", "conv3x3", "stem7x7", "stem_pool", "bneck_tail")), (5, ("pad_input", "maxpool", "lower_conv", "relu", "preprocess_u8"))):
                tr = [t for t in wl.trace if t["kind"] in kinds]
                buf = (ctypes.c_float * max(1, len(tr)))()
                n = lib.odtk_prof_get_list(tag, buf, len(tr)) if tr else 0
                if n == len(tr):
                    for t, v in zip(tr, buf):
                        key = "%s %dx%dx%d %s->%s%s%s%s" % (t["kind"], t["n"], t["h"], t["w"], t["cin"], t.get("cout", ""),
                                                          " s2" if t.get("stride") == 2 else "", " +res" if t.get("residual") else "",
                                                          " +up" if t.get("upsample") else "")
                        g = per.setdefault(key, {"n": 0, "ms": 0.0, "flops": 0, "bytes": 0})
                        g["n"] += 1; g["ms"] += float(v); g["flops"] += t["flops"]; g["bytes"] += t["bytes"]
            tot = sum(g["ms"] for g in per.values())
            rows = [dict(layer=k, n=g["n"], us=round(g["ms"] * 1e3, 1), share=round(g["ms"] / max(tot, 1e-9), 4),
                         tflops=round(g["flops"] / max(g["ms"], 1e-9) / 1e9, 1), gbs=round(g["bytes"] / max(g["ms"], 1e-9) / 1e6, 1))
                    for k, g in sorted(per.items(), key=lambda kv: -kv[1]["ms"])]
            json.dump({"sum_us": round(tot * 1e3, 1), "rows": rows}, open(os.environ["ODTK_BENCH_INSTEP"], "w"), indent=1)
        if roof is not None and getattr(wl, "layerwise", None):
            wl.layerwise["frac_of_step"] = round(wl.layerwise["ideal_ms_per_step"] / (ms / args.steps), 4)
            roof["layerwise"] = wl.layerwise
        ms_e2e = None
        if not args.no_e2e:
            for _ in range(2):
                wl.step_e2e()
            ms_e2e, _, _ = timed(wl.step_e2e, args.steps, profile=False)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    units = wl.units_per_step() * world
    cfg = wl.config()
    cfg.update({"global_batch": units,
                "parallelism": ("image-wise sharding over %d GPUs, detections of all ranks delivered to every rank each step (see config.gather)" % world)
                if world > 1 else "single GPU"})
    out = {
        "metric": wl.metric, "value": round(units * args.steps / (ms * 1e-3), 2), "unit": "images/sec",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
        "config": cfg,
        "us_per_image": round(ms * 1e3 / args.steps / wl.units_per_step(), 3),
        "clocks": clocks,
        "gpu_launches": wl.launches_per_step * args.steps,
        "roofline": roof,
    }
    if ms_e2e is not None:
        out["e2e"] = {"value": round(units * args.steps / (ms_e2e * 1e-3), 2), "unit": "images/sec",
                      "h2d_bytes_per_step": wl.h2d_bytes, "d2h_bytes_per_step": wl.d2h_bytes,
                      "ms_per_step": round(ms_e2e / args.steps, 4)}
    if world > 1 and args.workload == "full":
        out["config"]["gather"] = ("in-kernel: every rank's NMS kernel stores its packed detections into all ranks' buffers over "
                                   "NVLink peer memory, inside the CUDA graph (odtk_nms_gather)") if wl.peer is not None else \
            "one host-launched ncclAllGather of the packed detections per step"
    if world == 1 and args.workload == "full":
        with torch.no_grad():
            out["latency"] = wl.latency(args.steps)
    if world == 1 and args.workload == "full" and not args.no_postproc:
        with torch.no_grad():
            out["postproc"] = postproc_sub(device, peaks, lib, args.steps, rotated=args.rotated)
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = wl.cpu_baseline()
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def reference_arm(args, rank, world):
    """The reference's CPU implementation of the path on this box's host cores.  /root/reference (Python) cannot travel to
    the GPU box, so this is the oracle port: oracle/model_ref.py (the same torch CPU convolutions nn.Conv2d runs) +
    oracle decode/nms.  Protocol (BASELINE.md section 3): --warmup untimed and EXACTLY --steps timed single-image passes
    (one image of the configured workload per step: a bounded sample), a fixed thread count, the MEDIAN pass time is
    the reported step time.  Rank 0 only; other ranks exit 0."""
    if rank != 0:
        return
    import torch
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    if args.workload == "postproc":
        from retinanet_examples_b200 import box, synth
        wl = PostprocWorkload.__new__(PostprocWorkload)
        nimg = 1
        cls, deltas = synth.head_outputs(nimg, seed=0, rotated=args.rotated, anchors=27 if args.rotated else 9)
        wl.torch, wl.batch, wl.rotated = torch, nimg, args.rotated
        wl.host = list(zip(cls, deltas))
        wl.anchors = [(box.generate_anchors_rotated(s, box.DEFAULT_RATIOS, box.DEFAULT_SCALES, box.DEFAULT_ANGLES)[0] if args.rotated
                       else box.generate_anchors(s, box.DEFAULT_RATIOS, box.DEFAULT_SCALES)).reshape(-1).tolist() for s in synth.LEVEL_STRIDES]
        wl.strides, wl.top_n, wl.det = synth.LEVEL_STRIDES, 1000, 100
        for _ in range(warmup):
            wl.cpu_once(1)
        times = [wl.cpu_once(nimg) for _ in range(steps)]
        cores, metric, dtype = 1, PostprocWorkload.metric, "f32"
        name = "decode+nms only, ResNet50FPN head shapes 3x800x1280%s (BASELINE configs[%d])" % (
            ", rotated" if args.rotated else "", 4 if args.rotated else 1)
        what = "1 image, all 5 levels, oracle/odtk_oracle.c decode+nms, 1 thread"
    else:
        from oracle import model_ref
        from retinanet_examples_b200 import synth
        from retinanet_examples_b200.model import make_state_dict
        sd = make_state_dict(args.backbone, 80, 27 if args.rotated else 9, args.rotated, seed=0)
        torch.set_num_threads(FullWorkload.cpu_threads())
        probe = torch.randn((1, 3, 256, 384), generator=torch.Generator().manual_seed(3))
        sd = synth.calibrate_cls_head(sd, lambda s: model_ref.forward_heads(s, args.backbone, probe, sigmoid=False)[0])
        times, cores = FullWorkload.cpu_run(args.backbone, sd, 1, steps, rotated=args.rotated, warmup=warmup)
        metric, dtype = FullWorkload.metric, "f32"
        name = "%s%s, full backbone+FPN+heads+decode+NMS, 3x800x1280 (BASELINE configs[%d] workload on the CPU path)" % (
            args.backbone, " --rotated-bbox" if args.rotated else "", 4 if args.rotated else 2)
        what = "1 image 3x800x1280 fp32, oracle/model_ref.py torch-CPU convs + oracle decode/nms, %d threads" % cores
    med = sorted(times)[len(times) // 2]
    v = round(1.0 / med, 3)
    sample = "median of %d timed steps (%d warm-up) x %s" % (steps, warmup, what)
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": v, "unit": "images/sec", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": round(med * 1e3, 3), "mean_ms_per_step": round(sum(times) / len(times) * 1e3, 3),
        "min_ms_per_step": round(min(times) * 1e3, 3), "max_ms_per_step": round(max(times) * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {"workload": name, "images_per_step": 1, "host_threads": cores, "host_cpus": os.cpu_count()},
        "cpu_baseline": {"value": v, "unit": "images/sec", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


if __name__ == "__main__":
    main()
