"""Join an ncu per-launch CSV of one step (tools/capture_step.py) with the engine trace of the same step:
per-launch duration, DRAM bytes and tensor-pipe activity next to the launch's algorithmic FLOPs / bytes and its
layer-wise speed of light max(FLOPs / tensor peak, bytes / HBM peak).
    python tools/layer_table.py launches.csv step_trace.json [--out profiles/rNN_layer_table] [--tensor-tflops T --hbm-gbs B]
The peaks default to MEASURED_PEAKS.json at the repository root (bf16_tflops_sustained or bf16_tflops, hbm_gbs), measured on
the GPU the capture was taken on; a committed table records the peaks it was computed with."""
import argparse
import collections
import csv
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNEL_KIND = [("conv_gemm_kernel", ("conv1x1", "conv3x3", "stem7x7")), ("bottleneck_tail_kernel", ("bneck_tail",)), ("stem_pool_kernel", ("stem_pool",)), ("lower", ("lower_conv",)), ("maxpool", ("maxpool",)),
               ("pad_input", ("pad_input",)), ("preprocess", ("preprocess_u8",))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("csv")
    ap.add_argument("trace")
    ap.add_argument("--out", default=None)
    ap.add_argument("--tensor-tflops", type=float, default=None, help="tensor-pipe peak, TFLOP/s")
    ap.add_argument("--hbm-gbs", type=float, default=None, help="HBM peak, GB/s")
    args = ap.parse_args()
    tf, bw = args.tensor_tflops, args.hbm_gbs
    if tf is None or bw is None:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        tf = tf or peaks.get("bf16_tflops_sustained") or peaks["bf16_tflops"]
        bw = bw or peaks["hbm_gbs"]
    lines = [l for l in open(args.csv) if l.startswith('"')]
    rows = collections.OrderedDict()
    for r in csv.DictReader(lines):
        d = rows.setdefault(int(r["ID"]), {"kernel": r["Kernel Name"], "grid": r["Grid Size"]})
        v = float(r["Metric Value"].replace(",", ""))
        unit = r["Metric Unit"]
        name = r["Metric Name"]
        if name == "gpu__time_duration.sum":
            v *= {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}.get(unit, 1.0)
            d["us"] = v
        elif name.startswith("dram__bytes"):
            v *= {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)
            d["dram"] = d.get("dram", 0.0) + v
        elif "tensor" in name:
            d["tensor_pct"] = v
    launches = list(rows.values())
    trace = json.load(open(args.trace))
    # kernels outside the engine trace (decode, nms, memsets) are kept as they are
    ti, table = 0, []
    for l in launches:
        kinds = next((k for pat, k in KERNEL_KIND if pat in l["kernel"]), None)
        rec = {"kernel": l["kernel"].split("(")[0].split("::")[-1][:40], "us": round(l.get("us", 0.0), 2),
               "dram_MB": round(l.get("dram", 0.0) / 1e6, 2), "tensor_pct": l.get("tensor_pct")}
        if kinds and ti < len(trace):
            while ti < len(trace) and trace[ti]["kind"] not in kinds:
                ti += 1
            t = trace[ti]
            ti += 1
            ideal_us = max(t["flops"] / (tf * 1e12), t["bytes"] / (bw * 1e9)) * 1e6
            rec.update(layer="%s %dx%dx%d %s->%s%s%s%s" % (t["kind"], t["n"], t["h"], t["w"], t["cin"], t.get("cout", ""),
                                                          " s2" if t.get("stride") == 2 else "", " +res" if t.get("residual") else "",
                                                          " +up" if t.get("upsample") else ""),
                       gflop=round(t["flops"] / 1e9, 2), alg_MB=round(t["bytes"] / 1e6, 2), ideal_us=round(ideal_us, 2),
                       bound="tensor" if t["flops"] / (tf * 1e12) >= t["bytes"] / (bw * 1e9) else "hbm",
                       eff=round(ideal_us / max(l.get("us", 1e-9), 1e-9), 3),
                       tflops=round(t["flops"] / max(l.get("us", 1e-9), 1e-9) / 1e6, 1),
                       dram_over_alg=round(l.get("dram", 0.0) / max(t["bytes"], 1), 2))
        table.append(rec)
    tot = sum(r["us"] for r in table)
    ideal = sum(r.get("ideal_us", 0.0) for r in table)
    groups = collections.OrderedDict()
    for r in table:
        key = r.get("layer", r["kernel"])
        g = groups.setdefault(key, {"n": 0, "us": 0.0, "ideal_us": 0.0, "gflop": 0.0, "dram_MB": 0.0, "alg_MB": 0.0})
        g["n"] += 1
        for k in ("us", "ideal_us", "gflop", "dram_MB", "alg_MB"):
            g[k] += r.get(k, 0.0) or 0.0
    summary = {"launches": len(table), "sum_us": round(tot, 1), "sum_ideal_us": round(ideal, 1),
               "frac": round(ideal / tot, 4), "tensor_peak_tflops": tf, "hbm_peak_gbs": bw,
               "dram_bytes": sum(l.get("dram", 0.0) for l in launches),
               "conv_dram_bytes": sum(l.get("dram", 0.0) for l in launches
                                      if any(k in l["kernel"] for k in ("conv_gemm", "bottleneck_tail", "stem_pool"))),
               "groups": [dict(layer=k, share=round(g["us"] / tot, 4), eff=round(g["ideal_us"] / max(g["us"], 1e-9), 3),
                               **{a: round(b, 2) for a, b in g.items()})
                          for k, g in sorted(groups.items(), key=lambda kv: -kv[1]["us"])]}
    if args.out:
        json.dump({"summary": summary, "launches": table}, open(args.out + ".json", "w"), indent=1)
    print(json.dumps({k: v for k, v in summary.items() if k != "groups"}))
    for g in summary["groups"][:40]:
        print("%-46s n=%-3d %8.1f us  share %5.1f%%  eff %.2f  dram/alg %.2f" % (
            g["layer"][:46], g["n"], g["us"], 100 * g["share"], g["eff"], g["dram_MB"] / max(g["alg_MB"], 1e-9)))


if __name__ == "__main__":
    main()
