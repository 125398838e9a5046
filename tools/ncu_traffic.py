#!/usr/bin/env python
"""DRAM traffic and duration of one layer step per kernel class, from an ncu CSV of tools/layer_once.py:

    ncu --profile-from-start off --clock-control none --csv --log-file gpurun_out/layer_metrics.csv \
        --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum python tools/layer_once.py md17
    python tools/ncu_traffic.py gpurun_out/layer_metrics.csv profiles/ncu_traffic.json

Writes {csrc_digest, workload, classes: {class: {launches, dram_bytes, time_us}}, layer: {...}} -- bench.py attaches the
per-class DRAM bytes as roofline.traffic ONLY while csrc_digest equals the digest of the library it runs (build/stamp.txt),
so a capture can never outlive the kernels it was taken from."""
import collections
import csv
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLASSES = (("tc_f1", "tc_f1"), ("tc_f2", "tc_f2"), ("tc_b1", "tc_b1"), ("tc_bgemm", "tc_bgemm"),
           ("tc_b3", "tc_b3"), ("tc_dw", "tc_dw"), ("final_reduce", "final_reduce (both engines)"), ("tc_weight_images", "tc_weight_images"),
           ("block_fwd_kernel", "block_fwd (fp32 simt)"), ("block_bwd", "block_bwd (fp32 simt)"), ("segment_", "segment reduce / expand"),
           ("scatter_", "scatter (grad_h, table grads)"), ("add3_rows", "add3_rows"))


def classify(name):
    for key, cls in CLASSES:
        if key in name:
            return cls
    return "other (ATen)"


def main():
    src, dst = sys.argv[1], sys.argv[2]
    rows = list(csv.reader(open(src, errors="replace")))
    hdr = next(r for r in rows if len(r) > 5 and r[0] == "ID")
    per = collections.OrderedDict()
    for r in rows:
        if len(r) != len(hdr) or r[0] == "ID":
            continue
        d = dict(zip(hdr, r))
        val = float(d["Metric Value"].replace(",", ""))
        unit = d.get("Metric Unit", "")
        scale = {"Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "byte": 1.0, "usecond": 1.0, "us": 1.0, "msecond": 1e3, "ms": 1e3,
                 "nsecond": 1e-3, "ns": 1e-3, "second": 1e6, "s": 1e6}.get(unit, 1.0)
        k = per.setdefault(d["ID"], {"name": d["Kernel Name"], "dram": 0.0, "us": 0.0})
        if d["Metric Name"].startswith("dram__bytes"):
            k["dram"] += val * scale
        elif d["Metric Name"].startswith("gpu__time_duration"):
            k["us"] += val * scale
    classes = collections.OrderedDict()
    for k in per.values():
        c = classes.setdefault(classify(k["name"]), {"launches": 0, "dram_bytes": 0.0, "time_us": 0.0})
        c["launches"] += 1
        c["dram_bytes"] += k["dram"]
        c["time_us"] += k["us"]
    stamp = open(os.path.join(ROOT, "clifford-group-equivariant-simplicial-message-passing-networks_b200", "csrc", "build", "stamp.txt")).read().strip()
    out = {"csrc_digest": stamp, "source": os.path.basename(src),
           "note": "one EGCL layer forward + backward (tools/layer_once.py, md17 workload unless the file name says otherwise); ncu replays "
                   "each kernel alone with cold caches, so durations are serialised cold-cache figures: use the SHARES, not the absolutes",
           "classes": classes,
           "layer": {"launches": sum(c["launches"] for c in classes.values()), "dram_bytes": sum(c["dram_bytes"] for c in classes.values()),
                     "time_us": sum(c["time_us"] for c in classes.values())}}
    for name, c in classes.items():
        c["share_of_time"] = c["time_us"] / out["layer"]["time_us"]
    # flat view bench.py reads: class -> DRAM bytes per layer step
    out.update({name: c["dram_bytes"] for name, c in classes.items()})
    json.dump(out, open(dst, "w"), indent=1)
    for name, c in classes.items():
        print(f"{name:32s} n={c['launches']:3d} {c['time_us']:9.1f} us {100 * c['share_of_time']:5.1f} %  DRAM {c['dram_bytes'] / 1e6:9.1f} MB")
    print(f"layer: {out['layer']['launches']} launches, {out['layer']['time_us']:.0f} us (serialised, cold), DRAM {out['layer']['dram_bytes'] / 1e6:.0f} MB")


if __name__ == "__main__":
    main()
