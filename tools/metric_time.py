#!/usr/bin/env python
"""The md17-shaped EGCL layer step under three metrics, on the fused block engines and on the unit-kernel composition.

The step is bench.py's layer leg: bench.make_batch("md17", 100, ...) (8 777 simplices, 53 976 pairs, C = 32), forward +
backward + gradient pack as ONE CUDA-graph replay of csmpn_b200.graphs.GraphedLayerStep.  Metrics: Euclidean (1,1,1),
Cl(2,1) (1,1,-1) and Cl(2,1) with the negative square on the second basis vector (1,-1,1); each captured once with the
fused engines and once with CSMPN_FUSED=0 (the path every non-Euclidean layer took before the fused engines took them).
All six steps are warmed, then timed in alternation, ROUNDS times each; the medians are printed, with the max-norm
relative difference of each fused step's outputs from its unit-kernel step.  Prints the card name and power limit first.

    python tools/metric_time.py [--out DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

METRICS = [(1.0, 1.0, 1.0), (1.0, 1.0, -1.0), (1.0, -1.0, 1.0)]
PATHS = ("fused", "unit")
ROUNDS = 5
ITERS = 50


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def capture(metric, path, b, dev):
    """GraphedLayerStep of a seed-0 EGCL over `metric`, captured with the fused engines on or off"""
    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.graphs import GraphedLayerStep
    from csmpn_b200.models.cegnn_utils import EGCL

    os.environ["CSMPN_FUSED"] = "1" if path == "fused" else "0"
    torch.manual_seed(0)
    layer = EGCL(CliffordAlgebra(metric).to(dev), b["C"], b["C"], b["C"], edge_attr_features=2 * bench.T_TYPES,
                 node_attr_features=bench.T_TYPES, aggr=bench.WORKLOADS["md17"][2]).to(dev)
    g = GraphedLayerStep(layer, b["edge_index"].to(dev), b["h"].to(dev), b["node_attr"].to(dev), b["cot"].to(dev))
    out = tuple(t.clone() for t in g())
    return layer, g, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="also write the results as JSON lines to DIR/metric_time.jsonl")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("metric_time.py needs a CUDA device")
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {card[0] if card else torch.cuda.get_device_name(dev)}", flush=True)
    b = bench.make_batch("md17", 100, 1000)
    old = os.environ.get("CSMPN_FUSED")
    steps, outs, keep = {}, {}, []
    try:
        for metric in METRICS:
            for path in PATHS:
                layer, g, out = capture(metric, path, b, dev)
                steps[(metric, path)], outs[(metric, path)] = g, out
                keep.append(layer)
    finally:
        if old is None:
            os.environ.pop("CSMPN_FUSED", None)
        else:
            os.environ["CSMPN_FUSED"] = old
    for s in steps.values():
        for _ in range(5):
            s()
    ts = {k: [] for k in steps}
    for _ in range(ROUNDS):
        for k, s in steps.items():
            ts[k].append(timed(s, ITERS))
    results = []
    for metric in METRICS:
        fused, unit = (statistics.median(ts[(metric, p)]) for p in PATHS)
        err = {k: rel(a, c) for k, a, c in zip(("y", "grad_h", "param_grads"), outs[(metric, "fused")], outs[(metric, "unit")])}
        results.append({"metric": metric, "N": b["N"], "E": b["E"], "C": b["C"], "fused_ms": fused, "unit_ms": unit,
                        "fused_ms_rounds": ts[(metric, "fused")], "unit_ms_rounds": ts[(metric, "unit")],
                        "fused_vs_unit_rel_diff": err})
        print(json.dumps(results[-1]), flush=True)
    print(f"\nmd17 layer step, N = {b['N']}, E = {b['E']}, C = {b['C']}; medians of {ROUNDS} alternating rounds of {ITERS} "
          f"graph replays")
    print(f"{'metric':18s} {'fused ms':>9s} {'CSMPN_FUSED=0 ms':>17s} {'ratio':>7s}  fused vs unit rel diff")
    for r in results:
        errs = ", ".join(f"{k} {v:.1e}" for k, v in r["fused_vs_unit_rel_diff"].items())
        print(f"{str(tuple(r['metric'])):18s} {r['fused_ms']:9.3f} {r['unit_ms']:17.3f} {r['unit_ms'] / r['fused_ms']:6.2f}x  {errs}")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "metric_time.jsonl"), "w") as f:
            f.write(json.dumps({"card": card}) + "\n")
            for r in results:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
