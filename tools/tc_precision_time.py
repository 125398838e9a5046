#!/usr/bin/env python
"""Default (3xTF32, fp32-accurate) against single-pass TF32 mode of the tensor-core engine (csmpn_block_desc.tf32),
selected with torch.backends.cuda.matmul.fp32_precision.

Times one EGCL layer step (forward + backward + gradient pack, one CUDA-graph replay of csmpn_b200.graphs.GraphedLayerStep)
on the bench.py batches of md17, motion, nba and md17 at hidden 64 / 128 / 256, and the md17 training step (bench.py's
train leg: 100 complexes, graphed forward + backward + Adam).  Each mode is captured once; the two are then timed in
alternation, three times each, and the medians are printed with the max-norm relative error of each TF32 output against
the default run of the same step.  Prints the card name and power limit first.

    python tools/tc_precision_time.py [--out DIR]
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

LAYERS = [("md17", None), ("motion", None), ("nba", None), ("md17", 64), ("md17", 128), ("md17", 256)]
MODES = ("ieee", "tf32")
ROUNDS = 3


def set_mode(mode):
    torch.backends.cuda.matmul.fp32_precision = mode


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


def alternate(steps, iters, warm):
    """steps: {mode: callable}; per mode the median over ROUNDS of the mean time of `iters` calls, modes alternating"""
    for mode in MODES:
        for _ in range(warm):
            steps[mode]()
    ts = {m: [] for m in MODES}
    for _ in range(ROUNDS):
        for mode in MODES:
            ts[mode].append(timed(steps[mode], iters))
    return {m: statistics.median(v) for m, v in ts.items()}, ts


def layer_case(wl, hidden, dev):
    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.graphs import GraphedLayerStep
    from csmpn_b200.models.cegnn_utils import EGCL

    metric, C, aggr, ncx, _ = bench.WORKLOADS[wl]
    b = bench.make_batch(wl, ncx, 1000, hidden)
    C = b["C"]
    torch.manual_seed(0)
    layer = EGCL(CliffordAlgebra(metric).to(dev), C, C, C, edge_attr_features=2 * bench.T_TYPES,
                 node_attr_features=bench.T_TYPES, aggr=aggr).to(dev)
    ei = b["edge_index"].to(dev)
    steps, outs = {}, {}
    for mode in MODES:
        set_mode(mode)
        g = GraphedLayerStep(layer, ei, b["h"].to(dev), b["node_attr"].to(dev), b["cot"].to(dev))
        steps[mode] = g
        y, gh, flat = g()
        outs[mode] = (y.clone(), gh.clone(), flat.clone())
    set_mode("ieee")
    med, raw = alternate(steps, iters=50, warm=5)
    err = {k: rel(a, b) for k, a, b in zip(("y", "grad_h", "param_grads"), outs["tf32"], outs["ieee"])}
    return {"workload": wl, "hidden": C, "N": b["N"], "E": b["E"], "ms": med, "ms_rounds": raw,
            "tf32_vs_default_rel_err": err}


def train_case(dev):
    from csmpn_b200.data.modules.simplicial_data import SimplicialTransform
    from csmpn_b200.models.md17_cssmpnn import CliffordSharedSimplicialMPNN_md17
    from csmpn_b200.train_step import GraphedDataParallelStep

    lift = SimplicialTransform(dim=2, dis=2.5, label="md17", molecule_type="aspirin")
    batch = lift.lift(bench.make_md17_graphs(100, 2000, dev), device=dev)
    # accuracy: one eager forward + backward per mode from the same initialisation
    grads = {}
    for mode in MODES:
        set_mode(mode)
        torch.manual_seed(0)
        m = CliffordSharedSimplicialMPNN_md17().to(dev)
        loss = m(batch, 0, "train")[0]
        grads[mode] = [loss.detach()] + [g for g in torch.autograd.grad(loss, list(m.parameters()), allow_unused=True)]
    err = {"loss": rel(grads["tf32"][0], grads["ieee"][0]),
           "worst_param_grad": max(rel(a, b) for a, b in zip(grads["tf32"][1:], grads["ieee"][1:]) if b is not None)}
    steps = {}
    loc0 = batch.loc.clone()
    for mode in MODES:
        set_mode(mode)
        torch.manual_seed(0)
        m = CliffordSharedSimplicialMPNN_md17().to(dev)
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, fused=True, capturable=True)
        step = GraphedDataParallelStep(m, opt, batch)

        def run(step=step):
            batch.loc = loc0
            return step(batch)[0]

        steps[mode] = run
    set_mode("ieee")
    med, raw = alternate(steps, iters=20, warm=3)
    return {"workload": "md17 train step (100 complexes, graphed fwd + bwd + Adam)", "N": int(batch.x_ind.shape[0]),
            "E": int(batch.edge_index.shape[1]), "ms": med, "ms_rounds": raw, "tf32_vs_default_rel_err": err}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="also write the results as JSON lines to DIR/tc_precision_time.jsonl")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tc_precision_time.py needs a CUDA device")
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {card[0] if card else torch.cuda.get_device_name(dev)}", flush=True)
    old = torch.backends.cuda.matmul.fp32_precision
    results = []
    try:
        for wl, hidden in LAYERS:
            results.append(layer_case(wl, hidden, dev))
            r = results[-1]
            print(json.dumps(r), flush=True)
        results.append(train_case(dev))
        print(json.dumps(results[-1]), flush=True)
    finally:
        torch.backends.cuda.matmul.fp32_precision = old
    print(f"\n{'workload':24s} {'N':>7s} {'E':>7s} {'default ms':>11s} {'tf32 ms':>9s} {'speedup':>8s}  tf32 vs default rel err")
    for r in results:
        name = r["workload"] if len(r["workload"]) < 20 else "md17 train step"
        if "hidden" in r:
            name = f"{r['workload']} C={r['hidden']}"
        d, t = r["ms"]["ieee"], r["ms"]["tf32"]
        errs = ", ".join(f"{k} {v:.1e}" for k, v in r["tf32_vs_default_rel_err"].items())
        print(f"{name:24s} {r['N']:7d} {r['E']:7d} {d:11.3f} {t:9.3f} {d / t:7.3f}x  {errs}")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "tc_precision_time.jsonl"), "w") as f:
            f.write(json.dumps({"card": card}) + "\n")
            for r in results:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
