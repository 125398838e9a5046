#!/usr/bin/env python
"""bench.py -- the CSMPN hot path on B200: one EGCL layer forward+backward over a batch of synthetic complexes.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload md17|motion|nba|hulls] [--dump-outputs DIR]

Metric (BASELINE.json): simplices/sec fwd+bwd per CSMPN layer.  A step = one pass (forward + backward, all
parameter and input gradients) of one shared simplicial message layer (EGCL) over one batch of 100 complexes.
Default workload = BASELINE.json configs[1]: MD17-aspirin-shaped, 21 atoms, kNN(k=3) clique complex lifted to
edges + triangles, Cl(3,0), hidden width 32, aggr "sum".  ONE JSON line is printed; the other named configs
(motion, NBA) ride along under "workloads" (layer step, resident inputs), the lifting and train-step figures
under "lifting" and "train".

  value     whole-job simplices/s with inputs resident in HBM (CUDA events, L2 flushed between steps, max over ranks)
  e2e       the same step through the public layer API starting from HOST buffers: pinned H2D of
            (h, edge_index, node_attr), CSR build, forward, backward, D2H of the layer output AND of every gradient
  roofline  the dominant kernel CLASS of the layer step by time share (every kernel timed alone, CUDA events) against
            the measured HBM peak; roofline.layer = the whole layer against SURVEY 8d's fused-minimum bytes / FLOPs
  cpu_baseline / --impl reference   the reference's own EGCL (oracle/_ref, the unmodified Python reference behind
            oracle/refshim.py's PyG stand-in) on the host cores, same batch; the oracle port if oracle/_ref is absent
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree, which may be read-only

import numpy as np
import torch

WORKLOADS = {
    # name: (metric, hidden C, aggr, complexes per batch, description)
    "md17": ((1.0, 1.0, 1.0), 32, "sum", 100, "MD17-aspirin-shaped: 21 atoms, kNN(k=3) clique complex (edges+triangles), Cl(3,0), C=32"),
    "motion": ((1.0, 1.0, 1.0), 28, "mean", 100, "CMU-motion-shaped: fixed 31v+12e+4t complex, 226 pairs, Cl(3,0), C=28"),
    "nba": ((1.0, 1.0), 40, "sum", 100, "NBA-shaped: 10 players + ball, full Rips complex, Cl(2,0), C=40"),
    # BASELINE.json configs[0] (the reference's CPU-runnable case; csmpn/configs/hulls.yaml:20-23, hulls_cssmpnn.py:13-28):
    # 8 points ~ N(0,1)^5, all <=2-faces of the Qhull facets, batch 16, Cl(5,0), C=28, aggr mean
    "hulls": ((1.0, 1.0, 1.0, 1.0, 1.0), 28, "mean", 16, "convex-hulls-shaped: 8 points in R^5, faces of the Qhull facets, Cl(5,0), C=28, batch 16"),
}
T_TYPES = 3


# ----------------------------------------------------------------------------------------------- synthetic data
def _clique_complex(n, und_edges):
    """vertices, edges, triangles (sorted tuples, lexicographic) of the clique complex of an undirected graph."""
    nbr = [set() for _ in range(n)]
    for a, b in und_edges:
        if a != b:
            nbr[a].add(b), nbr[b].add(a)
    edges = sorted({(min(a, b), max(a, b)) for a, b in und_edges if a != b})
    tris = [(a, b, c) for (a, b) in edges for c in sorted(nbr[a] & nbr[b]) if c > b]
    return edges, tris


def _pairs_from_complex(n, edges, tris, extra_zero_zero):
    """adjacency pairs of the reference's lifting (SURVEY.md 8a L4/L6) as global ids: blocks 0_0,0_1,1_0,1_1,1_2,2_1.
    Only the multiset matters for the bench (parity of the lifting itself is tests/test_lifting*.py)."""
    eid = {e: i for i, e in enumerate(edges)}
    ne = len(edges)
    src, dst = [], []

    def add(a, b):
        src.append(a), dst.append(b)

    for (a, b) in edges:  # 0_0 upper adjacency (both directions)
        add(b, a), add(a, b)
    if extra_zero_zero:
        have = set(edges)
        for i in range(n):
            for j in range(n):
                if i != j and (i, j) not in have:
                    add(i, j)
    for k, (a, b) in enumerate(edges):  # 0_1 boundary and 1_0 coboundary
        add(a, n + k), add(b, n + k)
    for k, (a, b) in enumerate(edges):
        add(n + k, a), add(n + k, b)
    for t, (a, b, c) in enumerate(tris):  # 1_1 upper adjacency via triangles, 1_2, 2_1
        es = [eid[(a, b)], eid[(a, c)], eid[(b, c)]]
        for x in es:
            for y in es:
                if x != y:
                    add(n + y, n + x)
        for x in es:
            add(n + x, n + ne + t)
        for x in es:
            add(n + ne + t, n + x)
    return src, dst


def make_batch(workload, n_complexes, seed, hidden=None):
    """One batch: h [N,C,B], edge_index [2,E] int64, node_attr [N,T,B], edge_attr [E,2T,B], cotangent [N,C,B]."""
    metric, C, aggr, _, _ = WORKLOADS[workload]
    C = hidden or C
    rng = np.random.default_rng(seed)
    B = 1 << len(metric)
    srcs, dsts, types = [], [], []
    off = 0
    for _ in range(n_complexes):
        if workload == "md17":
            n = 21
            pos = rng.normal(0, 1.5, (n, 3))
            d = ((pos[:, None] - pos[None]) ** 2).sum(-1)
            np.fill_diagonal(d, np.inf)
            knn = np.argsort(d, axis=1)[:, :3]
            und = [(i, int(j)) for i in range(n) for j in knn[i]]
            edges, tris = _clique_complex(n, und)
            s, t = _pairs_from_complex(n, edges, tris, extra_zero_zero=False)
        elif workload == "nba":
            n = 11
            und = [(i, j) for i in range(n) for j in range(i + 1, n)]
            edges, tris = _clique_complex(n, und)
            s, t = _pairs_from_complex(n, edges, tris, extra_zero_zero=True)
        elif workload == "hulls":
            from scipy.spatial import ConvexHull

            n = 8
            facets = ConvexHull(rng.normal(0, 1, (n, 5))).simplices
            edges = sorted({(min(a, b), max(a, b)) for f in facets for a in f for b in f if a != b})
            tris = sorted({tuple(sorted((a, b, c))) for f in facets for a in f for b in f for c in f if a < b < c})
            edges = [(int(a), int(b)) for a, b in edges]
            tris = [(int(a), int(b), int(c)) for a, b, c in tris]
            s, t = _pairs_from_complex(n, edges, tris, extra_zero_zero=True)
        else:  # motion: 31 v, 12 e, 4 t; 130 skeleton pairs + 96 fixed pairs
            n = 31
            edges = [(6, 7), (7, 8), (6, 8), (1, 2), (2, 3), (1, 3), (24, 25), (25, 26), (24, 26), (22, 23), (21, 22), (21, 23)]
            tris = [(6, 7, 8), (1, 2, 3), (24, 25, 26), (21, 22, 23)]
            eid = {e: i for i, e in enumerate(edges)}
            s, t = [], []
            parent = {i: i - 1 for i in range(1, 25)}
            parent.update(dict(zip(range(25, 31), (3, 7, 11, 15, 19, 22))))
            adj = {i: set() for i in range(31)}
            for c_, p_ in parent.items():
                adj[c_].add(p_), adj[p_].add(c_)
            for i in range(31):
                for j in range(31):
                    if i != j and (j in adj[i] or any(j in adj[k] for k in adj[i])):
                        s.append(i), t.append(j)
            for k, (a, b) in enumerate(edges):
                for v in (a, b):
                    s.append(n + k), t.append(v)
                    s.append(v), t.append(n + k)
            for ti, (a, b, c) in enumerate(tris):
                es = [eid[(a, b)], eid[(a, c)] if (a, c) in eid else eid[(min(a, c), max(a, c))], eid[(b, c)]]
                for x in es:
                    s.append(n + 12 + ti), t.append(n + x)
                    s.append(n + x), t.append(n + 12 + ti)
                    for y in es:
                        if x != y:
                            s.append(n + x), t.append(n + y)
        nn = n + len(edges) + len(tris)
        srcs.append(np.asarray(s, dtype=np.int64) + off)
        dsts.append(np.asarray(t, dtype=np.int64) + off)
        types.append(np.concatenate([np.zeros(n), np.ones(len(edges)), 2 * np.ones(len(tris))]).astype(np.int64))
        off += nn
    edge_index = torch.from_numpy(np.stack([np.concatenate(srcs), np.concatenate(dsts)]))
    node_types = torch.from_numpy(np.concatenate(types))
    N = off
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(N, C, B, generator=g)
    emb = torch.randn(T_TYPES, T_TYPES, generator=g)
    node_attr = torch.zeros(N, T_TYPES, B)
    node_attr[..., 0] = emb[node_types]
    edge_attr = torch.cat([node_attr[edge_index[0]], node_attr[edge_index[1]]], dim=1)
    cot = torch.randn(N, C, B, generator=g)
    return dict(h=h, edge_index=edge_index, node_attr=node_attr, edge_attr=edge_attr, cot=cot, N=N,
                E=int(edge_index.shape[1]), C=C, B=B, metric=metric, aggr=aggr, n_complexes=n_complexes)


def layer_flops_bytes(N, E, C, B, T=T_TYPES):
    """SURVEY.md 8d: algorithmic bytes and FLOPs of one EGCL layer fwd+bwd."""
    f_blk = lambda cin: 2 * B * C * (cin + 2 * C) + 3 * B * B * C + 18 * B * C
    f_edge = f_blk(C + 2 * T) + f_blk(C) + B * C
    f_node = f_blk(2 * C + T) + f_blk(C) + B * C
    flops = 3 * (E * f_edge + N * f_node)
    nbytes = 4 * C * B * (5 * N + 3 * E) + 12 * E + 10 * N
    return flops, nbytes


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:  # reaped here: the sampler must not outlive the benchmark
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            self.proc.wait()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            p = [x.strip() for x in l.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])), (mx := float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU reference arm
def _reference_layer(b):
    """The reference's own EGCL (csmpn/models/cegnn_utils.py:216-284, UNMODIFIED, from oracle/_ref -- a verbatim copy made
    by oracle/make_ref.py) behind oracle/refshim.py's stand-in for PyG's MessagePassing; None if oracle/_ref is absent."""
    ref_root = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "csmpn")):
        return None
    os.environ["CSMPN_REFERENCE_ROOT"] = ref_root  # never /root/reference at run time
    from oracle import refshim

    refshim.REFERENCE_ROOT = ref_root
    refshim.install()
    from csmpn.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn.models.cegnn_utils import EGCL

    alg = CliffordAlgebra(b["metric"])
    return EGCL(alg, b["C"], b["C"], b["C"], edge_attr_features=2 * T_TYPES, node_attr_features=T_TYPES, aggr=b["aggr"])


def cpu_layer_time(workload, n_complexes, steps, warmup, seed=1000, hidden=None):
    """fwd + bwd (input and all parameter gradients) of one layer on the host cores: (N, E, times, kind)"""
    from oracle import layers_ref as R

    torch.set_num_threads(os.cpu_count() or 1)
    b = make_batch(workload, n_complexes, seed, hidden=hidden)
    ralg = R.RefAlgebra(b["metric"])
    init = R.init_egcl_params(ralg, b["C"], T_TYPES, torch.Generator().manual_seed(0))
    layer = _reference_layer(b)
    if layer is not None:
        missing, unexpected = layer.load_state_dict(init, strict=False)
        assert not unexpected and all("algebra" in k for k in missing), (missing, unexpected)
        plist = list(layer.parameters())
        run = lambda h: layer(h, b["edge_index"], b["edge_attr"], b["node_attr"])
        kind = "reference"
    else:
        params = {k: v.requires_grad_() for k, v in init.items()}
        plist = list(params.values())
        run = lambda h: R.egcl(ralg, h, b["edge_index"], b["edge_attr"], b["node_attr"], params, aggr=b["aggr"])
        kind = "port"
    times = []
    for it in range(warmup + steps):
        h = b["h"].clone().requires_grad_()
        t0 = time.perf_counter()
        y = run(h)
        torch.autograd.grad(y, [h] + plist, b["cot"])
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return b["N"], b["E"], times, kind


def _cpu_what(kind, cores):
    return ("the reference's own EGCL (oracle/_ref: unmodified csmpn/models/cegnn_utils.py behind the PyG stand-in of oracle/refshim.py)"
            if kind == "reference" else "oracle/layers_ref.py (port; oracle/_ref absent)") + f", torch CPU, {cores} threads"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    metric, C, aggr, ncx, desc = WORKLOADS[args.workload]
    ncx = args.complexes or ncx  # the SAME batch as the GPU arm
    N, E, times, kind = cpu_layer_time(args.workload, ncx, args.steps, args.warmup, hidden=args.hidden or None)
    ms = 1e3 * sum(times) / len(times)
    value = N / (ms * 1e-3)
    cores = os.cpu_count() or 1
    C = args.hidden or C
    line = {
        "impl": "reference", "metric": "simplices/sec fwd+bwd per CSMPN layer", "value": value, "unit": "simplices/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "aggr": aggr, "hidden": C, "complexes_per_step_per_gpu": ncx, "simplices_per_gpu": N, "pairs_per_gpu": E},
        "cpu_baseline": {"value": value, "unit": "simplices/s", "cores": cores, "kind": kind,
                         "sample": f"{ncx} complexes ({N} simplices, {E} pairs) per step, {_cpu_what(kind, cores)}"},
        "e2e": {"value": value, "unit": "simplices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- full-model train step
def make_md17_graphs(n_complexes, seed, dev, frames=10, atoms=21):
    """synthetic MD17-aspirin-shaped samples (SURVEY.md 8d config 2): positions ~ N(0, 1.5^2), kNN(k=3) graph"""
    from csmpn_b200.data.modules.simplicial_data import Data

    g = torch.Generator().manual_seed(seed)
    graphs = []
    for _ in range(n_complexes):
        loc = torch.randn(atoms, frames, 3, generator=g) * 1.5
        d = torch.cdist(loc[:, 0].double(), loc[:, 0].double())
        d.fill_diagonal_(float("inf"))
        nbr = torch.argsort(d, dim=1, stable=True)[:, :3]
        ei = torch.stack([nbr.reshape(-1), torch.arange(atoms).repeat_interleave(3)])
        graphs.append(Data(loc=loc, vel=torch.randn(atoms, frames, 3, generator=g), edge_index=ei,
                           charges=torch.randint(1, 9, (atoms,), generator=g).float(),
                           y=loc + 0.1 * torch.randn(atoms, frames, 3, generator=g)))
    return graphs


def _timed_region(fn, steps, dev, world):
    """K calls of fn between two CUDA events, barrier + synchronize on both sides, max over ranks -> ms per call"""
    import torch.distributed as dist

    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps


def train_leg(dev, world, rank, steps, warmup, lib, graphed=True):
    """train complexes/s: the md17 model (C=32, 5 layers, 10 frames) on 100 complexes per GPU, two ways:

    fixed   one batch trained on repeatedly: forward + backward (+ all-reduce + Adam, see `launch`) replayed from ONE CUDA
            graph -- what fixed-topology data (the motion skeleton) allows;
    stream  a DIFFERENT batch every step (MD17 / NBA complexes change from sample to sample): per step the raw samples'
            kNN pairs and features are copied from pinned host memory, lifted on the GPU (csmpn_lift_*), collated, CSR
            built, then forward -> zero_grad -> backward -> all-reduce -> Adam -> cosine schedule, eagerly, in the
            reference trainer's order (engineer/trainer/trainer.py:204-227)."""
    from csmpn_b200.data.modules.simplicial_data import SimplicialTransform
    from csmpn_b200.models.md17_cssmpnn import CliffordSharedSimplicialMPNN_md17
    from csmpn_b200.train_step import CosineAnnealingLR, DataParallelStep, GraphedDataParallelStep

    ncx = 100
    lift = SimplicialTransform(dim=2, dis=2.5, label="md17", molecule_type="aspirin")
    graphs = make_md17_graphs(ncx, 2000 + rank, dev)
    batch = lift.lift(graphs, device=dev)
    torch.manual_seed(0)
    model = CliffordSharedSimplicialMPNN_md17().to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, fused=True, capturable=True)
    lc0 = lib.csmpn_launch_count()
    model(batch, 0, "train")[0].backward()  # one eager pass: counts this library's launches per step
    launches_eager = lib.csmpn_launch_count() - lc0
    model.zero_grad(set_to_none=True)
    out = {"metric": "train complexes/sec (md17 model: Cl(3,0), C=32, 5 layers, 10 frames, Adam)", "unit": "complexes/s",
           "complexes_per_step_per_gpu": ncx, "params": sum(p.numel() for p in model.parameters()),
           "gpu_launches_per_step": launches_eager}
    # ---- (b) a stream of different batches, eager
    n_pool = 8
    pool = [make_md17_graphs(ncx, 3000 + 17 * k + rank, "cpu") for k in range(n_pool)]
    for gs in pool:
        for g in gs:
            for k in ("loc", "vel", "edge_index", "charges", "y"):
                setattr(g, k, getattr(g, k).pin_memory())
    sched = CosineAnnealingLR(opt, steps * 64, warmup_steps=steps, decay_steps=steps * 16)
    eager = DataParallelStep(model, opt)
    sizes = []

    def stream_step(i):
        b = lift.lift(pool[i % n_pool], device=dev)  # pinned H2D of the raw samples + GPU lifting + collation
        loss, _ = eager(b, i)
        sched.step()
        sizes.append(int(b.x_ind.shape[0]))
        return loss

    for i in range(warmup):
        stream_step(i)
    sizes.clear()
    ms_stream = _timed_region(stream_step, steps, dev, world)
    out["stream"] = {"value": ncx * world / (ms_stream * 1e-3), "ms_per_step": ms_stream,
                     "simplices_per_step_per_gpu": [min(sizes), max(sizes)],
                     "what": "different batch every step: pinned H2D of raw samples, GPU lifting, CSR build, forward, zero_grad, backward, "
                             "flat-bucket all-reduce, fused Adam, cosine schedule; eager launches"}
    # ---- (c) the same stream replayed from ONE CUDA graph: every batch padded to a bucket of simplex / pair counts
    if graphed:
        from csmpn_b200.data.padding import make_bucket
        from csmpn_b200.train_step import StreamGraphedStep

        lifted = [lift.lift(gs, device=dev) for gs in pool]
        bucket = make_bucket([b.sizes for b in lifted])  # a pass over the sampler's batches fixes the bucket
        sstep = StreamGraphedStep(model, opt, lifted[0], bucket)
        del lifted

        from csmpn_b200.pipeline import LiftPrefetcher

        pre = LiftPrefetcher(lambda samples: lift.lift(samples, device=dev), dev)
        pre.submit(pool[0])

        def stream_graphed_step(i):
            sstep.load(pre.take())   # batch i -> the graph's static tensors (padded in place), CSR rebuilt in place
            pre.consumed()
            loss, _ = sstep.run(i)   # one graph replay ...
            pre.submit(pool[(i + 1) % n_pool])  # ... under which the host lifts batch i + 1 on a side stream
            sched.step()
            return loss

        for i in range(warmup):
            stream_graphed_step(i)
        ms_sg = _timed_region(stream_graphed_step, steps, dev, world)
        out["stream_graphed"] = {"value": ncx * world / (ms_sg * 1e-3), "ms_per_step": ms_sg,
                                 "bucket": {"simplices": bucket.simplices, "edges": bucket.edges, "triangles": bucket.triangles,
                                            "pairs": bucket.pairs, "dummy_vertices": bucket.n_dummy_vertices},
                                 "what": "different batch every step: pinned H2D of raw samples + GPU lifting of batch i+1 on a side stream under "
                                         "step i (csmpn_b200.pipeline.LiftPrefetcher), in-place padding to one "
                                         "bucket of simplex / pair counts (one dummy complex, masked out of the loss), CSR rebuilt in "
                                         "place, then ONE graph replay: " + sstep.describe()}
        del sstep
    # ---- (a) fixed structure, graph replay
    loc0 = batch.loc.clone()
    batch.loc = loc0
    step = GraphedDataParallelStep(model, opt, batch) if graphed else DataParallelStep(model, opt)

    def fixed_step(i):
        batch.loc = loc0
        return step(batch)[0]

    for i in range(warmup):
        fixed_step(i)
    ms = _timed_region(fixed_step, steps, dev, world)
    loss = fixed_step(0)
    out.update({"value": ncx * world / (ms * 1e-3), "ms_per_step": ms, "simplices_per_gpu": int(batch.x_ind.shape[0]),
                "pairs_per_gpu": int(batch.edge_index.shape[1]), "final_loss": float(loss.detach()),
                "launch": getattr(step, "describe", lambda: "eager")()})
    return out


# ----------------------------------------------------------------------------------------------- lifting leg
def lifting_leg(dev, hbm_peak, iters=10):
    """GPU lifting throughput (SURVEY 8d lists lifting among the HBM-bound kernels): csmpn_lift_count + csmpn_lift_fill on
    100 md17-shaped complexes per call and on a 4 000-complex batch; bytes = every output the lifter writes once
    (edge_index int64, x_ind fp32, node_types / batch int64) + the pair lists it reads."""
    from csmpn_b200.data.modules.lifting import LIFT_CLIQUE, lift_batch

    res = {}
    for ncx in (100, 4000):
        base = make_md17_graphs(min(ncx, 200), 4000, "cpu")
        graphs = [base[i % len(base)] for i in range(ncx)]
        pairs = torch.cat([g.edge_index for g in graphs], 1).to(dev)
        ppc = [g.edge_index.shape[1] for g in graphs]
        nv = [g.loc.shape[0] for g in graphs]
        lb = lift_batch(LIFT_CLIQUE, nv, pairs=pairs, pairs_per_complex=ppc, dim=2, device=dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            lb = lift_batch(LIFT_CLIQUE, nv, pairs=pairs, pairs_per_complex=ppc, dim=2, device=dev)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        N, E = int(lb.x_ind.shape[0]), int(lb.edge_index.shape[1])
        nbytes = 16 * E + 12 * N + 16 * N + 16 * pairs.shape[1]
        res[f"{ncx}_complexes"] = {"complexes_per_s": ncx / (ms * 1e-3), "ms_per_call": ms, "simplices": N, "pairs": E,
                                   "algorithmic_bytes": nbytes, "hbm_gbs": nbytes / (ms * 1e-3) / 1e9,
                                   "hbm_frac": nbytes / (ms * 1e-3) / 1e9 / hbm_peak}
    res["note"] = ("one call = csmpn_lift_count + one host sync for the output sizes + csmpn_lift_fill (one warp per complex); at 100 "
                   "complexes the call is launch/sync-latency bound, at 4 000 it approaches the write bandwidth")
    return res


# ----------------------------------------------------------------------------------------------- GPU arm
def _traffic_for_build():
    """DRAM bytes per kernel class per layer step from an `ncu --set full` capture (tools/ncu_traffic.py writes
    profiles/ncu_traffic.json) -- used ONLY when the capture was made from this very build of csrc/ (digest match)"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        stamp = open(os.path.join(ROOT, "clifford-group-equivariant-simplicial-message-passing-networks_b200", "csrc", "build", "stamp.txt")).read().strip()
        return t if t.get("csrc_digest") == stamp else None
    except Exception:
        return None


def dump_outputs(out_dir, per_simplex, whole, budget=64 << 20, seed=0):
    """Write every array as <out_dir>/<name>.npy in float32.  If they exceed `budget` bytes in all, the per-simplex arrays
    ([N, ...], same N) keep only a fixed, seeded sample of their rows -- the same rows in each -- so that two builds
    run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu() for k, v in whole.items()}
    rows = {k: v.detach().float().cpu() for k, v in per_simplex.items()}
    n = next(iter(rows.values())).shape[0]
    row_bytes = sum(v[0].numel() * 4 for v in rows.values())
    headers = 256 * (len(arrays) + len(rows))  # an .npy header takes at most a few hundred bytes
    keep = max(0, budget - headers - sum(v.numel() * 4 for v in arrays.values())) // max(row_bytes, 1)
    if keep < n:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:keep].sort().values
        rows = {k: v[idx] for k, v in rows.items()}
    arrays.update(rows)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.numpy())


def layer_leg(workload, ncx, C, dev, world, rank, steps, warmup, lib, use_graph=True, with_e2e=True, with_roofline=True,
              hbm_peak=6553.0, peak_src="", dump_dir=None):
    """One workload: the layer step with resident inputs (`value`), from host buffers (`e2e`), its kernel roofline.
    `dump_dir`: write what the last timed step returned (dump_outputs)."""
    import torch.distributed as dist

    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.models.cegnn_utils import EGCL, PairedNodeAttr
    from csmpn_b200.models.ops import CSRGraph

    metric, _, aggr, _, desc = WORKLOADS[workload]
    b = make_batch(workload, ncx, 1000 + rank, hidden=C)
    N, E, B = b["N"], b["E"], b["B"]
    torch.manual_seed(0)
    alg = CliffordAlgebra(metric).to(dev)
    layer = EGCL(alg, C, C, C, edge_attr_features=2 * T_TYPES, node_attr_features=T_TYPES, aggr=aggr).to(dev)
    params = [p for p in layer.parameters()]
    n_par = sum(p.numel() for p in params)
    # device-resident inputs.  edge_attr = node_attr[src] | node_attr[dst] (md17_cssmpnn.py:131) is passed symbolically
    # (PairedNodeAttr): the message kernel gathers the two table rows itself, no [E, 2T, B] tensor exists
    d = {k: b[k].to(dev) for k in ("h", "edge_index", "node_attr", "cot")}
    graph = CSRGraph(d["edge_index"], N)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    l0 = lib.csmpn_launch_count()
    h_ = d["h"].detach().requires_grad_()
    torch.autograd.grad(layer(h_, graph, PairedNodeAttr(d["node_attr"]), d["node_attr"]), [h_] + params, d["cot"])
    launches_per_step = lib.csmpn_launch_count() - l0
    glayer = None
    flat = torch.empty(n_par, device=dev)

    def step(h, graph_, node_attr, pack=True):
        """one EAGER layer step (forward + backward through autograd); the graphed runs replay GraphedLayerStep instead.
        Returns the layer output, grad_h and the parameter gradients (packed into `flat` when it was packed)."""
        hh = h.detach().requires_grad_()
        y = layer(hh, graph_, PairedNodeAttr(node_attr), node_attr)
        grads = torch.autograd.grad(y, [hh] + params, d["cot"])
        packed = pack or world > 1
        if packed:  # one flat gradient buffer: the all-reduce bucket / the D2H payload of the e2e leg
            torch._foreach_copy_(list(flat.split([p.numel() for p in params])), [g.reshape(-1) for g in grads[1:]])
        if world > 1:
            dist.all_reduce(flat)
            flat.div_(world)
        return y, grads[0], flat if packed else grads[1:]

    # host-resident inputs (pinned) for the end-to-end leg
    # ONE pinned staging buffer holding h | edge_index | node_attr back to back: one H2D copy per step instead of three.
    # Wire format: the pair list as int32 (simplex ids of a batch fit easily) and, when node_attr only carries scalars -- the
    # simplex-type embedding of the models, md17_cssmpnn.py:122-129 -- its grade-0 part [N, T]; both are widened on the device
    # into per-slot int64 [2, E] / [N, T, B] tensors by the feeder (copy stream), so the layer is called with the reference's
    # argument types.  At 8 GPUs the step time of this leg is set by the bytes that cross the host link (DESIGN.md 4.4).
    compact_attr = bool((b["node_attr"][..., 1:] == 0).all()) and os.environ.get("CSMPN_BENCH_WIRE", "compact") == "compact"
    segs = [("h", b["h"]),
            ("edge_index", b["edge_index"].to(torch.int32) if compact_attr else b["edge_index"]),
            ("node_attr", b["node_attr"][..., 0].contiguous() if compact_attr else b["node_attr"])]
    offs, total_b = {}, 0
    for k, t in segs:
        offs[k] = total_b
        total_b += (t.numel() * t.element_size() + 255) // 256 * 256
    blob_host = torch.empty(total_b, dtype=torch.uint8).pin_memory()
    for k, t in segs:
        blob_host[offs[k]: offs[k] + t.numel() * t.element_size()].view(t.dtype).view(t.shape).copy_(t)
    host_in = {"blob": blob_host}

    def unpack(dv):
        out = {}
        for k, t in segs:
            out[k] = dv["blob"][offs[k]: offs[k] + t.numel() * t.element_size()].view(t.dtype).view(t.shape)
        return out

    y_host = torch.empty((N, C, B), dtype=torch.float32).pin_memory()
    gh_host = torch.empty((N, C, B), dtype=torch.float32).pin_memory()
    gp_host = torch.empty(n_par, dtype=torch.float32).pin_memory()
    h2d_bytes = sum(t.numel() * t.element_size() for _, t in segs)
    # what comes back every step: the layer output and every parameter gradient.  grad_h only with CSMPN_BENCH_D2H_GRAD_H=1: it
    # is the cotangent handed to the previous layer on the device, and at 8 GPUs the box's host I/O (~92 GB/s over all
    # GPUs, measured: 2.5 ms per step for ~29 MB per GPU in r01 and r02 alike) makes the e2e figure a function of bytes
    d2h_grad_h = os.environ.get("CSMPN_BENCH_D2H_GRAD_H", "0") == "1"
    d2h_bytes = (y_host.numel() + (gh_host.numel() if d2h_grad_h else 0) + gp_host.numel()) * 4

    from csmpn_b200.pipeline import HostFeeder

    # graphed runs: one captured layer per feeder slot, each with its own CSR buffers -- the CSR of batch i+1 is rebuilt on the
    # copy stream right after its H2D copy (HostFeeder.prepare), under the kernels of step i, instead of in front of step i+1
    glayers = []
    n_slots = 2
    ei_dev = [torch.empty((2, E), dtype=torch.int64, device=dev) for _ in range(n_slots)]
    na_dev = [torch.zeros((N, T_TYPES, B), dtype=torch.float32, device=dev) for _ in range(n_slots)]

    def prepare(k, bufs):
        """on the copy stream, right after the H2D copy of slot k: widen the wire format, rebuild the slot's CSR in place"""
        x = unpack(bufs)
        if compact_attr:
            ei_dev[k].copy_(x["edge_index"])
            na_dev[k][..., 0].copy_(x["node_attr"])
        else:
            ei_dev[k], na_dev[k] = x["edge_index"], x["node_attr"]
        if use_graph and glayers:
            glayers[k].set_graph(ei_dev[k])

    feeder = HostFeeder(dev, slots=n_slots, prepare=prepare)
    drained = [None] * n_slots

    def run_e2e(n_steps):
        """n_steps layer steps from HOST buffers through the public API: every step copies its inputs from pinned host
        memory (HostFeeder: the copy of step i+1 overlaps the kernels of step i), builds the CSR of its edge_index, runs
        forward + backward and copies the layer output, grad_h and all parameter gradients back to pinned host memory."""
        feeder.submit(host_in)
        for i in range(n_steps):
            dv = feeder.next()
            if i + 1 < n_steps:
                feeder.submit(host_in)
            flush.fill_(1.0)  # L2 flush, inside the timed region
            x, k = unpack(dv), dv["_index"]
            if drained[k] is not None:  # the graph's static outputs of this slot: their last D2H copies must have left
                torch.cuda.current_stream(dev).wait_event(drained[k])
            if glayer is not None:
                # batches of a fixed shape: ONE graph replay per step (forward + backward + gradient pack) that reads the
                # feeder's device buffers directly; the CSR was rebuilt in place by the feeder
                y, gh, gflat = glayers[k]()
                if world > 1:
                    dist.all_reduce(gflat)
                    gflat.div_(world)
            else:
                y, gh, _ = step(x["h"], CSRGraph(ei_dev[k], N), na_dev[k])
                gflat = flat
            feeder.drain(y, y_host)
            if d2h_grad_h:
                feeder.drain(gh, gh_host)
            feeder.drain(gflat, gp_host)
            drained[k] = feeder.last_drain_event
            feeder.release(dv)
        feeder.join()

    def timed_e2e(steps, warmup, regions=3):
        run_e2e(warmup)
        out = []
        host = []
        for _ in range(regions):
            out.append(_timed_block(lambda: run_e2e(steps), dev, world))
            host.append(_timed_block.host_ms / steps)
        timed_e2e.host_ms_per_step = statistics.median(host)
        return statistics.median(out), out

    gstep = None
    if use_graph:
        # `value`: inputs resident -> the step is ONE replay of the whole-step graph on the resident tensors (no per-call copies
        # into graph-private buffers); the gradient pack is part of it only where it is used (the all-reduce bucket, N > 1)
        from csmpn_b200.graphs import GraphedLayerStep

        gstep = GraphedLayerStep(layer, d["edge_index"], d["h"], d["node_attr"], d["cot"], pack=world > 1)

    def resident_step():
        """one step; returns the layer output, grad_h and the parameter gradients (one flat tensor or one per parameter)"""
        if gstep is None:
            return step(d["h"], graph, d["node_attr"], pack=False)
        y, gh, gflat = gstep()
        if world > 1:
            dist.all_reduce(gflat)
            gflat.div_(world)
            return y, gh, gflat
        return y, gh, gstep.param_grads

    def timed(steps, warmup):
        """(summed ms of `steps` timed steps, the outputs of the last one; None unless they are dumped)"""
        for _ in range(warmup):
            resident_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        evs = []
        for _ in range(steps):
            flush.fill_(1.0)  # L2 flush (256 MiB > 126 MB L2), outside the timed events
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last = resident_step()
            e1.record()
            evs.append((e0, e1))
            if dump_dir is None:
                last = None
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t = torch.tensor([sum(a.elapsed_time(bb) for a, bb in evs)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), last

    if use_graph:
        glayer = gstep  # (flag for the host-fed leg below: graphed)
        if with_e2e:
            # the e2e leg: one whole-step graph per feeder slot, reading that slot's device buffers (own CSR buffers each, same
            # parameters).  Two submits create the slots' device buffers (their addresses then stay fixed).
            from csmpn_b200.graphs import GraphedLayerStep

            for _ in range(n_slots):
                feeder.submit(host_in)
            torch.cuda.synchronize()
            for k in range(n_slots):
                x = unpack(feeder.slots[k]["bufs"])
                glayers.append(GraphedLayerStep(layer, ei_dev[k], x["h"], na_dev[k], d["cot"]))
            for _ in range(n_slots):   # hand the two submitted batches back: the timed loops start from an empty feeder
                feeder.release(feeder.next())
            feeder.join()
    res = {"workload": desc, "aggr": aggr, "hidden": C, "complexes_per_step_per_gpu": ncx, "simplices_per_gpu": N, "pairs_per_gpu": E,
           "gpu_launches_per_step": int(launches_per_step)}
    if with_e2e:
        e2e_ms, regions = timed_e2e(steps, max(3, warmup // 2))
        res["e2e_ms_per_step"] = e2e_ms / steps
        res["e2e_regions_ms_per_step"] = [r / steps for r in regions]
        res["e2e_host_enqueue_ms_per_step"] = timed_e2e.host_ms_per_step
        res["h2d_bytes_per_step"], res["d2h_bytes_per_step"] = h2d_bytes, d2h_bytes
    total_ms, last = timed(steps, warmup)
    if dump_dir is not None:
        y, gh, pgrads = last
        if torch.is_tensor(pgrads):
            pgrads = pgrads.split([p.numel() for p in params])
        names = [n for n, _ in layer.named_parameters()]
        dump_outputs(dump_dir, {"y": y, "grad_h": gh}, {f"grad.{n}": g.reshape(p.shape) for n, g, p in zip(names, pgrads, params)})
    res["ms_per_step"] = total_ms / steps
    nt = torch.tensor([N], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(nt)
    res["simplices_all_gpus"] = int(nt.item())
    res["value"] = res["simplices_all_gpus"] / (res["ms_per_step"] * 1e-3)
    if with_e2e:
        res["e2e_value"] = res["simplices_all_gpus"] / (res["e2e_ms_per_step"] * 1e-3)
    flops, nbytes = layer_flops_bytes(N, E, C, B)
    t_s = res["ms_per_step"] * 1e-3
    res["layer_roofline"] = {"algorithmic_bytes": nbytes, "algorithmic_flops": flops, "hbm_gbs": nbytes / t_s / 1e9,
                             "hbm_frac": nbytes / t_s / 1e9 / hbm_peak, "fp32_tflops": flops / t_s / 1e12,
                             "fp32_frac_of_74.4": flops / t_s / 1e12 / 74.4}
    if with_roofline and rank == 0:
        from csmpn_b200.models import fused

        try:
            res["roofline"] = fused.bench_layer_kernels(layer, d, graph, hbm_peak, peak_src, traffic=_traffic_for_build())
        except Exception as e:  # pragma: no cover
            res["roofline"] = {"bound": "hbm", "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None, "traffic": None,
                               "kernel": f"unavailable: {e}", "peak_source": peak_src}
    del glayer
    glayers.clear()
    return res


def _release_cached(dev):
    import gc

    gc.collect()
    torch.cuda.synchronize(dev)
    torch.cuda.empty_cache()


def _timed_block(fn, dev, world):
    import torch.distributed as dist

    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    h0 = time.perf_counter()
    fn()
    _timed_block.host_ms = (time.perf_counter() - h0) * 1e3  # wall time the host needed to ENQUEUE the region (before the sync)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_ours(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from csmpn_b200 import _lib

    lib = _lib.lib()
    metric, C, aggr, ncx, desc = WORKLOADS[args.workload]
    ncx = args.complexes or ncx  # scaling sweep (BASELINE.json configs[4]): same complexes, larger batch
    C = args.hidden or C
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"

    if args.train_only:  # diagnostics: the train leg alone, on a fresh allocator
        train = train_leg(dev, world, rank, max(3, args.steps // 2), 3, lib, graphed=not args.no_graph)
        if rank == 0:
            print(json.dumps({"train": train}))
        if world > 1:
            dist.destroy_process_group()
        return
    # the train leg runs first, on a fresh allocator: its streamed-batch part allocates differently sized tensors every step
    # and is several times slower once the CUDA-graph pools of the layer legs have fragmented the caching allocator
    train = None if args.no_train else train_leg(dev, world, rank, max(3, args.steps // 2), 3, lib, graphed=not args.no_graph)
    _release_cached(dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    main = layer_leg(args.workload, ncx, C, dev, world, rank, args.steps, args.warmup, lib, use_graph=not args.no_graph,
                     with_e2e=not args.no_e2e, with_roofline=not args.no_roofline, hbm_peak=hbm_peak, peak_src=peak_src,
                     dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None  # sampled over the e2e and layer-step timed regions of the headline workload
    _release_cached(dev)
    others = {}
    if args.workload == "md17" and not args.complexes and not args.hidden and not args.only:
        for w in ("motion", "nba"):  # the other named GPU configs (BASELINE.json configs[2], [3]): resident layer step
            r = layer_leg(w, WORKLOADS[w][3], WORKLOADS[w][1], dev, world, rank, max(5, args.steps // 2), 3, lib,
                          use_graph=not args.no_graph, with_e2e=False, with_roofline=True, hbm_peak=hbm_peak, peak_src=peak_src)
            if "roofline" in r:  # keep the line readable: class summary only
                r["roofline"] = {k: r["roofline"].get(k) for k in ("kernel", "achieved", "frac", "unit", "classes", "summed_kernel_ms")}
            others[w] = r
            _release_cached(dev)
    lifting = lifting_leg(dev, hbm_peak) if (rank == 0 and not args.only) else None

    if rank == 0:
        roof = main.pop("roofline", None) or {"bound": "hbm", "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None,
                                              "traffic": None, "kernel": "not timed (--no-roofline)", "peak_source": peak_src}
        lr = main.pop("layer_roofline")
        lr["note"] = ("the whole layer step (`value`) against SURVEY 8d's fused-minimum bytes / FLOPs; the tensor-core engine runs a block "
                      "as several kernels whose intermediates cross L2/HBM (per-kernel figures under roofline.kernels)")
        roof["layer"] = lr
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cN, cE, times, kind = cpu_layer_time(args.workload, ncx, 3, 1, hidden=args.hidden or None)
            cms = statistics.median(times)
            cores = os.cpu_count() or 1
            cpu = {"value": cN / cms, "unit": "simplices/s", "cores": cores, "kind": kind,
                   "sample": f"the same {ncx} complexes ({cN} simplices, {cE} pairs), median of 3 steps after 1 warm-up, {_cpu_what(kind, cores)}"}
        glaunch = ("ONE CUDA-graph replay per step: layer forward + backward on the resident tensors (csmpn_b200.graphs.GraphedLayerStep)"
                   if not args.no_graph else "eager")
        line = {
            "metric": "simplices/sec fwd+bwd per CSMPN layer", "value": main["value"], "unit": "simplices/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "aggr": aggr, "hidden": C, "complexes_per_step_per_gpu": ncx, "simplices_per_gpu": main["simplices_per_gpu"],
                       "pairs_per_gpu": main["pairs_per_gpu"], "simplices_processed_in_timed_region": main["simplices_all_gpus"] * args.steps,
                       "l2": "flushed between timed steps (256 MiB write)",
                       "parallelism": f"dp{world}" if world > 1 else "single", "path": fused_path_name(), "launch": glaunch,
                       "edge_attr": "PairedNodeAttr(node_attr): node_attr[src] | node_attr[dst] gathered inside the message kernel"},
            "e2e": None if args.no_e2e else {"value": main["e2e_value"], "unit": "simplices/s", "h2d_bytes_per_step": main["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": main["d2h_bytes_per_step"], "ms_per_step": main["e2e_ms_per_step"],
                    "regions_ms_per_step": main["e2e_regions_ms_per_step"],
                    "host_enqueue_ms_per_step": main["e2e_host_enqueue_ms_per_step"],
                    "how": "median of 3 regions of K steps, each timed as one region; per step: ONE pinned H2D copy of h | edge_index (int32 on the wire) | node_attr (its scalar part on the wire; both widened on the device to the reference's int64 [2, E] / [N, T, B]) "
                           "(csmpn_b200.pipeline.HostFeeder, copy AND in-place CSR rebuild of step i+1 overlap the kernels of step i), layer "
                           "forward + backward + gradient pack as ONE CUDA-graph replay reading the feeder's device buffers (csmpn_b200.graphs.GraphedLayerStep; eager with --no-graph), D2H of the layer output and every parameter gradient "
                           "(+ grad_h with CSMPN_BENCH_D2H_GRAD_H=1); 256 MiB L2 flush inside the region every step"},
            "gpu_launches": int(main["gpu_launches_per_step"] * args.steps), "gpu_launches_per_step": main["gpu_launches_per_step"],
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "workloads": others or None, "train": train, "lifting": lifting,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def fused_path_name():
    from csmpn_b200.models import fused

    return "fused block kernels: tcgen05 engine for blocks with >= %d rows, FP32 SIMT engine below" % fused.tc_min_rows()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="md17", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--complexes", type=int, default=0, help="complexes per GPU per step (default: the workload's batch of 100)")
    ap.add_argument("--hidden", type=int, default=0, help="hidden width C (default: the workload's)")
    ap.add_argument("--no-train", action="store_true", help="skip the full-model train-step leg")
    ap.add_argument("--no-graph", action="store_true", help="launch the layer step eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (sweep runs: 10^6-simplex batches)")
    ap.add_argument("--no-roofline", action="store_true", help="skip the per-kernel timing table")
    ap.add_argument("--train-only", action="store_true", help="only the full-model train-step leg")
    ap.add_argument("--only", action="store_true", help="only the named workload's layer legs (no motion/NBA side runs, no lifting leg)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (layer output, grad_h, every parameter gradient) "
                         "as DIR/<name>.npy, float32, at most 64 MB in all (a fixed, seeded sample of rows beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.train_only):
        ap.error("--dump-outputs writes what the layer step of --impl ours computed (not with --train-only)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
