"""GPU parity of the tensor-core engine IN THE REGIME THE BENCH TIMES: many more 128-row tiles than SMs, so that every
persistent CTA walks several tiles and carries its pipeline state (chunk counter, ring-slot parities, prefetch under the
epilogue, TMEM accumulator reuse) across them.  Batches are the exact ones `bench.py` builds (`bench.make_batch`),
default engine policy (no environment overrides), eager and through the CUDA-graph replay the bench uses.

Oracle: oracle/layers_ref.py on the CPU, fp32 (the north-star comparison: forward rel 1e-5, gradients rel 1e-4) and
fp64 (arbitration: where two fp32 evaluations differ, the fp64 one says which is right).
"""
import os
import sys

import pytest
import torch

from conftest import FWD_TOL, GRAD_TOL, ROOT, rel_err
from oracle import layers_ref as R

if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu
DEV = "cuda"
T = 3

# (id, bench workload, complexes, hidden override, env) -- rows per block in the comments are for the default seed
REGIME = [
    ("md17_bench", "md17", 100, None, {}),                          # 422 tiles of pairs, 69 tiles of simplices, C=32
    ("nba_bench", "nba", 100, None, {}),                            # 1 848 tiles of pairs, 181 of simplices, Cl(2,0), C=40
    ("motion_bench", "motion", 100, None, {}),                      # 177 tiles of pairs on tcgen05, node blocks on SIMT
    ("motion_all_tc", "motion", 100, None, {"CSMPN_TC_MIN_ROWS": "0"}),
    ("md17_1000_tiles", "md17", 250, None, {}),                     # > 1 000 tiles of pairs: 7 tiles per CTA
    ("md17_c16", "md17", 60, 16, {"CSMPN_TC_MIN_ROWS": "0"}),       # narrow block, ragged last tile
]


def _oracle(b, params, dtype):
    ralg = R.RefAlgebra(b["metric"])
    h = b["h"].to(dtype).requires_grad_()
    p = {k: v.to(dtype).requires_grad_() for k, v in params.items()}
    y = R.egcl(ralg, h, b["edge_index"], b["edge_attr"].to(dtype), b["node_attr"].to(dtype), p, aggr=b["aggr"])
    names = list(p)
    grads = torch.autograd.grad(y, [h] + [p[k] for k in names], b["cot"].to(dtype))
    return y.detach(), dict(zip(["h"] + names, grads))


def _ours(b, params, graphed=False):
    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.models.cegnn_utils import EGCL
    from csmpn_b200.models.ops import CSRGraph

    alg = CliffordAlgebra(b["metric"]).to(DEV)
    C = b["C"]
    m = EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=b["aggr"]).to(DEV)
    missing, unexpected = m.load_state_dict(params, strict=False)
    assert not unexpected and all("algebra" in k for k in missing), (missing, unexpected)
    d = {k: b[k].to(DEV) for k in ("h", "edge_index", "edge_attr", "node_attr", "cot")}
    graph = CSRGraph(d["edge_index"], b["N"])
    named = dict(m.named_parameters())
    names = list(params)
    h = d["h"].clone().requires_grad_()
    if graphed:
        from csmpn_b200.graphs import GraphedEGCL

        g = GraphedEGCL(m, graph, d["h"], d["edge_attr"], d["node_attr"])
        y = g(h, d["edge_attr"], d["node_attr"])
    else:
        y = m(h, graph, d["edge_attr"], d["node_attr"])
    grads = torch.autograd.grad(y, [h] + [named[k] for k in names], d["cot"])
    torch.cuda.synchronize()
    return y.detach().cpu(), {k: v.cpu() for k, v in zip(["h"] + names, grads)}


def _check(tag, got, ref32, ref64, tol):
    """ours within `tol` of the fp32 oracle; where the fp32 oracle itself is further than that from the fp64 one (long
    fp32 sums over 10^5 rows), the fp64 oracle arbitrates."""
    e32, e64 = rel_err(got, ref32), rel_err(got, ref64.float())
    assert min(e32, e64) <= tol, f"{tag}: rel err vs fp32 oracle {e32:.2e}, vs fp64 oracle {e64:.2e} > {tol:.0e}"
    return e32, e64


@pytest.fixture(scope="module")
def bench_mod():
    import bench

    return bench


@pytest.mark.parametrize("case", REGIME, ids=[c[0] for c in REGIME])
def test_layer_step_matches_oracle_in_bench_regime(case, bench_mod, monkeypatch):
    from csmpn_b200 import _lib
    from csmpn_b200.models import fused

    name, workload, ncx, hidden, env = case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    b = bench_mod.make_batch(workload, ncx, 1000, hidden=hidden)
    ralg = R.RefAlgebra(b["metric"])
    params = R.init_egcl_params(ralg, b["C"], T, torch.Generator().manual_seed(7))
    tiles = (b["E"] + 127) // 128
    assert tiles > 148, (name, tiles)  # several tiles per persistent CTA
    assert fused.tc_supported(len(b["metric"]), b["C"] + 2 * T, b["C"]) and b["E"] >= fused.tc_min_rows()
    y32, g32 = _oracle(b, params, torch.float32)
    y64, g64 = _oracle(b, params, torch.float64)
    n0 = _lib.lib().csmpn_launch_count()
    y, g = _ours(b, params)
    assert _lib.lib().csmpn_launch_count() - n0 >= 30  # 2 + 7 kernels per tensor-core block
    worst = {"fwd": _check(f"{name} fwd", y, y32, y64, FWD_TOL)}
    for k in g32:
        worst[k] = _check(f"{name} grad {k}", g[k], g32[k], g64[k], GRAD_TOL)
    print(f"[regime] {name}: N={b['N']} E={b['E']} tiles={tiles} fwd {worst['fwd'][0]:.1e}/{worst['fwd'][1]:.1e} "
          f"worst grad {max(v[0] for k, v in worst.items() if k != 'fwd'):.1e} (vs fp32 oracle)")


@pytest.mark.parametrize("workload", ["md17", "nba"])
def test_graph_replay_matches_eager_and_oracle_in_bench_regime(workload, bench_mod):
    """the launch path `bench.py` times: csmpn_b200.graphs.GraphedEGCL on the bench batch -- bit-identical to the eager
    step and within tolerance of the oracle"""
    b = bench_mod.make_batch(workload, 100, 1000)
    ralg = R.RefAlgebra(b["metric"])
    params = R.init_egcl_params(ralg, b["C"], T, torch.Generator().manual_seed(7))
    y_e, g_e = _ours(b, params, graphed=False)
    y_g, g_g = _ours(b, params, graphed=True)
    assert torch.equal(y_e, y_g)
    for k in g_e:
        assert torch.equal(g_e[k], g_g[k]), k
    y32, g32 = _oracle(b, params, torch.float32)
    y64, g64 = _oracle(b, params, torch.float64)
    _check(f"{workload} graphed fwd", y_g, y32, y64, FWD_TOL)
    for k in g32:
        _check(f"{workload} graphed grad {k}", g_g[k], g32[k], g64[k], GRAD_TOL)


def test_step_is_deterministic_in_bench_regime(bench_mod):
    """two runs of the same multi-tile step give bit-identical outputs and gradients (fixed-order reductions, no atomics)"""
    b = bench_mod.make_batch("md17", 100, 1000)
    params = R.init_egcl_params(R.RefAlgebra(b["metric"]), b["C"], T, torch.Generator().manual_seed(7))
    y1, g1 = _ours(b, params)
    y2, g2 = _ours(b, params)
    assert torch.equal(y1, y2)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k


def test_overlapped_epilogue_bitwise_in_bench_regime(bench_mod, monkeypatch):
    """three tiles per CTA, alternating TMEM buffers: the overlapped-epilogue kernels reproduce the plain kernels' layer
    output and every gradient bit for bit on the bench batch"""
    b = bench_mod.make_batch("md17", 100, 1000)
    params = R.init_egcl_params(R.RefAlgebra(b["metric"]), b["C"], T, torch.Generator().manual_seed(7))
    monkeypatch.setenv("CSMPN_TC_OVERLAP", "1")
    y1, g1 = _ours(b, params)
    monkeypatch.setenv("CSMPN_TC_OVERLAP", "0")
    y0, g0 = _ours(b, params)
    assert torch.equal(y1, y0)
    for k in g1:
        assert torch.equal(g1[k], g0[k]), k
