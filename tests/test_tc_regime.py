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
from egcl_harness import DEV, assert_all_equal, bench_inputs, egcl_model, oracle_egcl

if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu
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


def _ours(b, inp, graphed=False):
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    m = egcl_model(b["metric"], b["C"], T, b["aggr"], inp["params"])
    h0, ea, na, cot = (inp[k].to(DEV) for k in ("h", "ea", "na", "cot"))
    graph = CSRGraph(inp["ei"].to(DEV), b["N"])
    pd = dict(m.named_parameters())
    names = list(inp["params"])
    h = h0.clone().requires_grad_()
    y = GraphedEGCL(m, graph, h0, ea, na)(h, ea, na) if graphed else m(h, graph, ea, na)
    grads = torch.autograd.grad(y, [h] + [pd[k] for k in names], cot)
    torch.cuda.synchronize()
    return y.detach().cpu(), {k: v.cpu() for k, v in zip(["h"] + names, grads)}


def _check(tag, got, ref32, ref64, tol):
    """ours within `tol` of the fp32 oracle; where the fp32 oracle itself is further than that from the fp64 one (long
    fp32 sums over 10^5 rows), the fp64 oracle arbitrates."""
    e32, e64 = rel_err(got, ref32), rel_err(got, ref64.float())
    assert min(e32, e64) <= tol, f"{tag}: rel err vs fp32 oracle {e32:.2e}, vs fp64 oracle {e64:.2e} > {tol:.0e}"
    return e32, e64


def _check_vs_oracle(tag, got, inp):
    """_check of the forward output and every gradient; returns (error vs fp32, vs fp64) per name"""
    (y32, g32), (y64, g64) = (oracle_egcl(inp, dtype, ("h",), "tensor") for dtype in (torch.float32, torch.float64))
    worst = {"fwd": _check(f"{tag} fwd", got[0], y32, y64, FWD_TOL)}
    for k in g32:
        worst[k] = _check(f"{tag} grad {k}", got[1][k], g32[k], g64[k], GRAD_TOL)
    return worst


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
    inp = bench_inputs(b)
    tiles = (b["E"] + 127) // 128
    assert tiles > 148, (name, tiles)  # several tiles per persistent CTA
    assert fused.tc_supported(len(b["metric"]), b["C"] + 2 * T, b["C"]) and b["E"] >= fused.tc_min_rows()
    n0 = _lib.lib().csmpn_launch_count()
    got = _ours(b, inp)
    assert _lib.lib().csmpn_launch_count() - n0 >= 30  # 2 + 7 kernels per tensor-core block
    worst = _check_vs_oracle(name, got, inp)
    print(f"[regime] {name}: N={b['N']} E={b['E']} tiles={tiles} fwd {worst['fwd'][0]:.1e}/{worst['fwd'][1]:.1e} "
          f"worst grad {max(v[0] for k, v in worst.items() if k != 'fwd'):.1e} (vs fp32 oracle)")


@pytest.mark.parametrize("workload", ["md17", "nba"])
def test_graph_replay_matches_eager_and_oracle_in_bench_regime(workload, bench_mod):
    """the launch path `bench.py` times: csmpn_b200.graphs.GraphedEGCL on the bench batch -- bit-identical to the eager
    step and within tolerance of the oracle"""
    b = bench_mod.make_batch(workload, 100, 1000)
    inp = bench_inputs(b)
    eager = _ours(b, inp, graphed=False)
    graphed = _ours(b, inp, graphed=True)
    assert_all_equal(graphed, eager, f"{workload} graphed vs eager:")
    _check_vs_oracle(f"{workload} graphed", graphed, inp)


def test_step_is_deterministic_in_bench_regime(bench_mod):
    """two runs of the same multi-tile step give bit-identical outputs and gradients (fixed-order reductions, no atomics)"""
    b = bench_mod.make_batch("md17", 100, 1000)
    inp = bench_inputs(b)
    first = _ours(b, inp)
    assert_all_equal(_ours(b, inp), first, "md17 second run vs first:")


def test_overlapped_epilogue_bitwise_in_bench_regime(bench_mod, monkeypatch):
    """three tiles per CTA, alternating TMEM buffers: the overlapped-epilogue kernels reproduce the plain kernels' layer
    output and every gradient bit for bit on the bench batch"""
    b = bench_mod.make_batch("md17", 100, 1000)
    inp = bench_inputs(b)
    monkeypatch.setenv("CSMPN_TC_OVERLAP", "1")
    overlapped = _ours(b, inp)
    monkeypatch.setenv("CSMPN_TC_OVERLAP", "0")
    assert_all_equal(overlapped, _ours(b, inp), "md17 overlapped vs plain:")
