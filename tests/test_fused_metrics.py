"""CEMLP blocks and EGCL layers of non-degenerate Cl(p,q) and rescaled metrics on the fused engines.

fused.enabled admits every diagonal metric of dimension 2, 3 or 5 without a zero entry; the kernels fold the metric into
their elementwise stages (MVSiLU invariants, normalisation, weighted geometric product, MVLayerNorm).  Per metric and
regime (FP32 SIMT engine below 32 tiles, tensor-core engine with ragged row counts, the streamed / wide C = 64 plan) an
EGCL layer and a plain CEMLP run forward and every gradient; each block's engine is read from fused._RECORDER, the
result is held to the fp64 oracle and cross-checked against the unit-kernel composition (CSMPN_FUSED=0).

Rule for the metrics with a negative entry (fused.tc_metric): their quadratic forms are indefinite, and the tensor-core
engine does not meet the oracle bound for them at scale, so in the "tc" and "wide" regimes their blocks must run on the
FP32 SIMT engine (or, too wide for it, on unit kernels) and meet the bound there."""
import ctypes
import functools

import pytest
import torch

from conftest import rel_err, tols
from egcl_harness import (DEV, assert_all_equal, cemlp_model, egcl_inputs, egcl_model, grads, mods, oracle_egcl,
                          run_egcl)
from oracle import layers_ref as R

T = 3  # node-attribute types: edge_attr = node_attr[src] | node_attr[dst] has 2T channels
WRT = ("h", "node_attr")
METRICS = [(1.0, -1.0), (-1.0, -1.0), (1.0, 1.0, -1.0), (-1.0, -1.0, -1.0), (2.0, 1.0, 0.5)]
CL41 = (1.0, 1.0, 1.0, 1.0, -1.0)  # conformal algebra of 3-D space: dimension 5, FP32 SIMT engine only
SIMT, TC = 0, 1

# regime -> (engine of every block, EGCL shape (C, complexes, simplices / complex, pairs / complex),
#            CEMLP shape (c_in, C, rows), CSMPN_TC_MIN_ROWS or None for the default policy)
REGIMES = {
    "simt": (SIMT, (24, 3, 41, 120), (5, 24, 300), None),
    # >= 32 tiles in every block: 4 164 simplices (32 tiles + 68 rows), 4 800 pairs (37 tiles + 64 rows)
    "tc": (TC, (32, 12, 347, 400), (7, 32, 4133), None),
    # C = 64: streamed forward weights and the wide backward (csmpn_block_tc_plan bits 1-3); small on purpose
    "wide": (TC, (64, 2, 87, 300), (64, 64, 300), "0"),
}
CASES = [(m, r) for m in METRICS for r in REGIMES] + [(CL41, "simt")]


def _id(metric, regime):
    return "cl" + "_".join(f"{v:g}".replace("-", "m").replace(".", "p") for v in metric) + "-" + regime


IDS = [_id(*c) for c in CASES]


def _egcl_case(metric, regime):
    C, ncx, n, e = REGIMES[regime][1]
    if len(metric) == 5:
        C, ncx, n, e = 8, 2, 31, 90
    return (_id(metric, regime), metric, C, T, ncx, n, e, "sum" if len(metric) % 2 else "mean")


@functools.lru_cache(maxsize=None)
def _egcl_data(metric, regime):
    """inputs, fp32 and fp64 oracle of the EGCL case"""
    inp = egcl_inputs(_egcl_case(metric, regime))
    return inp, oracle_egcl(inp, torch.float32, WRT, "paired"), oracle_egcl(inp, torch.float64, WRT, "paired")


@functools.lru_cache(maxsize=None)
def _cemlp_data(metric, regime):
    """parameters, input, cotangent, fp32 and fp64 oracle of the 2-block CEMLP case"""
    cin, C, rows = REGIMES[regime][2] if len(metric) < 5 else (3, 8, 200)
    gen = torch.Generator().manual_seed(sum(map(ord, _id(metric, regime) + "mlp")))
    ralg = R.RefAlgebra(metric)
    params = R.init_cemlp_params(ralg, cin, C, C, 2, gen)
    x = torch.randn(rows, cin, ralg.B, generator=gen)
    cot = torch.randn(rows, C, ralg.B, generator=gen)

    def oracle(dtype):
        xl = x.to(dtype, copy=True).requires_grad_()
        p = {k: v.to(dtype, copy=True).requires_grad_() for k, v in params.items()}
        y = R.cemlp(ralg, xl, p)
        g = torch.autograd.grad(y, [xl] + list(p.values()), cot.to(dtype))
        return y.detach(), dict(zip(["x"] + list(p), g))

    return (cin, C, params, x, cot), oracle(torch.float32), oracle(torch.float64)


def _run_cemlp(metric, regime):
    (cin, C, params, x, cot), _, _ = _cemlp_data(metric, regime)
    m = cemlp_model(metric, cin, C, 2, params)
    xd = x.to(DEV).requires_grad_()
    y = m(xd)
    pd = dict(m.named_parameters())
    g = grads(y, cot, [xd] + [pd[k] for k in params])
    torch.cuda.synchronize()
    return m, (y.detach(), dict(zip(["x"] + list(params), g)))


def _engine(metric, regime):
    """engine every recorded block call must report: positive metrics follow the regime, the others never reach the
    tensor-core engine (fused.tc_metric)"""
    return REGIMES[regime][0] if all(m > 0 for m in metric) else SIMT


def _check_calls(calls, metric, regime, nblocks, addr):
    positive = all(m > 0 for m in metric)
    if positive or regime != "wide":  # indefinite wide blocks may be too wide for the SIMT engine: unit kernels then
        assert [k for k, _, _ in calls] == ["fwd"] * nblocks + ["bwd"] * nblocks, calls
    assert all(e == _engine(metric, regime) and a == addr for _, e, a in calls), calls


def _recorded(monkeypatch, run):
    """run() with every native block call recorded: (result, [(kind, engine, metric address)])"""
    from csmpn_b200.models import fused

    rec = []
    monkeypatch.setattr(fused, "_RECORDER", rec)
    out = run()
    monkeypatch.setattr(fused, "_RECORDER", None)
    return out, [(c["kind"], int(c["desc"].engine), c["desc"].metric) for c in rec]


def _check_vs_oracle(got, ref32, ref64, metric, tag, unit=None):
    """each tensor within max(conftest.tols for the metric, 4 x the fp32 oracle's own error) of the fp64 oracle;
    returns the per-tensor bounds.  unit (metrics with a negative entry): the unit-kernel result, whose own error
    counts like the fp32 oracle's -- indefinite forms cancel towards 0 where the normalisation derivatives are steepest,
    and there two correct fp32 evaluations already differ by more than conftest.tols (measured: up to 2.3x over
    4 x the fp32 oracle's error for the unit kernels themselves)."""
    fwd_tol, grad_tol = tols({"metric": metric})
    bounds = {}
    for k, g, r32, r64, tol in [("fwd", got[0], ref32[0], ref64[0], fwd_tol)] + [
            (k, got[1][k], ref32[1][k], ref64[1][k], grad_tol) for k in ref64[1]]:
        ref_err = rel_err(r32, r64)
        if unit is not None:
            ref_err = max(ref_err, rel_err(unit[0] if k == "fwd" else unit[1][k], r64))
        bound = max(tol, 4 * ref_err)
        e = rel_err(g, r64)
        assert e <= bound, f"{tag} {k}: rel err {e:.3e} vs fp64 oracle > bound {bound:.3e}"
        bounds[k] = bound
    return bounds


def _check_vs_unit(got, unit, bounds, tag):
    """fused against unit kernels: both within a bound of the fp64 oracle, so within twice that bound of each other"""
    for k, g, u in [("fwd", got[0], unit[0])] + [(k, got[1][k], unit[1][k]) for k in unit[1]]:
        e = rel_err(g, u)
        assert e <= 2 * bounds[k], f"{tag} {k}: fused vs unit kernels rel err {e:.3e} > {2 * bounds[k]:.3e}"


@pytest.fixture
def regime_env(monkeypatch):
    def set_(regime):
        monkeypatch.setenv("CSMPN_TC", "1")
        monkeypatch.delenv("CSMPN_FUSED", raising=False)
        if REGIMES[regime][3] is None:
            monkeypatch.delenv("CSMPN_TC_MIN_ROWS", raising=False)
        else:
            monkeypatch.setenv("CSMPN_TC_MIN_ROWS", REGIMES[regime][3])
    return set_


@pytest.fixture
def precision():
    """set torch.backends.cuda.matmul.fp32_precision for the test and restore it afterwards"""
    old = torch.backends.cuda.matmul.fp32_precision

    def set_(value):
        torch.backends.cuda.matmul.fp32_precision = value

    yield set_
    torch.backends.cuda.matmul.fp32_precision = old


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("metric", [(1, -1), (1, 1, -1), (2, 1, 0.5), (-1, -1, -1, -1, 1)])
def test_enabled_admits_non_degenerate_metrics(metric, monkeypatch):
    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.models import fused

    monkeypatch.delenv("CSMPN_FUSED", raising=False)
    alg = CliffordAlgebra(metric)
    assert fused.enabled(alg)
    monkeypatch.setenv("CSMPN_FUSED", "0")
    assert not fused.enabled(alg)


@pytest.mark.parametrize("metric", [(1, 1, 0), (0, 1), (1, 1, 1, 1), (1, 1, 1, -1), (1, -1, -1, -1)])
def test_enabled_rejects_degenerate_and_dim4_metrics(metric, monkeypatch):
    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.models import fused

    monkeypatch.delenv("CSMPN_FUSED", raising=False)
    assert not fused.enabled(CliffordAlgebra(metric))


def test_block_abi_rejects_a_zero_metric_entry():
    """csmpn_block_desc.metric: a zero entry is CSMPN_ERR_UNSUPPORTED on both engines, checked on the host before any
    launch; NULL, all ones and a non-degenerate metric pass the descriptor check"""
    import __graft_entry__ as ge

    ge.build()
    from csmpn_b200 import _lib
    from csmpn_b200.models import fused

    L = _lib.lib()
    d = fused.BlockDesc()
    d.mode, d.c0, d.c, d.rows = 0, 4, 4, 1
    for name in ("p0", "w1", "sa", "sb", "wr", "na", "wl", "bl", "wp", "la", "y"):
        setattr(d, name, 256)  # never dereferenced: the descriptor check fails first, or no kernel runs
    for engine in (0, 1):
        d.engine = engine
        for vals, ok in (((1, 1, 0), False), ((0, 1, 1), False), ((1, 1, -1), True), ((1, 1, 1), True), (None, True)):
            arr = None if vals is None else (ctypes.c_float * 3)(*vals)
            d.metric = None if arr is None else ctypes.addressof(arr)
            if engine == 0:
                assert (L.csmpn_block_fwd_workspace(3, ctypes.byref(d)) == 0) == ok, (engine, vals)
            if not ok:
                assert L.csmpn_block_fwd(3, ctypes.byref(d), None) == -3, (engine, vals)
                assert L.csmpn_block_bwd_workspace(3, ctypes.byref(d)) == -1, (engine, vals)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("metric,regime", CASES, ids=IDS)
def test_egcl_vs_fp64_oracle_and_unit_kernels(metric, regime, monkeypatch, regime_env):
    """EGCL layer (4 blocks): forward, gradients of h, node_attr and every parameter; engine of every block"""
    regime_env(regime)
    inp, ref32, ref64 = _egcl_data(metric, regime)
    case = _egcl_case(metric, regime)
    m = egcl_model(metric, case[2], T, case[7], inp["params"])
    got, calls = _recorded(monkeypatch, lambda: run_egcl(m, inp, WRT, "paired"))
    _check_calls(calls, metric, regime, 4, ctypes.addressof(m.algebra._metric_c))
    monkeypatch.setenv("CSMPN_FUSED", "0")
    unit, calls = _recorded(monkeypatch, lambda: run_egcl(m, inp, WRT, "paired"))
    assert calls == []
    bounds = _check_vs_oracle(got, ref32, ref64, metric, case[0], None if min(metric) > 0 else unit)
    _check_vs_unit(got, unit, bounds, case[0])


@pytest.mark.gpu
@pytest.mark.parametrize("metric,regime", CASES, ids=IDS)
def test_cemlp_vs_fp64_oracle_and_unit_kernels(metric, regime, monkeypatch, regime_env):
    """plain 2-block CEMLP on rows (mode 0): forward, gradients of x and every parameter; engine of every block"""
    regime_env(regime)
    _, ref32, ref64 = _cemlp_data(metric, regime)
    (m, got), calls = _recorded(monkeypatch, lambda: _run_cemlp(metric, regime))
    _check_calls(calls, metric, regime, 2, ctypes.addressof(m.algebra._metric_c))
    monkeypatch.setenv("CSMPN_FUSED", "0")
    (_, unit), calls = _recorded(monkeypatch, lambda: _run_cemlp(metric, regime))
    assert calls == []
    bounds = _check_vs_oracle(got, ref32, ref64, metric, _id(metric, regime) + " cemlp", None if min(metric) > 0 else unit)
    _check_vs_unit(got, unit, bounds, _id(metric, regime) + " cemlp")


@pytest.mark.gpu
def test_degenerate_metric_stays_on_unit_kernels(monkeypatch, regime_env):
    """Cl(2,0,1)-style (1, 1, 0): no fused block call, and the unit-kernel layer matches the fp64 oracle"""
    regime_env("simt")
    metric = (1.0, 1.0, 0.0)
    case = ("degenerate", metric, 16, T, 2, 41, 120, "sum")
    inp = egcl_inputs(case)
    m = egcl_model(metric, 16, T, "sum", inp["params"])
    got, calls = _recorded(monkeypatch, lambda: run_egcl(m, inp, WRT, "paired"))
    assert calls == []
    _check_vs_oracle(got, oracle_egcl(inp, torch.float32, WRT, "paired"), oracle_egcl(inp, torch.float64, WRT, "paired"),
                     metric, "degenerate")


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["simt", "tc"])
def test_graphed_replay_and_eager_runs_are_bitwise_equal(regime, regime_env):
    """Cl(2,1): a GraphedEGCL replay equals the eager step bit for bit, and so do two eager steps (fixed-order reductions
    on both engines).  The graph is captured before any eager autograd on the same leaves, as in test_tc_block.py."""
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    regime_env(regime)
    metric = (1.0, 1.0, -1.0)
    inp, _, _ = _egcl_data(metric, regime)
    case = _egcl_case(metric, regime)
    _, M = mods()
    m = egcl_model(metric, case[2], T, case[7], inp["params"])
    plist = list(m.parameters())
    hd, cotd = inp["h"].to(DEV), inp["cot"].to(DEV)
    nad = inp["na"].to(DEV).requires_grad_()
    graph = CSRGraph(inp["ei"].to(DEV), hd.shape[0])
    g = GraphedEGCL(m, graph, hd, M.PairedNodeAttr(nad), nad)
    h2 = hd.clone().requires_grad_()
    yg = g(h2, None, nad)
    replay = (yg.detach(), dict(enumerate(torch.autograd.grad(yg, [h2, nad] + plist, cotd))))
    eager = []
    for _ in range(2):
        h1 = hd.clone().requires_grad_()
        ye = m(h1, graph, M.PairedNodeAttr(nad), nad)
        eager.append((ye.detach(), dict(enumerate(torch.autograd.grad(ye, [h1, nad] + plist, cotd)))))
    torch.cuda.synchronize()
    assert_all_equal(eager[1], eager[0], "eager vs eager")
    assert_all_equal(replay, eager[0], "graph replay vs eager")


@pytest.mark.gpu
@pytest.mark.parametrize("metric", METRICS, ids=[_id(m, "tc") for m in METRICS])
def test_tf32_mode_follows_the_precision_setting(metric, monkeypatch, regime_env, precision):
    """Single-pass TF32 (torch.backends.cuda.matmul.fp32_precision = "tf32"): blocks of a positive non-Euclidean metric
    follow the setting like Euclidean ones -- they stay on the tensor-core engine and meet the TF32 tolerances of
    test_tc_precision.py (5e-3 forward, 2e-2 gradients) against the fp64 oracle.  Metrics with a negative entry stay on
    the FP32 SIMT engine in this mode too (on the tensor-core engine their TF32 gradient errors reach O(1)), which ignores
    the setting: the TF32-mode step equals the default-mode step bit for bit."""
    regime_env("tc")
    inp, _, ref64 = _egcl_data(metric, "tc")
    case = _egcl_case(metric, "tc")
    m = egcl_model(metric, case[2], T, case[7], inp["params"])
    precision("tf32")
    got, calls = _recorded(monkeypatch, lambda: run_egcl(m, inp, WRT, "paired"))
    precision("ieee")
    assert len(calls) == 8 and all(e == _engine(metric, "tc") for _, e, _ in calls), calls
    if min(metric) < 0:
        assert_all_equal(got, run_egcl(m, inp, WRT, "paired"), f"{case[0]} tf32 vs default mode")
        return
    e_fwd = rel_err(got[0], ref64[0])
    e_grad = {k: rel_err(got[1][k], ref64[1][k]) for k in ref64[1]}
    worst = max(e_grad, key=e_grad.get)
    print(f"[metric tf32] {case[0]}: fwd {e_fwd:.2e}, worst grad {worst} {e_grad[worst]:.2e}")
    assert e_fwd <= 5e-3 and e_grad[worst] <= 2e-2, (case[0], e_fwd, worst, e_grad[worst])
