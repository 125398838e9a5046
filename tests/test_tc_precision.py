"""Single-pass TF32 mode of the tensor-core engine (csmpn_block_desc.tf32), selected by PyTorch's float32 matmul precision
(models/fused.py tc_precision): the resolver on the CPU; on the GPU its accuracy against the fp64 oracle, that the mode
is really taken, fixed at forward time, leaves no state behind, is deterministic and survives CUDA-graph capture."""
import json
import os
import subprocess
import sys

import pytest
import torch

from conftest import ROOT, load_golden, rel_err
from egcl_harness import (CASES, DEV, WIDE, assert_all_equal, bench_inputs, egcl_inputs, egcl_model, mods, oracle_egcl,
                          run_egcl)
from oracle import layers_ref as R

PAIRED = ("h", "node_attr")

# max-norm relative error against the fp64 oracle in TF32 mode.  Largest values measured on a B200 over every case here
# (DESIGN.md 4.1): forward 1.3e-3, worst gradient 6.0e-3 (both NBA-shaped, Cl(2,0)); md17 model 7.1e-3.  Each bound has at
# least 3x headroom.
TF32_FWD_TOL = 5e-3
TF32_GRAD_TOL = 2e-2
TF32_MD17_TOL = 2.5e-2   # md17 model at the benched size against the golden (fp32 reference) loss / outputs / gradients


# ---------------------------------------------------------------------------------------------------------------- CPU
RESOLVER_CASES = [
    # name, statements run in a fresh interpreter, TF32 mode expected
    ("fresh", "", False),
    ("legacy_high", "torch.set_float32_matmul_precision('high')", True),
    ("legacy_medium", "torch.set_float32_matmul_precision('medium')", True),
    ("legacy_highest", "torch.set_float32_matmul_precision('highest')", False),
    ("allow_tf32", "torch.backends.cuda.matmul.allow_tf32 = True", True),
    ("allow_tf32_off", "torch.backends.cuda.matmul.allow_tf32 = False", False),
    ("generic_tf32", "torch.backends.fp32_precision = 'tf32'", True),
    ("generic_ieee", "torch.backends.fp32_precision = 'ieee'", False),
    ("cuda_matmul_tf32", "torch.backends.cuda.matmul.fp32_precision = 'tf32'", True),
    ("cuda_matmul_ieee", "torch.backends.cuda.matmul.fp32_precision = 'ieee'", False),
    ("mixed_legacy_then_new_tf32", "torch.set_float32_matmul_precision('highest'); torch.backends.cuda.matmul.fp32_precision = 'tf32'", True),
    ("mixed_legacy_then_new_ieee", "torch.set_float32_matmul_precision('high'); torch.backends.cuda.matmul.fp32_precision = 'ieee'", False),
    ("mixed_new_then_legacy", "torch.backends.cuda.matmul.fp32_precision = 'ieee'; torch.backends.cuda.matmul.allow_tf32 = True", True),
]

_RESOLVE = """
import json, sys, warnings
warnings.simplefilter("ignore")
sys.path.insert(0, {root!r})
import torch
{stmts}
from csmpn_b200.models import fused
try:
    torch.get_float32_matmul_precision()
    legacy_raises = False
except RuntimeError:
    legacy_raises = True
print(json.dumps({{"tf32": fused.tc_precision(), "legacy_raises": legacy_raises}}))
"""


@pytest.mark.parametrize("case", RESOLVER_CASES, ids=[c[0] for c in RESOLVER_CASES])
def test_precision_resolver(case):
    """Every way of asking PyTorch for TF32 matmuls selects TF32 mode, everything else the default; a mixed legacy + new
    API state (where torch.get_float32_matmul_precision() raises) does not make the resolver raise.  Each case runs in
    its own interpreter: the torch setting is process-global and the mixed state is sticky."""
    name, stmts, want = case
    r = subprocess.run([sys.executable, "-c", _RESOLVE.format(root=ROOT, stmts=stmts)], capture_output=True, text=True,
                       cwd=ROOT, timeout=300)
    assert r.returncode == 0, r.stderr
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert got["tf32"] is want, (name, got)
    if name.startswith("mixed_legacy_then_new_tf32"):
        assert got["legacy_raises"], "the case should exercise a mixed legacy + new API state"


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture
def precision(monkeypatch):
    """set torch.backends.cuda.matmul.fp32_precision for the test and restore it afterwards; small cases on the
    tensor-core engine as in test_tc_block.py"""
    monkeypatch.setenv("CSMPN_TC_MIN_ROWS", "0")
    monkeypatch.setenv("CSMPN_TC", "1")
    old = torch.backends.cuda.matmul.fp32_precision

    def set_(value):
        torch.backends.cuda.matmul.fp32_precision = value

    yield set_
    torch.backends.cuda.matmul.fp32_precision = old


def _step(m, inp):
    """layer forward + (grad h, grad node_attr, every parameter gradient); edge_attr = node_attr[src] | node_attr[dst]"""
    return run_egcl(m, inp, PAIRED, "paired")


def _layer(case):
    name, metric, C, T, ncx, n, e, aggr = case
    inp = egcl_inputs(case)
    return egcl_model(metric, C, T, aggr, inp["params"]), inp


def _oracle_gpu_tf32(inp):
    """the oracle itself in fp32 on the GPU under the current matmul precision (its linears are einsums): what a
    plain-PyTorch implementation computes with TF32 matmuls"""
    import copy

    ralg = inp["ralg"]
    g = copy.copy(ralg)
    for k, v in vars(ralg).items():
        if torch.is_tensor(v):
            setattr(g, k, v.to(DEV))
    p = {k: v.to(DEV) for k, v in inp["params"].items()}
    nd, eid = inp["na"].to(DEV), inp["ei"].to(DEV)
    with torch.no_grad(), torch.device(DEV):  # the oracle creates its scratch tensors without a device argument
        return R.egcl(g, inp["h"].to(DEV), eid, torch.cat([nd[eid[0]], nd[eid[1]]], 1), nd, p, aggr=inp["aggr"])


def _errors(res, ref):
    return rel_err(res[0], ref[0]), max(rel_err(res[1][k], r) for k, r in ref[1].items())


def _check_vs_oracle(name, m, inp, precision):
    ref = oracle_egcl(inp, torch.float64, PAIRED, "paired")
    res = {}
    for mode in ("ieee", "tf32"):
        precision(mode)
        res[mode] = _step(m, inp)
    e_ref = rel_err(_oracle_gpu_tf32(inp), ref[0])  # under TF32, the mode set last
    e_def, e_tf = _errors(res["ieee"], ref), _errors(res["tf32"], ref)
    print(f"[tf32] {name}: fp64-oracle error fwd / worst grad: default {e_def[0]:.2e} / {e_def[1]:.2e}, "
          f"tf32 {e_tf[0]:.2e} / {e_tf[1]:.2e}; oracle on the GPU with TF32 matmuls fwd {e_ref:.2e}")
    assert e_tf[0] <= TF32_FWD_TOL and e_tf[1] <= TF32_GRAD_TOL, (name, e_tf)
    # the path is really taken: different bits and a larger error than the error-compensated products
    assert not torch.equal(res["tf32"][0], res["ieee"][0])
    assert e_tf[0] > e_def[0] and e_tf[1] > e_def[1], (e_tf, e_def)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tf32_layer_vs_fp64_oracle(case, precision):
    _check_vs_oracle(case[0], *_layer(case), precision)


@pytest.mark.gpu
@pytest.mark.parametrize("case", WIDE, ids=[c[0] for c in WIDE])
def test_tf32_wide_layer_vs_fp64_oracle(case, precision):
    """streamed weights (the [pass][K chunk][grade][2][R][4] units) and the slab-wise weight-gradient launches"""
    _check_vs_oracle(case[0], *_layer(case), precision)


@pytest.mark.gpu
def test_tf32_md17_bench_batch_vs_fp64_oracle(precision):
    """the md17 batch of bench.py (100 complexes: 52 k pairs, several tiles per persistent CTA)"""
    sys.path.insert(0, ROOT)
    import bench

    b = bench.make_batch("md17", 100, 1000)
    inp = bench_inputs(b)
    _check_vs_oracle("md17_bench", egcl_model(b["metric"], b["C"], 3, b["aggr"], inp["params"]), inp, precision)


@pytest.mark.gpu
def test_no_state_survives_a_tf32_run(precision):
    """A default run after TF32 runs equals a default run of a fresh model bit for bit (no cached TF32 weight images,
    no sticky descriptor field); wide blocks included (streamed weight images in the workspace)."""
    for case in (CASES[1], WIDE[0]):
        m, inp = _layer(case)
        precision("ieee")
        first = _step(m, inp)
        precision("tf32")
        _step(m, inp)
        precision("ieee")
        after = _step(m, inp)
        fresh = _step(_layer(case)[0], inp)
        assert_all_equal(after, fresh, f"{case[0]} after TF32 vs fresh:")
        assert_all_equal(after, first, f"{case[0]} after TF32 vs before:")


@pytest.mark.gpu
def test_mode_is_fixed_at_forward_time(precision):
    """switching the setting between forward and backward does not change the backward: gradients equal an all-TF32
    step bit for bit (and the other way round)"""
    _, M = mods()
    m, inp = _layer(CASES[1])  # md17-shaped, several tiles
    pd = dict(m.named_parameters())
    for fwd_mode, bwd_mode in (("tf32", "ieee"), ("ieee", "tf32")):
        precision(fwd_mode)
        ref = _step(m, inp)
        hd, nad = inp["h"].to(DEV).requires_grad_(), inp["na"].to(DEV).requires_grad_()
        y = m(hd, inp["ei"].to(DEV), M.PairedNodeAttr(nad), nad)
        precision(bwd_mode)
        g = torch.autograd.grad(y, [hd, nad] + [pd[k] for k in inp["params"]], inp["cot"].to(DEV))
        assert torch.equal(y, ref[0])
        for a, b in zip(g, ref[1].values()):
            assert torch.equal(a, b), (fwd_mode, bwd_mode)


@pytest.mark.gpu
def test_tf32_is_deterministic_and_kernel_family_independent(precision, monkeypatch):
    """two TF32 runs, and the overlapped-epilogue kernels against the plain ones (CSMPN_TC_OVERLAP=0), bit for bit"""
    m, inp = _layer(CASES[1])
    precision("tf32")
    runs = [_step(m, inp) for _ in range(2)]
    monkeypatch.setenv("CSMPN_TC_OVERLAP", "0")
    runs.append(_step(m, inp))
    for r in runs[1:]:
        assert_all_equal(r, runs[0], "tf32")


@pytest.mark.gpu
def test_graphed_layer_captured_under_tf32_replays_tf32(precision):
    """GraphedEGCL captured under TF32 replays the eager TF32 step bit for bit, even with the setting switched back
    before the replay: the mode is part of the captured launches.  (Captured before any eager autograd on the same
    leaves, as in test_tc_block.py.)"""
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    _, M = mods()
    m, inp = _layer(CASES[1])
    plist = list(m.parameters())
    hd, cotd = inp["h"].to(DEV), inp["cot"].to(DEV)
    nad = inp["na"].to(DEV).requires_grad_()
    graph = CSRGraph(inp["ei"].to(DEV), hd.shape[0])
    precision("tf32")
    g = GraphedEGCL(m, graph, hd, M.PairedNodeAttr(nad), nad)
    precision("ieee")
    h2 = hd.clone().requires_grad_()
    yg = g(h2, None, nad)
    gg = torch.autograd.grad(yg, [h2, nad] + plist, cotd)
    precision("tf32")
    h1 = hd.clone().requires_grad_()
    ye = m(h1, graph, M.PairedNodeAttr(nad), nad)
    ge = torch.autograd.grad(ye, [h1, nad] + plist, cotd)
    assert torch.equal(ye, yg)
    for a, b in zip(ge, gg):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_graphed_layer_step_captured_under_tf32_replays_tf32(precision):
    """GraphedLayerStep (forward + backward + gradient pack as one graph) captured under TF32 replays the eager TF32 step
    bit for bit, with the setting switched back before the replay"""
    from csmpn_b200.graphs import GraphedLayerStep
    from csmpn_b200.models.ops import CSRGraph

    _, M = mods()
    m, inp = _layer(CASES[1])
    h, ei, na, cot = (inp[k] for k in ("h", "ei", "na", "cot"))
    plist = list(m.parameters())
    h_s, na_s, cot_s = h.to(DEV).clone(), na.to(DEV).clone(), cot.to(DEV).clone()
    precision("tf32")
    g = GraphedLayerStep(m, ei.to(DEV), h_s, na_s, cot_s)
    precision("ieee")
    y, gh, flat = g()
    precision("tf32")
    h1 = h.to(DEV).requires_grad_()
    ye = m(h1, CSRGraph(ei.to(DEV), h.shape[0]), M.PairedNodeAttr(na.to(DEV)), na.to(DEV))
    ge = torch.autograd.grad(ye, [h1] + plist, cot.to(DEV))
    assert torch.equal(y, ye) and torch.equal(gh, ge[0])
    assert torch.equal(flat, torch.cat([t.reshape(-1) for t in ge[1:]]))


@pytest.mark.gpu
def test_md17_model_at_benched_size_under_tf32(precision):
    """The md17 model at bench.py's training size (tests/golden/md17_bench.pt, the reference model's fp32 loss and
    sampled gradients) under TF32: within TF32_MD17_TOL, as test_models.py checks the default mode within 1e-5 / 1e-4"""
    import hashlib

    from csmpn_b200.data.modules.simplicial_data import SimplicialTransform
    from test_models import model_class

    sys.path.insert(0, ROOT)
    import bench

    precision("tf32")
    dev = torch.device("cuda:0")
    fx = load_golden("md17_bench.pt")
    graphs = bench.make_md17_graphs(fx["n_complexes"], fx["seed"], dev)
    batch = SimplicialTransform(dim=2, dis=2.5, label="md17", molecule_type="aspirin").lift(graphs, device=dev)
    sha = lambda t: hashlib.sha256(t.contiguous().cpu().numpy().tobytes()).hexdigest()
    assert sha(batch.edge_index) == fx["edge_index_sha256"]
    torch.manual_seed(fx["init_seed"])
    m = model_class("md17")().to(dev)
    loss, out = m(batch, 0, "train")
    named = list(m.named_parameters())
    grads = torch.autograd.grad(loss, [p for _, p in named], allow_unused=True)
    errs = {"loss": rel_err(loss, fx["loss"])}
    for k, v in fx["out"].items():
        errs[f"out[{k}]"] = rel_err(out[k], v)
    for (n, _), gr in zip(named, grads):
        ref = fx["grads"][n]
        if ref is None:
            continue
        flat = gr.detach().double().cpu().reshape(-1)
        errs[n] = float((flat[ref["index"].long()] - ref["value"].double()).abs().max()) / (ref["absmax"] + 1e-30)
    worst = max(errs, key=errs.get)
    print(f"[tf32] md17@{fx['n_complexes']}: loss rel err {errs['loss']:.2e}, worst {worst} {errs[worst]:.2e}")
    for k, e in errs.items():
        assert e <= TF32_MD17_TOL, f"md17 under TF32: {k} rel err {e:.3e} > {TF32_MD17_TOL:.1e}"
