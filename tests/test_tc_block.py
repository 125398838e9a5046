"""GPU parity of the tensor-core (tcgen05, 3xTF32) CEMLP-block engine: against the CPU oracle (fp32 tolerance of the
north star: forward rel 1e-5, gradients rel 1e-4) and against the FP32 SIMT engine on the same inputs."""
import pytest
import torch

from conftest import assert_close
from egcl_harness import (CASES, DEV, WIDE, assert_all_close, assert_all_equal, block_diag_graph, cemlp_model,
                          egcl_inputs, egcl_model, mods, oracle_egcl, run_egcl)
from oracle import layers_ref as R

pytestmark = pytest.mark.gpu
ALL_LEAVES = ("h", "edge_attr", "node_attr")
PAIRED = ("h", "node_attr")


@pytest.fixture(autouse=True)
def _force_tc_for_small_batches(monkeypatch):
    """the default policy keeps blocks with few rows on the SIMT engine; the parity cases here are small on purpose"""
    monkeypatch.setenv("CSMPN_TC_MIN_ROWS", "0")


def _layer(case):
    """seeded inputs of a case and its layer on the GPU"""
    name, metric, C, T, ncx, n, e, aggr = case
    inp = egcl_inputs(case)
    return egcl_model(metric, C, T, aggr, inp["params"]), inp


def test_tc_engine_is_selected():
    from csmpn_b200.models import fused

    assert fused.tc_supported(3, 38, 32) and fused.tc_supported(3, 67, 32) and fused.tc_supported(2, 46, 40)
    assert not fused.tc_supported(5, 28, 28)  # Cl(5,0): 32 blades do not fit the TMEM accumulator budget
    assert fused.tc_supported(3, 64, 64)  # wide block: streamed weights


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tc_forward_vs_oracle(case, monkeypatch):
    from csmpn_b200 import _lib

    name = case[0]
    m, inp = _layer(case)
    yr = R.egcl(inp["ralg"], inp["h"], inp["ei"], inp["ea"], inp["na"], inp["params"], aggr=inp["aggr"])
    outs = {}
    for tc in ("1", "0"):
        monkeypatch.setenv("CSMPN_TC", tc)
        n0 = _lib.lib().csmpn_launch_count()
        with torch.no_grad():
            outs[tc] = m(*(inp[k].to(DEV) for k in ("h", "ei", "ea", "na"))).cpu()
        outs["launches" + tc] = _lib.lib().csmpn_launch_count() - n0
    # the tensor-core engine launches two kernels per block (8 per layer) where the SIMT engine launches one
    assert outs["launches1"] == outs["launches0"] + 4, (outs["launches1"], outs["launches0"])
    assert_close(outs["1"], yr, 1e-5, f"{name} tensor-core fwd vs oracle")
    assert_close(outs["1"], outs["0"], 1e-5, f"{name} tensor-core fwd vs SIMT engine")


def test_tc_cemlp_dense_rows(monkeypatch):
    """CEMLP on plain rows (the models' embedding / projection MLPs): rows not a multiple of the 128-row tile."""
    gen = torch.Generator().manual_seed(5)
    ralg = R.RefAlgebra((1, 1, 1))
    for cin, c, rows in ((7, 32, 1000), (32, 32, 129), (3, 16, 1)):
        params = R.init_cemlp_params(ralg, cin, c, c, 2, gen)
        m = cemlp_model((1, 1, 1), cin, c, 2, params)
        x = torch.randn(rows, cin, 8, generator=gen)
        yr = R.cemlp(ralg, x, params)
        monkeypatch.setenv("CSMPN_TC", "1")
        with torch.no_grad():
            y = m(x.to(DEV))
        assert_close(y, yr, 1e-5, f"cemlp {cin}->{c} rows={rows}")


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tc_backward_vs_oracle(case, monkeypatch):
    """forward + every gradient of one EGCL layer on the tensor-core engine against the CPU oracle (autograd)."""
    from csmpn_b200 import _lib

    monkeypatch.setenv("CSMPN_TC", "1")
    m, inp = _layer(case)
    ref = oracle_egcl(inp, torch.float32, ALL_LEAVES, "tensor")
    n0 = _lib.lib().csmpn_launch_count()
    got = run_egcl(m, inp, ALL_LEAVES, "tensor")
    assert _lib.lib().csmpn_launch_count() - n0 > 30  # the tensor-core engine: 2 + 7 kernels per block
    assert_all_close(got, ref, 1e-5, 1e-4, case[0])


def test_graphed_layer_matches_eager():
    """CUDA-graph replay of a layer step (csmpn_b200.graphs.GraphedEGCL) reproduces the eager step bit for bit, for new
    input VALUES on the same complex structure."""
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    m, inp = _layer(CASES[1])
    plist = list(m.parameters())
    hd, ead, nad, cotd = (inp[k].to(DEV) for k in ("h", "ea", "na", "cot"))
    graph = CSRGraph(inp["ei"].to(DEV), hd.shape[0])
    g = GraphedEGCL(m, graph, hd, ead, nad)
    for scale in (1.0, -0.37):
        h1 = (hd * scale).requires_grad_()
        y = m(h1, graph, ead, nad)
        ge = torch.autograd.grad(y, [h1] + plist, cotd)
        h2 = (hd * scale).requires_grad_()
        yg = g(h2, ead, nad)
        gg = torch.autograd.grad(yg, [h2] + plist, cotd)
        assert torch.equal(y, yg)
        for a, b in zip(ge, gg):
            assert torch.equal(a, b)


def test_graphed_layer_step_matches_eager():
    """csmpn_b200.graphs.GraphedLayerStep: forward + backward + gradient pack as ONE graph over static tensors (what the host-fed
    leg of bench.py replays): new VALUES written into the static tensors and a new pair structure rebuilt in place give the
    output, grad_h and every parameter gradient of the eager step, bit for bit."""
    from csmpn_b200.graphs import GraphedLayerStep
    from csmpn_b200.models.ops import CSRGraph

    _, M = mods()
    name, metric, C, T, ncx, n, e, aggr = CASES[0]
    m, inp = _layer(CASES[0])
    h, ei, na, cot = (inp[k] for k in ("h", "ei", "na", "cot"))
    plist = list(m.parameters())
    h_s, na_s, cot_s = h.to(DEV).clone(), na.to(DEV).clone(), cot.to(DEV).clone()
    g = GraphedLayerStep(m, ei.to(DEV), h_s, na_s, cot_s)
    ei2 = block_diag_graph(ncx, n, e, torch.Generator().manual_seed(99))
    for scale, pairs in ((1.0, ei), (-0.41, ei), (0.7, ei2)):
        h_s.copy_(h.to(DEV) * scale)          # the feeder writes new values into the static tensors
        g.set_graph(pairs.to(DEV))
        y, gh, flat = g()
        h1 = (h.to(DEV) * scale).requires_grad_()
        ye = m(h1, CSRGraph(pairs.to(DEV), h.shape[0]), M.PairedNodeAttr(na.to(DEV)), na.to(DEV))
        ge = torch.autograd.grad(ye, [h1] + plist, cot.to(DEV))
        assert torch.equal(y, ye) and torch.equal(gh, ge[0])
        assert torch.equal(flat, torch.cat([t.reshape(-1) for t in ge[1:]]))


def test_graphed_layer_new_structure_same_shape():
    """GraphedEGCL.set_graph: a different complex structure with the same counts is rebuilt in place (CSR + sorted views)
    and the replayed graphs follow it."""
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    name, metric, C, T, ncx, n, e, aggr = CASES[0]
    m, inp = _layer(CASES[0])
    na = inp["na"]
    plist = list(m.parameters())
    hd, nad, cotd = (inp[k].to(DEV) for k in ("h", "na", "cot"))
    g = GraphedEGCL(m, inp["ei"].to(DEV), hd, inp["ea"].to(DEV), nad)
    ei2 = block_diag_graph(ncx, n, e, torch.Generator().manual_seed(4242))
    ea2 = torch.cat([na[ei2[0]], na[ei2[1]]], 1).to(DEV)
    h1 = hd.clone().requires_grad_()
    y = m(h1, CSRGraph(ei2.to(DEV), hd.shape[0]), ea2, nad)
    ge = torch.autograd.grad(y, [h1] + plist, cotd)
    g.set_graph(ei2.to(DEV))
    h2 = hd.clone().requires_grad_()
    yg = g(h2, ea2, nad)
    gg = torch.autograd.grad(yg, [h2] + plist, cotd)
    assert torch.equal(y, yg)
    for a, b in zip(ge, gg):
        assert torch.equal(a, b)


def test_forked_backward_is_bitwise_the_sequential_one(monkeypatch):
    """The side-stream fork of the weight-gradient kernels (fused._tc_backward_forked) only reorders launches: every
    gradient equals the single-stream backward bit for bit."""
    m, inp = _layer(CASES[1])
    out = []
    for fork in ("0", "1"):
        monkeypatch.setenv("CSMPN_TC_FORK", fork)
        out.append(run_egcl(m, inp, ("h",), "tensor"))
    assert_all_equal(out[1], out[0], "forked vs sequential")


def test_host_feeder_round_trip():
    """pipeline.HostFeeder: double-buffered pinned H2D / D2H delivers every step's tensors intact, in order"""
    from csmpn_b200.pipeline import HostFeeder

    feeder = HostFeeder(torch.device(DEV))
    steps = 5
    host = [{"a": torch.full((1 << 16,), float(i)).pin_memory(), "b": torch.arange(1024, dtype=torch.int64).add(i).pin_memory()}
            for i in range(steps)]
    outs = [torch.empty(1 << 16).pin_memory() for _ in range(steps)]
    feeder.submit(host[0])
    for i in range(steps):
        dv = feeder.next()
        if i + 1 < steps:
            feeder.submit(host[i + 1])
        y = dv["a"] * 2 + dv["b"][:1].float()
        feeder.drain(y, outs[i])
        feeder.release(dv)
    feeder.join()
    torch.cuda.synchronize()
    for i in range(steps):
        assert torch.equal(outs[i], torch.full((1 << 16,), 2.0 * i + i))


@pytest.mark.parametrize("engine", ["tc", "simt"])
@pytest.mark.parametrize("case", [CASES[0], CASES[2], CASES[3]], ids=["motion", "nba", "odd_c"])
def test_paired_node_attr_equals_materialised_edge_attr(case, engine, monkeypatch):
    """edge_attr = PairedNodeAttr(node_attr) (the kernel gathers node_attr[src] | node_attr[dst] itself) gives the layer
    output of the materialised torch.cat((node_attr[ei[0]], node_attr[ei[1]]), 1) of the reference models
    (md17_cssmpnn.py:131) bit for bit, and the same gradients -- node_attr's includes the part that flowed through
    edge_attr -- on both engines and against the CPU oracle."""
    name = case[0]
    monkeypatch.setenv("CSMPN_TC", "1" if engine == "tc" else "0")
    m, inp = _layer(case)
    ref = oracle_egcl(inp, torch.float32, PAIRED, "paired")
    paired = run_egcl(m, inp, PAIRED, "paired")
    # materialised on the device from the node_attr leaf, so its gradient takes the edge_attr part too
    hd, nad, eid = inp["h"].to(DEV).requires_grad_(), inp["na"].to(DEV).requires_grad_(), inp["ei"].to(DEV)
    y = m(hd, eid, torch.cat([nad[eid[0]], nad[eid[1]]], 1), nad)
    pd = dict(m.named_parameters())
    g = torch.autograd.grad(y, [hd, nad] + [pd[k] for k in inp["params"]], inp["cot"].to(DEV))
    materialised = (y, dict(zip(list(PAIRED) + list(inp["params"]), g)))
    assert torch.equal(paired[0], materialised[0])
    assert_all_close(paired, materialised, 1e-5, 1e-5, f"{name} paired vs materialised:")
    assert_all_close(paired, ref, 1e-5, 1e-4, f"{name} paired vs oracle:")


def test_graphed_layer_with_paired_node_attr():
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    _, M = mods()
    m, inp = _layer(CASES[1])
    plist = list(m.parameters())
    hd, nad, cotd = inp["h"].to(DEV), inp["na"].to(DEV).requires_grad_(), inp["cot"].to(DEV)
    graph = CSRGraph(inp["ei"].to(DEV), hd.shape[0])
    g = GraphedEGCL(m, graph, hd, M.PairedNodeAttr(nad), nad)
    h1 = hd.clone().requires_grad_()
    y = m(h1, graph, M.PairedNodeAttr(nad), nad)
    ge = torch.autograd.grad(y, [h1, nad] + plist, cotd)
    h2 = hd.clone().requires_grad_()
    yg = g(h2, None, nad)
    gg = torch.autograd.grad(yg, [h2, nad] + plist, cotd)
    assert torch.equal(y, yg)
    for a, b in zip(ge, gg):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# wide blocks: weights streamed with the K chunks (csmpn_block_tc_plan bits 1-3), hidden widths 64 / 128 / 256
def test_wide_plans():
    from csmpn_b200 import _lib

    plan = _lib.lib().csmpn_block_tc_plan
    assert plan(3, 38, 32) == 1 and plan(2, 46, 40) == 1          # resident weights
    for c in (64, 128, 256):
        assert plan(3, c + 6, c) == 0b1111 and plan(3, 2 * c + 3, c) == 0b1111 and plan(3, c, c) == 0b1111
    assert plan(2, 134, 128) == 0b1111
    assert plan(5, 28, 28) == 0 and plan(3, 102, 96) == 0         # Cl(5,0) and non-slab widths stay off the engine


@pytest.mark.parametrize("case", WIDE, ids=[c[0] for c in WIDE])
def test_wide_block_forward_backward_vs_oracle(case):
    """EGCL at hidden widths 64 / 128 / 256 on the tensor-core engine (streamed weights, channel passes, slab-wise
    weight-gradient launches): forward and every gradient against the CPU oracle"""
    from csmpn_b200 import _lib
    from csmpn_b200.models import fused

    _, M = mods()
    m, inp = _layer(case)
    ref = oracle_egcl(inp, torch.float32, PAIRED, "paired")
    assert all(fused._block_uses_tc(m.algebra, b, True, 1) for b in list(m.edge_model.layers) + list(m.node_model.layers))
    n0 = _lib.lib().csmpn_launch_count()
    got = run_egcl(m, inp, PAIRED, "paired")
    assert _lib.lib().csmpn_launch_count() - n0 > 40
    assert_all_close(got, ref, 1e-5, 1e-4, case[0])
    with torch.no_grad():   # inference path: no saved tensors, the product sum goes through a scratch tensor
        na = inp["na"].to(DEV)
        y2 = m(inp["h"].to(DEV), inp["ei"].to(DEV), M.PairedNodeAttr(na), na)
    assert torch.equal(y2, got[0])


@pytest.mark.parametrize("case", [CASES[0], CASES[1], CASES[2], CASES[3], CASES[4]], ids=["motion", "md17", "nba", "odd_c", "tiny"])
def test_overlapped_epilogue_kernels_match_plain_kernels(case, monkeypatch):
    """tc_f1db / tc_bgemmdb (two TMEM accumulator buffers, epilogue of tile t-1 interleaved with the K loop of tile t) against
    the plain kernels (CSMPN_TC_OVERLAP=0): same arithmetic, so the layer output and every gradient are bit-identical"""
    m, inp = _layer(case)
    out = {}
    for ov in ("1", "0"):
        monkeypatch.setenv("CSMPN_TC_OVERLAP", ov)
        out[ov] = run_egcl(m, inp, ("h",), "tensor")
    assert_all_equal(out["1"], out["0"], f"{case[0]} overlapped vs plain:")
