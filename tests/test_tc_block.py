"""GPU parity of the tensor-core (tcgen05, 3xTF32) CEMLP-block engine: against the CPU oracle (fp32 tolerance of the
north star: forward rel 1e-5, gradients rel 1e-4) and against the FP32 SIMT engine on the same inputs."""
import pytest
import torch

from conftest import assert_close, rel_err
from oracle import layers_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(autouse=True)
def _force_tc_for_small_batches(monkeypatch):
    """the default policy keeps blocks with few rows on the SIMT engine; the parity cases here are small on purpose"""
    monkeypatch.setenv("CSMPN_TC_MIN_ROWS", "0")

CASES = [
    # name, metric, C, T, complexes, simplices/complex, pairs/complex, aggr
    ("motion", (1, 1, 1), 28, 3, 6, 47, 226, "mean"),
    ("md17", (1, 1, 1), 32, 3, 4, 87, 527, "sum"),
    ("nba", (1, 1), 40, 3, 6, 41, 345, "sum"),
    ("odd_c", (1, 1, 1), 30, 2, 3, 19, 77, "mean"),
    ("tiny", (1, 1, 1), 8, 3, 1, 5, 3, "sum"),
    ("one_tile_exact", (1, 1, 1), 16, 3, 1, 128, 256, "mean"),
]


def _mods():
    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.models import cegnn_utils as M

    return CliffordAlgebra, M


def _load(module, params):
    missing, unexpected = module.load_state_dict({k: v for k, v in params.items()}, strict=False)
    assert not unexpected and all("algebra" in m for m in missing), (missing, unexpected)


def _graph(n_cplx, n, e, gen):
    src = torch.randint(0, n, (n_cplx, e), generator=gen)
    dst = torch.randint(0, n, (n_cplx, e), generator=gen)
    off = (torch.arange(n_cplx) * n).unsqueeze(1)
    return torch.stack([(src + off).reshape(-1), (dst + off).reshape(-1)])


def _inputs(case):
    name, metric, C, T, ncx, n, e, aggr = case
    gen = torch.Generator().manual_seed(sum(map(ord, name)))
    ralg = R.RefAlgebra(metric)
    B = ralg.B
    params = R.init_egcl_params(ralg, C, T, gen)
    N = ncx * n
    h = torch.randn(N, C, B, generator=gen)
    ei = _graph(ncx, n, e, gen)
    na = torch.zeros(N, T, B)
    na[..., 0] = torch.randn(T, T, generator=gen)[torch.randint(0, T, (N,), generator=gen)]
    ea = torch.cat([na[ei[0]], na[ei[1]]], 1)
    cot = torch.randn(N, C, B, generator=gen)
    return ralg, params, h, ei, ea, na, cot


def test_tc_engine_is_selected():
    from csmpn_b200.models import fused

    assert fused.tc_supported(3, 38, 32) and fused.tc_supported(3, 67, 32) and fused.tc_supported(2, 46, 40)
    assert not fused.tc_supported(5, 28, 28)  # Cl(5,0): 32 blades do not fit the TMEM accumulator budget
    assert fused.tc_supported(3, 64, 64)  # wide block: streamed weights


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tc_forward_vs_oracle(case, monkeypatch):
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, _ = _inputs(case)
    yr = R.egcl(ralg, h, ei, ea, na, params, aggr=aggr)
    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    from csmpn_b200 import _lib

    outs = {}
    for tc in ("1", "0"):
        monkeypatch.setenv("CSMPN_TC", tc)
        n0 = _lib.lib().csmpn_launch_count()
        with torch.no_grad():
            outs[tc] = m(h.to(DEV), ei.to(DEV), ea.to(DEV), na.to(DEV)).cpu()
        outs["launches" + tc] = _lib.lib().csmpn_launch_count() - n0
    # the tensor-core engine launches two kernels per block (8 per layer) where the SIMT engine launches one
    assert outs["launches1"] == outs["launches0"] + 4, (outs["launches1"], outs["launches0"])
    assert_close(outs["1"], yr, 1e-5, f"{name} tensor-core fwd vs oracle")
    assert_close(outs["1"], outs["0"], 1e-5, f"{name} tensor-core fwd vs SIMT engine")


def test_tc_cemlp_dense_rows(monkeypatch):
    """CEMLP on plain rows (the models' embedding / projection MLPs): rows not a multiple of the 128-row tile."""
    CliffordAlgebra, M = _mods()
    gen = torch.Generator().manual_seed(5)
    ralg = R.RefAlgebra((1, 1, 1))
    alg = CliffordAlgebra((1, 1, 1)).to(DEV)
    for cin, c, rows in ((7, 32, 1000), (32, 32, 129), (3, 16, 1)):
        params = R.init_cemlp_params(ralg, cin, c, c, 2, gen)
        m = M.CEMLP(alg, cin, c, c, n_layers=2).to(DEV)
        _load(m, params)
        x = torch.randn(rows, cin, 8, generator=gen)
        yr = R.cemlp(ralg, x, params)
        monkeypatch.setenv("CSMPN_TC", "1")
        with torch.no_grad():
            y = m(x.to(DEV))
        assert_close(y, yr, 1e-5, f"cemlp {cin}->{c} rows={rows}")


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_tc_backward_vs_oracle(case, monkeypatch):
    """forward + every gradient of one EGCL layer on the tensor-core engine against the CPU oracle (autograd)."""
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, cot = _inputs(case)
    hr, ear, nar = h.clone().requires_grad_(), ea.clone().requires_grad_(), na.clone().requires_grad_()
    pr = {k: v.clone().requires_grad_() for k, v in params.items()}
    yr = R.egcl(ralg, hr, ei, ear, nar, pr, aggr=aggr)
    names = list(pr)
    gr = torch.autograd.grad(yr, [hr, ear, nar] + [pr[k] for k in names], cot)

    monkeypatch.setenv("CSMPN_TC", "1")
    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    hd, ead, nad = (t.to(DEV).requires_grad_() for t in (h, ea, na))
    from csmpn_b200 import _lib

    n0 = _lib.lib().csmpn_launch_count()
    y = m(hd, ei.to(DEV), ead, nad)
    pd = dict(m.named_parameters())
    got = torch.autograd.grad(y, [hd, ead, nad] + [pd[k] for k in names], cot.to(DEV))
    assert _lib.lib().csmpn_launch_count() - n0 > 30  # the tensor-core engine: 2 + 7 kernels per block
    assert_close(y, yr, 1e-5, f"{name} fwd")
    for what, a, b in zip(["gh", "gedge_attr", "gnode_attr"] + names, got, gr):
        assert_close(a, b, 1e-4, f"{name} {what}")


def test_graphed_layer_matches_eager():
    """CUDA-graph replay of a layer step (csmpn_b200.graphs.GraphedEGCL) reproduces the eager step bit for bit, for new
    input VALUES on the same complex structure."""
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    case = CASES[1]
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, cot = _inputs(case)
    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    plist = list(m.parameters())
    hd, ead, nad, cotd = h.to(DEV), ea.to(DEV), na.to(DEV), cot.to(DEV)
    graph = CSRGraph(ei.to(DEV), h.shape[0])
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
    from csmpn_b200.models.cegnn_utils import PairedNodeAttr
    from csmpn_b200.models.ops import CSRGraph

    case = CASES[0]
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, cot = _inputs(case)
    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    plist = list(m.parameters())
    h_s, na_s, cot_s = h.to(DEV).clone(), na.to(DEV).clone(), cot.to(DEV).clone()
    g = GraphedLayerStep(m, ei.to(DEV), h_s, na_s, cot_s)
    ei2 = _graph(ncx, n, e, torch.Generator().manual_seed(99))
    for scale, pairs in ((1.0, ei), (-0.41, ei), (0.7, ei2)):
        h_s.copy_(h.to(DEV) * scale)          # the feeder writes new values into the static tensors
        g.set_graph(pairs.to(DEV))
        y, gh, flat = g()
        h1 = (h.to(DEV) * scale).requires_grad_()
        ye = m(h1, CSRGraph(pairs.to(DEV), h.shape[0]), PairedNodeAttr(na.to(DEV)), na.to(DEV))
        ge = torch.autograd.grad(ye, [h1] + plist, cot.to(DEV))
        assert torch.equal(y, ye) and torch.equal(gh, ge[0])
        assert torch.equal(flat, torch.cat([t.reshape(-1) for t in ge[1:]]))


def test_graphed_layer_new_structure_same_shape():
    """GraphedEGCL.set_graph: a different complex structure with the same counts is rebuilt in place (CSR + sorted views)
    and the replayed graphs follow it."""
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    case = CASES[0]
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, cot = _inputs(case)
    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    plist = list(m.parameters())
    hd, nad, cotd = h.to(DEV), na.to(DEV), cot.to(DEV)
    g = GraphedEGCL(m, ei.to(DEV), hd, ea.to(DEV), nad)
    ei2 = _graph(ncx, n, e, torch.Generator().manual_seed(4242))
    ea2 = torch.cat([na[ei2[0]], na[ei2[1]]], 1).to(DEV)
    h1 = hd.clone().requires_grad_()
    y = m(h1, CSRGraph(ei2.to(DEV), h.shape[0]), ea2, nad)
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
    case = CASES[1]
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, cot = _inputs(case)
    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    plist = list(m.parameters())
    out = []
    for fork in ("0", "1"):
        monkeypatch.setenv("CSMPN_TC_FORK", fork)
        hd = h.to(DEV).requires_grad_()
        y = m(hd, ei.to(DEV), ea.to(DEV), na.to(DEV))
        out.append(torch.autograd.grad(y, [hd] + plist, cot.to(DEV)))
        torch.cuda.synchronize()
    for a, b in zip(*out):
        assert torch.equal(a, b)


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
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    monkeypatch.setenv("CSMPN_TC", "1" if engine == "tc" else "0")
    ralg, params, h, ei, _, na, cot = _inputs(case)
    hr, nar = h.clone().requires_grad_(), na.clone().requires_grad_()
    pr = {k: v.clone().requires_grad_() for k, v in params.items()}
    yr = R.egcl(ralg, hr, ei, torch.cat([nar[ei[0]], nar[ei[1]]], 1), nar, pr, aggr=aggr)
    names = list(pr)
    gr = torch.autograd.grad(yr, [hr, nar] + [pr[k] for k in names], cot)

    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    pd = dict(m.named_parameters())
    eid = ei.to(DEV)
    out = {}
    for mode in ("paired", "materialised"):
        hd, nad = h.to(DEV).requires_grad_(), na.to(DEV).requires_grad_()
        ea = M.PairedNodeAttr(nad) if mode == "paired" else torch.cat([nad[eid[0]], nad[eid[1]]], 1)
        y = m(hd, eid, ea, nad)
        out[mode] = (y, torch.autograd.grad(y, [hd, nad] + [pd[k] for k in names], cot.to(DEV)))
    assert torch.equal(out["paired"][0], out["materialised"][0])
    assert_close(out["paired"][0], yr, 1e-5, f"{name} fwd")
    for what, a, b, c in zip(["gh", "gnode_attr"] + names, out["paired"][1], out["materialised"][1], gr):
        assert_close(a, b, 1e-5, f"{name} {what} paired vs materialised")
        assert_close(a, c, 1e-4, f"{name} {what} paired vs oracle")


def test_graphed_layer_with_paired_node_attr():
    from csmpn_b200.graphs import GraphedEGCL
    from csmpn_b200.models.ops import CSRGraph

    case = CASES[1]
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, cot = _inputs(case)
    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    plist = list(m.parameters())
    hd, nad, cotd = h.to(DEV), na.to(DEV).requires_grad_(), cot.to(DEV)
    graph = CSRGraph(ei.to(DEV), h.shape[0])
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
WIDE = [
    # name, metric, C, T, complexes, simplices/complex, pairs/complex, aggr
    ("cl3_c64", (1, 1, 1), 64, 3, 4, 87, 527, "sum"),
    ("cl3_c128", (1, 1, 1), 128, 3, 2, 87, 527, "mean"),
    ("cl3_c256", (1, 1, 1), 256, 3, 1, 60, 300, "sum"),
    ("cl2_c128", (1, 1), 128, 3, 3, 41, 345, "sum"),
    ("cl2_c64", (1, 1), 64, 3, 3, 41, 345, "mean"),
    ("cl3_c64_multi_tile", (1, 1, 1), 64, 3, 40, 87, 527, "sum"),   # 165 tiles of pairs: two tiles on some CTAs
]


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
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, cot = _inputs(case)
    hr, nar = h.clone().requires_grad_(), na.clone().requires_grad_()
    pr = {k: v.clone().requires_grad_() for k, v in params.items()}
    yr = R.egcl(ralg, hr, ei, torch.cat([nar[ei[0]], nar[ei[1]]], 1), nar, pr, aggr=aggr)
    names = list(pr)
    gr = torch.autograd.grad(yr, [hr, nar] + [pr[k] for k in names], cot)

    from csmpn_b200 import _lib
    from csmpn_b200.models import fused

    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    assert all(fused._block_uses_tc(alg, b, True, 1) for b in list(m.edge_model.layers) + list(m.node_model.layers))
    hd, nad = h.to(DEV).requires_grad_(), na.to(DEV).requires_grad_()
    n0 = _lib.lib().csmpn_launch_count()
    y = m(hd, ei.to(DEV), M.PairedNodeAttr(nad), nad)
    pd = dict(m.named_parameters())
    got = torch.autograd.grad(y, [hd, nad] + [pd[k] for k in names], cot.to(DEV))
    assert _lib.lib().csmpn_launch_count() - n0 > 40
    assert_close(y, yr, 1e-5, f"{name} fwd")
    for what, a, b in zip(["gh", "gnode_attr"] + names, got, gr):
        assert_close(a, b, 1e-4, f"{name} {what}")
    with torch.no_grad():   # inference path: no saved tensors, the product sum goes through a scratch tensor
        y2 = m(h.to(DEV), ei.to(DEV), M.PairedNodeAttr(na.to(DEV)), na.to(DEV))
    assert torch.equal(y2, y.detach())


@pytest.mark.parametrize("case", [CASES[0], CASES[1], CASES[2], CASES[3], CASES[4]], ids=["motion", "md17", "nba", "odd_c", "tiny"])
def test_overlapped_epilogue_kernels_match_plain_kernels(case, monkeypatch):
    """tc_f1db / tc_bgemmdb (two TMEM accumulator buffers, epilogue of tile t-1 interleaved with the K loop of tile t) against
    the plain kernels (CSMPN_TC_OVERLAP=0): same arithmetic, so the layer output and every gradient are bit-identical"""
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    ralg, params, h, ei, ea, na, cot = _inputs(case)
    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    names = [k for k, _ in m.named_parameters()]
    plist = [p for _, p in m.named_parameters()]
    out = {}
    for ov in ("1", "0"):
        monkeypatch.setenv("CSMPN_TC_OVERLAP", ov)
        hd = h.to(DEV).requires_grad_()
        y = m(hd, ei.to(DEV), ea.to(DEV), na.to(DEV))
        out[ov] = (y.detach().clone(), torch.autograd.grad(y, [hd] + plist, cot.to(DEV)))
        torch.cuda.synchronize()
    assert torch.equal(out["1"][0], out["0"][0])
    for what, a, b in zip(["gh"] + names, out["1"][1], out["0"][1]):
        assert torch.equal(a, b), f"{name} {what} overlapped vs plain"
