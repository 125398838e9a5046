"""GPU parity: the product layers (C ABI -> sm_100a kernels) against (a) the golden vectors the reference produced
and (b) the CPU oracle on larger seeded inputs.  Tolerances: forward rel 1e-5, gradients rel 1e-4 (fp32)."""
import math

import pytest
import torch

from conftest import LAYER_FIXTURES, assert_close, load_golden, tols
from oracle import layers_ref as R

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(params=["fused", "unit"])
def path(request, monkeypatch):
    """run the CEMLP / EGCL tests through both the fused block kernels and the unit-kernel composition"""
    monkeypatch.setenv("CSMPN_FUSED", "1" if request.param == "fused" else "0")
    return request.param


def _mods():
    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.models import cegnn_utils as M

    return CliffordAlgebra, M


def _load(module, params):
    missing, unexpected = module.load_state_dict({k: v for k, v in params.items()}, strict=False)
    assert not unexpected, unexpected
    assert all("algebra" in m for m in missing), missing


def _grads(out, cot, tensors):
    return torch.autograd.grad(out, tensors, cot.to(out.device), allow_unused=True)


@pytest.fixture(scope="module", params=LAYER_FIXTURES)
def fx(request):
    f = load_golden(request.param)
    CliffordAlgebra, _ = _mods()
    f["alg"] = CliffordAlgebra(f["metric"]).to(DEV)
    f["ralg"] = R.RefAlgebra(f["metric"])
    return f


def test_native_library_loaded():
    from csmpn_b200 import _lib

    _lib.lib()
    maps = open("/proc/self/maps").read()
    assert "libcsmpn_b200.so" in maps


def test_tables_match_reference(fx):
    alg = fx["alg"]
    assert torch.equal(alg.cayley.cpu(), fx["cayley"])
    assert torch.equal(alg.subspaces.cpu(), fx["subspaces"])
    assert torch.equal(alg.bbo_grades.cpu(), fx["bbo_grades"])
    assert torch.equal(alg.geometric_product_paths, fx["paths"])


def test_geometric_product(fx):
    FWD, GRAD = tols(fx)
    alg, g = fx["alg"], fx["gp"]
    a, b = g["a"].to(DEV).requires_grad_(), g["b"].to(DEV).requires_grad_()
    out = alg.geometric_product(a, b)
    assert_close(out, g["out"], FWD, "gp")
    ga, gb = _grads(out, g["cot"], [a, b])
    assert_close(ga, g["ga"], GRAD, "ga")
    assert_close(gb, g["gb"], GRAD, "gb")
    # forms
    assert_close(torch.cat(alg.qs(g["a"].to(DEV)), -1), fx["qs"], FWD, "qs")
    assert_close(torch.cat(alg.norms(g["a"].to(DEV)), -1), fx["norms"], FWD, "norms")
    assert_close(alg.norm(g["a"].to(DEV)), fx["norm_all"], FWD, "norm")


def test_geometric_product_broadcast_and_blades(fx):
    FWD, GRAD = tols(fx)
    alg, ralg = fx["alg"], fx["ralg"]
    gen = torch.Generator().manual_seed(5)
    a = torch.randn(1, ralg.B, generator=gen)
    b = torch.randn(37, ralg.B, generator=gen)
    ad, bd = a.to(DEV).requires_grad_(), b.to(DEV).requires_grad_()
    out = alg.geometric_product(ad, bd)
    ar, br = a.clone().requires_grad_(), b.clone().requires_grad_()
    ref = R.geometric_product(ralg, ar, br)
    assert_close(out, ref, FWD, "bcast gp")
    cot = torch.randn(37, ralg.B, generator=gen)
    ga, gb = _grads(out, cot, [ad, bd])
    gar, gbr = torch.autograd.grad(ref, [ar, br], cot)
    assert_close(ga, gar, GRAD, "bcast ga")
    assert_close(gb, gbr, GRAD, "bcast gb")


@pytest.mark.parametrize("sub", [1, 0])
def test_mvlinear(fx, sub):
    FWD, GRAD = tols(fx)
    _, M = _mods()
    alg, g = fx["alg"], fx[f"mvlinear_{sub}"]
    m = M.MVLinear(alg, g["x"].shape[1], g["y"].shape[1], subspaces=bool(sub)).to(DEV)
    with torch.no_grad():
        m.weight.copy_(g["weight"])
        m.bias.copy_(g["bias"])
    x = g["x"].to(DEV).requires_grad_()
    y = m(x)
    assert_close(y, g["y"], FWD, "mvlinear")
    gx, gw, gb = _grads(y, g["cot"], [x, m.weight, m.bias])
    assert_close(gx, g["gx"], GRAD, "gx")
    assert_close(gw, g["gw"], GRAD, "gw")
    assert_close(gb, g["gb"], GRAD, "gb")


def test_mvsilu(fx):
    FWD, GRAD = tols(fx)
    _, M = _mods()
    alg, g = fx["alg"], fx["mvsilu"]
    m = M.MVSiLU(alg, g["x"].shape[1]).to(DEV)
    with torch.no_grad():
        m.a.copy_(g["a"]); m.b.copy_(g["b"])
    x = g["x"].to(DEV).requires_grad_()
    y = m(x)
    assert_close(y, g["y"], FWD, "mvsilu")
    for got, key in zip(_grads(y, g["cot"], [x, m.a, m.b]), ("gx", "ga", "gb")):
        assert_close(got, g[key], GRAD, key)


def test_mvnorm(fx):
    FWD, GRAD = tols(fx)
    _, M = _mods()
    alg, g = fx["alg"], fx["mvnorm"]
    m = M.NormalizationLayer(alg, g["x"].shape[1]).to(DEV)
    with torch.no_grad():
        m.a.copy_(g["a"])
    x = g["x"].to(DEV).requires_grad_()
    y = m(x)
    assert_close(y, g["y"], FWD, "mvnorm")
    for got, key in zip(_grads(y, g["cot"], [x, m.a]), ("gx", "ga")):
        assert_close(got, g[key], GRAD, key)


def test_mvlayernorm(fx):
    FWD, GRAD = tols(fx)
    _, M = _mods()
    alg, g = fx["alg"], fx["mvlayernorm"]
    m = M.MVLayerNorm(alg, g["x"].shape[1]).to(DEV)
    with torch.no_grad():
        m.a.copy_(g["a"])
    x = g["x"].to(DEV).requires_grad_()
    y = m(x)
    assert_close(y, g["y"], FWD, "mvlayernorm")
    for got, key in zip(_grads(y, g["cot"], [x, m.a]), ("gx", "ga")):
        assert_close(got, g[key], GRAD, key)


def test_sgp(fx):
    FWD, GRAD = tols(fx)
    _, M = _mods()
    alg, g = fx["alg"], fx["sgp"]
    m = M.SteerableGeometricProductLayer(alg, g["x"].shape[1]).to(DEV)
    _load(m, g["params"])
    x = g["x"].to(DEV).requires_grad_()
    y = m(x)
    assert_close(y, g["y"], FWD, "sgp")
    plist = list(m.named_parameters())
    got = _grads(y, g["cot"], [x] + [p for _, p in plist])
    assert_close(got[0], g["gx"], GRAD, "gx")
    for (n, _), gi in zip(plist, got[1:]):
        assert_close(gi, g["grads"][n], GRAD, n)


def test_cemlp(fx, path):
    FWD, GRAD = tols(fx)
    _, M = _mods()
    alg, g = fx["alg"], fx["cemlp"]
    C = g["y"].shape[1]
    m = M.CEMLP(alg, g["x"].shape[1], C, C, n_layers=2).to(DEV)
    _load(m, g["params"])
    x = g["x"].to(DEV).requires_grad_()
    y = m(x)
    assert_close(y, g["y"], FWD, "cemlp")
    plist = list(m.named_parameters())
    got = _grads(y, g["cot"], [x] + [p for _, p in plist])
    assert_close(got[0], g["gx"], GRAD, "gx")
    for (n, _), gi in zip(plist, got[1:]):
        assert_close(gi, g["grads"][n], GRAD, n)


@pytest.mark.parametrize("aggr", ["sum", "mean"])
def test_egcl(fx, aggr, path):
    FWD, GRAD = tols(fx)
    _, M = _mods()
    alg, g = fx["alg"], fx[f"egcl_{aggr}"]
    C, T = g["h"].shape[1], g["node_attr"].shape[1]
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, g["params"])
    h, ea, na = (g[k].to(DEV).requires_grad_() for k in ("h", "edge_attr", "node_attr"))
    y = m(h, g["edge_index"].to(DEV), ea, na)
    assert_close(y, g["y"], FWD, "egcl")
    plist = list(m.named_parameters())
    got = _grads(y, g["cot"], [h, ea, na] + [p for _, p in plist])
    assert_close(got[0], g["gh"], GRAD, "gh")
    assert_close(got[1], g["gedge_attr"], GRAD, "gedge_attr")
    assert_close(got[2], g["gnode_attr"], GRAD, "gnode_attr")
    for (n, _), gi in zip(plist, got[3:]):
        assert_close(gi, g["grads"][n], GRAD, n)


# ------------------------------------------------------------------------------------------------
# larger seeded cases against the oracle: the BASELINE layer shapes (scaled-down batch so the CPU oracle stays fast)
CASES = [
    # name, metric, C, T, complexes, simplices/complex, pairs/complex, aggr
    ("motion", (1, 1, 1), 28, 3, 6, 47, 226, "mean"),
    ("md17", (1, 1, 1), 32, 3, 4, 87, 527, "sum"),
    ("nba", (1, 1), 40, 3, 6, 41, 345, "sum"),
    ("hulls", (1, 1, 1, 1, 1), 28, 3, 2, 30, 200, "mean"),
    ("odd_c", (1, 1, 1), 30, 2, 3, 19, 77, "mean"),
]


def _block_diag_graph(n_cplx, n, e, gen):
    src = torch.randint(0, n, (n_cplx, e), generator=gen)
    dst = torch.randint(0, n, (n_cplx, e), generator=gen)
    off = (torch.arange(n_cplx) * n).unsqueeze(1)
    return torch.stack([(src + off).reshape(-1), (dst + off).reshape(-1)])


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_egcl_vs_oracle(case, path):
    name, metric, C, T, ncx, n, e, aggr = case
    CliffordAlgebra, M = _mods()
    gen = torch.Generator().manual_seed(hash(name) % 1000)
    ralg = R.RefAlgebra(metric)
    B = ralg.B
    params = R.init_egcl_params(ralg, C, T, gen)
    N = ncx * n
    h = torch.randn(N, C, B, generator=gen)
    ei = _block_diag_graph(ncx, n, e, gen)
    types = torch.randint(0, T, (N,), generator=gen)
    emb = torch.randn(T, T, generator=gen)
    na = torch.zeros(N, T, B)
    na[..., 0] = emb[types]
    ea = torch.cat([na[ei[0]], na[ei[1]]], 1)
    cot = torch.randn(N, C, B, generator=gen)

    hr = h.clone().requires_grad_()
    pr = {k: v.clone().requires_grad_() for k, v in params.items()}
    yr = R.egcl(ralg, hr, ei, ea, na, pr, aggr=aggr)
    names = list(pr)
    gr = torch.autograd.grad(yr, [hr] + [pr[k] for k in names], cot)

    alg = CliffordAlgebra(metric).to(DEV)
    m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
    _load(m, params)
    hd = h.to(DEV).requires_grad_()
    y = m(hd, ei.to(DEV), ea.to(DEV), na.to(DEV))
    assert_close(y, yr, 1e-5, f"{name} fwd")
    pd = dict(m.named_parameters())
    got = _grads(y, cot, [hd] + [pd[k] for k in names])
    assert_close(got[0], gr[0], 1e-4, f"{name} gh")
    for k, a, b in zip(names, got[1:], gr[1:]):
        assert_close(a, b, 1e-4, f"{name} {k}")


def test_egcl_empty_and_ragged(path):
    """no pairs at all; a receiver with hundreds of pairs; N not a multiple of any tile."""
    CliffordAlgebra, M = _mods()
    gen = torch.Generator().manual_seed(9)
    ralg = R.RefAlgebra((1, 1, 1))
    C, T, N = 8, 3, 13
    params = R.init_egcl_params(ralg, C, T, gen)
    alg = CliffordAlgebra((1, 1, 1)).to(DEV)
    for aggr in ("sum", "mean"):
        m = M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV)
        _load(m, params)
        for ei in (torch.zeros(2, 0, dtype=torch.long),
                   torch.stack([torch.randint(0, N, (300,), generator=gen), torch.full((300,), 5)])):
            h = torch.randn(N, C, 8, generator=gen)
            na = torch.zeros(N, T, 8); na[..., 0] = torch.randn(N, T, generator=gen)
            ea = torch.cat([na[ei[0]], na[ei[1]]], 1)
            yr = R.egcl(ralg, h, ei, ea, na, params, aggr=aggr)
            y = m(h.to(DEV), ei.to(DEV), ea.to(DEV), na.to(DEV))
            assert_close(y, yr, 1e-5, f"ragged {aggr} E={ei.shape[1]}")


@pytest.mark.parametrize("small", ["1", "0"])
def test_csr_is_stable_sort(small, monkeypatch):
    """both builders -- the single-launch two-CTA kernel (csmpn_csr_build_pair) and the multi-launch path -- give the stable
    counting sort: rowptr = exclusive counts, perm = argsort(key, stable); the sorted views and the inverse permutation
    follow the receiver order; rebuild_ in place gives the same for new pairs."""
    from csmpn_b200.models import fused
    from csmpn_b200.models.ops import CSRGraph

    monkeypatch.setenv("CSMPN_CSR_SMALL", small)
    gen = torch.Generator().manual_seed(2)

    def verify(g, ei, N, E):
        for key, rowptr, perm in ((ei[1], g.rowptr_dst, g.perm_dst), (ei[0], g.rowptr_src, g.perm_src)):
            order = torch.argsort(key, stable=True)
            counts = torch.bincount(key, minlength=N)
            ref_ptr = torch.cat([torch.zeros(1, dtype=torch.long), counts.cumsum(0)])
            assert torch.equal(rowptr.cpu().long(), ref_ptr)
            assert torch.equal(perm.cpu().long()[:E], order)
        if E:
            sg = fused.sorted_graph(g)
            order = torch.argsort(ei[1], stable=True)
            assert torch.equal(sg.src_sorted.cpu().long()[:E], ei[0][order])
            assert torch.equal(sg.dst_sorted.cpu().long()[:E], ei[1][order])
            assert torch.equal(sg.rank.cpu().long()[:E][order], torch.arange(E))

    for N, E in ((1, 0), (7, 1), (50, 1000), (5000, 30000), (3, 5000), (1031, 4097), (40000, 100000), (60000, 90000)):
        ei = torch.randint(0, N, (2, E), generator=gen)
        g = CSRGraph(ei.to(DEV), N)
        verify(g, ei, N, E)
        if E:
            ei2 = torch.randint(0, N, (2, E), generator=gen)
            g.rebuild_(ei2.to(DEV))   # first call builds eagerly and captures, second call replays the captured rebuild
            verify(g, ei2, N, E)
            ei3 = torch.randint(0, N, (2, E), generator=gen)
            g.rebuild_(ei3.to(DEV))
            verify(g, ei3, N, E)


def test_equivariance_with_correct_inverse():
    """f(rho_w(x)) = rho_w(f(x)) for a random rotor, using w^-1 = beta(w)/q(w) (the reference's ``inverse`` is not
    norm-preserving, SURVEY.md appendix B)."""
    CliffordAlgebra, M = _mods()
    gen = torch.Generator().manual_seed(4)
    ralg = R.RefAlgebra((1, 1, 1))
    alg = CliffordAlgebra((1, 1, 1)).to(DEV)
    C = 8
    m = M.CEMLP(alg, C, C, C, n_layers=2).to(DEV)
    _load(m, R.init_cemlp_params(ralg, C, C, C, 2, gen))
    v1, v2 = torch.zeros(8), torch.zeros(8)
    v1[1:4] = torch.randn(3, generator=gen); v2[1:4] = torch.randn(3, generator=gen)
    w = R.geometric_product(ralg, v1, v2)
    beta = torch.tensor([(-1.0) ** (g * (g - 1) // 2) for g in ralg.grade])
    w_inv = beta * w / R.geometric_product(ralg, w, beta * w)[0]

    def rho(x):
        wd, wi = w.to(x.device), w_inv.to(x.device)
        return alg.geometric_product(alg.geometric_product(wd.expand_as(x).contiguous(), x), wi.expand_as(x).contiguous())

    x = torch.randn(33, C, 8, generator=gen).to(DEV)
    a = m(rho(x))
    b = rho(m(x))
    assert_close(a, b, 2e-5, "equivariance")


def test_versor_utilities_match_the_reference():
    """the off-path helpers of CliffordAlgebra (alpha_w, inverse, rho, sandwich, output_blades, parity, eta,
    reduce_geometric_product, random_vector / versor shapes) against the reference's definitions on the same inputs
    (tests/golden/versor.pt, made by tests/golden/make_golden_versor.py)."""
    CliffordAlgebra, _ = _mods()
    gold = load_golden("versor.pt")
    for metric in ((1, 1), (1, 1, 1)):
        ref = gold[metric]
        alg = CliffordAlgebra(metric).to(DEV)
        Bn = 2 ** len(metric)
        mv, vec, rot = ref["mv"], ref["vec"], ref["rot"]   # rot: an even element, vec: an odd one
        for w, r in zip((vec, rot), ref["elements"]):
            assert bool(alg.parity(w.to(DEV))) == r["parity"] and int(alg.eta(w.to(DEV))) == r["eta"]
            assert_close(alg.alpha_w(w.to(DEV), mv.to(DEV)), r["alpha_w"], 1e-6, "alpha_w")
            assert_close(alg.inverse(w.to(DEV)), r["inverse"], 1e-5, "inverse")
            assert_close(alg.rho(w.to(DEV), mv.to(DEV)), r["rho"], 1e-5, "rho")
        assert_close(alg.sandwich(mv.to(DEV), vec.to(DEV), mv.to(DEV)), ref["sandwich"], 1e-5, "sandwich")
        with pytest.raises(ValueError):
            alg.parity((vec + rot).to(DEV))
        ob = ref["output_blades"]
        assert torch.equal(alg.output_blades(ob["left"], ob["right"]), ob["blades"])
        chain = ref["chain"]
        assert_close(alg.reduce_geometric_product([c.to(DEV) for c in chain]), ref["reduce_geometric_product"], 1e-5, "reduce")
        rv = alg.random_vector(4)
        assert rv.shape == (4, Bn) and bool((rv[:, alg.bbo_grades.to(rv.device) != 1] == 0).all())
        v = alg.versor()
        assert v.shape == (1, Bn) and abs(float(alg.norm(v)[..., 0]) - 1.0) < 1e-5
        assert alg.rotor().shape == (1, Bn) and alg.random(3).shape == (3, Bn)
