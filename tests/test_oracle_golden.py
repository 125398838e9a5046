"""The CPU oracle (oracle/layers_ref.py) against the golden vectors produced by the reference's own code
(tests/golden/make_golden.py).  This is what pins the oracle; the GPU parity tests then compare against it."""
import pytest
import torch

from conftest import LAYER_FIXTURES, assert_close, load_golden, tols
from egcl_harness import grads
from oracle import layers_ref as R


@pytest.fixture(scope="module", params=LAYER_FIXTURES)
def fx(request):
    f = load_golden(request.param)
    f["alg"] = R.RefAlgebra(f["metric"])
    return f


def test_tables(fx):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg = fx["alg"]
    assert torch.equal(alg.dense_cayley(), fx["cayley"])
    assert alg.subspaces == fx["subspaces"].tolist()
    assert alg.grade == [int(g) for g in fx["bbo_grades"].tolist()]
    assert torch.equal(alg.paths, fx["paths"])
    assert alg.bitmap == fx["index_to_bitmap"].tolist()


def test_geometric_product(fx):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx["gp"]
    a, b = g["a"].clone().requires_grad_(), g["b"].clone().requires_grad_()
    out = R.geometric_product(alg, a, b)
    assert_close(out, g["out"], FWD_TOL, "gp")
    ga, gb = grads(out, g["cot"], [a, b])
    assert_close(ga, g["ga"], GRAD_TOL, "gp ga")
    assert_close(gb, g["gb"], GRAD_TOL, "gp gb")


def test_forms(fx):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx["gp"]
    q = R.grade_q(alg, g["a"])
    assert_close(q, fx["qs"], FWD_TOL, "qs")
    assert_close(R.smooth_abs_sqrt(q), fx["norms"], FWD_TOL, "norms")


@pytest.mark.parametrize("sub", [1, 0])
def test_mvlinear(fx, sub):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx[f"mvlinear_{sub}"]
    x, w, b = (g[k].clone().requires_grad_() for k in ("x", "weight", "bias"))
    y = R.mvlinear(alg, x, w, b)
    assert_close(y, g["y"], FWD_TOL, "mvlinear")
    gx, gw, gb = grads(y, g["cot"], [x, w, b])
    assert_close(gx, g["gx"], GRAD_TOL, "gx")
    assert_close(gw, g["gw"], GRAD_TOL, "gw")
    assert_close(gb, g["gb"], GRAD_TOL, "gb")


def test_mvsilu(fx):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx["mvsilu"]
    x, a, b = (g[k].clone().requires_grad_() for k in ("x", "a", "b"))
    y = R.mvsilu(alg, x, a, b)
    assert_close(y, g["y"], FWD_TOL, "mvsilu")
    for got, key in zip(grads(y, g["cot"], [x, a, b]), ("gx", "ga", "gb")):
        assert_close(got, g[key], GRAD_TOL, key)


def test_mvnorm(fx):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx["mvnorm"]
    x, a = (g[k].clone().requires_grad_() for k in ("x", "a"))
    y = R.normalization(alg, x, a)
    assert_close(y, g["y"], FWD_TOL, "mvnorm")
    for got, key in zip(grads(y, g["cot"], [x, a]), ("gx", "ga")):
        assert_close(got, g[key], GRAD_TOL, key)


def test_mvlayernorm(fx):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx["mvlayernorm"]
    x, a = (g[k].clone().requires_grad_() for k in ("x", "a"))
    y = R.mvlayernorm(alg, x, a)
    assert_close(y, g["y"], FWD_TOL, "mvlayernorm")
    for got, key in zip(grads(y, g["cot"], [x, a]), ("gx", "ga")):
        assert_close(got, g[key], GRAD_TOL, key)


def test_sgp(fx):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx["sgp"]
    p = {k: v.clone().requires_grad_() for k, v in g["params"].items()}
    x = g["x"].clone().requires_grad_()
    y = R.sgp(alg, x, p, "")
    assert_close(y, g["y"], FWD_TOL, "sgp")
    names = list(p)
    got = grads(y, g["cot"], [x] + [p[n] for n in names])
    assert_close(got[0], g["gx"], GRAD_TOL, "gx")
    for n, gi in zip(names, got[1:]):
        assert_close(gi, g["grads"][n], GRAD_TOL, n)


def test_cemlp(fx):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx["cemlp"]
    p = {k: v.clone().requires_grad_() for k, v in g["params"].items()}
    x = g["x"].clone().requires_grad_()
    y = R.cemlp(alg, x, p)
    assert_close(y, g["y"], FWD_TOL, "cemlp")
    names = list(p)
    got = grads(y, g["cot"], [x] + [p[n] for n in names])
    assert_close(got[0], g["gx"], GRAD_TOL, "gx")
    for n, gi in zip(names, got[1:]):
        assert_close(gi, g["grads"][n], GRAD_TOL, n)


@pytest.mark.parametrize("aggr", ["sum", "mean"])
def test_egcl(fx, aggr):
    FWD_TOL, GRAD_TOL = tols(fx)
    alg, g = fx["alg"], fx[f"egcl_{aggr}"]
    p = {k: v.clone().requires_grad_() for k, v in g["params"].items()}
    h, ea, na = (g[k].clone().requires_grad_() for k in ("h", "edge_attr", "node_attr"))
    y = R.egcl(alg, h, g["edge_index"], ea, na, p, aggr=aggr)
    assert_close(y, g["y"], FWD_TOL, "egcl")
    names = list(p)
    got = grads(y, g["cot"], [h, ea, na] + [p[n] for n in names])
    assert_close(got[0], g["gh"], GRAD_TOL, "gh")
    assert_close(got[1], g["gedge_attr"], GRAD_TOL, "gedge_attr")
    assert_close(got[2], g["gnode_attr"], GRAD_TOL, "gnode_attr")
    for n, gi in zip(names, got[3:]):
        assert_close(gi, g["grads"][n], GRAD_TOL, n)


def test_oracle_fp64_agrees_with_fp32():
    """fp64 run of the same oracle: tells fp32 noise from a wrong formula."""
    alg = R.RefAlgebra((1, 1, 1))
    gen = torch.Generator().manual_seed(3)
    p32 = R.init_egcl_params(alg, 8, 3, gen)
    p64 = {k: v.double() for k, v in p32.items()}
    h = torch.randn(10, 8, 8, generator=gen)
    ei = torch.randint(0, 10, (2, 40), generator=gen)
    na = torch.zeros(10, 3, 8)
    na[..., 0] = torch.randn(10, 3, generator=gen)
    ea = torch.cat([na[ei[0]], na[ei[1]]], 1)
    y32 = R.egcl(alg, h, ei, ea, na, p32, "sum")
    y64 = R.egcl(alg, h.double(), ei, ea.double(), na.double(), p64, "sum")
    assert_close(y32, y64.float(), 5e-5, "fp32 vs fp64 oracle")


def test_dense_and_table_weighted_product_agree():
    for metric in ((1, 1), (1, 1, 1), (1, -1, 1), (0, 1, 1)):
        alg = R.RefAlgebra(metric)
        gen = torch.Generator().manual_seed(1)
        x = torch.randn(7, 5, alg.B, generator=gen, dtype=torch.float64)
        r = torch.randn(7, 5, alg.B, generator=gen, dtype=torch.float64)
        w = torch.randn(5, alg.n_paths, generator=gen, dtype=torch.float64)
        assert_close(R.weighted_gp(alg, x, r, w), R.weighted_gp_tables(alg, x, r, w), 1e-12, str(metric))
