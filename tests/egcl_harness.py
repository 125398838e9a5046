"""Shared pieces of the GPU parity tests: the product's EGCL / CEMLP built on the GPU with reference parameters, seeded
EGCL inputs on a block-diagonal pair graph, the CPU oracle (oracle/layers_ref.py) and our layer run the same way, and
one comparison of a forward output and its gradients.  Imports without a GPU, so the suite still collects on a CPU."""
import torch

from conftest import assert_close
from oracle import layers_ref as R

DEV = "cuda"
# leaves of an EGCL step -> their key in an inputs dict
LEAVES = {"h": "h", "edge_attr": "ea", "node_attr": "na"}

CASES = [
    # name, metric, C, T, complexes, simplices/complex, pairs/complex, aggr
    ("motion", (1, 1, 1), 28, 3, 6, 47, 226, "mean"),
    ("md17", (1, 1, 1), 32, 3, 4, 87, 527, "sum"),
    ("nba", (1, 1), 40, 3, 6, 41, 345, "sum"),
    ("odd_c", (1, 1, 1), 30, 2, 3, 19, 77, "mean"),
    ("tiny", (1, 1, 1), 8, 3, 1, 5, 3, "sum"),
    ("one_tile_exact", (1, 1, 1), 16, 3, 1, 128, 256, "mean"),
]

# wide blocks: weights streamed with the K chunks (csmpn_block_tc_plan bits 1-3), hidden widths 64 / 128 / 256
WIDE = [
    ("cl3_c64", (1, 1, 1), 64, 3, 4, 87, 527, "sum"),
    ("cl3_c128", (1, 1, 1), 128, 3, 2, 87, 527, "mean"),
    ("cl3_c256", (1, 1, 1), 256, 3, 1, 60, 300, "sum"),
    ("cl2_c128", (1, 1), 128, 3, 3, 41, 345, "sum"),
    ("cl2_c64", (1, 1), 64, 3, 3, 41, 345, "mean"),
    ("cl3_c64_multi_tile", (1, 1, 1), 64, 3, 40, 87, 527, "sum"),   # 165 tiles of pairs: two tiles on some CTAs
]


def mods():
    """the product's CliffordAlgebra and layer module, imported when a test runs"""
    from csmpn_b200.algebra.cliffordalgebra import CliffordAlgebra
    from csmpn_b200.models import cegnn_utils as M

    return CliffordAlgebra, M


def load_params(module, params):
    """load reference parameters: nothing unexpected, and only the algebra's buffers missing"""
    missing, unexpected = module.load_state_dict(dict(params), strict=False)
    assert not unexpected and all("algebra" in k for k in missing), (missing, unexpected)
    return module


def egcl_model(metric, C, T, aggr, params):
    CliffordAlgebra, M = mods()
    alg = CliffordAlgebra(metric).to(DEV)
    return load_params(M.EGCL(alg, C, C, C, edge_attr_features=2 * T, node_attr_features=T, aggr=aggr).to(DEV), params)


def cemlp_model(metric, c_in, C, n_layers, params):
    CliffordAlgebra, M = mods()
    alg = CliffordAlgebra(metric).to(DEV)
    return load_params(M.CEMLP(alg, c_in, C, C, n_layers=n_layers).to(DEV), params)


def grads(out, cot, tensors):
    return torch.autograd.grad(out, tensors, cot.to(out.device), allow_unused=True)


def block_diag_graph(n_cplx, n, e, gen):
    """e random (sender, receiver) pairs inside each of n_cplx complexes of n simplices"""
    src = torch.randint(0, n, (n_cplx, e), generator=gen)
    dst = torch.randint(0, n, (n_cplx, e), generator=gen)
    off = (torch.arange(n_cplx) * n).unsqueeze(1)
    return torch.stack([(src + off).reshape(-1), (dst + off).reshape(-1)])


def egcl_inputs(case):
    """Seeded inputs of an EGCL case: the seed is the sum of the name's code points, so a test ID names its inputs
    whatever the interpreter's hash seed.  node_attr is a type embedding in the scalar blade and
    edge_attr = node_attr[src] | node_attr[dst], as the models build them."""
    name, metric, C, T, ncx, n, e, aggr = case
    gen = torch.Generator().manual_seed(sum(map(ord, name)))
    ralg = R.RefAlgebra(metric)
    params = R.init_egcl_params(ralg, C, T, gen)
    N = ncx * n
    h = torch.randn(N, C, ralg.B, generator=gen)
    ei = block_diag_graph(ncx, n, e, gen)
    na = torch.zeros(N, T, ralg.B)
    na[..., 0] = torch.randn(T, T, generator=gen)[torch.randint(0, T, (N,), generator=gen)]
    return {"ralg": ralg, "params": params, "aggr": aggr, "h": h, "ei": ei, "ea": torch.cat([na[ei[0]], na[ei[1]]], 1),
            "na": na, "cot": torch.randn(N, C, ralg.B, generator=gen)}


def bench_inputs(b):
    """inputs of a bench.make_batch batch, with seed-7 EGCL parameters"""
    ralg = R.RefAlgebra(b["metric"])
    params = R.init_egcl_params(ralg, b["C"], b["node_attr"].shape[1], torch.Generator().manual_seed(7))
    return {"ralg": ralg, "params": params, "aggr": b["aggr"], "h": b["h"], "ei": b["edge_index"], "ea": b["edge_attr"],
            "na": b["node_attr"], "cot": b["cot"]}


def oracle_egcl(inputs, dtype, wrt, edge):
    """CPU oracle in dtype: (y, {name: gradient}) for the leaves named in wrt and every parameter.  edge "tensor" feeds
    the materialised edge_attr leaf; "paired" builds node_attr[src] | node_attr[dst] from the node_attr leaf."""
    leaves = {k: inputs[v].to(dtype, copy=True).requires_grad_(k in wrt) for k, v in LEAVES.items()}
    p = {k: v.to(dtype, copy=True).requires_grad_() for k, v in inputs["params"].items()}
    ei, na = inputs["ei"], leaves["node_attr"]
    ea = leaves["edge_attr"] if edge == "tensor" else torch.cat([na[ei[0]], na[ei[1]]], 1)
    y = R.egcl(inputs["ralg"], leaves["h"], ei, ea, na, p, aggr=inputs["aggr"])
    g = torch.autograd.grad(y, [leaves[k] for k in wrt] + list(p.values()), inputs["cot"].to(dtype))
    return y.detach(), dict(zip(list(wrt) + list(p), g))


def run_egcl(model, inputs, wrt, edge):
    """our layer on the GPU, as oracle_egcl runs the oracle; edge "paired" passes PairedNodeAttr(node_attr)"""
    _, M = mods()
    leaves = {k: inputs[v].to(DEV).requires_grad_(k in wrt) for k, v in LEAVES.items()}
    na = leaves["node_attr"]
    y = model(leaves["h"], inputs["ei"].to(DEV), leaves["edge_attr"] if edge == "tensor" else M.PairedNodeAttr(na), na)
    pd = dict(model.named_parameters())
    g = torch.autograd.grad(y, [leaves[k] for k in wrt] + [pd[k] for k in inputs["params"]], inputs["cot"].to(DEV))
    torch.cuda.synchronize()
    return y.detach(), dict(zip(list(wrt) + list(inputs["params"]), g))


def _what(k):
    return "g" + k if k in LEAVES else k


def assert_all_close(got, ref, fwd_tol, grad_tol, tag):
    """(y, {name: gradient}) against a reference of the same shape: y within fwd_tol, each of ref's gradients within
    grad_tol (max-norm error relative to the reference)"""
    assert_close(got[0], ref[0], fwd_tol, f"{tag} fwd")
    for k, r in ref[1].items():
        assert_close(got[1][k], r, grad_tol, f"{tag} {_what(k)}")


def assert_all_equal(got, ref, tag):
    """(y, {name: gradient}) bit for bit"""
    assert torch.equal(got[0], ref[0]), f"{tag} fwd"
    for k, r in ref[1].items():
        assert torch.equal(got[1][k], r), f"{tag} {_what(k)}"
