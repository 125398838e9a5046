"""The four task models (csmpn_b200.models.*_cssmpnn) against fixtures produced by the reference's own models
(tests/golden/models.pt, made by tests/golden/make_golden_models.py): same state_dict keys and shapes (so reference
checkpoints load), loss / per-sample losses within rel 1e-5, parameter gradients within rel 1e-4 (fp32)."""
import types

import pytest
import torch

from conftest import FWD_TOL, GRAD_TOL, assert_close, load_golden


def model_class(name):
    from csmpn_b200.models.hulls_cssmpnn import HullsCliffordSharedSimplicialMPNN
    from csmpn_b200.models.md17_cssmpnn import CliffordSharedSimplicialMPNN_md17
    from csmpn_b200.models.motion_cssmpnn import MotionCliffordSharedSimplicialMPNN
    from csmpn_b200.models.nba_cssmpnn import NBACliffordSharedSimplicialMPNN

    return {"md17": CliffordSharedSimplicialMPNN_md17, "motion": MotionCliffordSharedSimplicialMPNN,
            "nba": NBACliffordSharedSimplicialMPNN, "hulls": HullsCliffordSharedSimplicialMPNN}[name]


@pytest.fixture(scope="module")
def gold():
    return load_golden("models.pt")


NAMES = ["md17", "motion", "nba", "hulls"]


@pytest.mark.parametrize("name", NAMES)
def test_state_dict_layout_matches_reference(gold, name):
    fx = gold[name]
    m = model_class(name)(**fx["kwargs"])
    ours = {k: tuple(v.shape) for k, v in m.state_dict().items() if "algebra" not in k}
    ref = {k: tuple(v.shape) for k, v in fx["state_dict"].items()}
    assert ours == ref
    assert [n for n, _ in m.named_parameters()] == list(fx["grads"].keys())


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_model_forward_backward_matches_reference(gold, name):
    dev = torch.device("cuda:0")
    fx = gold[name]
    m = model_class(name)(**fx["kwargs"]).to(dev)
    missing, unexpected = m.load_state_dict(fx["state_dict"], strict=False)
    assert not unexpected and all("algebra" in k for k in missing), (missing, unexpected)
    g = types.SimpleNamespace(**{k: v.clone().to(dev) for k, v in fx["batch"].items()})
    loss, out = m(g, 0, "train")
    assert_close(loss, fx["loss"], FWD_TOL, f"{name} loss")
    for k, v in fx["out"].items():
        assert_close(out[k], v, FWD_TOL, f"{name} out[{k}]")
    named = list(m.named_parameters())
    grads = torch.autograd.grad(loss, [p for _, p in named], allow_unused=True)
    for (n, _), gr in zip(named, grads):
        ref = fx["grads"][n]
        if ref is None:
            assert gr is None or float(gr.abs().max()) == 0.0, n
            continue
        assert gr is not None, n
        assert_close(gr, ref, GRAD_TOL, f"{name} grad {n}")


@pytest.mark.gpu
def test_model_on_gpu_lifted_batch_matches_fixture_batch(gold):
    """lifting + model end to end: the NBA batch lifted on the GPU gives the same loss as the oracle-lifted one"""
    from csmpn_b200.data.modules.simplicial_data import Data, SimplicialTransform

    dev = torch.device("cuda:0")
    fx = gold["nba"]
    b = fx["batch"]
    graphs = []
    for c in range(3):
        lo = int(b["ptr"][c])
        pos, vel = b["pos"][lo:lo + 6], b["vel"][lo:lo + 6]
        graphs.append(Data(pos=pos.to(dev), vel=vel.to(dev), init_pos=pos[:, 0].to(dev), y=b["y"][5 * c:5 * c + 5].to(dev)))
    g = SimplicialTransform(dim=2, dis=1e4, label="nba").lift(graphs, device=dev)
    assert torch.equal(g.edge_index.cpu(), b["edge_index"]) and torch.equal(g.x_ind.cpu(), b["x_ind"])
    m = model_class("nba")(**fx["kwargs"]).to(dev)
    m.load_state_dict(fx["state_dict"], strict=False)
    loss, _ = m(g, 0, "train")
    assert_close(loss, fx["loss"], FWD_TOL, "nba loss on the GPU-lifted batch")


@pytest.mark.gpu
def test_graphed_train_step_equals_eager(gold):
    """GraphedDataParallelStep (forward + backward replayed from one CUDA graph) follows the eager DataParallelStep:
    same losses and the same parameters after three Adam steps on the md17 fixture batch."""
    from csmpn_b200.train_step import DataParallelStep, GraphedDataParallelStep

    dev = torch.device("cuda:0")
    fx = gold["md17"]
    results = []
    for graphed in (False, True):
        m = model_class("md17")(**fx["kwargs"]).to(dev)
        m.load_state_dict(fx["state_dict"], strict=False)
        g = types.SimpleNamespace(**{k: v.clone().to(dev) for k, v in fx["batch"].items()})
        loc0 = g.loc.clone()
        # graphed: capturable fused Adam with a device-tensor learning rate, optimizer step INSIDE the graph
        opt = (torch.optim.Adam(m.parameters(), lr=torch.tensor(1e-3, device=dev), fused=True, capturable=True) if graphed
               else torch.optim.Adam(m.parameters(), lr=1e-3))
        step = GraphedDataParallelStep(m, opt, g) if graphed else DataParallelStep(m, opt)
        if graphed:
            assert step.captured_optimizer and "Adam" in step.describe()
        if graphed:  # the capture warm-up ran backward passes but no optimizer step: parameters are still the fixture's
            assert all(torch.equal(p.detach().cpu(), fx["state_dict"][n]) for n, p in m.named_parameters())
        losses = []
        for _ in range(3):
            g.loc = loc0
            loss, _ = step(g)
            losses.append(float(loss))
        results.append((losses, [p.detach().clone() for p in m.parameters()]))
    (l0, p0), (l1, p1) = results
    for a, b in zip(l0, l1):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (l0, l1)
    for a, b in zip(p0, p1):
        # Adam divides by sqrt(v): fp32 run-to-run noise (1e-7, torch's atomic index_add in the pooling) of near-zero
        # gradients is amplified to ~1e-5 of a parameter after three steps, in eager mode as well
        assert_close(b, a, 2e-4, "parameters after 3 steps")


@pytest.mark.gpu
def test_md17_model_at_benched_size_matches_reference():
    """The md17 model at the size `bench.py`'s train leg runs (100 complexes: ~8.6 k simplices, ~52 k pairs, so the layers'
    per-pair blocks run on the tensor-core engine with 3 tiles per persistent CTA) against the UNMODIFIED reference
    model's loss and parameter gradients (tests/golden/md17_bench.pt, made by tests/golden/make_golden_md17_bench.py).
    The batch is regenerated from the seed and lifted on the GPU, the parameters from the seed of the reference's
    initialisation; checksums tie both to what the reference saw.  The gradients are compared on a fixed sample of their
    entries, against the largest magnitude of the whole reference gradient (the scale of rel_err)."""
    import hashlib
    import os
    import sys

    from conftest import ROOT
    from csmpn_b200 import _lib
    from csmpn_b200.data.modules.simplicial_data import SimplicialTransform

    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench

    dev = torch.device("cuda:0")
    fx = load_golden("md17_bench.pt")
    graphs = bench.make_md17_graphs(fx["n_complexes"], fx["seed"], dev)
    batch = SimplicialTransform(dim=2, dis=2.5, label="md17", molecule_type="aspirin").lift(graphs, device=dev)
    sha = lambda t: hashlib.sha256(t.contiguous().cpu().numpy().tobytes()).hexdigest()
    assert sha(batch.edge_index) == fx["edge_index_sha256"] and sha(batch.x_ind) == fx["x_ind_sha256"]
    assert int(batch.edge_index.shape[1]) == fx["n_pairs"] >= 8192
    torch.manual_seed(fx["init_seed"])
    m = model_class("md17")()
    sd = hashlib.sha256()
    for k, v in m.state_dict().items():
        if "algebra" not in k:
            sd.update(k.encode() + b"\0" + v.contiguous().numpy().tobytes())
    assert sd.hexdigest() == fx["state_dict_sha256"], "the seeded initialisation no longer gives the reference's parameters"
    m = m.to(dev)
    n0 = _lib.lib().csmpn_launch_count()
    loss, out = m(batch, 0, "train")
    named = list(m.named_parameters())
    grads = torch.autograd.grad(loss, [p for _, p in named], allow_unused=True)
    assert _lib.lib().csmpn_launch_count() - n0 > 150
    assert_close(loss, fx["loss"], FWD_TOL, "md17@100 loss")
    for k, v in fx["out"].items():
        assert_close(out[k], v, FWD_TOL, f"md17@100 out[{k}]")
    for (n, _), gr in zip(named, grads):
        ref = fx["grads"][n]
        if ref is None:
            assert gr is None or float(gr.abs().max()) == 0.0, n
            continue
        assert gr is not None and tuple(gr.shape) == ref["shape"], n
        flat = gr.detach().double().cpu().reshape(-1)
        scale = ref["absmax"] + 1e-30
        e = float((flat[ref["index"].long()] - ref["value"].double()).abs().max()) / scale
        assert e <= GRAD_TOL, f"md17@100 grad {n}: rel err {e:.3e} > {GRAD_TOL:.1e}"
        # the largest magnitude of the whole gradient: within the same bound if every entry is
        e = abs(float(flat.abs().max()) - ref["absmax"]) / scale
        assert e <= GRAD_TOL, f"md17@100 grad {n}: max |g| rel err {e:.3e} > {GRAD_TOL:.1e}"


@pytest.mark.gpu
def test_graphed_motion_step_follows_updates(gold):
    """The motion model REBINDS graph.pos in forward (centring, motion_cssmpnn.py:146): the graphed step must keep reading
    the tensors it captured and take new input values through update().  Two steps with different positions, graphed vs
    eager: same losses, same parameters."""
    from csmpn_b200.train_step import CosineAnnealingLR, DataParallelStep, GraphedDataParallelStep

    dev = torch.device("cuda:0")
    fx = gold["motion"]
    pos1 = fx["batch"]["pos"].clone().to(dev)
    pos2 = (pos1 * 0.5 + 0.25).contiguous()
    results = []
    for graphed in (False, True):
        m = model_class("motion")(**fx["kwargs"]).to(dev)
        m.load_state_dict(fx["state_dict"], strict=False)
        g = types.SimpleNamespace(**{k: v.clone().to(dev) for k, v in fx["batch"].items()})
        if graphed:
            opt = torch.optim.Adam(m.parameters(), lr=torch.tensor(1e-3, device=dev), fused=True, capturable=True)
            step = GraphedDataParallelStep(m, opt, g)
        else:
            opt = torch.optim.Adam(m.parameters(), lr=1e-3)
            step = DataParallelStep(m, opt)
        sched = CosineAnnealingLR(opt, 8, warmup_steps=2, decay_steps=2)
        losses = []
        for pos in (pos1, pos2, pos1):
            if graphed:
                step.update(pos=pos)
                loss, _ = step()
            else:
                g.pos = pos.clone()
                loss, _ = step(g)
            sched.step()
            losses.append(float(loss.detach()))
        results.append((losses, [p.detach().clone() for p in m.parameters()]))
    (l0, p0), (l1, p1) = results
    assert abs(l0[0] - l0[1]) > 1e-4 * abs(l0[0])  # the update really changed the input
    for a, b in zip(l0, l1):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (l0, l1)
    for a, b in zip(p0, p1):
        assert_close(b, a, 2e-4, "motion parameters after 3 scheduled steps")


@pytest.mark.gpu
def test_csr_cache_eviction_does_not_invalidate_a_captured_step(gold):
    """ADVICE r01: the captured step holds its own references to the CSR of its batch; running many other batches eagerly
    between replays (which cycles the identity-keyed CSR cache) must not change what the replay computes."""
    from csmpn_b200.models.ops import get_csr
    from csmpn_b200.train_step import GraphedDataParallelStep

    dev = torch.device("cuda:0")
    fx = gold["md17"]
    m = model_class("md17")(**fx["kwargs"]).to(dev)
    m.load_state_dict(fx["state_dict"], strict=False)
    g = types.SimpleNamespace(**{k: v.clone().to(dev) for k, v in fx["batch"].items()})
    opt = torch.optim.SGD(m.parameters(), lr=0.0)
    step = GraphedDataParallelStep(m, opt, g)
    l0 = float(step()[0])
    keep = []
    for k in range(12):  # more distinct edge_index tensors than the cache holds
        ei = g.edge_index.clone()
        keep.append(ei)
        get_csr(ei, g.x_ind.shape[0])
    torch.cuda.synchronize()
    l1 = float(step()[0])
    assert l0 == l1


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["md17", "motion", "nba"])
def test_fused_permute_embed_equals_materialised_rows(gold, name, monkeypatch):
    """embed_simplicial_complex with the first block of cl_feature_embedding[d] gathering its (type, vertex slot, feature)
    channels from a per-vertex table (csmpn_block_desc mode 2, no permuted rows in memory) against the torch-indexing path
    (CSMPN_TC=0: rows materialised, SIMT engine): same embedding, same parameter gradients.  The fixture batch is
    replicated so that the per-dimension row counts cross the tensor-core threshold."""
    from csmpn_b200.models import fused

    dev = torch.device("cuda:0")
    fx = gold[name]
    b = fx["batch"]
    reps = 400
    n = b["x_ind"].shape[0]
    big = {}
    for k, v in b.items():
        if k == "edge_index":
            big[k] = torch.cat([v + i * n for i in range(reps)], 1)
        elif k in ("ptr", "x_ind_ptr"):
            big[k] = torch.cat([v[:-1] + i * n for i in range(reps)] + [v[-1:] + (reps - 1) * n])
        elif k in ("batch", "x_ind_batch"):
            big[k] = torch.cat([v + i * (int(v.max()) + 1) for i in range(reps)])
        else:
            big[k] = torch.cat([v] * reps, 0)
    m = model_class(name)(**fx["kwargs"]).to(dev)
    m.load_state_dict(fx["state_dict"], strict=False)
    out = {}
    for tc in ("1", "0"):
        monkeypatch.setenv("CSMPN_TC", tc)
        g = types.SimpleNamespace(**{k: v.clone().to(dev) for k, v in big.items()})
        if name == "md17":
            g.pos = g.loc
        calls = []
        orig = fused.embed_rows_forward
        def counted(*a, **k):
            r = orig(*a, **k)
            calls.append(r is not None)
            return r

        monkeypatch.setattr(fused, "embed_rows_forward", counted)
        x = m.embed_simplicial_complex(g, out_channels=m.num_input) if name == "nba" else m.embed_simplicial_complex(g)
        params = [p for e in m.cl_feature_embedding for p in e.parameters()]
        grads = torch.autograd.grad(x.square().sum(), params)
        monkeypatch.setattr(fused, "embed_rows_forward", orig)
        out[tc] = (x.detach(), grads, sum(calls))
    assert out["1"][2] >= 1 and out["0"][2] == 0  # the fused path ran for at least one simplex dimension / never without the engine
    assert_close(out["1"][0], out["0"][0], 1e-5, f"{name} embedding")
    for a, c in zip(out["1"][1], out["0"][1]):
        assert_close(a, c, 1e-4, f"{name} embedding parameter gradient")


# ---------------------------------------------------------------------------------------------- shape-padded stream
def _md17_samples(n, seed):
    import bench

    return bench.make_md17_graphs(n, seed, "cpu")


@pytest.mark.gpu
def test_padded_batch_leaves_loss_and_gradients_unchanged():
    """data/padding.py: one dummy complex absorbs the difference to the bucket sizes.  The md17 model on the padded batch gives
    the loss, the per-sample losses and every parameter gradient of the unpadded batch (dummy simplices only talk to
    dummy simplices and are masked out of the loss)."""
    from csmpn_b200.data.modules.simplicial_data import SimplicialTransform
    from csmpn_b200.data.padding import BucketOverflow, make_bucket, pad_to_bucket

    dev = torch.device("cuda:0")
    lift = SimplicialTransform(dim=2, dis=2.5, label="md17", molecule_type="aspirin")
    b = lift.lift(_md17_samples(12, 5), device=dev)
    torch.manual_seed(0)
    m = model_class("md17")().to(dev)
    loss, out = m(b, 0, "train")
    g_ref = torch.autograd.grad(loss, list(m.parameters()))
    bucket = make_bucket([b.sizes], margin=1.1)
    assert bucket.edges > b.sizes["edges"] and bucket.triangles > b.sizes["triangles"] and bucket.pairs > b.sizes["pairs"]
    pb = pad_to_bucket(b, bucket)
    assert pb.x_ind.shape[0] == bucket.simplices and pb.edge_index.shape[1] == bucket.pairs
    assert [int((pb.node_types == d).sum()) for d in range(3)] == list(bucket.counts())
    loss_p, out_p = m(pb, 0, "train")
    g_p = torch.autograd.grad(loss_p, list(m.parameters()))
    assert_close(loss_p, loss, FWD_TOL, "loss of the padded batch")
    assert out_p["loss"].shape == out["loss"].shape
    assert_close(out_p["loss"], out["loss"], FWD_TOL, "per-sample losses of the padded batch")
    for (n, _), a, r in zip(m.named_parameters(), g_p, g_ref):
        assert torch.isfinite(a).all(), n
        assert_close(a, r, GRAD_TOL, f"grad {n} (padded batch)")
    small = make_bucket([{**b.sizes, "edges": b.sizes["edges"] - 70}], margin=1.0, multiple=1)
    with pytest.raises(BucketOverflow):
        pad_to_bucket(b, small)


@pytest.mark.gpu
@pytest.mark.parametrize("optim", ["adam", "sgd"])
def test_padded_stream_step_follows_eager_on_different_batches(optim):
    """StreamGraphedStep: ONE captured graph (forward + backward [+ Adam]) replayed on three DIFFERENT md17 batches (different
    simplex and pair counts) tracks the eager DataParallelStep on the same batches.  adam: the optimizer step is inside the
    graph, losses of the three steps agree (Adam turns fp32 noise of near-zero gradients into +-lr, so the parameters are
    compared under plain SGD, where they must agree to the gradient tolerance)."""
    from csmpn_b200.data.modules.simplicial_data import SimplicialTransform
    from csmpn_b200.data.padding import make_bucket
    from csmpn_b200.train_step import DataParallelStep, StreamGraphedStep

    dev = torch.device("cuda:0")
    lift = SimplicialTransform(dim=2, dis=2.5, label="md17", molecule_type="aspirin")
    pools = [_md17_samples(10, 100 + k) for k in range(4)]
    sizes = [lift.lift(p, device=dev).sizes for p in pools]
    assert len({(s["simplices"], s["pairs"]) for s in sizes}) > 1, "the batches should differ in size"
    results = []
    for graphed in (False, True):
        torch.manual_seed(0)
        m = model_class("md17")().to(dev)
        if optim == "sgd":
            opt = torch.optim.SGD(m.parameters(), lr=1e-2)
        elif graphed:
            opt = torch.optim.Adam(m.parameters(), lr=torch.tensor(1e-3, device=dev), fused=True, capturable=True)
        else:
            opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        if graphed:
            step = StreamGraphedStep(m, opt, lift.lift(pools[0], device=dev), make_bucket(sizes))
            assert step.captured_optimizer == (optim == "adam")
        else:
            step = DataParallelStep(m, opt)
        losses = []
        for k in (1, 2, 3):
            loss, _ = step(lift.lift(pools[k], device=dev), k)
            losses.append(float(loss.detach()))
        results.append((losses, [p.detach().clone() for p in m.parameters()]))
    (l0, p0), (l1, p1) = results
    for a, b in zip(l0, l1):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (l0, l1)
    if optim == "sgd":
        for a, b in zip(p0, p1):
            assert_close(b, a, GRAD_TOL, "parameters after 3 SGD steps on different batches")


@pytest.mark.gpu
def test_padded_nba_batch_leaves_loss_and_gradients_unchanged(gold):
    """the same for the NBA model (Cl(2,0), Rips complexes, targets for all vertices but the last of each complex)"""
    from csmpn_b200.data.modules.simplicial_data import Data, SimplicialTransform
    from csmpn_b200.data.padding import make_bucket, pad_to_bucket

    dev = torch.device("cuda:0")
    fx = gold["nba"]
    b = fx["batch"]
    graphs = []
    for c in range(3):
        lo = int(b["ptr"][c])
        pos, vel = b["pos"][lo:lo + 6], b["vel"][lo:lo + 6]
        graphs.append(Data(pos=pos.to(dev), vel=vel.to(dev), init_pos=pos[:, 0].to(dev), y=b["y"][5 * c:5 * c + 5].to(dev)))
    g = SimplicialTransform(dim=2, dis=1e4, label="nba").lift(graphs, device=dev)
    m = model_class("nba")(**fx["kwargs"]).to(dev)
    m.load_state_dict(fx["state_dict"], strict=False)
    loss, out = m(g, 0, "train")
    g_ref = torch.autograd.grad(loss, [p for p in m.parameters() if p.requires_grad], allow_unused=True)
    pb = pad_to_bucket(g, make_bucket([g.sizes], margin=1.2, multiple=8))
    assert pb.y.shape[0] == g.y.shape[0] + 5 and pb.x_ind.shape[0] > g.x_ind.shape[0]
    loss_p, out_p = m(pb, 0, "train")
    g_p = torch.autograd.grad(loss_p, [p for p in m.parameters() if p.requires_grad], allow_unused=True)
    assert_close(loss_p, loss, FWD_TOL, "nba loss of the padded batch")
    assert_close(out_p["loss"], out["loss"], FWD_TOL, "nba per-sample losses of the padded batch")
    for a, r in zip(g_p, g_ref):
        assert (a is None) == (r is None)
        if a is not None:
            assert_close(a, r, GRAD_TOL, "nba grad (padded batch)")


@pytest.mark.gpu
def test_padded_stream_step_nba_follows_eager(gold):
    """the NBA model (Cl(2,0), Rips complexes whose edge / triangle counts change with the positions) trained from ONE graph
    on different batches: same losses and, under SGD, the same parameters as the eager step"""
    from csmpn_b200.data.modules.simplicial_data import Data, SimplicialTransform
    from csmpn_b200.data.padding import make_bucket
    from csmpn_b200.train_step import DataParallelStep, StreamGraphedStep

    dev = torch.device("cuda:0")
    fx = gold["nba"]
    frames = fx["batch"]["pos"].shape[1]
    lift = SimplicialTransform(dim=2, dis=1.6, label="nba")

    def samples(seed, n=4):
        g = torch.Generator().manual_seed(seed)
        out = []
        for _ in range(n):
            pos = torch.randn(6, frames, 2, generator=g)
            out.append(Data(pos=pos.to(dev), vel=torch.randn(6, frames, 2, generator=g).to(dev), init_pos=pos[:, 0].to(dev),
                            y=torch.randn(5, fx["batch"]["y"].shape[1], 2, generator=g).to(dev)))
        return out

    pools = [samples(500 + k) for k in range(4)]
    sizes = [lift.lift(p, device=dev).sizes for p in pools]
    assert len({(s["simplices"], s["pairs"]) for s in sizes}) > 1, "the batches should differ in size"
    results = []
    for graphed in (False, True):
        m = model_class("nba")(**fx["kwargs"]).to(dev)
        m.load_state_dict(fx["state_dict"], strict=False)
        opt = torch.optim.SGD(m.parameters(), lr=1e-2)
        step = StreamGraphedStep(m, opt, lift.lift(pools[0], device=dev), make_bucket(sizes, multiple=8)) if graphed \
            else DataParallelStep(m, opt)
        losses = []
        for k in (1, 2, 3):
            loss, _ = step(lift.lift(pools[k], device=dev), k)
            losses.append(float(loss.detach()))
        results.append((losses, [p.detach().clone() for p in m.parameters()]))
    (l0, p0), (l1, p1) = results
    for a, b in zip(l0, l1):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (l0, l1)
    for a, b in zip(p0, p1):
        assert_close(b, a, GRAD_TOL, "nba parameters after 3 SGD steps on different batches")
