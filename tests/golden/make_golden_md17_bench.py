#!/usr/bin/env python
"""Golden fixture for the md17 model AT THE BENCHED SIZE: the UNMODIFIED reference model
(csmpn/models/md17_cssmpnn.py: Cl(3,0), num_input=30, num_hidden=32, 5 layers -- csmpn/configs/md17.yaml:29-34) on the
exact 100-complex batch `bench.py`'s train leg uses (bench.make_md17_graphs(100, 2000)), run on the CPU of the build
container through oracle/refshim.py.

    python tests/golden/make_golden_md17_bench.py     (needs a copy of the reference, see oracle/refshim.py; writes
                                                       tests/golden/md17_bench.pt, ~0.25 MB)

Stored: the training loss, the per-sample losses, a fixed seeded sample of GRAD_SAMPLE entries of the gradient of the
loss w.r.t. every parameter (with the indices and the largest magnitude of the whole gradient, the scale the test
measures errors against), a checksum of the state_dict (the reference's initialisation under torch.manual_seed(0),
which the product's models reproduce; the test rebuilds it and checks the checksum) and a checksum of the collated
edge_index / x_ind (the batch itself is regenerated from the seed by the test and lifted on the GPU; the checksum proves
both sides saw the same complexes in the same order).  The sample keeps the file small.
"""
import hashlib
import os
import sys
import time
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import torch

from oracle import lift_ref as L
from oracle import refshim

refshim.install()

N_COMPLEXES, SEED = 100, 2000
INIT_SEED = 0
GRAD_SAMPLE = 128


def checksum(t: torch.Tensor) -> str:
    return hashlib.sha256(t.contiguous().cpu().numpy().tobytes()).hexdigest()


def state_dict_checksum(sd) -> str:
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode() + b"\0" + v.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def compact(fx):
    """the full fixture (state_dict, every gradient) -> the stored one (state_dict checksum, sampled gradients)"""
    fx = dict(fx)
    sd = fx.pop("state_dict")
    fx["init_seed"], fx["state_dict_sha256"] = INIT_SEED, state_dict_checksum(sd)
    picks = {}
    for i, (n, g) in enumerate(fx["grads"].items()):
        if g is not None:
            flat = g.reshape(-1)
            picks[n] = (flat, torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(i))[:GRAD_SAMPLE].sort().values)
    # every sample is a view of one index and one value tensor: torch.save then writes two storages, not two per parameter
    index = torch.cat([idx for _, idx in picks.values()]).to(torch.int32)
    value = torch.cat([flat[idx] for flat, idx in picks.values()])
    grads, off = {}, 0
    for n, g in fx["grads"].items():
        if g is None:
            grads[n] = None
            continue
        flat, idx = picks[n]
        k = idx.numel()
        grads[n] = {"shape": tuple(g.shape), "index": index[off:off + k], "value": value[off:off + k],
                    "absmax": float(flat.abs().max())}
        off += k
    fx["grads"] = grads
    return fx


def main():
    import bench
    from csmpn.models.md17_cssmpnn import CliffordSharedSimplicialMPNN_md17
    from make_golden_models import collate

    graphs = bench.make_md17_graphs(N_COMPLEXES, SEED, "cpu")
    parts, loc, vel, chg, ys = [], [], [], [], []
    for g in graphs:
        n, F = g.loc.shape[0], g.loc.shape[1]
        parts.append(L.merge_ref(*L.clique_lift_ref(n, g.edge_index)))
        loc.append(g.loc), vel.append(g.vel), ys.append(g.y)
        chg.append(g.charges.reshape(n, 1, 1).repeat(1, F, 1))
    b = collate(parts, dict(loc=loc, vel=vel, charges=chg))
    b["y"] = torch.cat(ys)
    torch.manual_seed(INIT_SEED)
    model = CliffordSharedSimplicialMPNN_md17()
    t0 = time.time()
    loss, out = model(types.SimpleNamespace(**{k: v.clone() for k, v in b.items()}), 0, "train")
    named = list(model.named_parameters())
    grads = torch.autograd.grad(loss, [p for _, p in named], allow_unused=True)
    print(f"reference md17 model fwd+bwd on {b['x_ind'].shape[0]} simplices / {b['edge_index'].shape[1]} pairs: {time.time() - t0:.1f} s")
    fx = dict(
        n_complexes=N_COMPLEXES, seed=SEED, loss=loss.detach(), out={k: v.detach() for k, v in out.items()},
        grads={n: (None if g is None else g.detach()) for (n, _), g in zip(named, grads)},
        state_dict={k: v.detach().clone() for k, v in model.state_dict().items() if "algebra" not in k},
        edge_index_sha256=checksum(b["edge_index"]), x_ind_sha256=checksum(b["x_ind"]),
        n_simplices=int(b["x_ind"].shape[0]), n_pairs=int(b["edge_index"].shape[1]))
    path = os.path.join(HERE, "md17_bench.pt")
    torch.save(compact(fx), path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB", "loss", float(loss))


if __name__ == "__main__":
    main()
