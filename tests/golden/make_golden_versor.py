#!/usr/bin/env python
"""Golden fixture for the off-path versor utilities of CliffordAlgebra (parity, eta, alpha_w, inverse, rho, sandwich,
output_blades, reduce_geometric_product): the reference's definitions (csmpn/algebra/cliffordalgebra.py:170-236)
restated over the tables of oracle/layers_ref.py and evaluated in fp64 on the CPU, on the seeded inputs
tests/test_gpu_layers.py::test_versor_utilities_match_the_reference has always used.

    python tests/golden/make_golden_versor.py        (writes tests/golden/versor.pt)

Restated as the reference has them, quirks included: ``b(x, y)`` is the scalar part of ``beta(x) y``; ``inverse(w)`` is
``beta(w) / b(w, beta(w))`` (not norm-preserving, SURVEY.md appendix B); ``alpha_w`` flips the odd grades of ``mv`` by
``eta(w) = (-1) ** parity(w)``; ``rho(w, mv) = w alpha_w(mv) inverse(w)``.
"""
import functools
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import torch

from oracle import layers_ref as R

METRICS = ((1, 1), (1, 1, 1))


def versor_case(metric, gen):
    ralg = R.RefAlgebra(metric)
    Bn = ralg.B
    grade = torch.tensor(ralg.grade)
    odd = grade % 2 == 1
    beta_sign = torch.tensor([(-1.0) ** (g * (g - 1) // 2) for g in ralg.grade], dtype=torch.float64)
    gp = lambda a, b: R.geometric_product(ralg, a, b)
    beta = lambda x: beta_sign * x
    inverse = lambda w: beta(w) / gp(beta(w), beta(w))[..., :1]

    def parity(w):
        no_even, no_odd = bool((w[..., ~odd] == 0).all()), bool((w[..., odd] == 0).all())
        assert no_even != no_odd
        return no_even

    def alpha_w(w, mv):
        return ~odd * mv + (-1.0 if parity(w) else 1.0) * odd * mv

    # the draws, in the order the test made them
    mv = torch.randn(5, Bn, generator=gen)
    vec = torch.zeros(1, Bn)
    vec[0, 1:1 + len(metric)] = torch.randn(len(metric), generator=gen)                      # odd element
    rot = gp(vec, torch.roll(vec, 1, dims=1) * (grade == 1))                                 # even element
    chain = [torch.randn(3, Bn, generator=gen) for _ in range(3)]

    d = lambda t: t.double()
    case = {"mv": mv, "vec": vec, "rot": rot, "chain": chain, "elements": []}
    for w in (vec, rot):
        case["elements"].append({
            "parity": parity(w), "eta": -1 if parity(w) else 1,
            "alpha_w": alpha_w(d(w), d(mv)), "inverse": inverse(d(w)),
            "rho": gp(gp(d(w), alpha_w(d(w), d(mv))), inverse(d(w))),
        })
    case["sandwich"] = gp(gp(d(mv), d(vec)), d(mv))
    left, right = [1, 2], list(range(Bn))
    index_of = {b: i for i, b in enumerate(ralg.bitmap)}
    case["output_blades"] = {"left": left, "right": right,
                             "blades": torch.tensor([index_of[ralg.bitmap[l] ^ ralg.bitmap[r]] for l in left for r in right])}
    case["reduce_geometric_product"] = functools.reduce(gp, [d(c) for c in chain])
    return case


def main():
    gen = torch.Generator().manual_seed(11)
    fx = {metric: versor_case(metric, gen) for metric in METRICS}
    path = os.path.join(HERE, "versor.pt")
    torch.save(fx, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
