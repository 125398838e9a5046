"""Every tensor-core block plan against the fp64 oracle.

The tensor-core engine picks a plan per block shape (dim, c_in, C): resident or streamed weights for f1 and for f2,
the pass widths ns1 / ns2, the resident or the wide backward (csmpn_block_tc_plan bits 0-3) -- or it rejects the shape,
and models/fused.py runs the block on the FP32 SIMT engine or composes it from unit kernels.  Each case below names the
branch it exists for and records the plan bits and the engine of every block it runs, so a failure points at a plan.

Checks per case: the plan bits; the engine each block actually ran (descriptors and launch counts of every native block
call); forward and every gradient against oracle/layers_ref.py in float64, globally and per slice (128-row tile, output
channel, blade; grade and output channel of [Cout, Cin, G] weights); bit-exact guard bands around the forward output
in the inference configuration; single-pass TF32 mode on the streamed, wide and padded plans."""
import ctypes
import functools

import pytest
import torch

from egcl_harness import DEV, block_diag_graph, cemlp_model, egcl_model, mods
from oracle import layers_ref as R

pytestmark = pytest.mark.gpu
T = 3  # node-attribute types of the EGCL cases: edge_attr has 2T channels

# global criterion (BASELINE.json north star): max-norm relative to the fp64 oracle
FWD_TOL, GRAD_TOL = 1e-5, 1e-4
# single-pass TF32 mode, as in test_tc_precision.py
TF32_FWD_TOL, TF32_GRAD_TOL = 5e-3, 2e-2

TC, SIMT, UNIT = "T", "S", "U"  # engine of a block: tensor-core, FP32 SIMT, unit kernels

# name, dim, C, shape, engine of each block, plan of each block, why the case exists
#   shape ("egcl", complexes, simplices per complex, pairs per complex, aggr): an EGCL layer with hidden width C; its
#     blocks are edge (C + 2T -> C, gather), edge (C -> C, BPT input), node (2C + T -> C), node (C -> C, residual)
#   shape ("mlp", c_in, rows): a 2-block CEMLP c_in -> C -> C on plain rows (mode 0)
# plan: (csmpn_block_tc_plan bits, ns1, ns2, np) -- bits 1 supported, 2 f1 streams its weights, 4 f2 streams its
#   weights, 8 wide backward; output channels per pass of f1, of f2 and of the wide backward GEMMs (csmpn_block_tc_passes)
NO = (0, 0, 0, 0)  # the tensor-core engine rejects the shape
MULTI = 300 * 128 + 1  # 300 tiles on 148 persistent CTAs: every CTA runs at least two tiles, four run three
CASES = [
    # ---- anchors: the classes test_tc_block.py already covers
    ("cl3_c32_anchor", 3, 32, ("egcl", 1, 129, 383, "sum"), "TTTT", ((0b1, 32, 32, 0),) * 4,
     "resident weights, resident backward (md17 width)"),
    ("cl2_c40_anchor", 2, 40, ("egcl", 3, 43, 43, "mean"), "TTTT", ((0b1, 48, 48, 0),) * 4,
     "Cl(2,0) resident weights at Cp = 48 (NBA width)"),
    ("cl3_c64_anchor", 3, 64, ("egcl", 1, 127, 255, "sum"), "TTTT", ((0b1111, 64, 32, 64),) * 4,
     "streamed f1 / f2 and wide backward at a whole slab, no padding"),
    # ---- Cl(3,0), C = 33..63: Cp = 48 or 64
    ("cl3_c40_egcl", 3, 40, ("egcl", 1, 129, 383, "mean"), "TTTT",
     ((0b1101, 48, 16, 64), (0b1101, 48, 16, 64), (0b1111, 48, 16, 64), (0b1101, 48, 16, 64)),
     "f2 streamed, ns2 = 16 at Cp = 48; wide backward with Cp < np = 64, partial 64-channel slab"),
    ("cl3_c33_rows", 3, 33, ("mlp", 7, 129), "TT", ((0b1101, 48, 16, 64),) * 2,
     "f2 streamed, ns2 = 16: the last pass holds one real channel and 15 padded ones"),
    ("cl3_c40_rows_multi", 3, 40, ("mlp", 40, MULTI), "TT", ((0b1101, 48, 16, 64),) * 2,
     "f2 streamed at Cp = 48 over more tiles than SMs: persistent CTAs carry streamed weights across tiles"),
    ("cl3_c63_rows", 3, 63, ("mlp", 63, 255), "TT", ((0b1111, 64, 32, 64),) * 2,
     "f1 / f2 streamed at Cp = 64, ns2 = 32: one padded output channel inside the last streamed pass"),
    # ---- Cl(3,0), Cp rounds to 128 or 256
    ("cl3_c120_egcl", 3, 120, ("egcl", 1, 127, 255, "sum"), "TTTT", ((0b1111, 64, 32, 64),) * 4,
     "streamed passes and weight-gradient slabs at Cp = 128 whose last slab is partly padding"),
    ("cl3_c120_rows_multi", 3, 120, ("mlp", 120, MULTI), "TT", ((0b1111, 64, 32, 64),) * 2,
     "streamed passes at Cp = 128 over more tiles than SMs"),
    ("cl3_c250_rows", 3, 250, ("mlp", 250, 129), "TT", ((0b1111, 64, 32, 64),) * 2,
     "Cp = 256: last streamed pass and last weight-gradient slab partly padding"),
    # ---- Cl(2,0), C = 49..63 and 113..127
    ("cl2_c60_egcl", 2, 60, ("egcl", 3, 43, 43, "sum"), "TTTT",
     ((0b1101, 64, 64, 128), (0b1101, 64, 64, 128), (0b1111, 64, 64, 128), (0b1101, 64, 64, 128)),
     "f2 at the 2 B Cp = 512 TMEM boundary with padding, streamed in one pass; wide backward with Cp < np = 128"),
    ("cl2_c120_rows", 2, 120, ("mlp", 120, 255), "TT", ((0b1111, 128, 64, 128),) * 2,
     "wide Cl(2,0) block at Cp = 128 with padding: streamed f1 / f2, wide backward"),
    # ---- dense CEMLP with a wide input
    ("cl3_cin300_c32", 3, 32, ("mlp", 300, 255), "TT", ((0b1011, 32, 32, 64), (0b1, 32, 32, 0)),
     "n16 > 4 nbw sends a narrow block to the wide backward; f1 streams at Cp = 32"),
    ("cl2_cin520_c16", 2, 16, ("mlp", 520, 129), "TT", ((0b1011, 16, 16, 128), (0b1, 16, 16, 0)),
     "Cl(2,0): n16 > 4 nbw, wide backward and streamed f1 at Cp = 16"),
    # ---- very narrow blocks
    ("cl3_c1_rows", 3, 1, ("mlp", 1, 129), "TT", ((0b1, 16, 16, 0),) * 2,
     "one real channel in a 16-lane Cp, MVLayerNorm over a single channel, kin8 = 8 with 7 zero lanes"),
    ("cl3_c17_rows", 3, 17, ("mlp", 1, 255), "TT", ((0b1, 32, 32, 0),) * 2,
     "one real channel in the second 16-lane group; c_in = 1"),
    ("cl3_c1_egcl", 3, 1, ("egcl", 3, 43, 43, "mean"), "TTTT", ((0b1, 16, 16, 0),) * 4,
     "C = 1 in the gather, BPT-input and residual block modes"),
    # ---- widths the engine rejects: the fallback engine and what the layer then computes
    ("cl3_c96_rows", 3, 96, ("mlp", 96, 129), "UU", (NO,) * 2,
     "Cp = 96 is no slab width; too wide for the SIMT engine: unit kernels"),
    ("cl3_c100_egcl", 3, 100, ("egcl", 3, 43, 43, "sum"), "UUUU", (NO,) * 4,
     "Cp = 112: the whole layer on unit kernels"),
    ("cl2_c65_rows", 2, 65, ("mlp", 65, 255), "SS", (NO,) * 2,
     "Cl(2,0) Cp = 80: the FP32 SIMT engine takes it"),
    ("cl2_c65_egcl", 2, 65, ("egcl", 3, 43, 43, "mean"), "USUS", (NO,) * 4,
     "Cl(2,0) C = 65: the first blocks (71 -> 65, 133 -> 65) fit neither engine and run on unit kernels inside the "
     "unfused layer; the 65 -> 65 blocks still run on the FP32 SIMT engine"),
    ("cl2_c100_rows", 2, 100, ("mlp", 100, 129), "UU", (NO,) * 2,
     "Cl(2,0) Cp = 112: unit kernels"),
]
IDS = [c[0] for c in CASES]
BY_NAME = dict(zip(IDS, CASES))
# the streamed, wide and padded plans (everything on the tensor-core engine but the resident anchors)
TF32_CASES = [c[0] for c in CASES if TC in c[4] and not c[0].endswith("_anchor")]
# one case of each streamed or wide class, and the narrow ones: CEMLPs on plain rows, so the block output is the
# reference-layout tensor a caller owns
GUARD_CASES = [c[0] for c in CASES if c[3][0] == "mlp" and c[4] == "TT"]


def _metric(dim):
    return (1.0,) * dim


def _block_shapes(case):
    name, dim, C, shape = case[:4]
    if shape[0] == "egcl":
        return [(C + 2 * T, C), (C, C), (2 * C + T, C), (C, C)]
    return [(shape[1], C), (C, C)]


# ------------------------------------------------------------------------------------------------ inputs and oracle
@functools.lru_cache(maxsize=None)
def _inputs(name):
    """seeded inputs of a case: parameters (reference state_dict names), leaves, index tensors and the cotangent"""
    _, dim, C, shape = BY_NAME[name][:4]
    gen = torch.Generator().manual_seed(sum(map(ord, name)))
    ralg = R.RefAlgebra(_metric(dim))
    B = ralg.B
    if shape[0] == "egcl":
        _, ncx, n, e, aggr = shape
        params = R.init_egcl_params(ralg, C, T, gen)
        N = ncx * n
        ei = block_diag_graph(ncx, n, e, gen)
        h = torch.randn(N, C, B, generator=gen)
        na = torch.zeros(N, T, B)
        na[..., 0] = torch.randn(T, T, generator=gen)[torch.randint(0, T, (N,), generator=gen)]
        return {"params": params, "leaves": {"h": h, "node_attr": na}, "ei": ei, "aggr": aggr,
                "cot": torch.randn(N, C, B, generator=gen)}
    _, cin, rows = shape
    params = R.init_cemlp_params(ralg, cin, C, C, 2, gen)
    return {"params": params, "leaves": {"x": torch.randn(rows, cin, B, generator=gen)},
            "cot": torch.randn(rows, C, B, generator=gen)}


@functools.lru_cache(maxsize=None)
def _oracle(name, dtype):
    """forward output and every gradient (dict keyed like the result of _ours) of the CPU oracle in dtype"""
    _, dim, C, shape = BY_NAME[name][:4]
    inp = _inputs(name)
    ralg = R.RefAlgebra(_metric(dim))
    leaves = {k: v.to(dtype, copy=True).requires_grad_() for k, v in inp["leaves"].items()}  # the cached inputs stay
    pr = {k: v.to(dtype, copy=True).requires_grad_() for k, v in inp["params"].items()}     # plain tensors
    if shape[0] == "egcl":
        ei, na = inp["ei"], leaves["node_attr"]
        y = R.egcl(ralg, leaves["h"], ei, torch.cat([na[ei[0]], na[ei[1]]], 1), na, pr, aggr=inp["aggr"])
    else:
        y = R.cemlp(ralg, leaves["x"], pr)
    keys = list(leaves) + list(pr)
    g = torch.autograd.grad(y, [leaves[k] for k in leaves] + [pr[k] for k in pr], inp["cot"].to(dtype))
    return y.detach(), dict(zip(keys, (t.detach() for t in g)))


def _model(name):
    _, dim, C, shape = BY_NAME[name][:4]
    params = _inputs(name)["params"]
    if shape[0] == "egcl":
        m = egcl_model(_metric(dim), C, T, shape[4], params)
        return m.algebra, m, list(m.edge_model.layers) + list(m.node_model.layers)
    m = cemlp_model(_metric(dim), shape[1], C, 2, params)
    return m.algebra, m, list(m.layers)


class _BlockCallSpy:
    """Stands in for _lib.lib() inside models/fused.py: every native block call is passed through and recorded with its
    engine (csmpn_block_desc.engine), shape and the kernels it launched (csmpn_launch_count delta).  A forked tensor-core
    backward (stage masks 1, 16, 2|4, 32|64, 8) is one call here."""

    def __init__(self, real):
        self.real, self.fwd, self.bwd = real, [], []

    def __getattr__(self, name):
        return getattr(self.real, name)

    def csmpn_block_fwd(self, dim, dref, stream):
        n0 = self.real.csmpn_launch_count()
        rc = self.real.csmpn_block_fwd(dim, dref, stream)
        d = dref._obj
        self.fwd.append({"engine": int(d.engine), "c_in": d.c0 + d.c1 + d.c2, "c": int(d.c), "rows": int(d.rows),
                         "launches": self.real.csmpn_launch_count() - n0})
        return rc

    def csmpn_block_bwd(self, dim, dref, gref, ws, nbytes, stream):
        n0 = self.real.csmpn_launch_count()
        rc = self.real.csmpn_block_bwd(dim, dref, gref, ws, nbytes, stream)
        d = dref._obj
        n = self.real.csmpn_launch_count() - n0
        if d.stage_mask in (0, 1):
            self.bwd.append({"engine": int(d.engine), "c_in": d.c0 + d.c1 + d.c2, "c": int(d.c), "launches": n})
        else:
            self.bwd[-1]["launches"] += n
        return rc


def _ours(name, monkeypatch):
    """forward + every gradient on the GPU, with the native block calls recorded"""
    from csmpn_b200 import _lib
    from csmpn_b200.models import fused

    _, dim, C, shape = BY_NAME[name][:4]
    inp = _inputs(name)
    alg, m, blocks = _model(name)
    spy = _BlockCallSpy(_lib.lib())
    monkeypatch.setattr(fused, "lib", lambda: spy)
    leaves = {k: v.to(DEV).requires_grad_() for k, v in inp["leaves"].items()}
    pd = dict(m.named_parameters())
    n0 = _lib.lib().csmpn_launch_count()
    if shape[0] == "egcl":
        _, M = mods()
        na = leaves["node_attr"]
        y = m(leaves["h"], inp["ei"].to(DEV), M.PairedNodeAttr(na), na)
    else:
        y = m(leaves["x"])
    keys = list(leaves) + list(inp["params"])
    g = torch.autograd.grad(y, [leaves[k] for k in leaves] + [pd[k] for k in inp["params"]], inp["cot"].to(DEV))
    torch.cuda.synchronize()
    launches = _lib.lib().csmpn_launch_count() - n0
    return alg, blocks, y.detach(), dict(zip(keys, (t.detach() for t in g))), spy, launches


# ------------------------------------------------------------------------------------------------ sliced error check
def _slice_errors(a, ref, dims):
    """max |a - ref| / max |ref| per index of each dim in dims (dim 0 of a row tensor: per 128-row tile)"""
    diff, scale = (a - ref).abs(), ref.abs()
    out = {}
    for dim in dims:
        if dim == "tile":
            pad = (-diff.shape[0]) % 128
            dv = torch.nn.functional.pad(diff.reshape(diff.shape[0], -1), (0, 0, 0, pad)).reshape(-1, 128 * diff[0].numel())
            sv = torch.nn.functional.pad(scale.reshape(scale.shape[0], -1), (0, 0, 0, pad)).reshape(-1, 128 * scale[0].numel())
        else:
            dv = diff.movedim(dim, 0).reshape(diff.shape[dim], -1)
            sv = scale.movedim(dim, 0).reshape(scale.shape[dim], -1)
        out[dim] = dv.amax(1) / (sv.amax(1) + 1e-30)
    return out


def _check(what, got, ref32, ref64, tol, kind=None):
    """Global max-norm error against the fp64 oracle <= tol, and per slice err <= max(tol, 4 x the fp32 oracle's error on
    that slice), each relative to the slice's own fp64 scale.  kind "rows" ([rows, C, B]): per 128-row tile, per channel
    and per blade; kind "weight" ([Cout, Cin, G]): per output channel and per grade; other tensors only globally.
    Returns (global error, worst sliced error, that slice's bound)."""
    got, ref32, ref64 = got.detach().double().cpu(), ref32.double(), ref64.double()
    assert got.shape == ref64.shape, (what, got.shape, ref64.shape)
    e = float((got - ref64).abs().max() / (ref64.abs().max() + 1e-30)) if got.numel() else 0.0
    assert e <= tol, f"{what}: global rel err {e:.3e} > {tol:.1e}"
    names = {"rows": {"tile": "128-row tile", 1: "channel", 2: "blade"},
             "weight": {0: "output channel", 2: "grade"}}.get(kind)
    if names is None or got.numel() == 0:
        return e, e, tol
    ours, fp32 = _slice_errors(got, ref64, names), _slice_errors(ref32, ref64, names)
    worst = (0.0, tol)
    for dim, label in names.items():
        bound = torch.clamp(4 * fp32[dim], min=tol)
        ratio = ours[dim] / bound
        k = int(ratio.argmax())
        assert float(ratio[k]) <= 1.0, (f"{what}: {label} {k}: rel err {float(ours[dim][k]):.3e} > bound "
                                        f"{float(bound[k]):.3e} (fp32 oracle on that slice {float(fp32[dim][k]):.3e})")
        if float(ratio[k]) > worst[0] / worst[1]:
            worst = (float(ours[dim][k]), float(bound[k]))
    return e, worst[0], worst[1]


def _kind(key, t):
    if key in ("x", "h", "node_attr"):
        return "rows"
    return "weight" if t.dim() == 3 and key.endswith("weight") else None


# ------------------------------------------------------------------------------------------------ tests
@pytest.fixture(autouse=True)
def _small_blocks_on_tc(monkeypatch):
    """the default policy keeps blocks with few rows on the SIMT engine; the cases here are small on purpose"""
    monkeypatch.setenv("CSMPN_TC_MIN_ROWS", "0")
    monkeypatch.setenv("CSMPN_TC", "1")


def test_case_table_covers_every_block():
    """the table is consistent with itself: one engine and one plan per block; pass widths divide the padded width,
    a streamed GEMM (bit 1 / 2) is the only way to a narrower pass, and np is set exactly for the wide backward"""
    for name, dim, C, shape, engines, plans, why in CASES:
        assert len(engines) == len(plans) == len(_block_shapes(BY_NAME[name])), name
        for e, (bits, ns1, ns2, np_) in zip(engines, plans):
            assert (bits != 0) == (e == TC), name
            if bits:
                cp = (C + 15) // 16 * 16
                assert cp % ns1 == 0 and cp % ns2 == 0 and (ns1 == cp or bits & 2) and (ns2 == cp or bits & 4), name
                assert (np_ != 0) == bool(bits & 8), name
            else:
                assert (ns1, ns2, np_) == (0, 0, 0), name


@pytest.mark.parametrize("name", IDS)
def test_plan_bits(name):
    """csmpn_block_tc_plan and csmpn_block_tc_passes of every block of the case equal the recorded plan: a plan change
    that moves a case into another class, or to other pass widths, fails here first"""
    from csmpn_b200 import _lib

    L = _lib.lib()
    _, dim, C, shape, engines, plans, why = BY_NAME[name]
    got = []
    for ci, c in _block_shapes(BY_NAME[name]):
        v = L.csmpn_block_tc_passes(dim, ci, c)
        got.append((L.csmpn_block_tc_plan(dim, ci, c), v & 1023, (v >> 10) & 1023, (v >> 20) & 1023))
    print(f"[plan] {name}: blocks {_block_shapes(BY_NAME[name])} (bits, ns1, ns2, np) "
          f"{[(bin(p[0]),) + p[1:] for p in got]} ({why})")
    assert tuple(got) == plans, (name, got, plans)


@pytest.mark.parametrize("name", IDS)
def test_plan_parity_vs_fp64_oracle(name, monkeypatch):
    """forward and every gradient against the fp64 oracle (global and sliced), on the engine each block is expected on"""
    from csmpn_b200.models import fused

    _, dim, C, shape, engines, plans, why = BY_NAME[name]
    alg, blocks, y, g, spy, launches = _ours(name, monkeypatch)
    # the engine each block is routed to ...
    for blk, e, (ci, c) in zip(blocks, engines, _block_shapes(BY_NAME[name])):
        assert (blk[0].in_features, blk[0].out_features) == (ci, c)
        assert fused._block_supported(blk) == (e != UNIT), (name, ci, c)
        if e != UNIT:
            assert fused._block_uses_tc(alg, blk, True, 1 << 30) == (e == TC), (name, ci, c)
            assert fused._fits_fused(dim, ci, c) or e == TC, (name, ci, c)
    # ... and the one it ran on: one native forward and one native backward per fused block, in block order, with two
    # kernels per tensor-core forward plus one weight-image kernel per streamed GEMM
    fused_blocks = [(e, p, s) for e, p, s in zip(engines, plans, _block_shapes(BY_NAME[name])) if e != UNIT]
    assert [(c["engine"], c["c_in"], c["c"]) for c in spy.fwd] == [(int(e == TC), s[0], s[1]) for e, _, s in fused_blocks]
    assert [(c["engine"], c["c_in"], c["c"]) for c in spy.bwd] == [(int(e == TC), s[0], s[1]) for e, _, s in fused_blocks][::-1]
    for c, (e, p, _) in zip(spy.fwd, fused_blocks):
        assert c["launches"] == (2 + bool(p[0] & 2) + bool(p[0] & 4) if e == TC else 1), (name, c)
    in_blocks = sum(c["launches"] for c in spy.fwd + spy.bwd)
    assert launches > in_blocks if UNIT in engines else launches >= in_blocks  # unit-kernel blocks run native kernels
    y32, g32 = _oracle(name, torch.float32)
    y64, g64 = _oracle(name, torch.float64)
    worst = {"fwd": _check(f"{name} fwd", y, y32, y64, FWD_TOL, "rows")}
    for k in g64:
        worst[k] = _check(f"{name} grad {k}", g[k], g32[k], g64[k], GRAD_TOL, _kind(k, g64[k]))
    ws = max((v for k, v in worst.items() if k != "fwd"), key=lambda v: v[1] / v[2])
    print(f"[plans] {name}: plan bits {[bin(p[0]) for p in plans]} engines {engines} "
          f"fwd launches {[c['launches'] for c in spy.fwd]} bwd launches {[c['launches'] for c in spy.bwd]}; "
          f"fwd global {worst['fwd'][0]:.1e} sliced {worst['fwd'][1]:.1e} (bound {worst['fwd'][2]:.1e}); "
          f"worst grad global {max(v[0] for k, v in worst.items() if k != 'fwd'):.1e} "
          f"sliced {ws[1]:.1e} (bound {ws[2]:.1e})")


def _fwd_inference(alg, blk, x, y):
    """csmpn_block_fwd through ctypes as TcBlockFn.forward fills the descriptor under no_grad (no saved tensors), mode 0,
    output in the reference layout written into y"""
    from csmpn_b200 import _lib
    from csmpn_b200.models import fused

    L = _lib.lib()
    dim, rows, c, cin = alg.dim, x.shape[0], blk[0].out_features, x.shape[1]
    params = tuple(None if t is None else t.detach().contiguous() for t in fused._block_params(blk))
    y2 = fused.bpt_empty(dim, rows, c, x.device)
    d = fused._fill_desc(dim, 0, [x, None, None], [cin, 0, 0], rows, c, params, None, y, None, None)
    d.engine, d.in_bpt, d.out_bpt, d.tf32 = 1, 0, 0, 0
    d.save_y2 = y2.data_ptr()
    keep = [y2]
    nws = L.csmpn_block_fwd_workspace(dim, ctypes.byref(d))
    assert nws >= 0
    if nws > 0:
        ws, scratch_o = _lib.workspace(nws, x.device), fused.bpt_empty(dim, rows, c, x.device)
        d.fwd_ws, d.fwd_ws_bytes, d.save_o = ws.data_ptr(), nws, scratch_o.data_ptr()
        keep += [ws, scratch_o]
    _lib.check(L.csmpn_block_fwd(dim, ctypes.byref(d), _lib.stream_ptr(x.device)), "block_fwd (inference)")
    torch.cuda.synchronize()


@pytest.mark.parametrize("name", GUARD_CASES)
def test_forward_output_guard_bands(name):
    """Each block of the CEMLP writes y = rows x C x B into a NaN-filled buffer with one 128-row tile of guard before and
    after it: the guards keep their bits (no write past `rows` from the tail tile, nor before row 0) and y equals the
    autograd path's output bit for bit."""
    from csmpn_b200.models import fused

    alg, m, blocks = _model(name)
    x = _inputs(name)["leaves"]["x"].to(DEV)
    B = alg.n_blades
    for k, blk in enumerate(blocks):
        rows, c = x.shape[0], blk[0].out_features
        assert rows % 128 != 0
        buf = torch.full((rows + 256, c, B), float("nan"), device=DEV)
        nan_bits = buf[:1].view(torch.int32).flatten()[0].item()
        y = buf[128:128 + rows]
        _fwd_inference(alg, blk, x, y)
        ref = fused.block_forward(alg, blk, x.detach().requires_grad_())  # autograd path: TcBlockFn with saved tensors
        torch.cuda.synchronize()
        for where, gband in (("before", buf[:128]), ("after", buf[128 + rows:])):
            assert bool((gband.view(torch.int32) == nan_bits).all()), f"{name} block {k}: guard {where} y overwritten"
        assert torch.equal(y, ref.detach()), f"{name} block {k}: inference output differs from the autograd path"
        x = ref.detach()


@pytest.fixture
def precision():
    """set torch.backends.cuda.matmul.fp32_precision for the test and restore it afterwards"""
    old = torch.backends.cuda.matmul.fp32_precision

    def set_(value):
        torch.backends.cuda.matmul.fp32_precision = value

    yield set_
    torch.backends.cuda.matmul.fp32_precision = old


@pytest.mark.parametrize("name", TF32_CASES)
def test_tf32_plan_vs_fp64_oracle(name, precision, monkeypatch):
    """Single-pass TF32 (halved streamed weight units, one MMA per product) on the streamed, wide and padded plans:
    forward and every gradient within 5e-3 / 2e-2 of the fp64 oracle, as in test_tc_precision.py.  Blocks of width 1 stay
    off the tensor-core engine in this mode (fused.tc_supported): their MVLayerNorm over one channel turns the TF32
    rounding of the GEMM operands into gradient errors up to 2.5e-2, so they run on the FP32 SIMT engine instead."""
    _, dim, C, shape, engines, plans, why = BY_NAME[name]
    res = {}
    for mode in ("ieee", "tf32"):
        precision(mode)
        res[mode] = _ours(name, monkeypatch)
    want = int(C > 1)  # engine of every block in TF32 mode: 1 tensor-core, 0 FP32 SIMT
    spy = res["tf32"][4]
    assert [c["engine"] for c in spy.fwd] == [want] * len(engines), (name, spy.fwd)
    assert [c["engine"] for c in spy.bwd] == [want] * len(engines), (name, spy.bwd)
    assert all(c["engine"] == 1 for c in res["ieee"][4].fwd)
    y64, g64 = _oracle(name, torch.float64)
    rel = lambda a, b: float((a.detach().double().cpu() - b).abs().max() / (b.abs().max() + 1e-30))
    y, g = res["tf32"][2:4]
    e_fwd = rel(y, y64)
    e_grad = {k: rel(g[k], g64[k]) for k in g64}
    worst = max(e_grad, key=e_grad.get)
    print(f"[plans tf32] {name}: engine {'tensor-core' if want else 'fp32 simt'}, fp64-oracle error fwd {e_fwd:.2e}, "
          f"worst grad {worst} {e_grad[worst]:.2e}")
    assert e_fwd <= TF32_FWD_TOL and e_grad[worst] <= TF32_GRAD_TOL, (name, e_fwd, worst, e_grad[worst])
    if want:
        assert not torch.equal(y, res["ieee"][2])  # the TF32 path is really taken
    else:  # the SIMT engine computes in fp32 whatever the setting: north-star tolerances
        assert e_fwd <= FWD_TOL and e_grad[worst] <= GRAD_TOL, (name, e_fwd, e_grad[worst])
