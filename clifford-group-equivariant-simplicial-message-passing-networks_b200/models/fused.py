"""Fused CEMLP-block / EGCL path: Python side of csrc/block_fused.cu (C ABI: csmpn_block_fwd / csmpn_block_bwd).

One autograd node per CEMLP block.  The EGCL layer becomes

    block(gather: h[dst]-h[src] | edge_attr)  ->  block(dense)  ->  CSR segment reduce (contiguous rows)
    block(concat: h | agg | node_attr)        ->  block(dense, + residual)

with every per-pair tensor kept in receiver-sorted order so the reduce reads contiguous rows and is
deterministic.  Enabled for Euclidean algebras of dimension 2, 3 and 5 (the reference's models); other
algebras use the unit kernels.  ``CSMPN_FUSED=0`` forces the unit-kernel composition (used by tests to
cross-check the two paths).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_float, c_int32, c_int64, c_void_p

import torch

from .. import _lib
from .._lib import check, f32c, lib, ptr, require_cuda, stream_ptr, workspace
from . import ops


class BlockDesc(ctypes.Structure):
    _fields_ = [
        ("mode", c_int32), ("c0", c_int32), ("c1", c_int32), ("c2", c_int32), ("c", c_int32), ("has_b1", c_int32),
        ("rows", c_int64),
        ("p0", c_void_p), ("p1", c_void_p), ("p2", c_void_p),
        ("src", c_void_p), ("dst", c_void_p), ("eid", c_void_p),
        ("w1", c_void_p), ("b1", c_void_p), ("sa", c_void_p), ("sb", c_void_p), ("wr", c_void_p), ("na", c_void_p),
        ("wl", c_void_p), ("bl", c_void_p), ("wp", c_void_p), ("la", c_void_p),
        ("y", c_void_p), ("res", c_void_p), ("save_y1", c_void_p), ("save_xr", c_void_p), ("save_o", c_void_p),
        ("engine", c_int32), ("in_bpt", c_int32), ("out_bpt", c_int32), ("stage_mask", c_int32),
        ("save_y2", c_void_p), ("save_x0", c_void_p),
        ("pair_attr", c_int32),
        ("vt_k", c_int32), ("vt_fp", c_int32),
        ("fwd_ws", c_void_p), ("fwd_ws_bytes", c_int64),
        ("tf32", c_int32),
    ]


class BlockGrads(ctypes.Structure):
    _fields_ = [
        ("grad_y", c_void_p), ("grad_x", c_void_p),
        ("g_w1", c_void_p), ("g_b1", c_void_p), ("g_sa", c_void_p), ("g_sb", c_void_p), ("g_wr", c_void_p),
        ("g_na", c_void_p), ("g_wl", c_void_p), ("g_bl", c_void_p), ("g_wp", c_void_p), ("g_la", c_void_p),
        ("gy_bpt", c_int32), ("gx_bpt", c_int32),
        ("gy_rows", c_void_p), ("gy_row_stride", ctypes.c_int64),
    ]


def _declare():
    """All C entry points are declared in _lib._declare; loading the library is all that is left to do."""
    lib()


FUSED_DIMS = (2, 3, 5)

# bench.py's per-kernel timing: when a list is bound here, every block call appends (kind, dim, descriptor copies and the
# tensors they point to); bench_layer_kernels() then replays each recorded call one kernel at a time (stage_mask)
_RECORDER = None


def _record(kind, dim, d, g=None, ws=None, keep=()):
    if _RECORDER is not None:
        _RECORDER.append({"kind": kind, "dim": dim, "desc": BlockDesc.from_buffer_copy(d),
                          "grads": None if g is None else BlockGrads.from_buffer_copy(g), "ws": ws, "keep": list(keep)})


def tc_enabled() -> bool:
    """Tensor-core (tcgen05) engine switch: CSMPN_TC=0 forces the FP32 SIMT kernels (tests cross-check the two)."""
    return os.environ.get("CSMPN_TC", "1") != "0"


def tc_precision() -> bool:
    """True when the tensor-core engine runs its channel GEMMs in single-pass TF32 (csmpn_block_desc.tf32): PyTorch's
    float32 matmul precision for CUDA is "tf32", i.e. ``torch.backends.cuda.matmul.fp32_precision == "tf32"``.  That
    is what ``torch.set_float32_matmul_precision("high")`` / ``("medium")``, ``torch.backends.cuda.matmul.allow_tf32 =
    True`` and ``torch.backends.fp32_precision = "tf32"`` select, and what makes the reference's einsum linears run in
    TF32.  Any other value keeps the default error-compensated fp32 products.  The attribute is read directly:
    ``torch.get_float32_matmul_precision()`` and ``allow_tf32`` raise once a program has mixed the legacy and the new API.
    Only the tensor-core engine follows the setting; the FP32 SIMT engine and the unit kernels always compute in fp32."""
    return torch.backends.cuda.matmul.fp32_precision == "tf32"


def tc_supported(dim: int, c_in: int, c: int) -> bool:
    return tc_enabled() and bool(lib().csmpn_block_tc_supported(dim, c_in, c))


def bpt_empty(dim: int, rows: int, channels: int, device, zero: bool = False) -> torch.Tensor:
    """A blade-plane tile tensor [ceil(rows/128), B, cp/4, 128, 4] (include/csmpn_b200.h, engine 1)."""
    cp = (channels + 15) // 16 * 16
    shape = ((rows + 127) // 128, 1 << dim, cp // 4, 128, 4)
    return (torch.zeros if zero else torch.empty)(shape, dtype=torch.float32, device=device)


def available() -> bool:
    try:
        _declare()
        return True
    except Exception:
        return False


def enabled(algebra) -> bool:
    if os.environ.get("CSMPN_FUSED", "1") == "0":
        return False
    return bool(getattr(algebra, "is_euclidean", False)) and algebra.dim in FUSED_DIMS


def _block_supported(layer) -> bool:
    from .cegnn_utils import MVLayerNorm, MVLinear, MVSiLU, NormalizationLayer, SteerableGeometricProductLayer

    if len(layer) != 4:
        return False
    lin, act, sgp, ln = layer[0], layer[1], layer[2], layer[3]
    if not (isinstance(lin, MVLinear) and lin.subspaces and isinstance(act, MVSiLU) and act.invariant == "mag2"
            and isinstance(sgp, SteerableGeometricProductLayer) and sgp.include_first_order
            and isinstance(sgp.normalization, NormalizationLayer) and isinstance(ln, MVLayerNorm)
            and lin.out_features <= 256):
        return False
    # wide blocks whose weights leave room for fewer than 4 rows per shared-memory tile of the SIMT engine run on the
    # tensor-core engine with streamed weights (csmpn_block_tc_plan); what neither engine takes is composed from unit kernels
    dim = lin.algebra.dim
    return _fits_fused(dim, lin.in_features, lin.out_features) or (dim in (2, 3) and tc_supported(dim, lin.in_features, lin.out_features))


_FITS: dict = {}


def _fits_fused(dim: int, c_in: int, c: int) -> bool:
    key = (dim, c_in, c)
    if key not in _FITS:
        _FITS[key] = lib().csmpn_block_simt_resident(dim, c_in, c) >= 4  # rows per shared-memory tile
    return _FITS[key]


def _block_params(layer):
    lin, act, sgp, ln = layer[0], layer[1], layer[2], layer[3]
    return (lin.weight, lin.bias, act.a, act.b, sgp.linear_right.weight, sgp.normalization.a, sgp.linear_left.weight,
            sgp.linear_left.bias, sgp.weight, ln.a)


class SortedGraph:
    """Receiver-sorted int32 views of a CSRGraph for the fused kernels (built once per batch)."""

    def __init__(self, g: ops.CSRGraph):
        _declare()
        self.csr = g
        dev = g.edge_index.device
        E = g.n_pairs
        self.src_sorted = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        self.dst_sorted = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        self.rank = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        self.refresh_()

    def refresh_(self):
        """(re)compute the sorted views in place from the CSR (CSRGraph.rebuild_ calls this)"""
        g = self.csr
        E = g.n_pairs
        s = stream_ptr(g.edge_index.device)
        check(lib().csmpn_csr_sorted_indices(ptr(g.src), ptr(g.dst), ptr(g.perm_dst), ptr(self.src_sorted),
                                             ptr(self.dst_sorted), E, s), "csr_sorted_indices")
        check(lib().csmpn_csr_rank(ptr(g.perm_dst), ptr(self.rank), E, s), "csr_rank")


def sorted_graph(g: ops.CSRGraph) -> SortedGraph:
    sg = getattr(g, "_sorted", None)
    if sg is None:
        sg = SortedGraph(g)
        g._sorted = sg
    return sg


def _fill_desc(dim, mode, srcs, chans, rows, c, params, sgraph, y, res, saves, pair_attr=False):
    w1, b1, sa, sb, wr, na, wl, bl, wp, la = params
    d = BlockDesc()
    d.pair_attr = int(bool(pair_attr))
    d.mode, d.c0, d.c1, d.c2, d.c = mode, chans[0], chans[1], chans[2], c
    d.has_b1 = int(b1 is not None)
    d.rows = rows
    d.p0, d.p1, d.p2 = (None if t is None else t.data_ptr() for t in srcs)
    if mode == 1:
        d.src, d.dst = sgraph.src_sorted.data_ptr(), sgraph.dst_sorted.data_ptr()
        d.eid = sgraph.csr.perm_dst.data_ptr()
    d.w1, d.sa, d.sb, d.wr, d.na = w1.data_ptr(), sa.data_ptr(), sb.data_ptr(), wr.data_ptr(), na.data_ptr()
    d.b1 = None if b1 is None else b1.data_ptr()
    d.wl, d.bl, d.wp, d.la = wl.data_ptr(), bl.data_ptr(), wp.data_ptr(), la.data_ptr()
    d.y = y.data_ptr()
    d.res = None if res is None else res.data_ptr()
    if saves is not None:
        d.save_y1, d.save_xr, d.save_o = (t.data_ptr() for t in saves)
    return d


class FusedBlockFn(torch.autograd.Function):
    """One CEMLP block.  inputs: p0, p1, p2 (sources), res, then the ten parameters."""

    @staticmethod
    def forward(ctx, cfg, p0, p1, p2, res, w1, b1, sa, sb, wr, na, wl, bl, wp, la):
        _declare()
        dim, mode, sgraph = cfg["dim"], cfg["mode"], cfg.get("sgraph")
        srcs = [None if t is None else f32c(t) for t in (p0, p1, p2)]
        require_cuda(*srcs, what="fused block")
        B = 1 << dim
        chans = [0 if t is None else t.shape[1] for t in srcs]
        pair = bool(cfg.get("pair_attr"))
        if pair:
            chans[1] *= 2  # p1 is the per-simplex table: every pair sees table[src] | table[dst]
        c = w1.shape[0]
        if sum(chans) != w1.shape[1]:
            raise ValueError(f"fused block: input channels {chans} do not match weight {tuple(w1.shape)}")
        rows = sgraph.csr.n_pairs if mode == 1 else srcs[0].shape[0]
        params = tuple(None if t is None else f32c(t) for t in (w1, b1, sa, sb, wr, na, wl, bl, wp, la))
        dev = srcs[0].device
        y = torch.empty((rows, c, B), dtype=torch.float32, device=dev)
        need_grad = cfg["need_grad"]
        saves = tuple(torch.empty((rows, c, B), dtype=torch.float32, device=dev) for _ in range(3)) if need_grad else None
        resc = None if res is None else f32c(res)
        d = _fill_desc(dim, mode, srcs, chans, rows, c, params, sgraph, y, resc, saves, pair)
        check(lib().csmpn_block_fwd(dim, ctypes.byref(d), stream_ptr(dev)), "block_fwd")
        _record("fwd", dim, d, keep=[srcs, params, y, resc, saves])
        if need_grad:
            ctx.save_for_backward(*[t for t in srcs if t is not None], *[t for t in params if t is not None], *saves)
            ctx.meta = (dim, mode, sgraph, chans, c, rows, [t is not None for t in srcs], [t is not None for t in params],
                        res is not None, [None if t is None else t.shape for t in (w1, b1, sa, sb, wr, na, wl, bl, wp, la)],
                        [None if t is None else t.shape for t in (p0, p1, p2)], pair)
        return y

    @staticmethod
    def backward(ctx, gy):
        dim, mode, sgraph, chans, c, rows, src_mask, par_mask, has_res, pshapes, sshapes, pair = ctx.meta
        saved = list(ctx.saved_tensors)
        srcs = [saved.pop(0) if m else None for m in src_mask]
        params = [saved.pop(0) if m else None for m in par_mask]
        saves = tuple(saved)
        gy = f32c(gy)
        dev = gy.device
        B = 1 << dim
        cin = sum(chans)
        y_dummy = gy  # desc.y is not written by the backward
        d = _fill_desc(dim, mode, srcs, chans, rows, c, params, sgraph, y_dummy, None, saves, pair)
        gx = torch.empty((rows, cin, B), dtype=torch.float32, device=dev)
        pg = [None if t is None else torch.empty_like(t) for t in params]
        g = BlockGrads()
        g.grad_y, g.grad_x = gy.data_ptr(), gx.data_ptr()
        names = ("g_w1", "g_b1", "g_sa", "g_sb", "g_wr", "g_na", "g_wl", "g_bl", "g_wp", "g_la")
        for n, t in zip(names, pg):
            setattr(g, n, None if t is None else t.data_ptr())
        nbytes = lib().csmpn_block_bwd_workspace(dim, ctypes.byref(d))
        if nbytes < 0:
            raise _lib.CsmpnError("fused block backward: unsupported configuration")
        ws = workspace(nbytes, dev)
        check(lib().csmpn_block_bwd(dim, ctypes.byref(d), ctypes.byref(g), ptr(ws), ws.numel(), stream_ptr(dev)), "block_bwd")
        _record("bwd", dim, d, g, ws, keep=[srcs, params, saves, gy, gx, pg])
        # split the gradient of the assembled input row back onto the sources
        gsrc = [None, None, None]
        if mode == 0:
            off = 0
            for k in range(3):
                if srcs[k] is not None:
                    gsrc[k] = gx[:, off:off + chans[k]] if (chans[k] != cin) else gx
                    off += chans[k]
        else:
            csr = sgraph.csr
            n_nodes, width = srcs[0].shape[0], chans[0] * B
            gh = torch.empty((n_nodes, chans[0], B), dtype=torch.float32, device=dev)
            check(lib().csmpn_scatter_diff_sorted(ptr(gx), cin * B, ptr(csr.rowptr_dst), ptr(csr.rowptr_src), ptr(csr.perm_src),
                                                  ptr(sgraph.rank), ptr(gh), n_nodes, width, 0, stream_ptr(dev)),
                  "scatter_diff_sorted")
            gsrc[0] = gh
            if srcs[1] is not None and ctx.needs_input_grad[2]:
                gsrc[1] = _extra_channel_grad(gx, cin, chans, B, sgraph, srcs[1], rows, pair, dev)
        gsrc = [None if t is None else t.reshape(s) for t, s in zip(gsrc, sshapes)]
        gres = gy if has_res else None
        pgr = [None if t is None else t.reshape(s) for t, s in zip(pg, pshapes)]
        return (None, gsrc[0], gsrc[1], gsrc[2], gres, *pgr)


def _extra_channel_grad(gx, cin, chans, B, sgraph, p1, rows, pair, dev):
    """gradient of the gathered extra channels of a mode-1 block: per pair in the original pair order (edge_attr), or --
    pair_attr -- summed onto the per-simplex table that entered every pair as table[src] | table[dst]"""
    csr = sgraph.csr
    if pair:
        half = chans[1] // 2
        gt = torch.empty((p1.shape[0], half, B), dtype=torch.float32, device=dev)
        check(lib().csmpn_scatter_pair_sorted(ptr(gx), cin * B, chans[0] * B, (chans[0] + half) * B, ptr(csr.rowptr_dst),
                                              ptr(csr.rowptr_src), ptr(csr.perm_src), ptr(sgraph.rank), ptr(gt), p1.shape[0],
                                              half * B, stream_ptr(dev)), "scatter_pair_sorted")
        return gt
    ge = torch.empty((rows, chans[1], B), dtype=torch.float32, device=dev)
    check(lib().csmpn_scatter_rows(ptr(gx), cin * B, chans[0] * B, ptr(csr.perm_dst), ptr(ge), rows, chans[1] * B,
                                   stream_ptr(dev)), "scatter_rows")
    return ge


class TcBlockFn(torch.autograd.Function):
    """One CEMLP block on the tensor-core engine (csrc/tc_block_fwd.cu, tc_block_bwd.cu).

    cfg: dim, mode, sgraph, rows, in_bpt (p0 is a BPT tensor with cfg["c_in"] channels), out_bpt, need_grad.
    Intermediates and saved tensors are BPT (blade-plane tile) tensors; only the block boundary facing the rest of the
    model (gathered h / edge_attr, the messages, the layer output and the residual) is in the reference layout.

    Numeric mode: the forward reads tc_precision() once and its backward runs in the same mode, even if the setting
    changes in between.  A captured CUDA graph (GraphedEGCL, GraphedLayerStep, the train-step graphs) keeps the mode that
    was set at capture time, like every other descriptor field."""

    @staticmethod
    def forward(ctx, cfg, p0, p1, p2, res, w1, b1, sa, sb, wr, na, wl, bl, wp, la):
        _declare()
        dim, mode, sgraph = cfg["dim"], cfg["mode"], cfg.get("sgraph")
        in_bpt, out_bpt = bool(cfg.get("in_bpt")), bool(cfg.get("out_bpt"))
        srcs = [None if t is None else f32c(t) for t in (p0, p1, p2)]
        require_cuda(*srcs, what="tensor-core block")
        B = 1 << dim
        chans = [cfg["c_in"], 0, 0] if in_bpt else [0 if t is None else t.shape[1] for t in srcs]
        pair = bool(cfg.get("pair_attr")) and not in_bpt
        if pair:
            chans[1] *= 2  # p1 is the per-simplex table: every pair sees table[src] | table[dst]
        vt = cfg.get("vertex_table") if mode == 2 else None  # (vertex ids int32 [rows, k], channels per (type, vertex))
        if vt is not None:
            chans = [srcs[0].shape[1] * vt[0].shape[1], 0, 0]  # p0 is the per-vertex table [V, types * fp, B]
        c = w1.shape[0]
        cin = sum(chans)
        if cin != w1.shape[1]:
            raise ValueError(f"tensor-core block: input channels {chans} do not match weight {tuple(w1.shape)}")
        rows = cfg["rows"] if in_bpt else (sgraph.csr.n_pairs if mode == 1 else (vt[0].shape[0] if vt is not None else srcs[0].shape[0]))
        params = tuple(None if t is None else f32c(t) for t in (w1, b1, sa, sb, wr, na, wl, bl, wp, la))
        dev = srcs[0].device
        y = bpt_empty(dim, rows, c, dev) if out_bpt else torch.empty((rows, c, B), dtype=torch.float32, device=dev)
        need_grad = cfg["need_grad"]
        y2 = bpt_empty(dim, rows, c, dev)
        saves = tuple(bpt_empty(dim, rows, c, dev) for _ in range(3)) if need_grad else None
        x0 = bpt_empty(dim, rows, cin, dev) if (need_grad and not in_bpt) else None
        resc = None if res is None else f32c(res)
        d = _fill_desc(dim, mode, srcs, chans, rows, c, params, sgraph, y, resc, saves, pair)
        d.engine, d.in_bpt, d.out_bpt = 1, int(in_bpt), int(out_bpt)
        d.tf32 = ctx.tf32 = int(tc_precision())
        d.save_y2 = y2.data_ptr()
        d.save_x0 = None if x0 is None else x0.data_ptr()
        if vt is not None:
            d.src, d.vt_k, d.vt_fp = vt[0].data_ptr(), vt[0].shape[1], vt[1]
        nws = lib().csmpn_block_fwd_workspace(dim, ctypes.byref(d))
        if nws < 0:
            raise _lib.CsmpnError("tensor-core block forward: unsupported configuration")
        wsf = scratch_o = None
        if nws > 0:  # wide block: pre-split weight images streamed with the K chunks
            wsf = workspace(nws, dev)
            d.fwd_ws, d.fwd_ws_bytes = wsf.data_ptr(), nws
            if saves is None:  # the scaling pass of the second kernel re-reads the product sum from this tensor
                scratch_o = bpt_empty(dim, rows, c, dev)
                d.save_o = scratch_o.data_ptr()
        check(lib().csmpn_block_fwd(dim, ctypes.byref(d), stream_ptr(dev)), "block_fwd (tensor-core)")
        _record("fwd", dim, d, keep=[srcs, params, y, resc, saves, y2, x0, wsf, scratch_o])
        red = cfg.get("reduce")   # (SortedGraph, mean): return the per-receiver aggregate of the rows instead of the rows
        if red is not None:
            csr = red[0].csr
            agg = torch.empty((csr.n_nodes, c, B), dtype=torch.float32, device=dev)
            check(lib().csmpn_segment_reduce_sorted(ptr(y), ptr(csr.rowptr_dst), ptr(agg), csr.n_nodes, c * B, int(red[1]),
                                                    stream_ptr(dev)), "segment_reduce_sorted")
            ctx.reduce = red
            y = agg
        else:
            ctx.reduce = None
        if need_grad:
            ctx.save_for_backward(*[t for t in srcs if t is not None], *[t for t in params if t is not None], *saves, y2,
                                  *([] if x0 is None else [x0]))
            ctx.meta = (dim, mode, sgraph, chans, c, rows, [t is not None for t in srcs], [t is not None for t in params],
                        res is not None, [None if t is None else t.shape for t in (w1, b1, sa, sb, wr, na, wl, bl, wp, la)],
                        [None if t is None else t.shape for t in (p0, p1, p2)], in_bpt, out_bpt, x0 is not None, pair, vt)
        return y

    @staticmethod
    def backward(ctx, gy):
        return _tc_block_backward(ctx, gy)


def _tc_block_backward(ctx, gy):
    (dim, mode, sgraph, chans, c, rows, src_mask, par_mask, has_res, pshapes, sshapes, in_bpt, out_bpt, has_x0, pair, vt) = ctx.meta
    saved = list(ctx.saved_tensors)
    srcs = [saved.pop(0) if m else None for m in src_mask]
    params = [saved.pop(0) if m else None for m in par_mask]
    y1, xr, o, y2 = saved[:4]
    x0 = saved[4] if has_x0 else None
    B = 1 << dim
    red = getattr(ctx, "reduce", None)
    gy_rows, gy_stride = None, 0
    if red is not None:
        # gy is the cotangent of the AGGREGATE [n_nodes, c, B]: row r of the block reads row dst_sorted[r] of it (the adjoint
        # of the segment sum folded into the first backward kernel; no [pairs, c, B] expansion).  A channel slice of a
        # wider gradient (the update block hands back grad_x[:, c:2c]) is read in place through its row pitch.
        rsg, mean = red
        if mean:
            deg = (rsg.csr.rowptr_dst[1:] - rsg.csr.rowptr_dst[:-1]).clamp(min=1).to(torch.float32)
            gy = gy.to(torch.float32) / deg.reshape(-1, 1, 1)
        if not (gy.dtype == torch.float32 and gy.dim() == 3 and gy.stride(2) == 1 and gy.stride(1) == B
                and gy.stride(0) % 4 == 0 and gy.data_ptr() % 16 == 0):
            gy = f32c(gy)
        gy_rows, gy_stride = rsg.dst_sorted, int(gy.stride(0))
    else:
        gy = f32c(gy)
    dev = gy.device
    cin = sum(chans)
    d = _fill_desc(dim, mode, srcs, chans, rows, c, params, sgraph, gy, None, (y1, xr, o), pair)
    d.engine, d.in_bpt, d.out_bpt = 1, int(in_bpt), int(out_bpt)
    d.tf32 = ctx.tf32  # the mode of the forward
    d.save_y2 = y2.data_ptr()
    d.save_x0 = None if x0 is None else x0.data_ptr()
    if vt is not None:
        if ctx.needs_input_grad[1]:
            raise _lib.CsmpnError("the vertex-table gather (mode 2) has no gradient w.r.t. the table: its rows are input data")
        d.src, d.vt_k, d.vt_fp = vt[0].data_ptr(), vt[0].shape[1], vt[1]
        gx = None  # no grad_x GEMM at all
    else:
        gx = bpt_empty(dim, rows, cin, dev) if in_bpt else torch.empty((rows, cin, B), dtype=torch.float32, device=dev)
    pg = [None if t is None else torch.empty_like(t) for t in params]
    g = BlockGrads()
    g.grad_y, g.grad_x = gy.data_ptr(), None if gx is None else gx.data_ptr()
    g.gy_bpt, g.gx_bpt = int(out_bpt), int(in_bpt)
    if gy_rows is not None:
        g.gy_rows, g.gy_row_stride = gy_rows.data_ptr(), gy_stride
    names = ("g_w1", "g_b1", "g_sa", "g_sb", "g_wr", "g_na", "g_wl", "g_bl", "g_wp", "g_la")
    for n, t in zip(names, pg):
        setattr(g, n, None if t is None else t.data_ptr())
    nbytes = lib().csmpn_block_bwd_workspace(dim, ctypes.byref(d))
    if nbytes < 0:
        raise _lib.CsmpnError("tensor-core block backward: unsupported configuration")
    ws = workspace(nbytes, dev)
    _record("bwd", dim, d, g, ws, keep=[srcs, params, y1, xr, o, y2, x0, gy, gx, pg])
    if _fork_enabled():
        _tc_backward_forked(dim, d, g, ws, dev)
    else:
        check(lib().csmpn_block_bwd(dim, ctypes.byref(d), ctypes.byref(g), ptr(ws), ws.numel(), stream_ptr(dev)),
              "block_bwd (tensor-core)")
    gsrc = [None, None, None]
    if vt is not None:
        pass
    elif in_bpt:
        gsrc[0] = gx
    elif mode == 0:
        off = 0
        for k in range(3):
            if srcs[k] is not None:
                gsrc[k] = gx[:, off:off + chans[k]] if (chans[k] != cin) else gx
                off += chans[k]
    else:
        csr = sgraph.csr
        n_nodes, width = srcs[0].shape[0], chans[0] * B
        gh = torch.empty((n_nodes, chans[0], B), dtype=torch.float32, device=dev)
        check(lib().csmpn_scatter_diff_sorted(ptr(gx), cin * B, ptr(csr.rowptr_dst), ptr(csr.rowptr_src), ptr(csr.perm_src),
                                              ptr(sgraph.rank), ptr(gh), n_nodes, width, 0, stream_ptr(dev)),
              "scatter_diff_sorted")
        gsrc[0] = gh
        if srcs[1] is not None and ctx.needs_input_grad[2]:
            gsrc[1] = _extra_channel_grad(gx, cin, chans, B, sgraph, srcs[1], rows, pair, dev)
    if not in_bpt and vt is None:
        gsrc = [None if t is None else t.reshape(s) for t, s in zip(gsrc, sshapes)]
    gres = gy if has_res else None
    pgr = [None if t is None else t.reshape(s) for t, s in zip(pg, pshapes)]
    return (None, gsrc[0], gsrc[1], gsrc[2], gres, *pgr)


_SIDE_STREAMS: dict = {}


def _fork_enabled() -> bool:
    return os.environ.get("CSMPN_TC_FORK", "1") != "0"


def _tc_backward_forked(dim, d, g, ws, dev):
    """csmpn_block_bwd (engine 1) as two concurrent chains, joined before returning:
         main:  b1 -> gemm(dy2) -> b3 -> gemm(grad_x)
         side:        dW(wl, wr) [after b1] -> dW(w1) [after b3] -> final reduce
    Every block forks, whatever its row count.  Measured on B200 (layer step, CUDA-graph replay): md17 1.63 -> 1.50 ms with
    the node blocks (69 tiles, each kernel fills half the GPU) on the tensor-core engine, and still 1.51 -> 1.48 ms from
    forking the per-pair blocks alone, whose persistent kernels leave SMs idle in their last wave (2.85 tiles per SM)."""
    main = torch.cuda.current_stream(dev)
    side = _SIDE_STREAMS.get(dev)
    if side is None:
        side = _SIDE_STREAMS[dev] = torch.cuda.Stream(dev)

    def run(mask, stream):
        d.stage_mask = mask
        check(lib().csmpn_block_bwd(dim, ctypes.byref(d), ctypes.byref(g), ptr(ws), ws.numel(), c_void_p(stream.cuda_stream)),
              "block_bwd (tensor-core, forked)")

    side.wait_stream(main)          # workspace and saved tensors were produced on the main stream
    run(1, main)
    e1 = torch.cuda.Event()
    e1.record(main)
    side.wait_event(e1)
    run(16, side)
    run(2 | 4, main)
    e2 = torch.cuda.Event()
    e2.record(main)
    side.wait_event(e2)
    run(32 | 64, side)
    run(8, main)
    main.wait_stream(side)
    d.stage_mask = 0


class SegmentReduceSortedFn(torch.autograd.Function):
    """[E_sorted, W] -> [N, W]; rows of a receiver are contiguous (deterministic, fixed order)."""

    @staticmethod
    def forward(ctx, msg, sgraph: SortedGraph, mean: bool):
        _declare()
        msg = f32c(msg)
        csr = sgraph.csr
        out = torch.empty((csr.n_nodes, msg.shape[1]), dtype=torch.float32, device=msg.device)
        check(lib().csmpn_segment_reduce_sorted(ptr(msg), ptr(csr.rowptr_dst), ptr(out), csr.n_nodes, msg.shape[1], int(mean),
                                                stream_ptr(msg.device)), "segment_reduce_sorted")
        ctx.sgraph, ctx.mean = sgraph, mean
        return out

    @staticmethod
    def backward(ctx, go):
        go = f32c(go)
        sg = ctx.sgraph
        gm = torch.empty((sg.csr.n_pairs, go.shape[1]), dtype=torch.float32, device=go.device)
        check(lib().csmpn_segment_expand_sorted(ptr(go), ptr(sg.dst_sorted), ptr(sg.csr.rowptr_dst), ptr(gm), sg.csr.n_pairs,
                                                go.shape[1], int(ctx.mean), stream_ptr(go.device)), "segment_expand_sorted")
        return gm, None, None


class FanoutFn(torch.autograd.Function):
    """h -> (h, h, h) for the three uses of the layer input in EGCL.forward (gather source of the messages, first source of
    the update, residual); the backward sums the three gradient contributions in ONE kernel (csmpn_add3_rows) instead of
    two autograd adds plus a copy of the strided slice."""

    @staticmethod
    def forward(ctx, h):
        return h.view_as(h), h.view_as(h), h.view_as(h)

    @staticmethod
    def backward(ctx, g1, g2, g3):
        gs = [g for g in (g1, g2, g3) if g is not None]
        if len(gs) == 3 and all(g.dim() == 3 and g.dtype == torch.float32 and g.stride(2) == 1 and g.stride(1) == g.shape[2]
                                and g.stride(0) % 4 == 0 and g.data_ptr() % 16 == 0 for g in gs):
            n, width = g1.shape[0], g1.shape[1] * g1.shape[2]
            out = torch.empty(g1.shape, dtype=torch.float32, device=g1.device)
            check(lib().csmpn_add3_rows(ptr(g1), g1.stride(0), ptr(g2), g2.stride(0), ptr(g3), g3.stride(0), ptr(out), n, width,
                                        stream_ptr(g1.device)), "add3_rows")
            return out
        if not gs:
            return None
        tot = gs[0]
        for g in gs[1:]:
            tot = tot + g
        return tot


def _need_grad(*tensors_and_params):
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors_and_params)


def tc_min_rows() -> int:
    """Rows below which a block stays on the FP32 SIMT engine: the tensor-core engine runs a block as several
    persistent kernels over 128-row tiles, each paying its prologue once per CTA.  With the batched weight staging
    (tc_block.cuh) the cross-over is near 32 tiles: motion-shaped batch, 4 700 simplices = 37 tiles per node block:
    0.796 ms with tensor-core node blocks vs 0.814 ms with SIMT ones (r01 prologues: 0.966 vs 0.935 ms)."""
    return int(os.environ.get("CSMPN_TC_MIN_ROWS", "4096"))  # 32 tiles; see DESIGN.md 4.4 for the measurements behind it


def _block_uses_tc(algebra, layer, need_grad, rows=None) -> bool:
    lin = layer[0]
    if algebra.dim not in (2, 3):
        return False
    if not tc_supported(algebra.dim, lin.in_features, lin.out_features):
        return False
    if not _fits_fused(algebra.dim, lin.in_features, lin.out_features):
        return True  # wide block: the SIMT engine cannot hold it, whatever the row count
    return rows is None or rows >= tc_min_rows()


def block_forward(algebra, layer, x, p1=None, p2=None, res=None, mode=0, sgraph=None, bpt_rows=None, out_bpt=False,
                  pair_attr=False, reduce=None):
    """Run one CEMLP block (nn.Sequential of the four sub-layers) through the fused kernels.

    bpt_rows: x is a BPT tensor (output of a previous tensor-core block) holding that many rows.
    out_bpt:  return a BPT tensor (only honoured on the tensor-core engine; the caller checks with is_bpt)."""
    in_bpt = bpt_rows is not None
    if not in_bpt and (not _block_supported(layer) or (x is not None and x.dim() != 3)):
        if reduce is not None:
            raise ValueError("block_forward(reduce=...) needs a block the fused kernels support")
        y = x if p1 is None else torch.cat([t for t in (x, p1, p2) if t is not None], dim=1)
        y = layer(y)
        return y if res is None else res + y
    params = _block_params(layer)
    need_grad = _need_grad(x, p1, p2, res, *params)
    cfg = {"dim": algebra.dim, "mode": mode, "sgraph": sgraph, "need_grad": need_grad, "pair_attr": pair_attr}
    rows_now = bpt_rows if in_bpt else (sgraph.csr.n_pairs if mode == 1 else x.shape[0])
    if in_bpt or _block_uses_tc(algebra, layer, need_grad, rows_now):
        cfg.update(in_bpt=in_bpt, out_bpt=out_bpt, rows=bpt_rows, c_in=layer[0].in_features)
        if reduce is not None and not out_bpt and res is None:
            cfg["reduce"] = reduce   # the block returns the aggregate; its backward gathers the aggregate's cotangent
            return TcBlockFn.apply(cfg, x, p1, p2, res, *params)
        y = TcBlockFn.apply(cfg, x, p1, p2, res, *params)
    else:
        y = FusedBlockFn.apply(cfg, x, p1, p2, res, *params)
    if reduce is not None:
        B = algebra.n_blades
        n_pairs = reduce[0].csr.n_pairs
        return SegmentReduceSortedFn.apply(y.reshape(n_pairs, -1), reduce[0], reduce[1]).reshape(reduce[0].csr.n_nodes, -1, B)
    return y


def embed_rows_forward(algebra, blocks, table, vertex_rows, fp):
    """The permute-embed step of ``embed_simplicial_complex`` (md17_cssmpnn.py:85-120) for one simplex dimension, without
    materialising the permuted feature rows: ``table`` [V, types * fp, B] holds every vertex' features once, ``vertex_rows``
    int32 [rows, k] the table rows of the k vertices of each (simplex, vertex order) row.  The first block of the CEMLP
    gathers its input channels ``(type, vertex slot, feature)`` itself (csmpn_block_desc mode 2); returns [rows, C, B], or
    None when these blocks do not run on the tensor-core engine (the caller then builds the rows with torch indexing)."""
    rows = vertex_rows.shape[0]
    need_grad = _need_grad(*[t for b in blocks for t in _block_params(b)])
    k = vertex_rows.shape[1]
    lin = blocks[0][0]
    if (not all(_block_supported(b) for b in blocks) or lin.in_features != table.shape[1] * k or table.requires_grad
            or not _chain_uses_tc(algebra, blocks, need_grad, rows)):
        return None
    cfg = {"dim": algebra.dim, "mode": 2, "sgraph": None, "need_grad": need_grad, "pair_attr": False,
           "vertex_table": (vertex_rows.contiguous(), int(fp)), "in_bpt": False, "out_bpt": len(blocks) > 1, "rows": None,
           "c_in": lin.in_features}
    u = TcBlockFn.apply(cfg, f32c(table), None, None, None, *_block_params(blocks[0]))
    for i, blk in enumerate(blocks[1:]):
        last = i == len(blocks) - 2
        u = block_forward(algebra, blk, u, bpt_rows=rows, out_bpt=not last)
    return u


def _chain_uses_tc(algebra, blocks, need_grad, rows) -> bool:
    return all(_block_supported(b) for b in blocks) and all(_block_uses_tc(algebra, b, need_grad, rows) for b in blocks)


def mlp_forward(algebra, blocks, x, p1=None, p2=None, res=None, mode=0, sgraph=None, rows=None, pair_attr=False, reduce=None):
    """A CEMLP (list of blocks): on the tensor-core engine the tensors between blocks stay in the BPT layout.
    reduce = (SortedGraph, mean): the rows are messages in receiver-sorted order and the CEMLP returns their per-receiver
    aggregate [n_nodes, C, B] (the last block folds the aggregation's adjoint into its backward on the tensor-core engine)."""
    need_grad = _need_grad(x, p1, p2, res, *[t for b in blocks for t in _block_params(b)])
    tc = len(blocks) > 1 and _chain_uses_tc(algebra, blocks, need_grad, rows)
    u = block_forward(algebra, blocks[0], x, p1, p2, res if len(blocks) == 1 else None, mode=mode, sgraph=sgraph, out_bpt=tc,
                      pair_attr=pair_attr, reduce=reduce if len(blocks) == 1 else None)
    for k, blk in enumerate(blocks[1:]):
        last = k == len(blocks) - 2
        u = block_forward(algebra, blk, u, res=res if last else None, bpt_rows=rows if tc else None, out_bpt=tc and not last,
                          reduce=reduce if last else None)
    return u


def egcl_forward(egcl, h, edge_index, edge_attr=None, node_attr=None):
    """EGCL.forward (cegnn_utils.py:277-284) on the fused path."""
    from .cegnn_utils import PairedNodeAttr

    alg = egcl.algebra
    blocks_e, blocks_n = list(egcl.edge_model.layers), list(egcl.node_model.layers)
    pair = isinstance(edge_attr, PairedNodeAttr)
    if not all(_block_supported(b) for b in blocks_e + blocks_n) or h.dim() != 3:
        if pair:
            edge_attr = edge_attr.materialize(edge_index)
        hf = alg.flatten(h)
        return alg.split(egcl.propagate(edge_index, h=hf, edge_attr=edge_attr, node_attr=node_attr))
    require_cuda(h, what="EGCL")
    B = alg.n_blades
    N = h.shape[0]
    csr = ops.get_csr(edge_index, N)
    sg = sorted_graph(csr)
    h = f32c(h)
    if h.requires_grad and torch.is_grad_enabled() and csr.n_pairs > 0 and egcl.residual:
        h_msg, h_upd, h_res = FanoutFn.apply(h)
    else:
        h_msg = h_upd = h_res = h
    if csr.n_pairs > 0:
        agg = mlp_forward(alg, blocks_e, h_msg, edge_attr.node_attr if pair else edge_attr, None, None, mode=1, sgraph=sg,
                          rows=csr.n_pairs, pair_attr=pair, reduce=(sg, egcl.aggr == "mean"))
    else:
        agg = h.new_zeros((N, egcl.out_features, B))
    return mlp_forward(alg, blocks_n, h_upd, agg, node_attr, h_res if egcl.residual else None, rows=N)


# ------------------------------------------------------------------------------------------------- bench helper
def _time_call(fn, flush, iters, warm=3):
    ts = []
    for it in range(iters + warm):
        flush.fill_(0.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if it >= warm:
            ts.append(e0.elapsed_time(e1))
    return sum(ts) / len(ts) * 1e-3


def _kernel_stages(d: BlockDesc, g, B: int):
    """(class, description, mask, algorithmic bytes, tensor-pipe FLOPs) of every kernel behind one recorded block call.
    Algorithmic bytes = every tensor the kernel must read or write, once (DESIGN.md section 4); T = one BPT [rows, Cp]
    tensor, Tin = one BPT [rows, c_in] tensor; tensor-pipe FLOPs count the three TF32 MMAs of a split product,
    or the one MMA of a single-pass TF32 product (d.tf32)."""
    rows, C = int(d.rows), int(d.c)
    cin = d.c0 + d.c1 + d.c2
    cp, cinp = (C + 15) // 16 * 16, (cin + 15) // 16 * 16
    tiles = (rows + 127) // 128
    T, Tin = tiles * 128 * B * cp * 4, tiles * 128 * B * cinp * 4
    ref = lambda ch: rows * ch * B * 4
    if d.engine == 0:  # FP32 SIMT engine: one kernel per direction
        src = ref(2 * d.c0 + d.c1) + 12 * rows if d.mode == 1 else ref(cin)
        if g is None:
            return [("block_fwd (fp32 simt)", "fused CEMLP block forward", 0, src + ref(4 * C), 0)]
        return [("block_bwd (fp32 simt)", "fused CEMLP block backward + parameter-gradient reduce", 0, src + ref(4 * C) + ref(cin), 0)]
    k = 1 if d.tf32 else 3  # TF32 MMAs per product
    if g is None:
        f1_in = Tin if d.in_bpt else (ref(2 * d.c0) + ref(d.c1) + 12 * rows if d.mode == 1 else ref(cin))
        f1_out = (0 if d.in_bpt else Tin) + 2 * T
        y_out = T if d.out_bpt else ref(C) * (2 if d.res else 1)
        return [("tc_f1", "input rows (gather | BPT) -> MVLinear W1 + bias -> y1, MVSiLU -> y2", 1, f1_in + f1_out, k * rows * 2 * B * C * cin),
                ("tc_f2", "linear_right/left + normalisation + weighted GP + MVLayerNorm (+residual)", 2, 4 * T + y_out, k * rows * 4 * B * C * C)]
    gy = T if g.gy_bpt else ref(C)
    gx = 0 if not g.grad_x else (Tin if g.gx_bpt else ref(cin))
    return [("tc_b1", "MVLayerNorm / weighted GP / normalisation adjoints", 1, 6 * T + gy, 0),
            ("tc_bgemm", "dy2 = dy2p + d WL + dxr WR", 2, 4 * T, k * rows * 4 * B * C * C),
            ("tc_b3", "MVSiLU adjoint", 4, 3 * T, 0),
            ("tc_bgemm", "grad_x = dy1 W1", 8, T + gx, k * rows * 2 * B * C * cin),
            ("tc_dw", "dWL, dWR = [d|dxr]^T y2", 16, 3 * T, k * rows * 4 * B * C * C),
            ("tc_dw", "dW1 = dy1^T x0", 32, T + Tin, k * rows * 2 * B * C * cin),
            ("tc_final", "fixed-order reduction of per-CTA partials", 64, 0, 0)]


def bench_layer_kernels(layer, d, graph, hbm_peak, peak_src, traffic=None, iters=8):
    """Per-kernel roofline of ONE layer step, measured live: one eager forward + backward is recorded (every block call of
    the layer with its descriptors), then every kernel behind every recorded call is launched ALONE (stage_mask) and
    timed with CUDA events on the launching stream, L2 flushed between launches.  Kernels are grouped by class; the
    DOMINANT class is the one with the largest share of the summed kernel time of the layer, and the reported figure is
    its algorithmic bytes over its time (all its launches in the layer).  ``traffic``: optional {class: DRAM bytes per
    layer step} from an ncu capture of this very build (bench.py passes it only when the build digest matches)."""
    global _RECORDER
    from .cegnn_utils import PairedNodeAttr

    alg = layer.algebra
    B = alg.n_blades
    dev = d["h"].device
    s = stream_ptr(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    h = d["h"].detach().requires_grad_()
    na = d["node_attr"]
    ea = d.get("edge_attr")
    ea = PairedNodeAttr(na) if ea is None else ea
    fork = os.environ.get("CSMPN_TC_FORK")
    os.environ["CSMPN_TC_FORK"] = "0"  # single-stream eager pass: the recorded descriptors carry stage_mask 0
    _RECORDER = rec = []
    try:
        y = layer(h, graph, ea, na)
        torch.autograd.grad(y, [h] + list(layer.parameters()), d["cot"])
        torch.cuda.synchronize()
    finally:
        _RECORDER = None
        if fork is None:
            os.environ.pop("CSMPN_TC_FORK", None)
        else:
            os.environ["CSMPN_TC_FORK"] = fork
    table = []
    for call in rec:
        desc, g, ws, dim = call["desc"], call["grads"], call["ws"], call["dim"]
        cin = desc.c0 + desc.c1 + desc.c2
        where = "%s block, c_in=%d, C=%d, %d rows" % ("per-pair" if desc.rows == graph.n_pairs else "per-simplex", cin, desc.c, desc.rows)
        for cls, what, mask, nbytes, tflops in _kernel_stages(desc, g, B):
            desc.stage_mask = mask
            if g is None:
                fn = lambda: check(lib().csmpn_block_fwd(dim, ctypes.byref(desc), s), "fwd")
            else:
                fn = lambda: check(lib().csmpn_block_bwd(dim, ctypes.byref(desc), ctypes.byref(g), ptr(ws), ws.numel(), s), "bwd")
            t = _time_call(fn, flush, iters)
            table.append({"class": cls, "kernel": what, "block": where, "launch_ms": t * 1e3, "algorithmic_bytes": nbytes,
                          "hbm_gbs": nbytes / t / 1e9, "hbm_frac": nbytes / t / 1e9 / hbm_peak,
                          "tensor_tflops_tf32x3": tflops / t / 1e12})
        desc.stage_mask = 0
    total = sum(r["launch_ms"] for r in table)
    classes = {}
    for r in table:
        c = classes.setdefault(r["class"], {"launches": 0, "ms": 0.0, "bytes": 0})
        c["launches"] += 1
        c["ms"] += r["launch_ms"]
        c["bytes"] += r["algorithmic_bytes"]
    for name, c in classes.items():
        c["share_of_layer_kernel_time"] = c["ms"] / total
        c["hbm_gbs"] = c["bytes"] / (c["ms"] * 1e-3) / 1e9
        c["hbm_frac"] = c["hbm_gbs"] / hbm_peak
        c["traffic"] = None if not traffic else traffic.get(name)
    dom_name = max(classes, key=lambda k: classes[k]["ms"])
    dom = classes[dom_name]
    return {
        "bound": "hbm", "achieved": dom["hbm_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": dom["hbm_frac"],
        "traffic": None if not dom["traffic"] else dom["traffic"] / dom["launches"], "peak_source": peak_src,
        "kernel": "%s (%d launches per layer step, %.0f %% of the layer's summed kernel time)" % (dom_name, dom["launches"], 100 * dom["share_of_layer_kernel_time"]),
        "launch_ms": dom["ms"] / dom["launches"], "algorithmic_bytes_per_launch": dom["bytes"] / dom["launches"],
        "how": "every kernel of one layer step launched alone (csmpn_block_desc.stage_mask) between CUDA events on the launching "
               "stream, L2 flushed before each launch, mean of %d; dominant = kernel class with the largest time share; achieved = its "
               "algorithmic bytes / its time over all its launches in the step; traffic = ncu dram bytes of the class per step "
               "(only when profiles/ holds a capture of this build, else null)" % iters,
        "classes": classes, "kernels": table, "summed_kernel_ms": total,
    }
