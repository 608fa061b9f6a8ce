"""torch-facing wrappers of the C-ABI kernels (PyTorch tensors in, PyTorch tensors out).

Each autograd Function mirrors one step of /root/reference/module/layer.py:44-51 and
its autograd; nothing here computes on the host or falls back to torch kernels for
the aggregate / exchange path.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _C
from .graph import CsrPlan, PartGraph, alloc_rows


def _rows(t: torch.Tensor):
    if t.dim() != 2 or (t.shape[1] > 1 and t.stride(1) != 1):
        raise _C.PgError(f"expected a row-major 2-D tensor, got shape {tuple(t.shape)} strides {t.stride()}")
    if not t.is_cuda:
        raise _C.PgError("the hot path runs on CUDA tensors only (no CPU fall-back)")
    return t


class DropSpec:
    """Key of a dropout mask (include/pipegcn_b200.h: pg_drop): probability, 64-bit seed, device-side step counter +
    offset.  The same key evaluated by different kernels gives the same mask, so the mask is never stored."""

    def __init__(self, p: float, seed: int, step: torch.Tensor = None, step_off: int = 0):
        self.p, self.seed, self.step, self.step_off = float(p), int(seed) & 0xFFFFFFFFFFFFFFFF, step, int(step_off)

    def shifted(self, off: int) -> "DropSpec":
        return DropSpec(self.p, self.seed, self.step, self.step_off + off)

    def c(self):
        return _C.pg_drop(self.p, self.seed, self.step.data_ptr() if self.step is not None else None, self.step_off)


def layer_seed(layer: int) -> int:
    """Dropout seed of graph layer `layer`: the same on every rank (all ranks seed torch identically, train.py:298)."""
    return (torch.initial_seed() * 0x9E3779B97F4A7C15 + (layer + 1) * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF


def _drop_ok(t: torch.Tensor) -> bool:
    """The mask is defined on 16-byte vectors of padded, aligned rows."""
    return t.dim() == 2 and t.is_cuda and t.stride(1) == 1 and (t.stride(0) * t.element_size()) % 16 == 0 \
        and t.data_ptr() % 16 == 0 and t.stride(0) >= (t.shape[1] + 7) // 8 * 8 and t.dtype in (torch.float32, torch.bfloat16)


def dropout_rows(x: torch.Tensor, spec: DropSpec, out: torch.Tensor = None, row0: int = 0) -> torch.Tensor:
    """out = dropout(x) under the key `spec`; rows are numbered from row0 (x may be a row slice of a larger tensor)."""
    if out is None:
        out = alloc_rows(x.shape[0], x.shape[1], x.dtype, x.device)
    _C.count()
    _C.check(_C.lib.pg_dropout_rows(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), int(row0), x.shape[0],
                                    x.shape[1], _C.dtype_code(x.dtype), C.byref(spec.c()), _C.stream_ptr()),
             "pg_dropout_rows")
    return out


def aggregate(plan: CsrPlan, x: torch.Tensor, out: torch.Tensor = None, row_div: torch.Tensor = None,
              acc_rows: int = 0, drop: DropSpec = None) -> torch.Tensor:
    """out[r] = sum_{e in row r} x[indices[e]] (/ row_div[r]) (+ out[r] for r < acc_rows); with `drop` the mask of that
    key is applied to every row as it is written."""
    _rows(x)
    d = x.shape[1]
    if out is None:
        out = alloc_rows(plan.n_rows, d, x.dtype, x.device)
    _rows(out)
    assert out.shape[0] == plan.n_rows and out.shape[1] == d and out.dtype == x.dtype
    scratch = plan.scratch(d)
    prof = PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    _C.count(2 if plan.n_long else 1)
    if drop is not None and drop.p > 0:
        _C.check(_C.lib.pg_aggregate_drop(C.byref(plan.c), x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), d,
                                          _C.dtype_code(x.dtype), row_div.data_ptr() if row_div is not None else None,
                                          int(acc_rows), scratch.data_ptr() if scratch is not None else None,
                                          C.byref(drop.c()), _C.stream_ptr()), "pg_aggregate_drop")
    else:
        _C.check(_C.lib.pg_aggregate(C.byref(plan.c), x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), d,
                                     _C.dtype_code(x.dtype), row_div.data_ptr() if row_div is not None else None,
                                     int(acc_rows), scratch.data_ptr() if scratch is not None else None,
                                     _C.stream_ptr()), "pg_aggregate")
    if prof is not None:
        e1.record()
        prof.append((e0, e1, aggregate_bytes(plan, x, row_div is not None)))
    return out


# when a list, every aggregate launch appends (start event, end event, algorithmic bytes)
PROFILE = None


def aggregate_bytes(plan: CsrPlan, x: torch.Tensor, has_div: bool) -> int:
    """ALGORITHMIC bytes of one launch (SURVEY.md §8d): column ids + row pointers + divisor +
    every source row once + every output row once."""
    s, d = x.element_size(), x.shape[1]
    return 4 * plan.nnz + 4 * (plan.n_rows + 1) + (4 * plan.n_rows if has_div else 0) \
        + s * d * x.shape[0] + s * d * plan.n_rows


def row_div(x: torch.Tensor, div: torch.Tensor, out: torch.Tensor = None) -> torch.Tensor:
    _rows(x)
    if out is None:
        out = alloc_rows(x.shape[0], x.shape[1], x.dtype, x.device)
    _C.count()
    _C.check(_C.lib.pg_row_div(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), x.shape[0], x.shape[1],
                               _C.dtype_code(x.dtype), div.data_ptr(), _C.stream_ptr()), "pg_row_div")
    return out


class SageAggregate(torch.autograd.Function):
    """ah = (A @ feat) / in_deg   (layer.py:47-50) and its gradient  g_feat = A^T @ (g_ah / in_deg)."""

    @staticmethod
    def forward(ctx, feat, graph: PartGraph, deg_f):
        ctx.graph, ctx.deg_f = graph, deg_f
        if feat.stride(1) != 1:
            feat = feat.contiguous()
        return aggregate(graph.fwd, feat, row_div=deg_f)

    @staticmethod
    def backward(ctx, g_ah):
        graph = ctx.graph
        if g_ah.stride(1) != 1:
            g_ah = g_ah.contiguous()
        gs = row_div(g_ah, ctx.deg_f)
        return aggregate(graph.bwd, gs), None, None


def sage_aggregate(feat: torch.Tensor, graph: PartGraph, deg_f: torch.Tensor = None) -> torch.Tensor:
    return SageAggregate.apply(feat, graph, graph.in_deg_f if deg_f is None else deg_f)


# ---- dense part: hand-written tcgen05 GEMM (csrc/linear_tcgen05.cu) -----------------------------
LINEAR_IMPL = "tcgen05 (pg_linear / pg_wgrad: TMA + tcgen05.mma kind::f16 / 3xTF32, TMEM accumulators; dW MN-major split-K)"


def _tma_ready(t: torch.Tensor) -> torch.Tensor:
    """Row-major view whose rows start on 16-byte boundaries (what a TMA descriptor needs)."""
    if t.dim() == 2 and t.stride(1) == 1 and (t.stride(0) * t.element_size()) % 16 == 0 \
            and t.data_ptr() % 16 == 0 and t.stride(0) >= t.shape[1]:
        return t
    out = alloc_rows(t.shape[0], t.shape[1], t.dtype, t.device)
    out.copy_(t)
    return out


def padded_weight(w: torch.Tensor, dtype, transpose: bool = False) -> torch.Tensor:
    """[n, k] copy of a weight (or of its transpose) in the activation dtype with 16-byte aligned rows."""
    src = w.detach().t() if transpose else w.detach()
    out = alloc_rows(src.shape[0], src.shape[1], dtype, w.device)
    out.copy_(src)
    return out


def split_tf32(x: torch.Tensor):
    """(hi, lo) with hi = x truncated to tf32 and lo = x - hi, both padded row-major fp32 (pg_split_tf32)."""
    _rows(x)
    hi = alloc_rows(x.shape[0], x.shape[1], torch.float32, x.device)
    lo = alloc_rows(x.shape[0], x.shape[1], torch.float32, x.device)
    if x.shape[0]:
        _C.count()
        _C.check(_C.lib.pg_split_tf32(x.data_ptr(), x.stride(0), hi.data_ptr(), lo.data_ptr(), hi.stride(0),
                                      x.shape[0], x.shape[1], _C.stream_ptr()), "pg_split_tf32")
    return hi, lo


# fp32 activations: "3xtf32" = hi*hi + hi*lo + lo*hi on the tf32 tensor cores (fp32-grade accuracy, the
# parity mode); "tf32" = one pass (rel. error ~1e-3).  bf16 activations always use one kind::f16 pass.
FP32_GEMM = os.environ.get("PG_FP32_GEMM", "3xtf32")


class Split:
    """An fp32 operand together with its tf32 (hi, lo) halves, so that one split serves every product that uses the
    operand (a gradient feeds two dX GEMMs and two weight-gradient GEMMs)."""

    def __init__(self, x: torch.Tensor):
        self.x = _rows(x)
        self.hi, self.lo = split_tf32(x)

    def rows(self, lo: int, hi: int = None) -> "Split":
        out = Split.__new__(Split)
        out.x, out.hi, out.lo = self.x[lo:hi], self.hi[lo:hi], self.lo[lo:hi]
        return out


def presplit(x: torch.Tensor):
    """`Split(x)` when x is an fp32 operand of the 3xTF32 product, else x itself."""
    if isinstance(x, torch.Tensor) and x.dtype == torch.float32 and FP32_GEMM == "3xtf32":
        return Split(x)
    return x


def _plain(t):
    return t.x if isinstance(t, Split) else t


def _halves(t):
    return (t.hi, t.lo) if isinstance(t, Split) else split_tf32(t)


def gemm_nt(a0, b0, a1=None, b1=None, bias=None, row_div=None, out=None, out_dtype=None, drop=None,
            drop_row0: int = 0) -> torch.Tensor:
    """out[m, n] = a0 @ b0^T (+ a1 @ b1^T) (+ bias) (/ row_div[:, None]) on the tcgen05 tensor cores.  Operands may be
    `Split` objects (fp32 operands split once by the caller).  `drop`: dropout mask applied to `out` as it is written
    (out's first row is row `drop_row0` of the tensor the mask is defined on)."""
    raw = [(a0, b0)] + ([(a1, b1)] if a1 is not None else [])
    a0, b0 = _plain(a0), _plain(b0)
    pairs = [(_rows(_plain(a)), _rows(_plain(b))) for a, b in raw]
    m, n = a0.shape[0], b0.shape[0]
    for a, b in pairs:
        assert a.shape[0] == m and b.shape[0] == n and a.shape[1] == b.shape[1] and a.dtype == b.dtype == a0.dtype
    if n > 256:
        # one N tile holds at most 256 columns: split the weight rows
        outs = [gemm_nt(raw[0][0], b0[i:i + 256], raw[1][0] if len(raw) > 1 else None,
                        None if len(raw) == 1 else _plain(raw[1][1])[i:i + 256],
                        None if bias is None else bias[i:i + 256], row_div, None, out_dtype)
                for i in range(0, n, 256)]
        assert drop is None or drop.p == 0, "fused dropout with n > 256 is not supported"
        res = torch.cat(outs, dim=1)
        if out is not None:
            out.copy_(res)
            return out
        return res
    if out is None:
        out = alloc_rows(m, n, out_dtype or a0.dtype, a0.device)
    assert out.shape == (m, n) and out.stride(1) == 1
    if m == 0:
        return out
    if a0.dtype == torch.float32 and FP32_GEMM == "3xtf32":
        split = []
        for a, b in raw:
            (ah, al), (bh, bl) = _halves(a), _halves(b)
            split += [(ah, bh), (ah, bl), (al, bh)]
        pairs = split
    else:
        pairs = [(_tma_ready(a), _tma_ready(b)) for a, b in pairs]
    srcs = (_C.pg_gemm_src * len(pairs))(*[_C.pg_gemm_src(a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0),
                                                            a.shape[1]) for a, b in pairs])
    if bias is not None:
        bias = bias.detach().to(torch.float32).contiguous()
    _C.count()
    if drop is not None and drop.p > 0:
        _C.check(_C.lib.pg_linear_drop(_C.dtype_code(a0.dtype), _C.dtype_code(out.dtype), srcs, len(pairs),
                                       bias.data_ptr() if bias is not None else None,
                                       row_div.data_ptr() if row_div is not None else None,
                                       out.data_ptr(), out.stride(0), m, n, C.byref(drop.c()), int(drop_row0),
                                       _C.stream_ptr()), "pg_linear_drop")
        return out
    _C.check(_C.lib.pg_linear(_C.dtype_code(a0.dtype), _C.dtype_code(out.dtype), srcs, len(pairs),
                              bias.data_ptr() if bias is not None else None,
                              row_div.data_ptr() if row_div is not None else None,
                              out.data_ptr(), out.stride(0), m, n, _C.stream_ptr()), "pg_linear")
    return out


# fp32 weight gradients: "3xtf32" = MN-major kind::tf32 with hi/lo splits, "bf16x3" = six MN-major kind::f16 products
WGRAD_FP32 = os.environ.get("PG_WGRAD_FP32", "3xtf32")


def _split_bf16x3(x: torch.Tensor):
    out, r = [], x.float()
    for _ in range(3):
        b = alloc_rows(x.shape[0], x.shape[1], torch.bfloat16, x.device)
        b.copy_(r)
        out.append(b)
        r = r - b.float()
    return out



def wgrad(g: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """g^T @ x  -> fp32 [n, k]: the weight gradient of `x @ W^T` on the tcgen05 tensor cores (pg_wgrad: MN-major
    operands straight from the row-major activations, split-K over the rows, fixed-order reduction)."""
    gs, xs = g, x
    g, x = _rows(_plain(g)), _rows(_plain(x))
    m, n, k = g.shape[0], g.shape[1], x.shape[1]
    assert x.shape[0] == m and g.dtype == x.dtype
    out = torch.empty(n, k, dtype=torch.float32, device=g.device)
    if m == 0:
        return out.zero_()
    if g.dtype == torch.float32 and FP32_GEMM == "3xtf32" and WGRAD_FP32 == "3xtf32":
        (gh, gl), (xh, xl) = _halves(gs), _halves(xs)
        pairs = [(gh, xh), (gh, xl), (gl, xh)]
    elif g.dtype == torch.float32 and FP32_GEMM == "3xtf32":
        # fp32 = b0 + b1 + b2 exactly (three bf16 terms): six bf16 products carry the product to ~2^-24
        g3, x3 = _split_bf16x3(g), _split_bf16x3(x)
        pairs = [(g3[0], x3[0]), (g3[0], x3[1]), (g3[1], x3[0]), (g3[0], x3[2]), (g3[2], x3[0]), (g3[1], x3[1])]
    else:
        pairs = [(_tma_ready(g), _tma_ready(x))]
    code = _C.dtype_code(pairs[0][0].dtype)
    for n0 in range(0, n, 256):
        for k0 in range(0, k, 256):
            nn, kk = min(256, n - n0), min(256, k - k0)
            # split-K partials: a fresh block per call (the caching allocator is stream-aware; several simulated
            # ranks run on their own streams in one process and must not share scratch)
            ws = torch.empty(int(_C.lib.pg_wgrad_workspace(m, nn, kk, code)), dtype=torch.float32, device=g.device)
            es = pairs[0][0].element_size()
            srcs = (_C.pg_gemm_src * len(pairs))(*[
                _C.pg_gemm_src(a.data_ptr() + n0 * es, a.stride(0), b.data_ptr() + k0 * es, b.stride(0), m)
                for a, b in pairs])
            o = out[n0:n0 + nn, k0:k0 + kk]
            _C.count(2)
            _C.check(_C.lib.pg_wgrad(code, srcs, len(pairs), o.data_ptr(), o.stride(0), m, nn, kk, ws.data_ptr(),
                                     ws.numel(), _C.stream_ptr()), "pg_wgrad")
    return out


class _Linear(torch.autograd.Function):
    """y = x @ W^T + b   (plain `nn.Linear` layers: use_pp layer 0 and the trailing n_linear layers)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        wp = padded_weight(weight, x.dtype)
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return gemm_nt(x, wp, bias=bias)

    @staticmethod
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        colsum = _take_colsum(g)
        g = _tma_ready(g if g.dtype == x.dtype else g.to(x.dtype))
        gsp = presplit(g)
        gx = gemm_nt(gsp, padded_weight(weight, x.dtype, transpose=True)) if ctx.needs_input_grad[0] else None
        gw = wgrad(gsp, x).to(weight.dtype)
        gb = (colsum if colsum is not None else g.float().sum(0)) if ctx.has_bias else None
        return gx, gw, gb


def linear(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor = None) -> torch.Tensor:
    return _Linear.apply(x, weight, bias)


class SageLayerFn(torch.autograd.Function):
    """The whole training branch of GraphSAGELayer.forward (layer.py:44-51) and its gradient:

        ah  = (A @ feat) / in_deg                         pg_aggregate
        out = feat[:N_in] @ W1^T + ah @ W2^T + (b1 + b2)  pg_linear, two sources, one kernel

        g_feat[:N_in] = g @ W1                            pg_linear
        gs            = (g @ W2) / in_deg                 pg_linear with the row scale fused
        g_feat       += A^T @ gs                          pg_aggregate accumulating into rows < N_in
        gW1 = g^T feat[:N_in], gW2 = g^T ah, gb = sum g   library GEMM / reduction
    """

    @staticmethod
    def forward(ctx, feat, graph, deg_f, w1, b1, w2, b2, drop_bwd=None):
        # drop_bwd: `feat` already IS dropout(F) (written that way by its producers); the gradient returned is the one
        # with respect to F, i.e. the dropout backward is applied to g_feat as the transposed aggregate writes it
        ctx.drop_bwd = drop_bwd
        if feat.stride(1) != 1:
            feat = feat.contiguous()
        n_in = graph.num_in
        ah = aggregate(graph.fwd, feat, row_div=deg_f)
        x = feat[:n_in]
        bias = None
        if b1 is not None:
            bias = b1.detach().float() + b2.detach().float()
        out = gemm_nt(x, padded_weight(w1, feat.dtype), ah, padded_weight(w2, feat.dtype), bias=bias)
        ctx.graph, ctx.deg_f = graph, deg_f
        ctx.has_bias = b1 is not None
        ctx.save_for_backward(x, ah, w1, w2)
        ctx.num_all = feat.shape[0]
        return out

    @staticmethod
    def backward(ctx, g):
        x, ah, w1, w2 = ctx.saved_tensors
        graph, deg_f = ctx.graph, ctx.deg_f
        colsum = _take_colsum(g)
        g = _tma_ready(g if g.dtype == x.dtype else g.to(x.dtype))
        gsp = presplit(g)                      # fp32: one split of g serves the two dX and the two dW products
        g_feat = None
        if ctx.needs_input_grad[0]:
            d_in = x.shape[1]
            g_feat = alloc_rows(ctx.num_all, d_in, x.dtype, x.device)
            gemm_nt(gsp, padded_weight(w1, x.dtype, transpose=True), out=g_feat[:graph.num_in])
            gs = gemm_nt(gsp, padded_weight(w2, x.dtype, transpose=True), row_div=deg_f)
            aggregate(graph.bwd, gs, out=g_feat, acc_rows=graph.num_in, drop=ctx.drop_bwd)
        gw1 = wgrad(gsp, x).to(w1.dtype)
        gw2 = wgrad(gsp, ah).to(w2.dtype)
        gb = (colsum if colsum is not None else g.float().sum(0)) if ctx.has_bias else None
        return g_feat, None, None, gw1, gb, gw2, gb, None


class SageLayerNarrowFn(torch.autograd.Function):
    """The same function as `SageLayerFn`, evaluated TRANSFORM-FIRST when the layer narrows (d_out < d_in):

        z   = feat @ W2^T                          [num_all, d_out]   pg_linear over all rows (inner + halo)
        out = feat[:N_in] @ W1^T + (b1 + b2)       [N_in, d_out]      pg_linear
        out += (A @ z) / in_deg                                       pg_aggregate, accumulating, division fused

    (A F) W = A (F W): the aggregate -- the HBM/L2-bound part of /root/reference/module/layer.py:47-51 -- moves
    d_out-wide rows instead of d_in-wide ones (4x fewer bytes for the 256 -> 64 output layer of the headline config).
    Backward: dz = A^T (g / in_deg) [num_all, d_out], g_feat = dz @ W2 (+ g @ W1 on the inner rows),
    gW2 = dz^T feat, gW1 = g^T feat[:N_in].  Same sums, different association: fp32 results agree with the
    aggregate-first form to rounding (parity tests compare against the oracle, which aggregates first).
    """

    @staticmethod
    def forward(ctx, feat, graph, deg_f, w1, b1, w2, b2, drop_bwd=None):
        ctx.drop_bwd = drop_bwd
        if feat.stride(1) != 1:
            feat = feat.contiguous()
        n_in = graph.num_in
        fsp = presplit(feat)                   # fp32: one split of feat for both products
        bias = None
        if b1 is not None:
            bias = b1.detach().float() + b2.detach().float()
        na, nb = w2.shape[0], w1.shape[0]
        v = 16 // feat.element_size()
        na_pad = -(-na // v) * v
        if MERGE_NARROW and na_pad + nb <= 256:
            # ONE product reads feat once: [z | self part] = feat @ [W2 ; W1]^T (+ [0 | b1 + b2]); the self part of
            # the halo rows is computed and never read.  W1 starts at a 16-byte aligned column.
            wc = alloc_rows(na_pad + nb, feat.shape[1], feat.dtype, feat.device)
            if na_pad != na:
                wc[na:na_pad].zero_()
            wc[:na].copy_(w2.detach())
            wc[na_pad:].copy_(w1.detach())
            bias_c = None
            if bias is not None:
                bias_c = torch.zeros(na_pad + nb, dtype=torch.float32, device=feat.device)
                bias_c[na_pad:].copy_(bias)
            zc = gemm_nt(fsp, wc, bias=bias_c)
            z, out = zc[:, :na], zc[:n_in, na_pad:]
        else:
            z = gemm_nt(fsp, padded_weight(w2, feat.dtype))
            out = gemm_nt(fsp.rows(0, n_in) if isinstance(fsp, Split) else feat[:n_in], padded_weight(w1, feat.dtype),
                          bias=bias)
        aggregate(graph.fwd, z, out=out, row_div=deg_f, acc_rows=n_in)
        ctx.graph, ctx.deg_f = graph, deg_f
        ctx.has_bias = b1 is not None
        ctx.save_for_backward(feat, w1, w2)
        return out

    @staticmethod
    def backward(ctx, g):
        feat, w1, w2 = ctx.saved_tensors
        graph, deg_f = ctx.graph, ctx.deg_f
        n_in = graph.num_in
        colsum = _take_colsum(g)
        g = _tma_ready(g if g.dtype == feat.dtype else g.to(feat.dtype))
        gs = row_div(g, deg_f)
        dz = aggregate(graph.bwd, gs)                                   # [num_all, d_out]
        gsp, dzsp, fsp = presplit(g), presplit(dz), presplit(feat)
        is_split = isinstance(fsp, Split)
        g_feat = None
        if ctx.needs_input_grad[0]:
            g_feat = alloc_rows(feat.shape[0], feat.shape[1], feat.dtype, feat.device)
            w1t, w2t = padded_weight(w1, feat.dtype, transpose=True), padded_weight(w2, feat.dtype, transpose=True)
            db = ctx.drop_bwd if (ctx.drop_bwd is not None and ctx.drop_bwd.p > 0 and feat.shape[1] <= 256
                                  and _drop_ok(g_feat)) else None   # dropout backward in the GEMM's epilogue
            gemm_nt(dzsp.rows(0, n_in) if is_split else dz[:n_in], w2t, gsp, w1t, out=g_feat[:n_in], drop=db)
            if feat.shape[0] > n_in:
                gemm_nt(dzsp.rows(n_in) if is_split else dz[n_in:], w2t, out=g_feat[n_in:], drop=db, drop_row0=n_in)
            if db is None and ctx.drop_bwd is not None and ctx.drop_bwd.p > 0:
                dropout_rows(g_feat, ctx.drop_bwd, out=g_feat)
        gw1 = wgrad(gsp, fsp.rows(0, n_in) if is_split else feat[:n_in]).to(w1.dtype)
        gw2 = wgrad(dzsp, fsp).to(w2.dtype)
        gb = (colsum if colsum is not None else g.float().sum(0)) if ctx.has_bias else None
        return g_feat, None, None, gw1, gb, gw2, gb, None


# transform-first when the layer narrows (PG_NARROW=0 keeps the reference's aggregate-first association everywhere)
NARROW = os.environ.get("PG_NARROW", "1") != "0"
# ... with the neighbour and self products of its forward in one GEMM (PG_MERGE_NARROW=0: two GEMMs)
MERGE_NARROW = os.environ.get("PG_MERGE_NARROW", "1") != "0"


def sage_layer(feat, graph, deg_f, w1, b1, w2, b2, drop_bwd=None) -> torch.Tensor:
    if NARROW and w1.shape[0] < feat.shape[1]:
        return SageLayerNarrowFn.apply(feat, graph, deg_f, w1, b1, w2, b2, drop_bwd)
    return SageLayerFn.apply(feat, graph, deg_f, w1, b1, w2, b2, drop_bwd)


def sage_linear(x, ah, w1, b1, w2, b2) -> torch.Tensor:
    """x @ W1^T + b1 + ah @ W2^T + b2   (layer.py:51) -- un-fused composition (eval branch)."""
    return linear(x, w1, b1) + linear(ah, w2, b2)


# ---- row-wise epilogues (csrc/rowops.cu) -------------------------------------------------------------------
# column sums of a gradient tensor computed as a by-product by the kernel that produced it, keyed by the
# tensor's address: the bias gradient of the linear upstream (saves a full pass over [N, d])
_COLSUM = {}


def _stash_colsum(t: torch.Tensor, colsum: torch.Tensor):
    if len(_COLSUM) > 64:
        _COLSUM.clear()
    _COLSUM[(t.data_ptr(), tuple(t.shape))] = colsum


def reset_colsum():
    """Drop by-products of an earlier backward (called at the start of every backward pass): an entry that was
    never consumed must not be picked up by a later gradient that happens to reuse the address."""
    _COLSUM.clear()


def _take_colsum(t: torch.Tensor):
    return _COLSUM.pop((t.data_ptr(), tuple(t.shape)), None)


def ln_relu_supported(y: torch.Tensor) -> bool:
    v = 16 // y.element_size()
    d = y.shape[1]
    return y.is_cuda and y.dim() == 2 and d % v == 0 and d // v <= 128 and y.stride(1) == 1 \
        and (y.stride(0) * y.element_size()) % 16 == 0 and y.data_ptr() % 16 == 0


class LayerNormReLU(torch.autograd.Function):
    """relu(LayerNorm(y)) in one pass (model.py:53-56); the backward also yields d gamma, d beta and the column
    sums of g_y, which is the bias gradient of the linear that produced y."""

    @staticmethod
    def forward(ctx, y, gamma, beta, eps, relu, out, clean=None, drop=None):
        # clean / drop: `out` receives dropout(result) under the key `drop` (the next layer's dropout, fused), `clean`
        # the result itself (source of the halo push, ReLU mask of the backward)
        n, d = y.shape
        if out is None:
            out = alloc_rows(n, d, y.dtype, y.device)
        mean = torch.empty(n, dtype=torch.float32, device=y.device)
        rstd = torch.empty(n, dtype=torch.float32, device=y.device)
        g32, b32 = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        _C.count()
        if clean is not None or drop is not None:
            _C.check(_C.lib.pg_ln_relu_drop_fwd(y.data_ptr(), y.stride(0), g32.data_ptr(), b32.data_ptr(), float(eps),
                                                int(relu), out.data_ptr(), out.stride(0),
                                                clean.data_ptr() if clean is not None else None,
                                                clean.stride(0) if clean is not None else 0,
                                                mean.data_ptr(), rstd.data_ptr(), n, d, _C.dtype_code(y.dtype),
                                                C.byref(drop.c()) if drop is not None else None, _C.stream_ptr()),
                     "pg_ln_relu_drop_fwd")
        else:
            _C.check(_C.lib.pg_ln_relu_fwd(y.data_ptr(), y.stride(0), g32.data_ptr(), b32.data_ptr(), float(eps), int(relu),
                                           out.data_ptr(), out.stride(0), mean.data_ptr(), rstd.data_ptr(), n, d,
                                           _C.dtype_code(y.dtype), _C.stream_ptr()), "pg_ln_relu_fwd")
        ctx.save_for_backward(y, mean, rstd, g32, b32)
        ctx.relu = bool(relu)
        ctx.param_dtype = gamma.dtype
        return out

    @staticmethod
    def backward(ctx, g):
        y, mean, rstd, g32, b32 = ctx.saved_tensors
        n, d = y.shape
        if g.dtype != y.dtype or g.stride(1) != 1 or (g.stride(0) * g.element_size()) % 16 or g.data_ptr() % 16:
            g = _tma_ready(g.to(y.dtype))
        g_y = alloc_rows(n, d, y.dtype, y.device)
        grid = _C.lib.pg_row_grid(n)
        partial = torch.empty(grid * 3 * d, dtype=torch.float32, device=y.device)
        red = torch.empty(3, d, dtype=torch.float32, device=y.device)
        _C.count(2)
        # the ReLU mask is recomputed from y (beta given): the forward output is neither kept nor read
        _C.check(_C.lib.pg_ln_relu_bwd2(g.data_ptr(), g.stride(0), None, 0, y.data_ptr(), y.stride(0),
                                        mean.data_ptr(), rstd.data_ptr(), g32.data_ptr(), b32.data_ptr(), int(ctx.relu),
                                        g_y.data_ptr(), g_y.stride(0), red[0].data_ptr(), red[1].data_ptr(),
                                        red[2].data_ptr(), partial.data_ptr(), n, d, _C.dtype_code(y.dtype),
                                        _C.stream_ptr()), "pg_ln_relu_bwd")
        _stash_colsum(g_y, red[2])
        return g_y, red[0].to(ctx.param_dtype), red[1].to(ctx.param_dtype), None, None, None, None, None


def layer_norm_relu(y, gamma, beta, eps=1e-5, relu=True, out=None, clean=None, drop=None):
    return LayerNormReLU.apply(y, gamma, beta, eps, relu, out, clean, drop)


class KeyedDropout(torch.autograd.Function):
    """dropout(x) under an explicit key, forward and backward (the un-fused form of what the fused producers do:
    PG_FUSED_DROPOUT=0, and the reference the fused kernels are tested against)."""

    @staticmethod
    def forward(ctx, x, spec):
        ctx.spec = spec
        return dropout_rows(x, spec)

    @staticmethod
    def backward(ctx, g):
        if not _drop_ok(g):
            gp = alloc_rows(g.shape[0], g.shape[1], g.dtype, g.device)
            gp.copy_(g)
            g = gp
        return dropout_rows(g, ctx.spec, out=g), None


def keyed_dropout(x, spec: DropSpec):
    return KeyedDropout.apply(x, spec) if spec.p > 0 else x


# dropout of graph layers >= 1 applied by the producers of the dropped tensor (LayerNorm epilogue, halo push,
# transposed aggregate) instead of by [num_all, d] passes; PG_FUSED_DROPOUT=0: the same masks by separate passes
FUSED_DROPOUT = os.environ.get("PG_FUSED_DROPOUT", "1") != "0"


class CrossEntropySum(torch.autograd.Function):
    """CrossEntropyLoss(reduction='sum') over the first n_train rows of the logits (train.py:320,351); the gradient
    is zero on the remaining rows (train rows come first after move_train_first)."""

    @staticmethod
    def forward(ctx, logits, labels, n_train):
        n, c = logits.shape
        dev = logits.device
        lse = torch.empty(max(n_train, 1), dtype=torch.float32, device=dev)
        grid = _C.lib.pg_row_grid(max(n, 1))
        partial = torch.empty(grid * max(c, 1), dtype=torch.float32, device=dev)
        loss = torch.zeros(1, dtype=torch.float32, device=dev)
        if n_train:
            _C.count(2)
            _C.check(_C.lib.pg_ce_fwd(logits.data_ptr(), logits.stride(0), labels.data_ptr(), n_train, c,
                                      _C.dtype_code(logits.dtype), lse.data_ptr(), partial.data_ptr(), loss.data_ptr(),
                                      _C.stream_ptr()), "pg_ce_fwd")
        ctx.save_for_backward(logits, labels, lse, partial)
        ctx.n_train = n_train
        return loss[0]

    @staticmethod
    def backward(ctx, up):
        logits, labels, lse, partial = ctx.saved_tensors
        n, c = logits.shape
        g = alloc_rows(n, c, logits.dtype, logits.device)
        colsum = torch.empty(c, dtype=torch.float32, device=logits.device)
        up = up.detach().float().reshape(1).contiguous()
        _C.count(2)
        _C.check(_C.lib.pg_ce_bwd(logits.data_ptr(), logits.stride(0), labels.data_ptr(), lse.data_ptr(), up.data_ptr(),
                                  ctx.n_train, n, c, _C.dtype_code(logits.dtype), g.data_ptr(), g.stride(0),
                                  colsum.data_ptr(), partial.data_ptr(), _C.stream_ptr()), "pg_ce_bwd")
        _stash_colsum(g, colsum)
        return g, None, None


def cross_entropy_sum(logits, labels, n_train):
    if logits.stride(1) != 1:
        logits = logits.contiguous()
    return CrossEntropySum.apply(logits, labels, int(n_train))


# ---- multi-label targets (train.py:11-17,317-318): bit-packed on the device ----------------------------------------
def pack_multilabel(y: torch.Tensor) -> torch.Tensor:
    """[rows, C] 0/1 labels -> [rows, ceil(C / 32)] 32-bit words; label j is bit j % 32 of word j // 32, bits >= C are
    0.  The words are held in an int32 tensor (torch's uint32 lacks the copy / add kernels the input pipeline uses);
    the kernels read them as uint32.  Set-up work (torch ops, any device); the kernels are the only readers."""
    if y.dim() != 2:
        raise _C.PgError(f"multi-label targets are [rows, C], got shape {tuple(y.shape)}")
    rows, c = y.shape
    lw = (c + 31) // 32
    bits = torch.zeros(rows, lw * 32, dtype=torch.int64, device=y.device)
    bits[:, :c] = (y != 0).to(torch.int64)
    words = (bits.view(rows, lw, 32) << torch.arange(32, device=y.device)).sum(dim=2)
    return torch.where(words >= 1 << 31, words - (1 << 32), words).to(torch.int32).contiguous()


def unpack_multilabel(ybits: torch.Tensor, c: int) -> torch.Tensor:
    """Inverse of `pack_multilabel`: float32 [rows, c] 0/1."""
    w = ybits.to(torch.int64) & 0xFFFFFFFF
    bits = (w.unsqueeze(2) >> torch.arange(32, device=w.device)) & 1
    return bits.reshape(w.shape[0], -1)[:, :c].to(torch.float32)


def _ml_logits(z: torch.Tensor) -> torch.Tensor:
    """Logits as the multi-label kernels read them: CUDA, fp32/bf16, 16-byte aligned rows (copied only if not)."""
    _rows(z)
    if z.dtype not in (torch.float32, torch.bfloat16):
        z = z.float()
    return _tma_ready(z)


class BceWithLogitsSum(torch.autograd.Function):
    """BCEWithLogitsLoss(reduction='sum') over the first n_train rows of the logits against bit-packed targets
    (train.py:317-318); the gradient is zero on the remaining rows (train rows come first after move_train_first)."""

    @staticmethod
    def forward(ctx, logits, ybits, n_train, c):
        dev = logits.device
        n = logits.shape[0]
        grid = _C.lib.pg_row_grid(max(n_train, 1))
        partial = torch.empty(grid * max(c, 1), dtype=torch.float32, device=dev)
        loss = torch.zeros(1, dtype=torch.float32, device=dev)
        if n_train:
            _C.count(2)
            _C.check(_C.lib.pg_bce_fwd(logits.data_ptr(), logits.stride(0), ybits.data_ptr(), ybits.shape[1], n_train,
                                       c, _C.dtype_code(logits.dtype), partial.data_ptr(), loss.data_ptr(),
                                       _C.stream_ptr()), "pg_bce_fwd")
        ctx.save_for_backward(logits, ybits)
        ctx.n_train, ctx.c, ctx.n = n_train, c, n
        return loss[0]

    @staticmethod
    def backward(ctx, up):
        logits, ybits = ctx.saved_tensors
        n, c = ctx.n, ctx.c
        g = alloc_rows(n, c, logits.dtype, logits.device)
        colsum = torch.empty(c, dtype=torch.float32, device=logits.device)
        partial = torch.empty(_C.lib.pg_row_grid(n) * c, dtype=torch.float32, device=logits.device)
        up = up.detach().float().reshape(1).contiguous()
        _C.count(2)
        _C.check(_C.lib.pg_bce_bwd(logits.data_ptr(), logits.stride(0), ybits.data_ptr(), ybits.shape[1], up.data_ptr(),
                                   ctx.n_train, n, c, _C.dtype_code(logits.dtype), g.data_ptr(), g.stride(0),
                                   colsum.data_ptr(), partial.data_ptr(), _C.stream_ptr()), "pg_bce_bwd")
        _stash_colsum(g, colsum)
        return g, None, None, None


def bce_with_logits_sum(logits, ybits, n_train, c):
    """Summed sigmoid cross-entropy of the first n_train rows; `ybits` from `pack_multilabel` (>= n_train rows)."""
    logits = _ml_logits(logits)
    assert logits.shape[1] == c and ybits.shape[1] == (c + 31) // 32 and ybits.shape[0] >= n_train
    return BceWithLogitsSum.apply(logits, ybits, int(n_train), int(c))


def f1_counts(logits: torch.Tensor, ybits: torch.Tensor, rows: torch.Tensor = None) -> torch.Tensor:
    """Device int64 [3] = micro (TP, FP, FN) of `logits > 0` against `ybits` over `rows` (all rows when None)."""
    z = _ml_logits(logits)
    n, c = (z.shape[0] if rows is None else int(rows.numel())), z.shape[1]
    assert ybits.shape[0] == z.shape[0] and ybits.shape[1] == (c + 31) // 32
    idx = None if rows is None else rows.to(device=z.device, dtype=torch.int32).contiguous()
    counts = torch.zeros(3, dtype=torch.int64, device=z.device)
    if n:
        _C.count()
        _C.check(_C.lib.pg_f1_counts(z.data_ptr(), z.stride(0), ybits.data_ptr(), ybits.shape[1],
                                     idx.data_ptr() if idx is not None else None, n, c, _C.dtype_code(z.dtype),
                                     counts.data_ptr(), _C.stream_ptr()), "pg_f1_counts")
    return counts


def multilabel_f1(logits: torch.Tensor, ybits: torch.Tensor, rows: torch.Tensor = None) -> float:
    """f1_score(y, logits > 0, average='micro') = 2 TP / (2 TP + FP + FN), one host read.  With no positive label and
    no positive prediction the score is 0.0, which is what sklearn returns there (zero_division='warn').  A single
    label column is a binary target to sklearn, whose micro average over the classes {0, 1} is the accuracy."""
    tp, fp, fn = (int(v) for v in f1_counts(logits, ybits, rows).tolist())
    if logits.shape[1] == 1:
        n = logits.shape[0] if rows is None else int(rows.numel())
        return (n - fp - fn) / n if n else 0.0
    den = 2 * tp + fp + fn
    return 2 * tp / den if den else 0.0


class Dropout(torch.autograd.Function):
    """Dropout whose mask is regenerated from (seed, element index) in the backward (csrc/rowops.cu)."""

    @staticmethod
    def forward(ctx, x, p, seed):
        out = alloc_rows(x.shape[0], x.shape[1], x.dtype, x.device)
        _C.count()
        step = STEP_DEV.data_ptr() if STEP_DEV is not None else None
        _C.check(_C.lib.pg_dropout(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), x.shape[0], x.shape[1],
                                   _C.dtype_code(x.dtype), float(p), int(seed), step, _C.stream_ptr()), "pg_dropout")
        ctx.p, ctx.seed, ctx.step = p, seed, step
        return out

    @staticmethod
    def backward(ctx, g):
        if g.stride(1) != 1 or (g.stride(0) * g.element_size()) % 16 or g.data_ptr() % 16 \
                or g.stride(0) < (g.shape[1] + 7) // 8 * 8:
            gp = alloc_rows(g.shape[0], g.shape[1], g.dtype, g.device)
            gp.copy_(g)
            g = gp
        _C.count()
        _C.check(_C.lib.pg_dropout(g.data_ptr(), g.stride(0), g.data_ptr(), g.stride(0), g.shape[0], g.shape[1],
                                   _C.dtype_code(g.dtype), float(ctx.p), int(ctx.seed), ctx.step, _C.stream_ptr()),
                 "pg_dropout")
        return g, None, None


_dropout_calls = 0
# device int32 step counter mixed into every dropout seed (set while epochs are replayed from a CUDA graph, where
# the host-side call counter is frozen at capture time)
STEP_DEV = None


def dropout(x: torch.Tensor, p: float, training: bool = True) -> torch.Tensor:
    """model.py:47.  Padded, 16-byte aligned rows go through the mask-free kernel; anything else through torch."""
    global _dropout_calls
    if not training or p == 0.0:
        return x
    ld_ok = x.dim() == 2 and x.is_cuda and x.stride(1) == 1 and (x.stride(0) * x.element_size()) % 16 == 0 \
        and x.data_ptr() % 16 == 0 and x.stride(0) >= (x.shape[1] + 7) // 8 * 8 and x.dtype in (torch.float32, torch.bfloat16)
    if not ld_ok:
        return torch.nn.functional.dropout(x, p, True)
    _dropout_calls += 1
    seed = (torch.initial_seed() * 0x9E3779B97F4A7C15 + _dropout_calls * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF
    return Dropout.apply(x, p, seed)
