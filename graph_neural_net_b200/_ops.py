"""torch.autograd glue over the C ABI: one Function per reference operator.

Each forward/backward is a single call into libfgnn_b200.so on the caller's current CUDA
stream.  Inputs must be CUDA float32 tensors; anything else raises (no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import torch

from . import _lib as L


def _npg(n_dev: Optional[torch.Tensor], G: Optional[int] = None):
    """Device pointer of the int32 per-graph vertex counts (or NULL).  The kernels index other planes with these
    values, so the tensor is checked here: CUDA, int32, contiguous, one entry per graph."""
    if n_dev is None:
        return None
    if not isinstance(n_dev, torch.Tensor) or not n_dev.is_cuda:
        raise L.FgnnError("sizes must be a CUDA tensor (there is no CPU fallback)")
    if n_dev.dtype != torch.int32 or n_dev.dim() != 1 or not n_dev.is_contiguous():
        raise L.FgnnError(f"sizes must be a contiguous 1-D int32 tensor, got {n_dev.dtype} {tuple(n_dev.shape)}")
    if G is not None and n_dev.numel() != G:
        raise L.FgnnError(f"sizes has {n_dev.numel()} entries for a batch of {G} graphs")
    return L.ptr(n_dev)


def check_user_sizes(n_dev: torch.Tensor, G: int, N: int) -> torch.Tensor:
    """Validate caller-supplied vertex counts (one host round trip): 1 <= n_g <= N for every graph."""
    _npg(n_dev, G)
    lo, hi = int(n_dev.min()), int(n_dev.max())
    if lo < 1 or hi > N:
        raise L.FgnnError(f"sizes must satisfy 1 <= n <= {N}; got range [{lo}, {hi}]")
    return n_dev


def make_mlp_params(weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor],
                    gn_w: Optional[torch.Tensor], gn_b: Optional[torch.Tensor], eps: float,
                    keep: list, constant_n: bool = True) -> L.MlpParams:
    """Fill an fgnn_mlp_params from Conv2d/GraphNorm tensors.  `keep` receives every temporary
    that must outlive the C call (contiguous copies)."""
    p = L.MlpParams()
    depth = len(weights)
    if depth > L.FGNN_MAX_DEPTH:
        raise L.FgnnError(f"depth_of_mlp {depth} > {L.FGNN_MAX_DEPTH}")
    w0 = weights[0]
    p.c_in = int(w0.shape[1])
    p.c_out = int(w0.shape[0])
    p.depth = depth
    for k in range(depth):
        w = L.require_cuda_f32(weights[k].detach().reshape(weights[k].shape[0], -1), f"convs[{k}].weight")
        b = biases[k]
        if b is None:
            b = torch.zeros(w.shape[0], device=w.device, dtype=torch.float32)
        b = L.require_cuda_f32(b.detach(), f"convs[{k}].bias")
        keep += [w, b]
        p.w[k] = w.data_ptr()
        p.b[k] = b.data_ptr()
    if gn_w is not None:
        gw = L.require_cuda_f32(gn_w.detach().reshape(-1), "gn.weight")
        gb = L.require_cuda_f32(gn_b.detach().reshape(-1), "gn.bias")
        keep += [gw, gb]
        p.gn_w = gw.data_ptr()
        p.gn_b = gb.data_ptr()
    else:
        p.gn_w = None
        p.gn_b = None
    p.eps = float(eps)
    p.constant_n = 1 if constant_n else 0
    return p


class MlpFunction(torch.autograd.Function):
    """MlpBlock_Real forward/backward (reference models/layers.py:109-131)."""

    @staticmethod
    def forward(ctx, x, n_dev, eps, depth, constant_n, gn_w, gn_b, *wb):
        lib = L.get_lib()
        x = L.require_cuda_f32(x, "x")
        weights, biases = wb[:depth], wb[depth:]
        keep = []
        p = make_mlp_params(weights, biases, gn_w, gn_b, eps, keep, constant_n)
        G, Ci, N, N2 = x.shape
        if N != N2 or Ci != p.c_in:
            raise L.FgnnError(f"MlpBlock_Real: bad input shape {tuple(x.shape)} for c_in={p.c_in}")
        y = torch.empty((G, p.c_out, N, N), device=x.device, dtype=torch.float32)
        stats = torch.empty((G, p.c_out, 2), device=x.device, dtype=torch.float32)
        nbytes = lib.fgnn_mlp_workspace_bytes(G, p.c_in, p.c_out, p.depth, N)
        ws = L.workspace(x.device, nbytes)
        L.check(lib.fgnn_mlp_fwd_f32(C.byref(p), L.ptr(x), L.ptr(y), L.ptr(stats), G, N, _npg(n_dev),
                                     L.ptr(ws), ws.numel(), L.stream_ptr(x.device)), "fgnn_mlp_fwd_f32")
        ctx.save_for_backward(x, stats, n_dev if n_dev is not None else torch.empty(0), gn_w, gn_b, *wb)
        ctx.has_n = n_dev is not None
        ctx.eps, ctx.depth, ctx.constant_n = eps, depth, constant_n
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = L.get_lib()
        x, stats, n_dev, gn_w, gn_b, *wb = ctx.saved_tensors
        n_dev = n_dev if ctx.has_n else None
        depth = ctx.depth
        weights, biases = wb[:depth], wb[depth:]
        keep = []
        p = make_mlp_params(weights, biases, gn_w, gn_b, ctx.eps, keep, ctx.constant_n)
        g = L.MlpGrads()
        dws = [torch.zeros_like(w, dtype=torch.float32).reshape(w.shape[0], -1).contiguous() for w in weights]
        dbs = [torch.zeros(w.shape[0], device=x.device, dtype=torch.float32) for w in weights]
        dgw = torch.zeros(p.c_out, device=x.device, dtype=torch.float32)
        dgb = torch.zeros(p.c_out, device=x.device, dtype=torch.float32)
        for k in range(depth):
            g.w[k] = dws[k].data_ptr()
            g.b[k] = dbs[k].data_ptr()
        g.gn_w, g.gn_b = dgw.data_ptr(), dgb.data_ptr()
        G, Ci, N, _ = x.shape
        dy = L.require_cuda_f32(dy, "dy")
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        nbytes = lib.fgnn_mlp_workspace_bytes(G, p.c_in, p.c_out, p.depth, N)
        ws = L.workspace(x.device, nbytes)
        L.check(lib.fgnn_mlp_bwd_f32(C.byref(p), C.byref(g), L.ptr(x), L.ptr(stats), L.ptr(dy), L.ptr(dx),
                                     G, N, _npg(n_dev), L.ptr(ws), ws.numel(), L.stream_ptr(x.device)),
                "fgnn_mlp_bwd_f32")
        grads_w = [dws[k].reshape(weights[k].shape) for k in range(depth)]
        grads_b = [dbs[k] if biases[k] is not None else None for k in range(depth)]
        return (dx, None, None, None, None,
                dgw.reshape(gn_w.shape) if gn_w is not None else None,
                dgb.reshape(gn_b.shape) if gn_b is not None else None, *grads_w, *grads_b)


class MatmulFunction(torch.autograd.Function):
    """Matmul.forward = torch.matmul over the last two dims (reference models/layers.py:161-162)."""

    @staticmethod
    def forward(ctx, a, b, n_dev):
        lib = L.get_lib()
        a = L.require_cuda_f32(a, "xs1")
        b = L.require_cuda_f32(b, "xs2")
        if a.shape != b.shape or a.dim() != 4 or a.shape[-1] != a.shape[-2]:
            raise L.FgnnError(f"Matmul: expected two (B,C,N,N) tensors, got {tuple(a.shape)} {tuple(b.shape)}")
        G, Cc, N, _ = a.shape
        out = torch.empty_like(a)
        L.check(lib.fgnn_matmul_fwd_f32(L.ptr(a), L.ptr(b), L.ptr(out), G, Cc, N, _npg(n_dev),
                                        L.stream_ptr(a.device)), "fgnn_matmul_fwd_f32")
        ctx.save_for_backward(a, b, n_dev if n_dev is not None else torch.empty(0))
        ctx.has_n = n_dev is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = L.get_lib()
        a, b, n_dev = ctx.saved_tensors
        n_dev = n_dev if ctx.has_n else None
        dout = L.require_cuda_f32(dout, "dout")
        G, Cc, N, _ = a.shape
        da = torch.empty_like(a) if ctx.needs_input_grad[0] else None
        db = torch.empty_like(b) if ctx.needs_input_grad[1] else None
        L.check(lib.fgnn_matmul_bwd_f32(L.ptr(a), L.ptr(b), L.ptr(dout), L.ptr(da), L.ptr(db), G, Cc, N,
                                        _npg(n_dev), L.stream_ptr(a.device)), "fgnn_matmul_bwd_f32")
        return da, db, None


class ColMaxFunction(torch.autograd.Function):
    """ColumnMaxPooling.forward = torch.max(x, -1)[0] (reference models/layers.py:194-203)."""

    @staticmethod
    def forward(ctx, x, n_dev):
        lib = L.get_lib()
        x = L.require_cuda_f32(x, "x")
        G, Cc, N, M = x.shape
        if N != M:
            raise L.FgnnError("ColumnMaxPooling: expected (B,C,N,N)")
        out = torch.empty((G, Cc, N), device=x.device, dtype=torch.float32)
        arg = torch.empty((G, Cc, N), device=x.device, dtype=torch.int32)
        L.check(lib.fgnn_colmax_fwd_f32(L.ptr(x), L.ptr(out), L.ptr(arg), G, Cc, N, _npg(n_dev),
                                        L.stream_ptr(x.device)), "fgnn_colmax_fwd_f32")
        ctx.save_for_backward(arg, n_dev if n_dev is not None else torch.empty(0))
        ctx.has_n = n_dev is not None
        ctx.shape = x.shape
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = L.get_lib()
        arg, n_dev = ctx.saved_tensors
        n_dev = n_dev if ctx.has_n else None
        dout = L.require_cuda_f32(dout, "dout")
        G, Cc, N, _ = ctx.shape
        dx = torch.empty(ctx.shape, device=dout.device, dtype=torch.float32)
        L.check(lib.fgnn_colmax_bwd_f32(L.ptr(dout), L.ptr(arg), L.ptr(dx), G, Cc, N, _npg(n_dev),
                                        L.stream_ptr(dout.device)), "fgnn_colmax_bwd_f32")
        return dx, None


def _save_sizes(*sizes):
    """Size tensors for ctx.save_for_backward (an empty placeholder for None) and which of them were given."""
    return [n if n is not None else torch.empty(0) for n in sizes], [n is not None for n in sizes]


def _saved_sizes(saved, given):
    return [n if g else None for n, g in zip(saved, given)]


def _pair_shapes(e1: torch.Tensor, e2: torch.Tensor, what: str):
    """(G, C, N1, N2) of graph 1's (G,C,N1) and graph 2's (G,C,N2) node vectors."""
    if e1.dim() != 3 or e2.dim() != 3 or e1.shape[:2] != e2.shape[:2]:
        raise L.FgnnError(f"{what}: embeddings must be (G,C,N1) and (G,C,N2) with the same G and C, got "
                          f"{tuple(e1.shape)} and {tuple(e2.shape)}")
    return e1.shape[0], e1.shape[1], e1.shape[2], e2.shape[2]


class ScoresFunction(torch.autograd.Function):
    """scores[b] = e1[b]^T e2[b] (reference models/trainers.py:67): e1 (G,C,N1), e2 (G,C,N2) -> (G,N1,N2), zero outside
    each graph's n1 x n2 block.  n2_dev (graph 2's sizes) defaults to n_dev."""

    @staticmethod
    def forward(ctx, e1, e2, n_dev, n2_dev=None):
        lib = L.get_lib()
        e1 = L.require_cuda_f32(e1, "e1")
        e2 = L.require_cuda_f32(e2, "e2")
        G, Cc, N1, N2 = _pair_shapes(e1, e2, "siamese head")
        n2_dev = n_dev if n2_dev is None else n2_dev
        s = torch.empty((G, N1, N2), device=e1.device, dtype=torch.float32)
        L.check(lib.fgnn_scores_pair_fwd_f32(L.ptr(e1), L.ptr(e2), L.ptr(s), G, Cc, N1, N2, _npg(n_dev, G), _npg(n2_dev, G),
                                             L.stream_ptr(e1.device)), "fgnn_scores_pair_fwd_f32")
        saved, ctx.given = _save_sizes(n_dev, n2_dev)
        ctx.save_for_backward(e1, e2, *saved)
        return s

    @staticmethod
    def backward(ctx, ds):
        lib = L.get_lib()
        e1, e2, *saved = ctx.saved_tensors
        n_dev, n2_dev = _saved_sizes(saved, ctx.given)
        ds = L.require_cuda_f32(ds, "dscores")
        G, Cc, N1, N2 = _pair_shapes(e1, e2, "siamese head")
        de1, de2 = torch.empty_like(e1), torch.empty_like(e2)
        L.check(lib.fgnn_scores_pair_bwd_f32(L.ptr(e1), L.ptr(e2), L.ptr(ds), L.ptr(de1), L.ptr(de2), G, Cc, N1, N2,
                                             _npg(n_dev), _npg(n2_dev), L.stream_ptr(e1.device)), "fgnn_scores_pair_bwd_f32")
        return de1, de2, None, None


def ce_argmax(scores: torch.Tensor, n_dev=None, n2_dev=None, want_argmax: bool = False):
    """fgnn_ce_pair_argmax_fwd_f32 on (G,N1,N2) scores -> (ce_sum[G], correct[G], row_lse (G,N1), row_argmax (G,N1) or
    None).  Row i's target is column i; rows i >= n2 have none.  n2_dev defaults to n_dev."""
    lib = L.get_lib()
    scores = L.require_cuda_f32(scores, "raw_scores")
    if scores.dim() != 3:
        raise L.FgnnError(f"raw_scores must be (B,N1,N2), got {tuple(scores.shape)}")
    G, N1, N2 = scores.shape
    n2_dev = n_dev if n2_dev is None else n2_dev
    ce = torch.empty(G, device=scores.device, dtype=torch.float32)
    correct = torch.empty(G, device=scores.device, dtype=torch.int32)
    lse = torch.empty((G, N1), device=scores.device, dtype=torch.float32)
    arg = torch.empty((G, N1), device=scores.device, dtype=torch.int32) if want_argmax else None
    ws = L.workspace(scores.device, lib.fgnn_ce_workspace_bytes(G, N1))
    L.check(lib.fgnn_ce_pair_argmax_fwd_f32(L.ptr(scores), L.ptr(ce), L.ptr(correct), L.ptr(lse), L.ptr(arg), G, N1, N2,
                                            _npg(n_dev, G), _npg(n2_dev, G), L.ptr(ws), ws.numel(),
                                            L.stream_ptr(scores.device)), "fgnn_ce_pair_argmax_fwd_f32")
    return ce, correct, lse, arg


class CrossEntropyIdentityFunction(torch.autograd.Function):
    """Per-graph sum_i CE(scores[i,:], i) (reference toolbox/losses.py:27-31), with the row argmax
    count as a by-product (toolbox/metrics.py:125-134).  Returns (ce_sum[G], correct[G]).  scores (G,N1,N2); the
    softmax of row i runs over graph 2's n2 valid columns (n2_dev, default n_dev) and rows i >= n2 have no target."""

    @staticmethod
    def forward(ctx, scores, n_dev, n2_dev=None):
        n2_dev = n_dev if n2_dev is None else n2_dev
        ce, correct, lse, _ = ce_argmax(scores, n_dev, n2_dev)
        saved, ctx.given = _save_sizes(n_dev, n2_dev)
        ctx.save_for_backward(scores, lse, *saved)
        ctx.mark_non_differentiable(correct)
        return ce, correct

    @staticmethod
    def backward(ctx, dce, _dcorrect):
        lib = L.get_lib()
        scores, lse, *saved = ctx.saved_tensors
        n_dev, n2_dev = _saved_sizes(saved, ctx.given)
        G, N1, N2 = scores.shape
        coef = L.require_cuda_f32(dce, "dce")
        ds = torch.empty_like(scores)
        L.check(lib.fgnn_ce_pair_bwd_f32(L.ptr(scores), L.ptr(lse), L.ptr(coef), L.ptr(ds), G, N1, N2, _npg(n_dev),
                                         _npg(n2_dev), L.stream_ptr(scores.device)), "fgnn_ce_pair_bwd_f32")
        return ds, None, None


def generate_pairs(generator: int, G: int, N: int, edge_density: float, noise: float, seed: int, n_dev=None, device="cuda"):
    """fgnn_generate_pairs_u8: (adj1, adj2) uint8 (G,N,N) CUDA tensors (reference loaders/data_generator.py:39-87)."""
    lib = L.get_lib()
    dev = torch.device(device)
    if dev.type != "cuda":
        raise L.FgnnError("graph pairs are generated by a CUDA kernel (there is no CPU fallback)")
    if n_dev is not None:
        check_user_sizes(n_dev, G, N)
    adj1 = torch.empty((G, N, N), dtype=torch.uint8, device=dev)
    adj2 = torch.empty((G, N, N), dtype=torch.uint8, device=dev)
    ws = L.workspace(dev, lib.fgnn_generate_workspace_bytes(G, N, generator))
    L.check(lib.fgnn_generate_pairs_u8(L.ptr(adj1), L.ptr(adj2), G, N, _npg(n_dev, G), generator, edge_density, noise,
                                       seed & 0xFFFFFFFFFFFFFFFF, L.ptr(ws), ws.numel(), L.stream_ptr(dev)),
            "fgnn_generate_pairs_u8")
    return adj1, adj2


def _head_operands(e1: torch.Tensor, e2: torch.Tensor, precision: str, what: str):
    """Checked (G,C,N1), (G,C,N2) fp32 operands of the tensor-core head, C zero-padded to a multiple of 16 (K of the
    MMA; zero channels add nothing to e1^T e2) -> (e1, e2, padded C)."""
    e1 = L.require_cuda_f32(e1, "e1")
    e2 = L.require_cuda_f32(e2, "e2")
    _pair_shapes(e1, e2, what)
    if precision not in ("bf16", "fp16"):
        raise L.FgnnError(f"{what} is the tensor-core head (bf16 / fp16 operand splitting); fp32 uses the CUDA-core operators")
    Cc = e1.shape[1]
    if Cc % 16:
        pad = 16 - Cc % 16
        e1 = torch.nn.functional.pad(e1, (0, 0, 0, pad)).contiguous()
        e2 = torch.nn.functional.pad(e2, (0, 0, 0, pad)).contiguous()
        Cc += pad
    return e1, e2, Cc


def head_fused(e1: torch.Tensor, e2: torch.Tensor, n_dev, precision: str = "fp16", want_scores: bool = False, n2_dev=None):
    """Fused siamese head on tensor cores (fgnn_head_pair_fwd): e1 (G,C,N1), e2 (G,C,N2) -> (ce_sum[G], correct[G],
    scores (G,N1,N2) or None).  scores = e1^T e2 (reference models/trainers.py:67), ce_sum / correct as
    CrossEntropyIdentityFunction (toolbox/losses.py:27-33, toolbox/metrics.py:125-134); the scores are only materialised
    on request.  n2_dev (graph 2's sizes) defaults to n_dev.  Forward only: under autograd use HeadFunction (or
    ScoresFunction + CrossEntropyIdentityFunction)."""
    lib = L.get_lib()
    e1, e2, Cc = _head_operands(e1, e2, precision, "head_fused")
    G, _, N1 = e1.shape
    N2 = e2.shape[2]
    n2_dev = n_dev if n2_dev is None else n2_dev
    ce = torch.empty(G, device=e1.device, dtype=torch.float32)
    correct = torch.empty(G, device=e1.device, dtype=torch.int32)
    scores = torch.empty((G, N1, N2), device=e1.device, dtype=torch.float32) if want_scores else None
    ws = L.workspace(e1.device, lib.fgnn_head_pair_workspace_bytes(G, N1))
    L.check(lib.fgnn_head_pair_fwd(L.PRECISIONS[precision], L.ptr(e1), L.ptr(e2), L.ptr(scores) if want_scores else None,
                                   L.ptr(ce), L.ptr(correct), G, Cc, N1, N2, _npg(n_dev, G), _npg(n2_dev, G), L.ptr(ws),
                                   ws.numel(), L.stream_ptr(e1.device)), "fgnn_head_pair_fwd")
    return ce, correct, scores


class HeadFunction(torch.autograd.Function):
    """Differentiable fused head (fgnn_head_pair_fwd_train / fgnn_head_pair_bwd): e1 (G,C,N1), e2 (G,C,N2) ->
    (ce_sum[G], correct[G]), what ScoresFunction + CrossEntropyIdentityFunction compute (models/trainers.py:67,
    toolbox/losses.py:27-31, toolbox/metrics.py:125-134) without the (G,N1,N2) scores or their gradient.  16-bit
    precisions only; correct is not differentiable; n2_dev (graph 2's sizes) defaults to n_dev."""

    @staticmethod
    def forward(ctx, e1, e2, n_dev, precision, n2_dev=None):
        lib = L.get_lib()
        c_in = e1.shape[1] if e1.dim() == 3 else None
        e1, e2, Cc = _head_operands(e1, e2, precision, "HeadFunction")
        G, _, N1 = e1.shape
        N2 = e2.shape[2]
        n2_dev = n_dev if n2_dev is None else n2_dev
        ce = torch.empty(G, device=e1.device, dtype=torch.float32)
        correct = torch.empty(G, device=e1.device, dtype=torch.int32)
        lse = torch.empty((G, N1), device=e1.device, dtype=torch.float32)
        ws = L.workspace(e1.device, lib.fgnn_head_pair_workspace_bytes(G, N1))
        L.check(lib.fgnn_head_pair_fwd_train(L.PRECISIONS[precision], L.ptr(e1), L.ptr(e2), L.ptr(ce), L.ptr(correct),
                                             L.ptr(lse), G, Cc, N1, N2, _npg(n_dev, G), _npg(n2_dev, G), L.ptr(ws),
                                             ws.numel(), L.stream_ptr(e1.device)), "fgnn_head_pair_fwd_train")
        saved, ctx.given = _save_sizes(n_dev, n2_dev)
        ctx.save_for_backward(e1, e2, lse, *saved)
        ctx.precision, ctx.c_in = precision, c_in
        ctx.mark_non_differentiable(correct)
        return ce, correct

    @staticmethod
    def backward(ctx, dce, _dcorrect):
        lib = L.get_lib()
        e1, e2, lse, *saved = ctx.saved_tensors
        n_dev, n2_dev = _saved_sizes(saved, ctx.given)
        G, Cc, N1 = e1.shape
        N2 = e2.shape[2]
        coef = L.require_cuda_f32(dce, "dce")
        de1, de2 = torch.empty_like(e1), torch.empty_like(e2)
        L.check(lib.fgnn_head_pair_bwd(L.PRECISIONS[ctx.precision], L.ptr(e1), L.ptr(e2), L.ptr(lse), L.ptr(coef),
                                       L.ptr(de1), L.ptr(de2), G, Cc, N1, N2, _npg(n_dev, G), _npg(n2_dev, G), None, 0,
                                       L.stream_ptr(e1.device)), "fgnn_head_pair_bwd")
        if Cc != ctx.c_in:
            de1, de2 = de1[:, :ctx.c_in], de2[:, :ctx.c_in]
        return de1, de2, None, None, None


def graphnorm_fwd(x: torch.Tensor, n_dev, gn_w, gn_b, eps: float, constant_n: bool = True) -> torch.Tensor:
    """GraphNorm / normalize forward (reference models/layers.py:68-80); no autograd (use MlpBlock_Real
    for training -- the standalone norm is not on the training path)."""
    lib = L.get_lib()
    x = L.require_cuda_f32(x, "b")
    G, Cc, N, M = x.shape
    if N != M:
        raise L.FgnnError("GraphNorm expects (B,C,N,N)")
    y = torch.empty_like(x)
    stats = torch.empty((G, Cc, 2), device=x.device, dtype=torch.float32)
    gw = L.require_cuda_f32(gn_w.detach().reshape(-1), "weight") if gn_w is not None else None
    gb = L.require_cuda_f32(gn_b.detach().reshape(-1), "bias") if gn_b is not None else None
    L.check(lib.fgnn_graphnorm_fwd_f32(L.ptr(x), L.ptr(y), L.ptr(stats), L.ptr(gw), L.ptr(gb), float(eps),
                                       1 if constant_n else 0, G, Cc, N, _npg(n_dev, G), L.stream_ptr(x.device)),
            "fgnn_graphnorm_fwd_f32")
    return y


def features_from_adjacency(adj: torch.Tensor, n_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Batch of adjacency matrices (G,N,N) uint8/bool on the GPU -> padded (G,2,N,N) float32 features
    B[0]=W, B[1]=diag(W.sum(1)) (reference loaders/data_generator.py:118-125 + maskedtensor.from_list padding)."""
    lib = L.get_lib()
    if not adj.is_cuda:
        raise L.FgnnError("adjacency must be a CUDA tensor (there is no CPU fallback)")
    if adj.dtype == torch.bool:
        adj = adj.view(torch.uint8)
    if adj.dtype != torch.uint8 or adj.dim() != 3 or adj.shape[1] != adj.shape[2]:
        raise L.FgnnError("adjacency must be (G,N,N) uint8 or bool")
    adj = adj.contiguous()
    G, N, _ = adj.shape
    out = torch.empty((G, 2, N, N), device=adj.device, dtype=torch.float32)
    L.check(lib.fgnn_features_from_adjacency_u8(L.ptr(adj), L.ptr(out), G, N, _npg(n_dev), L.stream_ptr(adj.device)),
            "fgnn_features_from_adjacency_u8")
    return out


def embed_fwd(params: L.EmbedParams, precision: int, x: torch.Tensor, c_out: int,
              n_dev: Optional[torch.Tensor]) -> torch.Tensor:
    """Fused node_embedding forward: x (G,c_in,N,N) -> (G,C,N)."""
    lib = L.get_lib()
    x = L.require_cuda_f32(x, "input")
    G, _, N, M = x.shape
    if N != M:
        raise L.FgnnError("input must be (B,F,N,N)")
    emb = torch.empty((G, c_out, N), device=x.device, dtype=torch.float32)
    nbytes = lib.fgnn_embed_workspace_bytes(C.byref(params), precision, G, N)
    if nbytes == 0:
        raise L.FgnnError("fgnn_embed_workspace_bytes returned 0: " + lib.fgnn_last_error().decode())
    ws = L.workspace(x.device, nbytes)
    L.check(lib.fgnn_embed_fwd(C.byref(params), precision, L.ptr(x), L.ptr(emb), G, N, _npg(n_dev), L.ptr(ws),
                               ws.numel(), L.stream_ptr(x.device)), "fgnn_embed_fwd")
    return emb


def embed_fwd_adjacency(params: L.EmbedParams, precision: int, adj: torch.Tensor, c_out: int,
                        n_dev: Optional[torch.Tensor]) -> torch.Tensor:
    """Fused node_embedding forward fed from a (G,N,N) uint8/bool adjacency batch (16-bit precisions only): the
    input features W, diag(deg) are built on the device directly in the kernels' plane layout."""
    lib = L.get_lib()
    if not adj.is_cuda:
        raise L.FgnnError("adjacency must be a CUDA tensor (there is no CPU fallback)")
    if adj.dtype == torch.bool:
        adj = adj.view(torch.uint8)
    if adj.dtype != torch.uint8 or adj.dim() != 3 or adj.shape[1] != adj.shape[2]:
        raise L.FgnnError("adjacency must be (G,N,N) uint8 or bool")
    adj = adj.contiguous()
    G, N, _ = adj.shape
    emb = torch.empty((G, c_out, N), device=adj.device, dtype=torch.float32)
    nbytes = lib.fgnn_embed_workspace_bytes(C.byref(params), precision, G, N)
    if nbytes == 0:
        raise L.FgnnError("fgnn_embed_workspace_bytes returned 0: " + lib.fgnn_last_error().decode())
    ws = L.workspace(adj.device, nbytes)
    L.check(lib.fgnn_embed_fwd_adjacency_u8(C.byref(params), precision, L.ptr(adj), L.ptr(emb), G, N, _npg(n_dev),
                                            L.ptr(ws), ws.numel(), L.stream_ptr(adj.device)),
            "fgnn_embed_fwd_adjacency_u8")
    return emb


def embed_params_from_flat(spec, flat, keep) -> L.EmbedParams:
    """spec: per block a 3-tuple of (depth, eps, constant_n, has_gn) for mlp1, mlp2, mlp3; flat: the tensors in the
    order [weights[0..d-1], biases[0..d-1], (gn.weight, gn.bias)] per MLP."""
    p = L.EmbedParams()
    p.num_blocks = len(spec)
    it = iter(flat)
    for i, trio in enumerate(spec):
        for name, (depth, eps, cst, has_gn) in zip(("mlp1", "mlp2", "mlp3"), trio):
            ws = [next(it) for _ in range(depth)]
            bs = [next(it) for _ in range(depth)]
            gw, gb = (next(it), next(it)) if has_gn else (None, None)
            setattr(p.block[i], name, make_mlp_params(ws, bs, gw, gb, eps, keep, cst))
    return p


class GradScale:
    """Loss scale of the 16-bit backward, the reference's AMP GradScaler in power-of-two form (Lightning precision=16,
    commander_explore.py:120): fgnn_embed_bwd scales max |d emb| to 2^log2; a step whose gradients overflowed is
    skipped and log2 is lowered by `backoff`; after `growth_interval` clean steps it is raised by one again."""
    log2 = 9
    max_log2 = 9
    min_log2 = -24
    backoff = 3
    growth_interval = 200
    _good = 0

    @classmethod
    def update(cls, found_inf: bool):
        if found_inf:
            cls.log2 = max(cls.min_log2, cls.log2 - cls.backoff)
            cls._good = 0
        else:
            cls._good += 1
            if cls._good >= cls.growth_interval and cls.log2 < cls.max_log2:
                cls.log2 += 1
                cls._good = 0


# Gradient sink of the flat trainer (training.FlatAdam): data_ptr of a parameter -> the fp32 view of the flat gradient
# buffer that receives its gradient.  fgnn_embed_bwd ACCUMULATES into its output buffers, so the 16-bit backward
# writes straight into the flat buffer (no per-parameter zeros / adds / copies) and returns no autograd gradient.
GRAD_SINK = {}


class EmbedTrainFunction(torch.autograd.Function):
    """node_embedding forward + backward in a 16-bit precision with every contraction on tcgen05
    (fgnn_embed_fwd_train / fgnn_embed_bwd): what autograd does to Network.forward under the reference's
    precision=16 trainer (models/trainers.py:70-76, commander_explore.py:120-123).  The forward's workspace holds the
    activations until backward; parameter gradients come back in fp32."""

    @staticmethod
    def forward(ctx, x, n_dev, spec, precision, c_out, *flat):
        lib = L.get_lib()
        x = L.require_cuda_f32(x, "input")
        G, _, N, M = x.shape
        if N != M:
            raise L.FgnnError("input must be (B,F,N,N)")
        keep = []
        params = embed_params_from_flat(spec, flat, keep)
        nbytes = lib.fgnn_embed_train_workspace_bytes(C.byref(params), precision, G, N)
        if nbytes == 0:
            raise L.FgnnError("fgnn_embed_train_workspace_bytes returned 0: " + lib.fgnn_last_error().decode())
        ws = L.private_workspace(x.device, nbytes)
        emb = torch.empty((G, c_out, N), device=x.device, dtype=torch.float32)
        L.check(lib.fgnn_embed_fwd_train(C.byref(params), precision, L.ptr(x), L.ptr(emb), G, N, _npg(n_dev, G),
                                         L.ptr(ws), ws.numel(), L.stream_ptr(x.device)), "fgnn_embed_fwd_train")
        ctx.ws, ctx.spec, ctx.precision, ctx.shape = ws, spec, precision, (G, N)
        ctx.has_n = n_dev is not None
        ctx.save_for_backward(n_dev if n_dev is not None else torch.empty(0), *flat)
        return emb

    @staticmethod
    def backward(ctx, demb):
        lib = L.get_lib()
        n_dev, *flat = ctx.saved_tensors
        n_dev = n_dev if ctx.has_n else None
        G, N = ctx.shape
        keep = []
        params = embed_params_from_flat(ctx.spec, flat, keep)
        grads = L.EmbedGrads()
        grads.num_blocks = len(ctx.spec)
        out = []
        it = iter(flat)
        for i, trio in enumerate(ctx.spec):
            for name, (depth, eps, cst, has_gn) in zip(("mlp1", "mlp2", "mlp3"), trio):
                mg = getattr(grads.block[i], name)
                ws_ = [next(it) for _ in range(depth)]
                bs_ = [next(it) for _ in range(depth)]
                tensors = ws_ + bs_ + ([next(it), next(it)] if has_gn else [])
                bufs = []
                for t in tensors:
                    if t is None:
                        bufs.append(None)
                        out.append(None)
                        continue
                    sink = GRAD_SINK.get(t.data_ptr())
                    if sink is not None and sink.numel() == t.numel():
                        bufs.append(sink)                 # accumulate in place in the trainer's flat buffer
                        out.append(None)
                    else:
                        g = torch.zeros(t.numel(), device=demb.device, dtype=torch.float32)
                        bufs.append(g)
                        out.append(g.reshape(t.shape))
                for k in range(depth):
                    mg.w[k] = bufs[k].data_ptr()
                    mg.b[k] = bufs[depth + k].data_ptr() if bufs[depth + k] is not None else None
                if has_gn:
                    mg.gn_w, mg.gn_b = bufs[2 * depth].data_ptr(), bufs[2 * depth + 1].data_ptr()
                keep += bufs
        demb = L.require_cuda_f32(demb, "d emb")
        ws = ctx.ws
        L.check(lib.fgnn_embed_bwd(C.byref(params), C.byref(grads), ctx.precision, L.ptr(demb), GradScale.log2, G, N, _npg(n_dev, G),
                                   L.ptr(ws), ws.numel(), L.stream_ptr(demb.device)), "fgnn_embed_bwd")
        ctx.ws = None
        return (None, None, None, None, None, *out)
