"""Data-parallel training step for the siamese 2-FGNN (BASELINE.json configs[4]).

The reference trains through pytorch_lightning.Trainer (commander_explore.py:120-123), whose only
multi-GPU mechanism is Lightning's default DDP.  Here one process drives one GPU, the batch of graph
pairs is sharded across ranks, and a training step issues exactly ONE collective: an all-reduce (sum)
of a flat fp32 buffer holding every parameter gradient plus the two scalars of the loss
(sum of row cross-entropies, number of rows).  The loss of toolbox/losses.py:20-34 divides by the
GLOBAL number of rows, so each rank back-propagates its un-normalised local sum and the division
happens once, after the reduction -- exact for ragged shards too.  Forward needs no collective:
GraphNorm statistics are per (graph, channel) (models/layers.py:72-73).
"""
from __future__ import annotations

from typing import Iterable, List, Optional, Tuple

import torch
import torch.distributed as dist


def flat_gradient_allreduce(params: Iterable[torch.nn.Parameter], extras: torch.Tensor,
                            group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """All-reduce (sum) every `p.grad` and the 1-D tensor `extras` in ONE flat buffer.

    Gradients are written back in place; the reduced extras are returned.  Works on any backend
    (NCCL over NVLink on the GPU box, gloo in the CPU tests)."""
    plist: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
    if not plist:
        raise ValueError("no trainable parameters")
    dev = plist[0].device
    sizes = [p.numel() for p in plist]
    flat = torch.empty(sum(sizes) + extras.numel(), dtype=torch.float32, device=dev)
    off = 0
    for p, n in zip(plist, sizes):
        if p.grad is None:
            flat[off:off + n].zero_()
        else:
            flat[off:off + n].copy_(p.grad.reshape(-1))
        off += n
    flat[off:].copy_(extras.to(device=dev, dtype=torch.float32))
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    off = 0
    for p, n in zip(plist, sizes):
        g = flat[off:off + n].view_as(p)
        if p.grad is None:
            p.grad = g.clone()
        else:
            p.grad.copy_(g)
        off += n
    return flat[off:].clone()


class FlatAdam(torch.optim.Optimizer):
    """torch.optim.Adam(lr) of the reference's configure_optimizers (models/trainers.py:92-104) over ONE flat fp32
    buffer (SURVEY 8(f) row 3).  Parameters, gradients and both moments live in flat device buffers (every
    parameter / p.grad is a view), so a data-parallel step is: one memset of the gradient buffer, backward writing
    straight into it (fgnn_embed_bwd accumulates in place), ONE all-reduce of [gradients | sum CE, rows, correct,
    overflow flag], ONE fgnn_adam_step_f32 launch that reads the row count and the overflow flag from the buffer
    itself.  A torch.optim.Optimizer subclass, so ReduceLROnPlateau drives param_groups[0]['lr'] as in the reference."""

    N_EXTRAS = 4      # sum CE, rows, correct, overflow flag (appended to the gradients)

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        params = [p for p in params if p.requires_grad]
        if not params:
            raise ValueError("no trainable parameters")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        from . import _lib as L
        dev = params[0].device
        if dev.type != "cuda":
            raise L.FgnnError("FlatAdam updates parameters with a CUDA kernel (there is no CPU fallback)")
        self.plist = params
        self.sizes = [p.numel() for p in params]
        n = sum(self.sizes)
        self.n = n
        self.flat_p = torch.empty(n, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(n + self.N_EXTRAS, dtype=torch.float32, device=dev)
        self.flat_m = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flat_v = torch.zeros(n, dtype=torch.float32, device=dev)
        self.grad_views = []
        off = 0
        for p, k in zip(params, self.sizes):
            self.flat_p[off:off + k].copy_(p.data.reshape(-1))
            p.data = self.flat_p[off:off + k].view_as(p)          # the parameter now lives in the flat buffer
            self.grad_views.append(self.flat_g[off:off + k].view_as(p))
            off += k
        self.steps_done = 0

    @property
    def extras(self):
        return self.flat_g[self.n:]

    def begin_step(self):
        """Zero the flat gradient buffer, point every p.grad at its view and publish the views as the sink of the
        16-bit backward."""
        from . import _ops
        self.flat_g.zero_()
        _ops.GRAD_SINK.clear()
        for p, gv in zip(self.plist, self.grad_views):
            p.grad = gv
            _ops.GRAD_SINK[p.data_ptr()] = gv.reshape(-1)

    @torch.no_grad()
    def step(self, closure=None):
        """One fused launch.  The gradient divisor (extras[1] = global rows) and the skip flag (extras[3]) are read on
        the device; call after the all-reduce of flat_g."""
        from . import _lib as L
        g = self.param_groups[0]
        L.check(L.get_lib().fgnn_adam_step_f32(L.ptr(self.flat_p), L.ptr(self.flat_g), L.ptr(self.flat_m), L.ptr(self.flat_v),
                                               self.n, float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]),
                                               float(g["eps"]), float(g["weight_decay"]), self.steps_done + 1,
                                               L.ptr(self.flat_g[self.n + 1:]), L.ptr(self.flat_g[self.n + 3:]),
                                               L.stream_ptr(self.flat_p.device)), "fgnn_adam_step_f32")


def train_step_flat(model, opt: "FlatAdam", x1, x2, group: Optional[dist.ProcessGroup] = None, fused_head: bool = False):
    """train_step with the flat trainer: same arithmetic, three framework launches instead of several per parameter
    around the forward / backward (memset, all-reduce, fused Adam).  Returns (global loss, #correct, #rows).
    fused_head (16-bit precisions): the head and its backward run as the fused tensor-core kernels (_ops.HeadFunction)
    instead of the scores, the cross-entropy and their gradients as (B,N,N) tensors; the same loss and gradients."""
    from . import _ops
    from .maskedtensors.maskedtensor import MaskedTensor
    from .toolbox.losses import _as_batch
    from .models.trainers import _head_sizes

    if fused_head and getattr(model, "precision", "fp32") == "fp32":
        raise _ops.L.FgnnError("fused_head is the tensor-core head of the 16-bit precisions; fp32 trains through the "
                               "CUDA-core scores and cross-entropy")
    opt.begin_step()
    try:
        if fused_head:
            e1, e2 = model.embed(x1), model.embed(x2)
            n_dev, n2_dev, sizes = _head_sizes(e1, e2)
            if isinstance(e1, MaskedTensor):
                e1, e2 = e1.tensor.rename(None), e2.tensor.rename(None)
            ce, correct = _ops.HeadFunction.apply(e1, e2, n_dev, model.precision, n2_dev)
        else:
            scores = model(x1, x2)
            plain, n_dev, n2_dev, sizes = _as_batch(scores, loss=True)
            ce, correct = _ops.CrossEntropyIdentityFunction.apply(plain, n_dev, n2_dev)
        local_sum = ce.sum()
        local_sum.backward()                                   # gradients land in opt.flat_g (in place)
    finally:
        # the sink maps parameter addresses of THIS model to its flat buffer: left behind, it would capture the
        # gradients of whatever later reuses those addresses (another model's parameters) and return none to autograd
        _ops.GRAD_SINK.clear()
    grads = opt.flat_g[:opt.n]
    ex = opt.extras
    ex[0] = local_sum.detach()
    ex[1] = sizes.sum()
    ex[2] = correct.sum()
    ex[3] = (~torch.isfinite(grads)).any()                 # fp16 gradient planes overflowed for the current loss scale
    torch.nan_to_num_(grads, nan=0.0, posinf=0.0, neginf=0.0)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(opt.flat_g, op=dist.ReduceOp.SUM, group=group)
    opt.step()                                             # divides by the global row count, skips on overflow (device side)
    ce_all, n_all, ok_all, bad_all = ex.tolist()           # the step's only host synchronisation
    found_inf = bad_all > 0
    if getattr(model, "precision", "fp32") != "fp32":
        _ops.GradScale.update(found_inf)
    if not found_inf:
        opt.steps_done += 1
    return ce_all / max(n_all, 1.0), int(round(ok_all)), int(round(n_all))


def shard_bounds(total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous shard [lo, hi) of `total` pairs for `rank` (sizes differ by at most one)."""
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def train_step(model, optimizer, x1, x2, group: Optional[dist.ProcessGroup] = None):
    """One data-parallel step on this rank's shard (x1, x2: {'input': (b,2,N,N)} dicts or MaskedTensor
    dicts).  Returns (global loss, global #correct, global #rows) as Python numbers."""
    from . import _ops
    from .toolbox.losses import _as_batch

    optimizer.zero_grad(set_to_none=True)
    scores = model(x1, x2)
    plain, n_dev, n2_dev, sizes = _as_batch(scores, loss=True)
    ce, correct = _ops.CrossEntropyIdentityFunction.apply(plain, n_dev, n2_dev)
    local_sum = ce.sum()
    local_sum.backward()                                   # un-normalised: d(sum CE_local)/d theta
    extras = torch.stack((local_sum.detach(), sizes.sum(), correct.sum().to(torch.float32)))
    # fourth extra: 1 if any local gradient is non-finite (fp16 gradient planes overflowed for the current loss scale)
    bad = torch.zeros((), device=local_sum.device)
    for p in model.parameters():
        if p.grad is not None:
            bad = bad + (~torch.isfinite(p.grad)).any().to(bad.dtype)
    for p in model.parameters():                           # keep the flat buffer finite so the loss scalars survive the sum
        if p.grad is not None:
            torch.nan_to_num_(p.grad, nan=0.0, posinf=0.0, neginf=0.0)
    extras = torch.cat((extras, bad.reshape(1)))
    ce_all, n_all, ok_all, bad_all = flat_gradient_allreduce(model.parameters(), extras, group).tolist()
    inv = 1.0 / max(n_all, 1.0)
    found_inf = bad_all > 0
    if getattr(model, "precision", "fp32") != "fp32":
        _ops.GradScale.update(found_inf)                   # every rank sees the same flag: scales stay in lock step
    if found_inf:
        optimizer.zero_grad(set_to_none=True)              # AMP semantics: skip the step, retry with a lower scale
    else:
        for p in model.parameters():
            if p.grad is not None:
                p.grad.mul_(inv)                           # loss = sum CE / sum n  (losses.py:12-13, 34)
        optimizer.step()
    return ce_all * inv, int(round(ok_all)), int(round(n_all))
