"""Row-softmax cross-entropy against the identity matching, one fused CUDA pass for the batch.

Mirror of the reference toolbox/losses.py:8-34: triplet_loss(loss_reduction='mean'|'mean_of_mean').
The reference loops over graphs in Python and launches one CrossEntropyLoss per graph; here the
whole (B,N1,N2) batch (dense or MaskedTensor) goes through fgnn_ce_pair_argmax_fwd_f32, which returns the
per-graph CE sums; the reduction over graphs is a handful of scalar ops.
"""
import torch
import torch.nn as nn

from .. import _ops
from ..maskedtensors.maskedtensor import MaskedTensor


def check_loss_sizes(n1, n2):
    """The loss keeps the reference's ground truth, row i <-> column i, so it is defined when every graph 1 has at
    most as many vertices as its graph 2 (CrossEntropyLoss(out, arange(n1)) over n2 columns).  n1, n2: per-pair sizes."""
    for g, (a, b) in enumerate(zip(n1, n2)):
        if a > b:
            raise ValueError(f"the identity-matching loss needs n1 <= n2 for every pair (row i's target is column i); "
                             f"pair {g} has n1={a} > n2={b}")


def _as_batch(raw_scores, loss=False):
    """-> (scores (B,N1,N2) plain tensor, row sizes, column sizes (int32 device tensors or None), float row sizes (B,)).
    loss=True refuses pairs whose rows outnumber their columns (check_loss_sizes)."""
    if isinstance(raw_scores, MaskedTensor):
        t = raw_scores.tensor.rename(None)
        rows, cols = raw_scores.tensor.names[1], raw_scores.tensor.names[2]
        n_dev = raw_scores.sizes_i32(t.device, name=rows)
        n2_dev = raw_scores.sizes_i32(t.device, name=cols)
        if loss:
            check_loss_sizes(raw_scores.sizes_host(rows), raw_scores.sizes_host(cols))
        return t, n_dev, n2_dev, n_dev.to(torch.float32)
    if isinstance(raw_scores, (list, tuple)):
        raise TypeError("pass a (B,N1,N2) tensor or a MaskedTensor (build one with maskedtensor.from_list)")
    if loss:
        check_loss_sizes([raw_scores.shape[1]], [raw_scores.shape[2]])
    sizes = torch.full((raw_scores.shape[0],), float(raw_scores.shape[1]), device=raw_scores.device)
    return raw_scores, None, None, sizes


class triplet_loss(nn.Module):
    def __init__(self, loss_reduction='mean', loss=None):
        super().__init__()
        if loss is not None and not (isinstance(loss, nn.CrossEntropyLoss) and loss.reduction == 'sum'):
            raise NotImplementedError("only CrossEntropyLoss(reduction='sum') is fused")
        if loss_reduction not in ('mean', 'mean_of_mean'):
            raise ValueError('Unknown loss_reduction parameters {}'.format(loss_reduction))
        self.loss_reduction = loss_reduction

    def forward(self, raw_scores):
        """raw_scores: (bs, n1, n2) tensor or MaskedTensor, n1 <= n2 per pair -> scalar (rows = the loss's divisor)."""
        scores, n_dev, n2_dev, sizes = _as_batch(raw_scores, loss=True)
        ce, _ = _ops.CrossEntropyIdentityFunction.apply(scores, n_dev, n2_dev)
        if self.loss_reduction == 'mean':
            return ce.sum() / sizes.sum()
        return (ce / sizes).sum() / ce.shape[0]
