"""Alignment accuracy metrics (reference toolbox/metrics.py:92-141).

accuracy_max is computed on the device in the same pass as the loss (row argmax == row index);
accuracy_linear_assignment (the metric training_step actually calls, trainers.py:53,74) runs a batched
shortest-augmenting-path solver on the device (csrc/fgnn_lap.cu) instead of one host scipy call per graph.
"""
import numpy as np
import torch

from .. import _ops
from .losses import _as_batch


def _labels_dev(labels, rows, N1, device):
    """Per-graph index arrays of graph-2 vertices (rows < n1 of graph g) -> (B, N1) int32 on the device, -2 elsewhere."""
    lab = np.full((len(rows), N1), -2, dtype=np.int32)
    for g, n in enumerate(rows):
        lg = np.asarray(labels[g]).reshape(-1)[:n]
        lab[g, :lg.size] = lg
    return torch.from_numpy(lab).to(device)


def _report(hits, sizes, aggregate_score):
    hits = hits.cpu().numpy().astype(np.int64)
    sizes = sizes.cpu().numpy().astype(np.int64)
    if aggregate_score:
        return int(hits.sum()), int(sizes.sum())
    return [h / n for h, n in zip(hits, sizes)]


def accuracy_max(weights, labels=None, aggregate_score=True):
    """(#rows whose arg-max column is the row's label, #rows) or the per-graph accuracies.  weights (B,N1,N2) tensor or
    MaskedTensor; labels: per-graph index arrays of graph-2 vertices, one per row of graph 1 (default: the identity,
    row i <-> column i), compared with the device row arg-max on the device."""
    scores, n_dev, n2_dev, sizes = _as_batch(weights)
    with torch.no_grad():
        _, correct, _, arg = _ops.ce_argmax(scores.detach(), n_dev, n2_dev, want_argmax=labels is not None)
    if labels is not None:
        rows = sizes.cpu().numpy().astype(np.int64)
        correct = (arg == _labels_dev(labels, rows, scores.shape[1], scores.device)).sum(dim=1)
    return _report(correct, sizes, aggregate_score)


def linear_assignment(rawscores):
    """Optimal matchings of a batch on the device (fgnn_lap_pair_fwd): (B,N1,N2) scores -> (col_of_row (B,N1) int32,
    -1 in padded rows and rows left without a column, correct (B,) int32, total_cost (B,) float64).  One CTA per graph
    runs the shortest-augmenting-path algorithm scipy uses, in double precision with scipy's tie rule (transposed when
    n1 > n2, as scipy's rectangular solver does), on cost = -log_softmax(scores) formed in the kernel."""
    from .. import _lib as L
    scores, n_dev, n2_dev, _ = _as_batch(rawscores)
    scores = L.require_cuda_f32(scores.detach(), "rawscores")
    if scores.dim() != 3:
        raise L.FgnnError(f"rawscores must be (B,N1,N2), got {tuple(scores.shape)}")
    G, N1, N2 = scores.shape
    cols = torch.empty((G, N1), dtype=torch.int32, device=scores.device)
    correct = torch.empty(G, dtype=torch.int32, device=scores.device)
    cost = torch.empty(G, dtype=torch.float64, device=scores.device)
    L.check(L.get_lib().fgnn_lap_pair_fwd(L.ptr(scores), L.ptr(cols), L.ptr(correct), L.ptr(cost), G, N1, N2,
                                          _ops._npg(n_dev, G), _ops._npg(n2_dev, G), L.stream_ptr(scores.device)),
            "fgnn_lap_pair_fwd")
    return cols, correct, cost


def accuracy_linear_assignment(rawscores, labels=None, aggregate_score=True):
    """Hungarian matching accuracy (reference toolbox/metrics.py:92-116) computed on the device on
    -log_softmax(scores) as the reference does; only the per-graph hit counts (B int32) travel to the host.  `labels`
    (per-graph index arrays of graph-2 vertices, one per row of graph 1) is compared with the matching on the device."""
    scores, _, _, sizes = _as_batch(rawscores)
    cols, correct, _ = linear_assignment(rawscores)
    if labels is not None:
        rows = sizes.cpu().numpy().astype(np.int64)
        correct = (cols == _labels_dev(labels, rows, scores.shape[1], scores.device)).sum(dim=1)
    return _report(correct, sizes, aggregate_score)
