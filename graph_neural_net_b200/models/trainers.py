"""Siamese node-embedding model: shared 2-FGNN embedder on both graphs, E1^T E2 scores.

Mirror of the reference models/trainers.py:8-104 (same constructor, registries, step functions and
optimizer recipe).  pytorch_lightning is optional: when it is not installed the class derives from
nn.Module and `log` is a no-op, which is all the hot path needs.
"""
import torch
import torch.nn as nn

from .. import _ops
from ..toolbox.losses import triplet_loss, _as_batch, check_loss_sizes
from ..toolbox.metrics import accuracy_max, accuracy_linear_assignment
from ..maskedtensors.maskedtensor import MaskedTensor
from .blocks_emb import node_embedding, block_emb, block
from .utils import Network

try:                                     # pragma: no cover - not installed in this image
    import pytorch_lightning as pl
    _Base = pl.LightningModule
except Exception:                        # noqa: BLE001
    class _Base(nn.Module):
        def log(self, *args, **kwargs):
            pass

get_node_emb = {'node_embedding': node_embedding}
get_block_init = {'block_emb': block_emb}
get_block_inside = {'block': block}


def _lookup(table, key, what):
    if key not in table:
        raise NotImplementedError(f"{what} {key} is not implemented")
    return table[key]


def _head_sizes(e1, e2):
    """Embeddings of both sides -> (graph 1's sizes, graph 2's sizes (int32 device tensors or None), float sizes of
    graph 1 (B,)), after refusing pairs the identity loss is not defined on (n1 > n2)."""
    if isinstance(e1, MaskedTensor):
        check_loss_sizes(e1.sizes_host(), e2.sizes_host())
        n_dev = e1.sizes_i32()
        return n_dev, e2.sizes_i32(), n_dev.to(torch.float32)
    check_loss_sizes([e1.shape[-1]], [e2.shape[-1]])
    return None, None, torch.full((e1.shape[0],), float(e1.shape[-1]), device=e1.device)


class Siamese_Node_Exp(_Base):
    def __init__(self, original_features_num, node_emb, lr=1e-3, scheduler_decay=0.5, scheduler_step=3,
                 lr_stop=1e-5):
        """(bs, original_features, n, n) x 2 -> (bs, n, n) node similarities."""
        super().__init__()
        # the reference resolves these three names in place in the caller's dict (trainers.py:31-43);
        # callables left by an earlier construction are accepted so a dict can be reused
        builder = _lookup(get_node_emb, node_emb['type'], "node embedding")
        for key, table, what in (('block_inside', get_block_inside, "block inside"),
                                 ('block_init', get_block_init, "block init")):
            if not callable(node_emb[key]):
                node_emb[key] = _lookup(table, node_emb[key], what)
        self.out_features = node_emb['out_features']
        self.node_embedder_dic = {'input': (None, []),
                                  'ne': builder(original_features_num, **node_emb)}
        self.node_embedder = Network(self.node_embedder_dic)
        self.loss = triplet_loss()
        self.metric = accuracy_linear_assignment
        self.lr = lr
        self.scheduler_decay = scheduler_decay
        self.scheduler_step = scheduler_step
        self.lr_stop = lr_stop

    @property
    def precision(self):
        return self.node_embedder.precision

    def set_precision(self, precision):
        self.node_embedder.set_precision(precision)
        return self

    def set_checkpoint_blocks(self, on=True):
        """Train the 16-bit embedder with block-level activation checkpoints (Network.set_checkpoint_blocks)."""
        self.node_embedder.set_checkpoint_blocks(on)
        return self

    def embed(self, x):
        return self.node_embedder(x)['ne/suffix']

    def forward(self, x1, x2):
        """Graph 1 padded to N1, graph 2 to N2 (the two may differ) -> (B,N1,N2) scores, zero outside each pair's n1 x n2
        block; for MaskedTensor inputs the rows carry graph 1's mask and the columns graph 2's."""
        e1 = self.embed(x1)
        e2 = self.embed(x2)
        # inference in a 16-bit mode: E1^T E2 on tensor cores (fgnn_head_pair_fwd with the scores requested)
        fused = (not torch.is_grad_enabled()) and self.precision != "fp32"
        if isinstance(e1, MaskedTensor):
            n_dev, n2_dev = e1.sizes_i32(), e2.sizes_i32()
            t1, t2 = e1.tensor.rename(None), e2.tensor.rename(None)
            if fused:
                s = _ops.head_fused(t1, t2, n_dev, self.precision, want_scores=True, n2_dev=n2_dev)[2]
            else:
                s = _ops.ScoresFunction.apply(t1, t2, n_dev, n2_dev)
            bname, nname = e1.tensor.names[0], e1.tensor.names[2]
            masks = {nname: e1.mask_dict[nname],
                     nname + '_': e2.mask_dict[e2.tensor.names[2]].rename(None).rename(bname, nname + '_')}
            out = MaskedTensor(s.rename(bname, nname, nname + '_'), masks, adjust_mask=False, apply_mask=False)
            # the embedders validated and uploaded both sides' sizes already
            out._dim_sizes = {nname: e1.sizes_host(), nname + '_': e2.sizes_host()}
            out._dim_sizes_dev = {nname: n_dev, nname + '_': n2_dev}
            return out
        if fused:
            return _ops.head_fused(e1, e2, None, self.precision, want_scores=True)[2]
        return _ops.ScoresFunction.apply(e1, e2, None)

    @torch.no_grad()
    def loss_and_accuracy(self, x1, x2):
        """Inference step without materialising the (B,N1,N2) scores: both embedders, then the fused tensor-core head
        (E1^T E2, row softmax cross-entropy against the identity matching, row argmax; models/trainers.py:67 +
        toolbox/losses.py:27-34 + toolbox/metrics.py:118-141 in one pass).  Returns device tensors
        (loss 'mean' = sum CE / sum n1, #correct rows, #rows = sum n1).  Graph 2's sizes come from x2; every pair needs
        n1 <= n2.  16-bit precisions; fp32 goes through forward()."""
        if self.precision == "fp32":
            scores = self(x1, x2)
            plain, n_dev, n2_dev, sizes = _as_batch(scores, loss=True)
            ce, correct = _ops.CrossEntropyIdentityFunction.apply(plain, n_dev, n2_dev)
        else:
            e1, e2 = self.embed(x1), self.embed(x2)
            n_dev, n2_dev, sizes = _head_sizes(e1, e2)
            if isinstance(e1, MaskedTensor):
                e1, e2 = e1.tensor.rename(None), e2.tensor.rename(None)
            ce, correct, _ = _ops.head_fused(e1, e2, n_dev, self.precision, n2_dev=n2_dev)
        rows = sizes.sum()
        return ce.sum() / rows, correct.sum(), rows

    @torch.no_grad()
    def loss_and_accuracy_from_adjacency(self, adj1, adj2, sizes=None, sizes2=None):
        """loss_and_accuracy fed from two CUDA (B,N1,N1) and (B,N2,N2) uint8 / bool adjacency batches (`sizes`, `sizes2`:
        optional CUDA int32 vertex counts of graph 1 and graph 2 in a padded ragged batch; `sizes2` defaults to `sizes`):
        the reference's input construction (loaders/data_generator.py:118-125) happens on the device, so a step ships
        1 byte per matrix entry instead of the 8 bytes of the (B,2,N,N) fp32 features.  16-bit precisions."""
        if self.precision == "fp32":
            raise _ops.L.FgnnError("loss_and_accuracy_from_adjacency needs precision 'fp16' or 'bf16'")
        sizes2 = sizes if sizes2 is None else sizes2
        e1 = self.node_embedder.forward_fused_adjacency(adj1, sizes=sizes)
        e2 = self.node_embedder.forward_fused_adjacency(adj2, sizes=sizes2)
        B, N1, N2 = e1.shape[0], e1.shape[-1], e2.shape[-1]
        if sizes2 is not sizes or N1 != N2:
            n1 = sizes.tolist() if sizes is not None else [N1] * B
            n2 = sizes2.tolist() if sizes2 is not None else [N2] * B
            check_loss_sizes(n1, n2)
        ce, correct, _ = _ops.head_fused(e1, e2, sizes, self.precision, n2_dev=sizes2)
        rows = sizes.sum().to(torch.float32) if sizes is not None else torch.tensor(float(B * N1), device=e1.device)
        return ce.sum() / rows, correct.sum(), rows

    def _step(self, batch, tag):
        raw_scores = self(batch[0], batch[1])
        loss = self.loss(raw_scores)
        self.log(tag + '_loss', loss)
        acc, n = self.metric(raw_scores)
        self.log(tag + '_acc', acc / n)
        return loss

    def training_step(self, batch, batch_idx):
        return self._step(batch, 'train')

    def validation_step(self, batch, batch_idx):
        self._step(batch, 'val')

    def test_step(self, batch, batch_idx):
        self._step(batch, 'test')

    def configure_optimizers(self):
        optimizer = torch.optim.Adam(self.parameters(), lr=self.lr, amsgrad=False)
        scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(
            optimizer, factor=self.scheduler_decay, patience=self.scheduler_step, min_lr=self.lr_stop)
        return {"optimizer": optimizer,
                "lr_scheduler": {"scheduler": scheduler, "monitor": "val_loss", "frequency": 1}}
