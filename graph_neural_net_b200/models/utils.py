"""Nested-dict -> DAG -> nn.Module executor, with a fused fast path for the 2-FGNN embedder.

API mirror of the reference models/utils.py (Network :53-75, build_graph :48-51, pipeline :45-46,
path_iter :11-14, normpath :34-41).  Node paths are joined with '/', modules are registered under
the path with '/' -> '_' (that is where the reference's state-dict keys come from), a node without
explicit inputs consumes the previous node of the flattened order, string inputs are resolved
relative to the node's parent.

Execution differs: with precision 'fp32' every node runs as its own CUDA operator and forward()
returns every node's output like the reference; with 'bf16'/'fp16' a Network whose graph is the
standard node_embedding DAG runs ONE fused call (fgnn_embed_fwd) and returns only the inputs and
'.../suffix' (SURVEY.md H7) -- intermediates never exist in HBM in the reference layout.
"""
from __future__ import annotations

import os
from collections import OrderedDict, defaultdict

import torch
import torch.nn as nn

from .. import _lib as L
from .. import _ops

sep = '/'

union = lambda *dicts: {k: v for d in dicts for (k, v) in d.items()}  # noqa: E731


def path_iter(nested_dict, pfx=()):
    """Depth-first (path tuple, leaf) pairs in insertion order."""
    for name, val in nested_dict.items():
        here = pfx + (name,)
        if isinstance(val, dict):
            yield from path_iter(val, here)
        else:
            yield here, val


def map_nested(func, nested_dict):
    return {k: (map_nested(func, v) if isinstance(v, dict) else func(v)) for k, v in nested_dict.items()}


def group_by_key(items):
    out = defaultdict(list)
    for k, v in items:
        out[k].append(v)
    return out


def split(path):
    head, _, tail = path.rpartition(sep)
    return head, tail


def normpath(path):
    out = []
    for part in path.split(sep):
        if part == '..':
            out.pop()
        else:
            out.append(part)
    return sep.join(out)


def has_inputs(node):
    return type(node) is tuple


def pipeline(net):
    flat = []
    for path, node in path_iter(net):
        flat.append((sep.join(path), node if has_inputs(node) else (node, [-1])))
    return flat


def build_graph(net):
    flat = pipeline(net)
    graph = OrderedDict()
    for idx, (path, (node, refs)) in enumerate(flat):
        ins = []
        for r in refs:
            if isinstance(r, str):
                ins.append(normpath(sep.join((path, '..', r))))
            else:
                ins.append(flat[idx + r][0])
        graph[path] = (node, ins)
    return graph


_DEFAULT_PRECISION = os.environ.get("FGNN_PRECISION", "fp32")


class Network(nn.Module):
    def __init__(self, net):
        super().__init__()
        self.graph = build_graph(net)
        for path, (val, _) in self.graph.items():
            setattr(self, path.replace(sep, '_'), val)
        self.precision = _DEFAULT_PRECISION
        self._fused = self._match_embedder()

    def set_precision(self, precision: str):
        if precision not in L.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(L.PRECISIONS)}")
        self.precision = precision
        return self

    def nodes(self):
        return (node for node, _ in self.graph.values())

    # ---- fused path ---------------------------------------------------------------------------
    def _match_embedder(self):
        """Recognise input -> [in] -> bm/{in, block_i/{in,mlp1,mlp2,mult,cat,mlp3}} -> suffix and
        return (input_key, suffix_key, [(mlp1, mlp2, mlp3), ...]) or None."""
        from .layers import MlpBlock_Real, ColumnMaxPooling, Matmul, Concat
        keys = list(self.graph.keys())
        sfx = [k for k in keys if split(k)[1] == 'suffix' and isinstance(self.graph[k][0], ColumnMaxPooling)]
        if len(sfx) != 1:
            return None
        root = split(sfx[0])[0]
        blocks = []
        i = 1
        while True:
            base = sep.join(x for x in (root, 'bm', f'block{i}') if x)
            trio = [self.graph.get(base + sep + n, (None,))[0] for n in ('mlp1', 'mlp2', 'mlp3')]
            if trio[0] is None:
                break
            if not all(isinstance(m, MlpBlock_Real) for m in trio):
                return None
            if not isinstance(self.graph.get(base + sep + 'mult', (None,))[0], Matmul):
                return None
            if not isinstance(self.graph.get(base + sep + 'cat', (None,))[0], Concat):
                return None
            blocks.append(tuple(trio))
            i += 1
        if not blocks:
            return None
        n_expected = 3 + 6 * len(blocks) + 1          # input, ne/in, bm/in, blocks, suffix
        if len(keys) != n_expected or keys[0] != 'input':
            return None
        return ('input', sfx[0], blocks)

    def _embed_params(self, keep):
        """fgnn_embed_params of the fused embedder, real shapes: the C library zero-pads the widths it runs
        (fgnn_tc.cu make_plan)."""
        p = L.EmbedParams()
        _, _, blocks = self._fused
        p.num_blocks = len(blocks)
        for i, trio in enumerate(blocks):
            for name, mlp in zip(('mlp1', 'mlp2', 'mlp3'), trio):
                mp = _ops.make_mlp_params([c.weight for c in mlp.convs], [c.bias for c in mlp.convs], mlp.gn.weight,
                                          mlp.gn.bias, mlp.gn.eps, keep, bool(mlp.cst_vertices))
                setattr(p.block[i], name, mp)
        return p

    def _flat_params(self):
        """(spec, tensors) of the fused embedder in the order _ops.embed_params_from_flat expects."""
        spec, flat = [], []
        for trio in self._fused[2]:
            row = []
            for mlp in trio:
                row.append((len(mlp.convs), float(mlp.gn.eps), bool(mlp.cst_vertices), True))
                flat += [c.weight for c in mlp.convs] + [c.bias for c in mlp.convs] + [mlp.gn.weight, mlp.gn.bias]
            spec.append(tuple(row))
        return spec, flat

    def forward_fused_train(self, x, precision=None):
        """Differentiable 16-bit embedder (fgnn_embed_fwd_train / fgnn_embed_bwd): x Tensor (B,F,N,N) or MaskedTensor
        -> (B,C,N) embeddings that carry autograd history to every parameter."""
        from .layers import _unwrap
        from ..maskedtensors.maskedtensor import MaskedTensor
        if self._fused is None:
            raise L.FgnnError("this Network is not a node_embedding DAG; fused execution unavailable")
        prec_name = precision or self.precision
        if prec_name == 'fp32':
            raise L.FgnnError("forward_fused_train is the 16-bit training path; fp32 trains through the per-operator Functions")
        plain, n_dev, rewrap = _unwrap(x)
        spec, flat = self._flat_params()
        if any(t is None for t in flat):
            raise L.FgnnError("the fused training path needs conv biases and an affine GraphNorm (the reference's modules)")
        c_out = self._fused[2][-1][2].convs[-1].weight.shape[0]
        emb = _ops.EmbedTrainFunction.apply(plain, n_dev, spec, L.PRECISIONS[prec_name], c_out, *flat)
        if isinstance(x, MaskedTensor):
            return rewrap(emb, x.tensor.names[:-1])
        return emb

    def forward_fused(self, x, precision=None):
        """One fgnn_embed_fwd call: x Tensor (B,F,N,N) or MaskedTensor -> (B,C,N) embeddings."""
        from .layers import _unwrap
        from ..maskedtensors.maskedtensor import MaskedTensor
        if self._fused is None:
            raise L.FgnnError("this Network is not a node_embedding DAG; fused execution unavailable")
        prec = L.PRECISIONS[precision or self.precision]
        plain, n_dev, rewrap = _unwrap(x)
        keep = []
        params = self._embed_params(keep)
        c_out = self._fused[2][-1][2].convs[-1].weight.shape[0]
        emb = _ops.embed_fwd(params, prec, plain, c_out, n_dev)
        if isinstance(x, MaskedTensor):
            return rewrap(emb, x.tensor.names[:-1])
        return emb

    def forward_fused_adjacency(self, adj, precision=None, sizes=None):
        """Embeddings straight from a CUDA (B,N,N) uint8/bool adjacency batch (`sizes`: optional CUDA int32 vertex
        counts of a padded ragged batch) -- the reference's input construction (loaders/data_generator.py:118-125)
        happens on the device.  16-bit precisions only; returns the plain (B,C,N) tensor."""
        if self._fused is None:
            raise L.FgnnError("this Network is not a node_embedding DAG; fused execution unavailable")
        prec_name = precision or self.precision
        if prec_name == 'fp32':
            raise L.FgnnError("forward_fused_adjacency needs precision 'bf16' or 'fp16' "
                              "(for fp32 build the features with loaders.data_generator.adjacency_batch_to_tensor_representation)")
        keep = []
        params = self._embed_params(keep)
        c_out = self._fused[2][-1][2].convs[-1].weight.shape[0]
        return _ops.embed_fwd_adjacency(params, L.PRECISIONS[prec_name], adj, c_out, sizes)

    # ---- reference-compatible execution ----------------------------------------------------------
    def forward(self, inputs):
        outputs = dict(inputs)
        if self._fused is not None and self.precision != 'fp32' and self._fused[0] in outputs:
            if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
                outputs[self._fused[1]] = self.forward_fused_train(outputs[self._fused[0]])
            else:
                outputs[self._fused[1]] = self.forward_fused(outputs[self._fused[0]])
            return outputs
        for key, (node, ins) in self.graph.items():
            if key not in outputs:                      # nodes supplied by the caller are not recomputed
                outputs[key] = node(*[outputs[name] for name in ins])
        return outputs

    def half(self):
        for node in self.nodes():
            if isinstance(node, nn.Module) and not isinstance(node, nn.BatchNorm2d):
                node.half()
        return self
