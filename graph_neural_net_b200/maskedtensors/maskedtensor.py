"""Ragged batches of graphs: zero-padded data + per-dimension prefix masks.

Host-side mirror of the reference's maskedtensors/maskedtensor.py (same public names:
from_list, MaskedTensor, implements, SPECIAL_FUNCTIONS, dispatch_cat, dispatch_stack,
get_sizes, get_dtype_min_value).  What differs is where the arithmetic happens: the reference
re-multiplies by the masks after every torch call (maskedtensor.py:87-112, 54 % of its masked
run time); here a MaskedTensor whose masks are prefix masks carries one int32 size per graph
(`sizes_i32()`), and the fgnn_b200 CUDA operators (models/layers.py, toolbox/losses.py) take
that vector and mask in-kernel.  Generic torch functions still work through
__torch_function__ (unwrap -> call -> re-mask) for API compatibility; they are not on the
hot path.
"""
from __future__ import annotations

import functools
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

SPECIAL_FUNCTIONS = {}


def implements(torch_function):
    """Register an override of `torch_function` for MaskedTensor arguments
    (reference maskedtensor.py:189-200)."""
    def decorator(func):
        functools.update_wrapper(func, torch_function)
        SPECIAL_FUNCTIONS[torch_function] = func
        return func
    return decorator


def get_dtype_min_value(dtype):
    """Smallest representable value of a float or int dtype (reference :202-211)."""
    if dtype.is_floating_point:
        return torch.finfo(dtype).min
    try:
        return torch.iinfo(dtype).min
    except TypeError:
        raise TypeError("dtype is neither float nor int")


def from_list(tensor_list: Sequence[torch.Tensor], dims: Iterable[int], batch_name: str = 'B',
              base_name: str = 'N') -> "MaskedTensor":
    """Pad a list of tensors to a common size along `dims` and record prefix masks.

    Reference maskedtensor.py:8-48: masked dim number i is named base_name + '_'*i, the batch
    dim `batch_name`; data is zero padded; mask[name] is (B, size) with ones on the valid prefix.
    """
    dims = list(dims)
    first = tensor_list[0]
    nd = first.dim()
    bsz = len(tensor_list)
    names: List[Optional[str]] = [batch_name] + [None] * nd
    for k, d in enumerate(dims):
        names[d + 1] = base_name + '_' * k
    full = [bsz] + [max(int(t.size(d)) for t in tensor_list) for d in range(nd)]
    data = torch.zeros(full, dtype=first.dtype, device=first.device)
    for b, t in enumerate(tensor_list):
        data[(b,) + tuple(slice(0, int(s)) for s in t.shape)] = t
    masks: Dict[str, torch.Tensor] = {}
    for d in range(nd):
        nm = names[d + 1]
        if nm is None:
            continue
        lens = torch.tensor([int(t.size(d)) for t in tensor_list], device=first.device)
        m = (torch.arange(full[d + 1], device=first.device)[None, :] < lens[:, None]).to(first.dtype)
        masks[nm] = m.refine_names(batch_name, nm)
    return MaskedTensor(data.refine_names(*names), masks, adjust_mask=False, apply_mask=False)


class MaskedTensor:
    """Padded named tensor + {dim name: (B, size) mask}.  Reference maskedtensor.py:50-184."""

    def __init__(self, data, mask, adjust_mask=True, apply_mask=False, copy=False, batch_name='B'):
        self.tensor = data.clone() if copy else data
        self.mask_dict = dict(mask)
        self._batch_name = batch_name
        self.dtype = self.tensor.dtype
        self.device = self.tensor.device
        self._sizes_cache = None
        self._sizes_dev = None        # int32 device copy of the sizes, uploaded once per batch
        self._dim_sizes = {}          # per-dim sizes_host(name) / sizes_i32(name=name)
        self._dim_sizes_dev = {}
        if adjust_mask:
            self._adjust_mask_()
        if apply_mask:
            self.mask_()

    def __repr__(self):
        return "Data:\n{}\nMask:\n{}".format(self.tensor, self.mask_dict)

    # ---- masks ---------------------------------------------------------------------------
    def _adjust_mask_(self):
        """Drop masks whose dim no longer exists; check sizes of the others (reference :75-85)."""
        present = set(n for n in self.tensor.names if n)
        for name in list(self.mask_dict):
            if name not in present:
                del self.mask_dict[name]
            else:
                assert self.mask_dict[name].size(name) == self.tensor.size(name)

    def mask_(self):
        """Zero the padding in place (reference :87-90)."""
        for m in self.mask_dict.values():
            self.tensor = self.tensor * m.align_as(self.tensor)

    def mask(self):
        return MaskedTensor(self.tensor, self.mask_dict, adjust_mask=False, apply_mask=True, copy=True)

    @staticmethod
    def _prefix_sizes(m: torch.Tensor) -> torch.Tensor:
        """(B, size) mask -> int64 sizes; the CUDA operators address padding by size: masks must be prefix masks."""
        m = m.rename(None)
        sz = m.sum(dim=1).round().to(torch.int64)
        pref = (torch.arange(m.shape[1], device=m.device)[None, :] < sz[:, None]).to(m.dtype)
        if not torch.equal(pref, m):
            raise ValueError("fgnn_b200 supports prefix masks only (as built by from_list)")
        return sz

    def sizes_host(self, name: Optional[str] = None) -> List[int]:
        """True size of each graph along the masked dim `name`.  Without a name: the one size all masked dims of a graph
        share (from_list data); scores of graphs of unequal sizes have one size per dim, ask for each by name."""
        if name is not None:
            if name not in self._dim_sizes:
                if name not in self.mask_dict:
                    raise KeyError(f"no mask for dim {name!r} (masked dims: {list(self.mask_dict)})")
                self._dim_sizes[name] = [int(v) for v in self._prefix_sizes(self.mask_dict[name]).tolist()]
            return self._dim_sizes[name]
        if self._sizes_cache is None:
            sz = self._prefix_sizes(next(iter(self.mask_dict.values())))
            for other in self.mask_dict.values():
                if not torch.equal(other.rename(None).sum(dim=1).round().to(torch.int64), sz):
                    raise ValueError("all masked dims of a graph must have the same size")
            self._sizes_cache = [int(v) for v in sz.tolist()]
        return self._sizes_cache

    def sizes_i32(self, device=None, name: Optional[str] = None) -> torch.Tensor:
        """sizes_host(name) as an int32 tensor on `device` (default: the data's), uploaded once."""
        dev = torch.device(self.device if device is None else device)
        if name is not None:
            t = self._dim_sizes_dev.get(name)
            if t is None or t.device != dev:
                t = self._dim_sizes_dev[name] = torch.tensor(self.sizes_host(name), dtype=torch.int32, device=dev)
            return t
        if self._sizes_dev is None or self._sizes_dev.device != dev:
            self._sizes_dev = torch.tensor(self.sizes_host(), dtype=torch.int32, device=dev)
        return self._sizes_dev

    def _inherit_sizes(self, other: "MaskedTensor") -> "MaskedTensor":
        """Operator outputs keep the masks of their input: reuse its validated sizes (no re-validation, no
        device synchronisation, no second upload)."""
        self._sizes_cache = other._sizes_cache
        self._sizes_dev = other._sizes_dev
        return self

    # ---- torch function protocol ---------------------------------------------------------
    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        kwargs = {} if kwargs is None else kwargs
        special = SPECIAL_FUNCTIONS.get(func)
        if special is not None:
            return special(*args, **kwargs)
        raw = [a.tensor if isinstance(a, MaskedTensor) else a for a in args]
        merged = {}
        for a in args:
            if isinstance(a, MaskedTensor):
                merged.update(a.mask_dict)
        return MaskedTensor(func(*raw, **kwargs), merged, adjust_mask=True, apply_mask=True)

    # ---- container protocol: iterate over un-padded graphs (reference :115-128) ------------
    def __getitem__(self, index):
        item = self.tensor[index]
        for d, name in enumerate(item.names):
            if name:
                length = int(self.mask_dict[name][index].sum().item())
                item = torch.narrow(item, d, 0, length)
        return item.rename(None)

    def __len__(self):
        return self.tensor.size(self._batch_name)

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    # ---- tensor-like helpers ---------------------------------------------------------------
    def size(self, *args):
        return self.tensor.size(*args)

    def dim(self):
        return self.tensor.dim()

    @property
    def shape(self):
        return self.tensor.size()

    @property
    def is_cuda(self):
        return self.tensor.is_cuda

    @property
    def get_device(self):
        return self.tensor.get_device()

    def contiguous(self, *args):
        self.tensor = self.tensor.contiguous(*args)
        return self

    def _renamed(self, plain, names):
        return MaskedTensor(plain.rename(*names), self.mask_dict, adjust_mask=False, apply_mask=False)

    def view(self, *dims):
        """Reshape trailing un-named dims only (reference :139-150)."""
        old = self.tensor.names
        names = [old[i] if i < len(old) else None for i in range(len(dims))]
        return self._renamed(self.tensor.rename(None).view(*dims), names)

    def permute(self, *dims):
        if len(dims) != self.tensor.dim():
            raise ValueError
        old = self.tensor.names
        return self._renamed(self.tensor.rename(None).permute(*dims), [old[d] for d in dims])

    def to(self, *args, **kwargs):
        masks = {k: v.to(*args, **kwargs) for k, v in self.mask_dict.items()}
        out = MaskedTensor(self.tensor.to(*args, **kwargs), masks, adjust_mask=False, apply_mask=False)
        out._sizes_cache = self._sizes_cache
        return out

    def cuda(self, device=None):
        return self.to(torch.device('cuda') if device is None else device)


# ---- overrides (reference maskedtensor.py:213-384) ---------------------------------------------
def _merge_masks(items):
    merged = {}
    for a in items:
        if isinstance(a, MaskedTensor):
            merged.update(a.mask_dict)
    return merged


@implements(torch.max)
def torch_max(masked_tensor, dim=None):
    if dim is None:
        return torch.max(masked_tensor.tensor)      # whole-batch max, as the reference (:216-218)
    t = masked_tensor.tensor
    lowest = get_dtype_min_value(t.dtype)
    for m in masked_tensor.mask_dict.values():
        am = m.align_as(t)
        t = t * am + lowest * (1 - am)
    values, indices = torch.max(t, dim)
    return MaskedTensor(values, masked_tensor.mask_dict, adjust_mask=True, apply_mask=True), indices


def _nameless_call(fn, inp, *args, **kwargs):
    names = inp.tensor.names
    res = fn(inp.tensor.rename(None), *args, **kwargs)
    return MaskedTensor(res.rename(*names), inp.mask_dict, adjust_mask=False, apply_mask=True)


@implements(F.conv2d)
def torch_conv2d(inp, *args, **kwargs):
    return _nameless_call(F.conv2d, inp, *args, **kwargs)


@implements(F.linear)
def torch_linear(inp, *args, **kwargs):
    return _nameless_call(F.linear, inp, *args, **kwargs)


@implements(F.layer_norm)
def torch_layer_norm(inp, *args, **kwargs):
    return _nameless_call(F.layer_norm, inp, *args, **kwargs)


@implements(torch.cat)
def torch_cat(tensors, dim=0):
    raw = [a.tensor if isinstance(a, MaskedTensor) else a for a in tensors]
    return MaskedTensor(torch.cat(raw, dim=dim), _merge_masks(tensors), adjust_mask=False, apply_mask=False)


def dispatch_cat(tensors, dim=0):
    head = tensors[0]
    if isinstance(head, torch.Tensor):
        return torch.cat(tensors, dim=dim)
    return head.__torch_function__(torch.cat, [type(t) for t in tensors], (tensors,), {'dim': dim})


@implements(torch.stack)
def torch_stack(tensors, dim=0):
    raw = [a.tensor.rename(None) if isinstance(a, MaskedTensor) else a for a in tensors]
    names = [a.tensor.names for a in tensors if isinstance(a, MaskedTensor)][0]
    out_names = names[:dim] + (None,) + names[dim:]
    return MaskedTensor(torch.stack(raw, dim=dim).refine_names(*out_names), _merge_masks(tensors),
                        adjust_mask=True, apply_mask=False)


def dispatch_stack(tensors, dim=0):
    head = tensors[0]
    if isinstance(head, torch.Tensor):
        return torch.stack(tensors, dim=dim)
    return head.__torch_function__(torch.stack, [type(t) for t in tensors], (tensors,), {'dim': dim})


@implements(torch.flatten)
def torch_flatten(inp, start_dim=0, end_dim=-1):
    names = inp.tensor.names
    end = end_dim if end_dim >= 0 else len(names) + end_dim
    out_names = names[:start_dim] + (None,) + names[end + 1:]
    res = torch.flatten(inp.tensor.rename(None), start_dim=start_dim, end_dim=end_dim)
    return MaskedTensor(res.refine_names(*out_names), inp.mask_dict, adjust_mask=True, apply_mask=False)


def get_sizes(masked_tensor, keepdim=False):
    """Number of un-masked entries per (batch, free dims) (reference :310-317)."""
    ones = torch.ones_like(masked_tensor.tensor)
    for m in masked_tensor.mask_dict.values():
        ones = ones * m.align_as(ones)
    return torch.sum(ones, dim=tuple(masked_tensor.mask_dict.keys()), keepdim=keepdim)


@implements(torch.mean)
def torch_mean(masked_tensor, keepdim=False, *args, **kwargs):
    """Mean over ALL masked dims, whatever `dim` says (reference :319-326)."""
    total = torch.sum(masked_tensor.tensor, dim=tuple(masked_tensor.mask_dict.keys()), keepdim=keepdim)
    return total / get_sizes(masked_tensor, keepdim=keepdim)


@implements(torch.var)
def torch_var(masked_tensor, keepdim=False, *args, **kwargs):
    mu = torch_mean(masked_tensor, keepdim=True)
    sq = MaskedTensor((masked_tensor.tensor - mu) ** 2, masked_tensor.mask_dict, adjust_mask=False,
                      apply_mask=True)
    total = torch.sum(sq.tensor, dim=tuple(sq.mask_dict.keys()), keepdim=keepdim)
    return total / get_sizes(masked_tensor, keepdim=keepdim)


@implements(F.instance_norm)
def torch_instance_norm(masked_tensor, eps=1e-05, weight=None, bias=None, *args, **kwargs):
    mu = torch_mean(masked_tensor, keepdim=True)
    var = torch_var(masked_tensor, keepdim=True)
    res = (masked_tensor.tensor - mu) / torch.sqrt(var + eps)
    if weight is not None and bias is not None:
        res = weight.reshape(1, -1, 1, 1) * res + bias.reshape(1, -1, 1, 1)
    return MaskedTensor(res, masked_tensor.mask_dict, adjust_mask=False, apply_mask=True)


@implements(torch.diag_embed)
def torch_diag_embed(inp, offset=0, dim1=-2, dim2=-1, *args, **kwargs):
    names = inp.tensor.names
    extra = names[-1] + '_'
    res = torch.diag_embed(inp.tensor.rename(None), offset=offset, dim1=dim1, dim2=dim2)
    masks = dict(inp.mask_dict)
    src = inp.mask_dict[names[-1]]
    masks[extra] = src.rename(None).rename(*(src.names[:-1] + (extra,)))
    return MaskedTensor(res.rename(*(names + (extra,))), masks, adjust_mask=False, apply_mask=True)


@implements(F.nll_loss)
def torch_nll_loss(masked_tensor, target, *args, **kwargs):
    return F.nll_loss(masked_tensor.tensor.rename(None), target, *args, **kwargs)


@implements(F.cross_entropy)
def torch_cross_entropy(masked_tensor, target, *args, **kwargs):
    return F.cross_entropy(masked_tensor.tensor.rename(None), target, *args, **kwargs)
