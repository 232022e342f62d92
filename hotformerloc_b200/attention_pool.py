"""Differentiable pyramid attention-pooling head, fp32 on the kernels of csrc/attn_pool_train.cu.

:func:`attention_pool` is the AdaptivePooling of the reference's ``PyramidAttnPoolWrapper``
(models/layers/pooling.py:183-233, salsa.py:25-55) for one pyramid level: the learned queries attend
over each submap's tokens.  It takes the level's per-submap token counts instead of padded
``(B, Nmax, C)`` features and a ``(B, N, N)`` mask, and keeps only a per-(submap, query) log-sum-exp
for the backward.  :class:`PyramidAttnPool` is the whole head with the reference module's parameters:
one :func:`attention_pool` per level, then the Mixer in torch.  Every op runs on the current torch
stream and raises ``HflError`` on bad input, before any launch.
"""
from __future__ import annotations

from typing import Dict, Sequence, Union

import torch

from . import native as N
from .models.hotformerloc import PyramidAttnPoolWrapper
from .native import HflError
from .octree import Octree

__all__ = ['attention_pool', 'AttentionPoolFunction', 'PyramidAttnPool']

MAX_K = 256
MIN_C, MAX_C = 32, 512
MAX_B = 1 << 24
_INT_DTYPES = (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8)


def _require(cond: bool, msg: str):
    if not cond:
        raise HflError(msg)


def _host_offsets(counts, n: int) -> torch.Tensor:
    """(B + 1,) int64 CPU prefix offsets of the per-submap token counts, checked against n."""
    if isinstance(counts, torch.Tensor):
        _require(not counts.is_cuda, 'counts must be a host tensor or sequence (reading a device tensor would '
                                     'synchronise)')
        c = counts
    else:
        try:
            c = torch.as_tensor(counts)
        except (TypeError, ValueError, RuntimeError) as e:
            raise HflError(f'counts must be a sequence of integers: {e}') from None
    _require(c.dtype in _INT_DTYPES, f'counts must be integers, got {c.dtype}')
    _require(c.dim() == 1 and 1 <= c.numel() <= MAX_B, f'counts must be 1-D with 1 to {MAX_B} entries, '
                                                         f'got shape {tuple(c.shape)}')
    c = c.to(torch.int64)
    _require(bool((c >= 0).all()), 'counts must be non-negative')
    total = int(c.sum())
    _require(total == n, f'counts must sum to the token count n = {n}, got {total}')
    return torch.cat([c.new_zeros(1), c.cumsum(0)])


def _check_args(x, counts, query):
    """Validates the arguments on the host; returns the CPU offsets."""
    _require(isinstance(x, torch.Tensor) and x.dim() == 2, 'x must be an (n, C) tensor')
    _require(isinstance(query, torch.Tensor) and query.dim() == 2, 'query must be a (k, C) tensor')
    _require(x.dtype == torch.float32, f'x must be torch.float32, got {x.dtype}')
    _require(query.dtype == torch.float32, f'query must be torch.float32, got {query.dtype}')
    k, C = query.shape
    _require(1 <= k <= MAX_K, f'the number of queries k must be in [1, {MAX_K}], got {k}')
    _require(MIN_C <= C <= MAX_C and C % 32 == 0, f'C must be a multiple of 32 in [{MIN_C}, {MAX_C}], got {C}')
    _require(x.shape[1] == C, f'x has {x.shape[1]} channels, query has {C}')
    off = _host_offsets(counts, x.shape[0])
    _require(x.is_contiguous() and query.is_contiguous(), 'x and query must be contiguous')
    _require(x.is_cuda and query.is_cuda, 'x and query must be CUDA tensors')
    _require(x.device == query.device, 'x and query must be on the same device')
    return off


def _aligned(t: torch.Tensor) -> torch.Tensor:
    """t itself, or a copy in a fresh (16-byte aligned) allocation when a view's offset leaves it misaligned:
    the kernels read rows as float4."""
    return t.clone() if t.data_ptr() % 16 else t


def _upload(off: torch.Tensor, device) -> torch.Tensor:
    """Host offsets -> device through the pinned staging pool: one asynchronous copy, no synchronisation."""
    stage = N.pinned.take(8 * off.numel()).view(torch.int64)
    stage.copy_(off)
    dev = stage.to(device, non_blocking=True)
    N.pinned.mark()
    return dev


def _workspace(nbytes: int, device):
    return torch.empty(nbytes, dtype=torch.uint8, device=device) if nbytes else None


class AttentionPoolFunction(torch.autograd.Function):
    """out[b] = softmax(C^-0.5 query x_b^T) x_b per segment b; gradients for x and query."""

    @staticmethod
    def forward(ctx, x, query, counts):
        off = _check_args(x, counts, query)
        x, query = _aligned(x), _aligned(query)
        (n, C), (k, B) = x.shape, (query.shape[0], off.numel() - 1)
        L = N.lib()
        dev = x.device
        with torch.cuda.device(dev):
            off_dev = _upload(off, dev)
            out = torch.empty((B, k, C), dtype=torch.float32, device=dev)
            lse = torch.empty((B, k), dtype=torch.float32, device=dev)
            nb = int(L.hfl_attn_pool_train_fwd_workspace_bytes(n, B, k, C))
            ws = _workspace(nb, dev)
            N.check(L.hfl_attn_pool_train_fwd(N.ptr(x), N.ptr(off_dev), N.ptr(query), n, B, k, C, N.ptr(out),
                                              N.ptr(lse), N.ptr(ws), nb, N.stream()))
        ctx.save_for_backward(x, query, off_dev, out, lse)
        return out

    @staticmethod
    def backward(ctx, grad):
        x, query, off_dev, out, lse = ctx.saved_tensors
        _require(grad.dtype == torch.float32 and grad.shape == out.shape, 'grad must match out')
        grad = _aligned(grad.contiguous())
        (n, C), (B, k) = x.shape, lse.shape
        L = N.lib()
        dev = x.device
        with torch.cuda.device(dev):
            dx = torch.empty_like(x)
            dq = torch.empty_like(query)
            nb = int(L.hfl_attn_pool_train_bwd_workspace_bytes(n, B, k, C))
            ws = _workspace(nb, dev)
            N.check(L.hfl_attn_pool_train_bwd(N.ptr(x), N.ptr(off_dev), N.ptr(query), N.ptr(out), N.ptr(lse),
                                              N.ptr(grad), n, B, k, C, N.ptr(dx), N.ptr(dq), N.ptr(ws), nb,
                                              N.stream()))
        return (dx if ctx.needs_input_grad[0] else None, dq if ctx.needs_input_grad[1] else None, None)


def attention_pool(x: torch.Tensor, counts: Union[torch.Tensor, Sequence[int]], query: torch.Tensor) -> torch.Tensor:
    """Attention pooling of one pyramid level over its per-submap token segments.

    x (n, C) float32 CUDA, the level's tokens with submap b's tokens at rows
    [sum(counts[:b]), sum(counts[:b + 1])); counts (B,) per-submap token counts on the host (a CPU
    tensor or a sequence: ``octree.batch_nnum_nempty[depth]``), non-negative, summing to n; query
    (k, C) float32 on x's device, 1 <= k <= 256, C a multiple of 32 in [32, 512].  Returns (B, k, C)
    float32: row q of submap b is ``softmax(C^-0.5 query[q] . x_b^T) x_b``, zero for a submap
    without tokens.  Differentiable in x and query, with outputs and gradients that are
    bit-identical run to run."""
    return AttentionPoolFunction.apply(x, query, counts)


class PyramidAttnPool(PyramidAttnPoolWrapper):
    """``PyramidAttnPoolWrapper`` + Mixer (pooling.py:183-233, salsa.py:25-111) on :func:`attention_pool`.
    Parameters are those of the reference module -- ``attpool.{j}.query`` and ``descriptor_extractor.*`` --
    so the ``pooling.pooling.*`` tensors of a checkpoint load into it.  ``F.normalize`` of the descriptor
    stays with the caller (HOTFormerLoc.forward), as in the reference."""

    def __init__(self, feature_size: int, output_dim: int, num_pyramid_levels: int, k_pooled_tokens: Sequence[int]):
        super().__init__(feature_size, output_dim, num_pyramid_levels, k_pooled_tokens)
        if not (MIN_C <= feature_size <= MAX_C and feature_size % 32 == 0):
            raise ValueError(f'feature_size must be a multiple of 32 in [{MIN_C}, {MAX_C}], got {feature_size}')
        if not all(1 <= k <= MAX_K for k in self.k_pooled_tokens):
            raise ValueError(f'every k_pooled_tokens entry must be in [1, {MAX_K}], got {self.k_pooled_tokens}')
        self.feature_size, self.output_dim, self.num_pyramid_levels = feature_size, output_dim, num_pyramid_levels

    def forward(self, local_feat_dict: Dict[int, torch.Tensor], octree) -> torch.Tensor:
        """local_feat_dict {depth: (n_d, C)} (the first output of ``HOTFormer.forward``), level j = the j-th
        largest depth; octree a native ``Octree`` or an ocnn octree, of which only ``batch_nnum_nempty`` is
        read.  Returns the (B, output_dim) descriptor before normalisation."""
        depths = sorted(local_feat_dict, reverse=True)
        if len(depths) != len(self.attpool):
            raise ValueError(f'expected {len(self.attpool)} pyramid levels, got depths {depths}')
        if isinstance(octree, Octree):
            octree.finalize()
        counts = octree.batch_nnum_nempty
        x = torch.cat([attention_pool(local_feat_dict[d], counts[d], ap.query)
                       for d, ap in zip(depths, self.attpool)], 1)                   # (B, ktot, C)
        de = self.descriptor_extractor
        for layer in de.mix:
            x = x + layer.mix(x)
        x = de.channel_proj(x.permute(0, 2, 1)).permute(0, 2, 1)
        return de.row_proj(x).flatten(1)

    def extra_repr(self) -> str:
        return (f'feature_size={self.feature_size}, output_dim={self.output_dim}, '
                f'num_pyramid_levels={self.num_pyramid_levels}, k_pooled_tokens={self.k_pooled_tokens}')
