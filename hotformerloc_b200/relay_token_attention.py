"""Differentiable relay-token self-attention (RTSA) core, fp32 on the kernels of csrc/rt_attn_train.cu.

The reference's ``RelayTokenTransformerBlock`` (hotformerloc_backbone.py:83-119, 275-295) concatenates
each submap's relay tokens (RTs) of the pyramid levels, pads them to ``(B, Nmax, C)`` with a
``(B, Nmax, Nmax)`` mask (``concat_and_pad_rt``, relay_token_utils.py:12-40; models/octree.py:229-265),
runs dense attention and splits the result back (``unpad_and_split_rt``, :42-79), with host
synchronisations in the Python loops.  Here:

- :func:`rt_layout` computes the per-submap RT sequences once per octree on the host, from the node
  counts (the ownership rule of :func:`~hotformerloc_b200.models.hotformerloc.rt_ownership`, shared
  with the inference engine), and uploads them in one asynchronous copy;
- :meth:`RelayTokenLayout.pack` / :meth:`RelayTokenLayout.unpack` are single gathers between the
  level RT tensors and the packed ``(T, C)`` rows, with autograd passing through;
- :func:`relay_token_attention` is the attention core over the ragged sequences, which keeps one
  log-sum-exp per (row, head) for the backward: no ``(B, H, Nmax, Nmax)`` tensor exists;
- :class:`RTAttention` wraps it with the reference module's parameters.

Every op runs on the current torch stream and raises ``HflError`` on bad input, before any launch.
"""
from __future__ import annotations

import numbers
from typing import List, Sequence

import numpy as np
import torch

from . import native as N
from .models.hotformerloc import _RTAttention, rt_ownership
from .native import HflError

__all__ = ['rt_layout', 'RelayTokenLayout', 'relay_token_attention', 'RelayTokenAttentionFunction',
           'RTAttention']

HEAD_DIM = 16
MAX_HEADS = 16
MAX_B = 1 << 24
_INT_DTYPES = (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8)


def _require(cond: bool, msg: str):
    if not cond:
        raise HflError(msg)


def _host_counts(c, j: int) -> np.ndarray:
    """Level j's per-submap node counts as a non-negative int64 numpy array, without touching a device."""
    if isinstance(c, torch.Tensor):
        _require(not c.is_cuda, f'level_counts[{j}] must be a host tensor or sequence (reading a device tensor '
                                f'would synchronise)')
        _require(c.dtype in _INT_DTYPES, f'level_counts[{j}] must be integers, got {c.dtype}')
        a = c.numpy()
    else:
        try:
            a = np.asarray(c)
        except (TypeError, ValueError) as e:
            raise HflError(f'level_counts[{j}] must be a sequence of integers: {e}') from None
    _require(a.ndim == 1 and 1 <= a.size <= MAX_B,
             f'level_counts[{j}] must be 1-D with 1 to {MAX_B} entries, got shape {a.shape}')
    _require(a.dtype.kind in 'iu', f'level_counts[{j}] must be integers, got {a.dtype}')
    a = a.astype(np.int64)
    _require(bool((a >= 0).all()), f'level_counts[{j}] must be non-negative')
    return a


class RelayTokenLayout:
    """The packed RT sequences of one octree's pyramid; built by :func:`rt_layout`.

    Device tensors (int32): ``cu`` (B + 1,) sequence offsets into the T packed rows, ``ids`` (T,)
    attention ids (the submap, or B for windows that hold only padding), ``index`` (T,) the row of
    ``torch.cat`` of the level RT tensors that each packed row takes, ``inverse`` (T,) its inverse.
    Host: ``num_windows`` per level (B,) RTs owned per submap, ``windows`` per level RT counts,
    ``total`` = T, ``max_len`` the longest sequence, ``batch_size`` = B."""

    def __init__(self, cu, ids, index, inverse, num_windows: List[np.ndarray], total: int, max_len: int):
        self.cu, self.ids, self.index, self.inverse = cu, ids, index, inverse
        self.num_windows = num_windows
        self.windows = [int(nw.sum()) for nw in num_windows]
        self.total, self.max_len = total, max_len
        self.batch_size = len(cu) - 1
        self.device = cu.device

    def pack(self, rts: Sequence[torch.Tensor]) -> torch.Tensor:
        """``concat_and_pad_rt`` without the padding: rts[j] (windows[j], C), the level RT tensors (all
        windows, padding windows included: ``relay_token_dict`` of ``HOTFormer.forward``) -> (T, C), submap
        b's sequence at rows [cu[b], cu[b + 1])."""
        _require(len(rts) == len(self.windows), f'expected {len(self.windows)} levels, got {len(rts)}')
        for j, (r, n) in enumerate(zip(rts, self.windows)):
            _require(isinstance(r, torch.Tensor) and r.dim() == 2 and r.shape[0] == n,
                     f'rts[{j}] must be a ({n}, C) tensor, got {tuple(r.shape) if isinstance(r, torch.Tensor) else r}')
            _require(r.device == self.device, f'rts[{j}] must be on {self.device}')
        return torch.cat(list(rts)).index_select(0, self.index)

    def unpack(self, x: torch.Tensor) -> List[torch.Tensor]:
        """``unpad_and_split_rt`` of packed rows: x (T, C) -> [(windows[j], C)] per level."""
        _require(isinstance(x, torch.Tensor) and x.dim() == 2 and x.shape[0] == self.total,
                 f'x must be a ({self.total}, C) tensor')
        _require(x.device == self.device, f'x must be on {self.device}')
        return list(x.index_select(0, self.inverse).split(self.windows))


def _layout_tables(level_counts, patch_size, dilation):
    """Checks rt_layout's arguments; returns the host tables (rt_ownership, index, inverse)."""
    _require(isinstance(patch_size, numbers.Integral) and patch_size >= 1,
             f'patch_size must be a positive int, got {patch_size!r}')
    _require(isinstance(dilation, numbers.Integral) and dilation >= 1,
             f'dilation must be a positive int, got {dilation!r}')
    _require(isinstance(level_counts, (list, tuple)) and len(level_counts) >= 1,
             'level_counts must be a non-empty list of per-level counts')
    counts = [_host_counts(c, j) for j, c in enumerate(level_counts)]
    B = counts[0].size
    _require(all(c.size == B for c in counts),
             f'every level must have the same number of submaps, got {[c.size for c in counts]}')
    blk = int(patch_size) * int(dilation)
    own = rt_ownership(counts, int(patch_size), [-(-int(c.sum()) // blk) * blk for c in counts])
    T = own.total
    _require(T < (1 << 31) // (3 * HEAD_DIM * MAX_HEADS), f'too many relay tokens ({T})')
    inverse = np.concatenate(own.pos)                  # row of the level concatenation -> packed row
    index = np.empty(T, dtype=np.int64)
    index[inverse] = np.arange(T)                      # packed row -> row of the level concatenation
    return own, index, inverse


def rt_layout(level_counts, patch_size: int, dilation: int, device) -> RelayTokenLayout:
    """Per-submap RT sequences of a pyramid, for :meth:`RelayTokenLayout.pack` and
    :func:`relay_token_attention`.

    level_counts: per level, fine to coarse, the per-submap node counts on the host (a CPU tensor or a
    sequence; for a native or ocnn octree ``octree.batch_nnum_nempty[depth]``).  Level tokens are padded to
    a multiple of patch_size * dilation, as ``OctreeT`` does.  Computed on the host and uploaded through
    the pinned staging buffer in one asynchronous copy: no synchronisation."""
    _require(torch.device(device).type == 'cuda', f'device must be a CUDA device, got {device!r}')
    own, index, inverse = _layout_tables(level_counts, patch_size, dilation)
    T = own.total
    parts = [own.cu, own.ids, index, inverse]
    stage = N.pinned.take(4 * sum(p.size for p in parts)).view(torch.int32)
    o = 0
    for p in parts:
        stage[o:o + p.size] = torch.from_numpy(p.astype(np.int32))
        o += p.size
    dev = torch.device(device)
    with torch.cuda.device(dev):
        buf = stage.to(dev, non_blocking=True)
        N.pinned.mark()
    views, o = [], 0
    for p in parts:
        views.append(buf[o:o + p.size])
        o += p.size
    return RelayTokenLayout(*views, own.num_windows, T, own.max_len)


def _check_args(qkv, cu, ids, num_heads):
    _require(isinstance(num_heads, numbers.Integral) and 1 <= num_heads <= MAX_HEADS,
             f'num_heads must be an int in [1, {MAX_HEADS}], got {num_heads!r}')
    C = HEAD_DIM * int(num_heads)
    T = ids.shape[0]
    _require(isinstance(qkv, torch.Tensor), 'qkv must be a tensor')
    _require(qkv.dtype == torch.float32, f'qkv must be torch.float32, got {qkv.dtype}')
    _require(tuple(qkv.shape) == (T, 3 * C),
             f'qkv must have shape (layout.total, 3C) = {(T, 3 * C)} for C = 16 num_heads, got {tuple(qkv.shape)}')
    _require(qkv.is_contiguous(), 'qkv must be contiguous')
    _require(qkv.is_cuda, 'qkv must be a CUDA tensor')
    _require(qkv.device == cu.device, f'qkv must be on the layout\'s device {cu.device}, got {qkv.device}')


def _aligned(t: torch.Tensor) -> torch.Tensor:
    """t itself, or a copy in a fresh (16-byte aligned) allocation when a view's offset leaves it misaligned:
    the kernels read rows as float4."""
    return t.clone() if t.data_ptr() % 16 else t


def _workspace(T: int, B: int, H: int, device):
    nb = int(N.lib().hfl_rt_attn_train_workspace_bytes(T, B, H))
    return torch.empty(nb, dtype=torch.uint8, device=device), nb


class RelayTokenAttentionFunction(torch.autograd.Function):
    """o = softmax(0.25 q k^T + mask) v per sequence and head; gradient for qkv."""

    @staticmethod
    def forward(ctx, qkv, cu, ids, num_heads):
        _check_args(qkv, cu, ids, num_heads)
        qkv = _aligned(qkv)
        T, H, B = ids.shape[0], int(num_heads), cu.shape[0] - 1
        dev = qkv.device
        with torch.cuda.device(dev):
            o = torch.empty((T, HEAD_DIM * H), dtype=torch.float32, device=dev)
            lse = torch.empty((T, H), dtype=torch.float32, device=dev)
            ws, nb = _workspace(T, B, H, dev)
            N.check(N.lib().hfl_rt_attn_train_fwd(N.ptr(qkv), N.ptr(cu), N.ptr(ids), int(ids.dtype == torch.int64),
                                                  B, T, H, N.ptr(o), N.ptr(lse), N.ptr(ws), nb, N.stream()))
        ctx.save_for_backward(qkv, cu, ids, o, lse)
        ctx.num_heads = H
        return o

    @staticmethod
    def backward(ctx, grad):
        qkv, cu, ids, o, lse = ctx.saved_tensors
        _require(grad.dtype == torch.float32 and grad.shape == o.shape, 'grad must match o')
        grad = _aligned(grad.contiguous())
        T, H, B = ids.shape[0], ctx.num_heads, cu.shape[0] - 1
        dev = qkv.device
        with torch.cuda.device(dev):
            dqkv = torch.empty_like(qkv)
            ws, nb = _workspace(T, B, H, dev)
            N.check(N.lib().hfl_rt_attn_train_bwd(N.ptr(qkv), N.ptr(cu), N.ptr(ids), int(ids.dtype == torch.int64),
                                                  N.ptr(o), N.ptr(lse), N.ptr(grad), B, T, H, N.ptr(dqkv), N.ptr(ws),
                                                  nb, N.stream()))
        return dqkv, None, None, None


def relay_token_attention(qkv: torch.Tensor, layout: RelayTokenLayout, num_heads: int) -> torch.Tensor:
    """Attention core of ``RTAttention.forward`` over the packed RT sequences of ``layout``.

    qkv (layout.total, 3C) float32 on the layout's device, the output of ``Linear(C, 3C)`` applied to
    packed rows, with C = 16 num_heads and 1 <= num_heads <= 16.  Within submap b's sequence, rows attend
    with bias 0 when their ids are equal and -1000 otherwise, as the reference's mask does (the padding
    windows' RTs, id B, among themselves).  Returns o (layout.total, C) float32, the layout of
    ``(att @ v).transpose(1, 2).reshape(B, Nmax, C)`` at the real rows.  Differentiable in qkv, with an
    output and a gradient that are bit-identical run to run."""
    _require(isinstance(layout, RelayTokenLayout), 'layout must be a RelayTokenLayout (see rt_layout)')
    return RelayTokenAttentionFunction.apply(qkv, layout.cu, layout.ids, num_heads)


class RTAttention(_RTAttention):
    """``RTAttention`` (hotformerloc_backbone.py:83-119) on :func:`relay_token_attention`.  Parameters are
    those of the reference module -- ``qkv.*`` and ``proj.*`` -- so the ``rt_attention.*`` tensors of a
    checkpoint load into it."""

    def __init__(self, dim: int, num_heads: int):
        super().__init__(dim)
        if not (1 <= num_heads <= MAX_HEADS and dim == HEAD_DIM * num_heads):
            raise ValueError(f'dim must be 16 num_heads with 1 <= num_heads <= {MAX_HEADS}, got dim={dim}, '
                             f'num_heads={num_heads}')
        self.dim, self.num_heads = dim, num_heads

    def forward(self, x: torch.Tensor, layout: RelayTokenLayout) -> torch.Tensor:
        """x (layout.total, C): packed RT rows (:meth:`RelayTokenLayout.pack`) -> (layout.total, C)."""
        return self.proj(relay_token_attention(self.qkv(x), layout, self.num_heads))

    def extra_repr(self) -> str:
        return f'dim={self.dim}, num_heads={self.num_heads}'
