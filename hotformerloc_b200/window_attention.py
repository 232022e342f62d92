"""Differentiable octree window attention core, fp32 on the kernels of csrc/window_attn_train.cu.

:func:`window_attention` is the part of the reference's ``OctreeAttention.forward`` between ``qkv``
and ``proj`` (octformer_backbone.py:52-93): the relative position bias (octformer_layers.py:156-170),
the submap mask and, for H-OSA, the relay token at window position 0 (hotformerloc_backbone.py:197-236).
It takes the window tokens' integer coordinates and submap ids instead of ``rel_pos`` and a dense
mask, and keeps only a per-row log-sum-exp for the backward, so no (N_win, H, L, L) tensor exists.
:class:`OctreeAttention` wraps it with the reference module's parameters.  Every op runs on the
current torch stream and raises ``HflError`` on bad input, before any launch.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import native as N
from .models.hotformerloc import _Attention
from .native import HflError

__all__ = ['window_attention', 'WindowAttentionFunction', 'OctreeAttention']

HEAD_DIM = 16
MAX_HEADS = 16
MAX_L = 128
MAX_BND = 1 << 20


def _require(cond: bool, msg: str):
    if not cond:
        raise HflError(msg)


def _check(name: str, t, dtypes, shape):
    _require(isinstance(t, torch.Tensor), f'{name} must be a tensor')
    _require(t.is_cuda, f'{name} must be a CUDA tensor')
    _require(t.dtype in dtypes, f'{name} must be {" or ".join(str(d) for d in dtypes)}, got {t.dtype}')
    _require(tuple(t.shape) == tuple(shape), f'{name} must have shape {tuple(shape)}, got {tuple(t.shape)}')
    _require(t.is_contiguous(), f'{name} must be contiguous')


def _check_args(qkv, xyz, ids, rpe_table, bnd, hat, num_heads):
    """Validates the forward's arguments; returns (n_win, L)."""
    _require(isinstance(num_heads, int) and 1 <= num_heads <= MAX_HEADS,
             f'num_heads must be an int in [1, {MAX_HEADS}], got {num_heads!r}')
    _require(hat in (0, 1, False, True), f'hat must be 0 or 1, got {hat!r}')
    _require(isinstance(bnd, int) and 0 <= bnd <= MAX_BND, f'bnd must be an int in [0, {MAX_BND}], got {bnd!r}')
    _require(isinstance(qkv, torch.Tensor) and qkv.dim() == 3,
             'qkv must be a (N_win, L, 3C) tensor')
    n_win, L, C3 = qkv.shape
    C = HEAD_DIM * num_heads
    _require(C3 == 3 * C, f'qkv must have 3C = {3 * C} columns for C = 16 num_heads, got {C3}')
    _require(1 <= L <= MAX_L, f'L must be in [1, {MAX_L}], got {L}')
    _check('qkv', qkv, (torch.float32,), (n_win, L, C3))
    _check('ids', ids, (torch.int32, torch.int64), (n_win, L))
    _check('xyz', xyz, (torch.int32, torch.int64), (n_win, L - int(hat), 3))
    if rpe_table is not None:
        _check('rpe_table', rpe_table, (torch.float32,), (3 * (2 * bnd + 1), num_heads))
    dev = qkv.device
    _require(all(t.device == dev for t in (xyz, ids) + ((rpe_table,) if rpe_table is not None else ())),
             'all tensors must be on the same device')
    return n_win, L


class WindowAttentionFunction(torch.autograd.Function):
    """o = softmax(q k^T 0.25 + mask + rpe) v per window and head; gradients for qkv and rpe_table."""

    @staticmethod
    def forward(ctx, qkv, xyz, ids, rpe_table, bnd, hat, num_heads):
        n_win, L = _check_args(qkv, xyz, ids, rpe_table, bnd, hat, num_heads)
        H, hat = num_heads, int(hat)
        o = torch.empty((n_win, L, HEAD_DIM * H), dtype=torch.float32, device=qkv.device)
        lse = torch.empty((n_win, H, L), dtype=torch.float32, device=qkv.device)
        with torch.cuda.device(qkv.device):
            N.check(N.lib().hfl_window_attn_train_fwd(
                N.ptr(qkv), N.ptr(xyz), int(xyz.dtype == torch.int64), N.ptr(ids), int(ids.dtype == torch.int64),
                N.ptr(rpe_table), n_win, L, H, hat, bnd, N.ptr(o), N.ptr(lse), N.stream()))
        ctx.save_for_backward(qkv, xyz, ids, rpe_table, o, lse)
        ctx.args = (bnd, hat, H)
        return o

    @staticmethod
    def backward(ctx, grad):
        qkv, xyz, ids, rpe_table, o, lse = ctx.saved_tensors
        bnd, hat, H = ctx.args
        grad = grad.contiguous()
        _check('grad', grad, (torch.float32,), o.shape)
        n_win, L = qkv.shape[0], qkv.shape[1]
        L_ = N.lib()
        dqkv = torch.empty_like(qkv)
        dtable = torch.empty_like(rpe_table) if rpe_table is not None else None
        ws_bytes = int(L_.hfl_window_attn_train_bwd_workspace_bytes(H, bnd, int(rpe_table is not None)))
        with torch.cuda.device(qkv.device):
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=qkv.device) if ws_bytes else None
            N.check(L_.hfl_window_attn_train_bwd(
                N.ptr(qkv), N.ptr(xyz), int(xyz.dtype == torch.int64), N.ptr(ids), int(ids.dtype == torch.int64),
                N.ptr(rpe_table), N.ptr(o), N.ptr(lse), N.ptr(grad), n_win, L, H, hat, bnd, N.ptr(dqkv),
                N.ptr(dtable), N.ptr(ws), ws_bytes, N.stream()))
        return (dqkv if ctx.needs_input_grad[0] else None, None, None,
                dtable if rpe_table is not None and ctx.needs_input_grad[3] else None, None, None, None)


def window_attention(qkv: torch.Tensor, xyz: torch.Tensor, ids: torch.Tensor, rpe_table: Optional[torch.Tensor],
                     bnd: int, hat: bool, num_heads: int) -> torch.Tensor:
    """Attention core of ``OctreeAttention.forward`` over windows of L = K + hat positions.

    qkv (N_win, L, 3C) float32, the output of ``Linear(C, 3C)`` with C = 16 num_heads;
    xyz (N_win, K, 3) int32/int64 integer cell coordinates of the window tokens (after any dilation
    gather); ids (N_win, L) int32/int64, tokens attend with bias 0 iff their ids are equal (else -1000,
    as the reference); rpe_table (3 (2 bnd + 1), num_heads) float32 or None; with ``hat`` the relay
    token is position 0 and gets no RPE term.  Returns o (N_win, L, C) float32, the layout of
    ``(att @ v).transpose(1, 2).reshape(N, L, C)``.  Differentiable in qkv and rpe_table, with
    gradients that are bit-identical run to run."""
    return WindowAttentionFunction.apply(qkv, xyz, ids, rpe_table, bnd, hat, num_heads)


class OctreeAttention(_Attention):
    """``OctreeAttention`` (octformer_backbone.py:52-93) on :func:`window_attention`.  Parameters are
    those of the reference module -- ``qkv.*``, ``proj.*`` and, with ``use_rpe``, ``rpe.rpe_table`` of
    shape (3 (2 pos_bnd + 1), num_heads) with pos_bnd = int(0.8 patch_size sqrt(dilation)) -- so the
    ``attention.*`` tensors of a pretrained block load into it.  ``hat`` makes window position 0 the
    relay token (HOTFormerBlock)."""

    def __init__(self, dim: int, patch_size: int, num_heads: int, dilation: int = 1, use_rpe: bool = True,
                 hat: bool = False):
        super().__init__(dim, patch_size, num_heads, dilation, use_rpe)
        if dim != HEAD_DIM * num_heads:
            raise ValueError(f'dim must be 16 num_heads = {HEAD_DIM * num_heads}, got {dim}')
        self.dim, self.patch_size, self.num_heads = dim, patch_size, num_heads
        self.dilation, self.use_rpe, self.hat = dilation, use_rpe, hat

    def forward(self, x: torch.Tensor, xyz: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
        """x (N_win, L, C) windows, xyz (N_win, L - hat, 3) token coordinates, ids (N_win, L) submap ids."""
        rpe = self.rpe if self.use_rpe else None
        o = window_attention(self.qkv(x), xyz, ids, rpe.rpe_table if rpe is not None else None,
                             rpe.pos_bnd if rpe is not None else 0, self.hat, self.num_heads)
        return self.proj(o)

    def extra_repr(self) -> str:
        return (f'dim={self.dim}, patch_size={self.patch_size}, num_heads={self.num_heads}, '
                f'dilation={self.dilation}, use_rpe={self.use_rpe}, hat={self.hat}')
